// msa.cpp -- see msa.hpp.  Behavioural reference: src/msa.cpp:18-88 (file
// formats), :621-632 (compression), :641-667 (consistency check).
#include "msa.hpp"

#include <algorithm>
#include <cctype>
#include <fstream>
#include <limits>
#include <numeric>
#include <sstream>
#include <stdexcept>

namespace {

bool parse_fasta(std::istream &in, std::vector<std::string> &labels, std::vector<std::string> &seqs) {
  std::string line;
  bool        any = false;
  while (std::getline(in, line)) {
    if (!line.empty() && line.back() == '\r') line.pop_back();
    if (line.empty()) continue;
    if (line[0] == '>') {
      std::string l = line.substr(1);
      while (!l.empty() && std::isspace((unsigned char)l.back())) l.pop_back();
      labels.push_back(l);
      seqs.emplace_back();
      any = true;
    } else {
      if (!any) return false;
      for (char c : line)
        if (!std::isspace((unsigned char)c)) seqs.back().push_back(c);
    }
  }
  return any;
}

bool phylip_interleaved(const std::vector<std::string> &lines, size_t n, size_t len,
                        std::vector<std::string> &labels, std::vector<std::string> &seqs) {
  if (lines.size() < n) return false;
  labels.assign(n, "");
  seqs.assign(n, "");
  for (size_t i = 0; i < lines.size(); ++i) {
    std::istringstream ls(lines[i]);
    std::string        tok;
    size_t             row = i % n;
    if (i < n) {
      if (!(ls >> tok)) return false;
      labels[row] = tok;
    }
    while (ls >> tok) seqs[row] += tok;
  }
  for (auto &s : seqs)
    if (s.size() != len) return false;
  return true;
}

bool phylip_sequential(const std::vector<std::string> &lines, size_t n, size_t len,
                       std::vector<std::string> &labels, std::vector<std::string> &seqs) {
  labels.assign(n, "");
  seqs.assign(n, "");
  std::vector<std::string> toks;
  for (auto &l : lines) {
    std::istringstream ls(l);
    std::string        t;
    while (ls >> t) toks.push_back(t);
  }
  size_t q = 0;
  for (size_t r = 0; r < n; ++r) {
    if (q >= toks.size()) return false;
    labels[r] = toks[q++];
    while (seqs[r].size() < len && q < toks.size()) seqs[r] += toks[q++];
    if (seqs[r].size() != len) return false;
  }
  return q == toks.size();
}

bool parse_phylip(std::istream &in, std::vector<std::string> &labels, std::vector<std::string> &seqs) {
  size_t n = 0, len = 0;
  if (!(in >> n >> len) || n == 0 || len == 0) return false;
  std::string              line;
  std::vector<std::string> lines;
  std::getline(in, line);
  while (std::getline(in, line)) {
    if (!line.empty() && line.back() == '\r') line.pop_back();
    if (line.find_first_not_of(" \t") == std::string::npos) continue;
    lines.push_back(line);
  }
  // as the reference does (src/msa.cpp:24-27): interleaved first, then sequential
  return phylip_interleaved(lines, n, len, labels, seqs) || phylip_sequential(lines, n, len, labels, seqs);
}

}  // namespace

msa_t::msa_t(const std::string &filename, const rdk_state_t *map, unsigned int states, bool do_compress)
    : _map(map), _states(states) {
  {
    std::ifstream in(filename);
    if (!in) throw std::invalid_argument("Could not parse msa file");
    if (!parse_phylip(in, _labels, _sequences)) {
      _labels.clear();
      _sequences.clear();
      in.clear();
      in.seekg(0);
      if (!parse_fasta(in, _labels, _sequences)) throw std::invalid_argument("Could not parse msa file");
    }
  }
  for (auto &s : _sequences)
    if (s.size() != _sequences[0].size()) throw std::invalid_argument("Sequences don't match in size");
  _weights.assign(length(), 1u);
  if (do_compress) compress();
}

msa_t::msa_t(std::vector<std::string> labels, std::vector<std::string> sequences, const rdk_state_t *map,
             unsigned int states, bool do_compress)
    : _labels(std::move(labels)), _sequences(std::move(sequences)), _map(map), _states(states) {
  if (_labels.size() != _sequences.size()) throw std::invalid_argument("labels and sequences differ in count");
  for (auto &s : _sequences)
    if (s.size() != _sequences[0].size()) throw std::invalid_argument("Sequences don't match in size");
  _weights.assign(length(), 1u);
  if (do_compress) compress();
}

msa_t::msa_t(const msa_t &o, size_t begin, size_t end) : _labels(o._labels), _map(o._map), _states(o._states) {
  if (begin > end || end > o.length()) throw std::out_of_range("column slice out of range");
  for (auto &s : o._sequences) _sequences.push_back(s.substr(begin, end - begin));
  _weights.assign(o._weights.begin() + (long)begin, o._weights.begin() + (long)end);
}

msa_t::msa_t(const msa_t &o, const partition_info_t &part) : _labels(o._labels), _map(o._map), _states(o._states) {
  size_t total = 0;
  for (auto &r : part.parts) {
    if (r.first == 0) throw std::runtime_error("Partition ranges start at 1, but we encountered a 0");
    if (r.second < r.first || r.second > o.length())
      throw std::runtime_error("Partition range " + std::to_string(r.first) + "-" + std::to_string(r.second) +
                               " of '" + part.partition_name + "' is outside the alignment (" +
                               std::to_string(o.length()) + " columns)");
    total += r.second - r.first + 1;
  }
  if (total > (size_t)std::numeric_limits<int>::max()) throw std::runtime_error("Partition range is too large");
  _sequences.reserve(o._sequences.size());
  for (auto &s : o._sequences) {
    std::string t;
    t.reserve(total);
    for (auto &r : part.parts) t.append(s, r.first - 1, r.second - r.first + 1);
    _sequences.push_back(std::move(t));
  }
  _weights.assign(total, 1u);
  compress();
}

std::vector<msa_t> msa_t::partition(const msa_partitions_t &parts) const {
  std::vector<msa_t> out;
  out.reserve(parts.size());
  for (auto &p : parts) out.emplace_back(*this, p);
  return out;
}

const char *msa_t::sequence(int i) const {
  if (i < 0 || i >= count()) throw std::out_of_range("Requested sequence does not exist");
  return _sequences[(size_t)i].c_str();
}
const char *msa_t::label(int i) const {
  if (i < 0 || i >= count()) throw std::out_of_range("Requested label does not exist");
  return _labels[(size_t)i].c_str();
}

unsigned int msa_t::total_weight() const {
  return std::accumulate(_weights.begin(), _weights.end(), 0u);
}

// corax_compress_site_patterns: identical columns (compared through the state
// map, so 'a' == 'A') are merged and their weights added; the surviving
// patterns come out in sorted order.
void msa_t::compress() {
  const size_t n = _sequences.size(), L = length();
  if (n == 0 || L == 0) return;
  std::vector<size_t> order(L);
  std::iota(order.begin(), order.end(), 0);
  auto code = [&](size_t r, size_t c) { return (unsigned)_map[(unsigned char)_sequences[r][c]]; };
  auto less = [&](size_t a, size_t b) {
    for (size_t r = 0; r < n; ++r) {
      unsigned x = code(r, a), y = code(r, b);
      if (x != y) return x < y;
    }
    return false;
  };
  std::stable_sort(order.begin(), order.end(), less);
  std::vector<size_t>   keep;
  std::vector<unsigned> w;
  for (size_t i = 0; i < L; ++i) {
    if (!keep.empty() && !less(keep.back(), order[i]) && !less(order[i], keep.back()))
      w.back() += _weights[order[i]];
    else {
      keep.push_back(order[i]);
      w.push_back(_weights[order[i]]);
    }
  }
  // column -> pattern: the columns of this alignment first, then those it was compressed from
  std::vector<unsigned> group(L);
  for (size_t i = 0, g = 0; i < L; ++i) {
    if (i && (less(order[i - 1], order[i]) || less(order[i], order[i - 1]))) ++g;
    group[order[i]] = (unsigned)g;
  }
  if (_column_pattern.empty()) _column_pattern.assign(group.begin(), group.end());
  else
    for (auto &c : _column_pattern) c = group[c];
  std::vector<std::string> out(n);
  for (size_t r = 0; r < n; ++r) {
    out[r].reserve(keep.size());
    for (size_t c : keep) out[r].push_back(_sequences[r][c]);
  }
  _sequences.swap(out);
  _weights.swap(w);
}

std::vector<unsigned int> msa_t::pattern_of_column() const {
  if (!_column_pattern.empty()) return _column_pattern;
  std::vector<unsigned int> id(length());
  std::iota(id.begin(), id.end(), 0u);
  return id;
}

bool msa_t::constiency_check(std::unordered_set<std::string> labels) const {
  std::unordered_set<std::string> taxa(_labels.begin(), _labels.end());
  bool                            ok = true;
  for (const auto &k : labels)
    if (!taxa.count(k)) ok = false;
  for (const auto &k : taxa)
    if (!labels.count(k)) ok = false;
  return ok;
}

void msa_t::valid_data() const {
  for (size_t i = 0; i < _sequences.size(); ++i)
    for (size_t j = 0; j < _sequences[i].size(); ++j) {
      char c = _sequences[i][j];
      if (c < 0)
        throw std::runtime_error("Encountered an invalid character in sequence " + std::to_string(i) +
                                 " at position " + std::to_string(j) + ".");
      if (_map[(size_t)c] == 0)
        throw std::runtime_error("Found unrecognized character sequence " + std::to_string(i) +
                                 " position " + std::to_string(j) + ".");
    }
}
