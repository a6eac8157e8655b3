// msa.hpp -- alignment container of the model_t mirror (interface of the
// reference's msa_t, src/msa.hpp:21-68: sequence/label/weights/map/states/
// count/length/total_weight, pattern compression, taxa consistency check).
// PHYLIP (sequential or interleaved) and FASTA are read; partition files and
// model strings are parsed by partition_file.hpp (SURVEY 8f, row N3).
#ifndef RD_HOST_MSA_HPP_
#define RD_HOST_MSA_HPP_

#include <rdk.h>

#include "partition_file.hpp"

#include <string>
#include <unordered_set>
#include <vector>

class msa_t {
public:
  msa_t(const std::string &msa_filename, const rdk_state_t *map = rdk_map_nt, unsigned int states = 4,
        bool compress = true);
  // in-memory construction (synthetic alignments, site shards)
  msa_t(std::vector<std::string> labels, std::vector<std::string> sequences,
        const rdk_state_t *map = rdk_map_nt, unsigned int states = 4, bool compress = true);
  // contiguous column slice [begin, end) of another alignment, weights carried over
  msa_t(const msa_t &other, size_t begin, size_t end);
  // the columns named by a partition's 1-based inclusive ranges, in range order,
  // weights reset and patterns re-compressed (src/msa.cpp:505-587)
  msa_t(const msa_t &other, const partition_info_t &partition);
  std::vector<msa_t> partition(const msa_partitions_t &parts) const;
  msa_t(const msa_t &) = delete;
  msa_t(msa_t &&) = default;

  const char        *sequence(int i) const;
  const char        *label(int i) const;
  const unsigned    *weights() const { return _weights.data(); }
  unsigned int       total_weight() const;
  const rdk_state_t *map() const { return _map; }
  unsigned int       states() const { return _states; }
  int                count() const { return (int)_sequences.size(); }
  unsigned int       length() const { return _sequences.empty() ? 0u : (unsigned)_sequences[0].size(); }

  void compress();
  // the pattern each column of the alignment this one was built from became (compress merges
  // identical columns; a partition's columns are in the order of its ranges): [column] -> pattern
  std::vector<unsigned int> pattern_of_column() const;
  bool constiency_check(std::unordered_set<std::string> labels) const;
  void valid_data() const;

private:
  std::vector<std::string>  _labels, _sequences;
  std::vector<unsigned int> _weights;
  std::vector<unsigned int> _column_pattern;  // empty: the identity (never compressed)
  const rdk_state_t        *_map;
  unsigned int              _states;
};

#endif
