// checkpoint.cpp -- the reference's "<prefix>.ckp" format (src/checkpoint.{hpp,cpp}),
// restated: see checkpoint.hpp for the byte layout.  Everything is serialised into a
// byte string first and appended with ONE write(2) under the file lock, so a record is
// either wholly in the log or (after a crash) a detectable torn tail.
#include "checkpoint.hpp"

#include <cerrno>
#include <cstring>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

namespace {

// ---- checksum: the reference's Adler-32 variant (src/checkpoint.hpp:34-48) ----
constexpr uint32_t kModAdler = 65521;

struct adler_t {
  uint32_t a = 1, b = 0;
  void     bytes(const void *p, size_t n) {
    const uint8_t *d = static_cast<const uint8_t *>(p);
    for (size_t i = 0; i < n; ++i) {
      a = (a + d[i]) % kModAdler;
      b = b + a;  // the reference writes `b + a % MOD_ADLER`: b is never reduced
    }
  }
  void doubles(const std::vector<double> &v) {
    for (double x : v) bytes(&x, sizeof(x));
  }
  uint32_t value() const { return (b << 16) | a; }
};

void checksum_params(adler_t &s, const partition_parameters_t &pp) {
  s.doubles(pp.subst_rates);
  s.doubles(pp.freqs);
  s.doubles(pp.gamma_alpha);
  s.doubles(pp.gamma_weights);
  // tail of the reference's variadic overload (src/checkpoint.hpp:80-85): the last call
  // compute_checksum_components(a, b) binds to the single-value template with
  // val = a, a0 = b, b0 = 0
  adler_t  t;
  uint32_t val = s.a;
  t.a = s.b;
  t.b = 0;
  t.bytes(&val, sizeof(val));
  s = t;
}

// ---- serialisation ----
struct out_t {
  std::string s;
  template <typename T> void pod(const T &v) { s.append(reinterpret_cast<const char *>(&v), sizeof(T)); }
  void str(const std::string &v) {
    pod<uint64_t>(v.size());
    s.append(v);
  }
  void doubles(const std::vector<double> &v) {
    pod<uint64_t>(v.size());
    for (double x : v) pod(x);
  }
};

// Positional reads (pread) on the checkpoint's OWN descriptor: opening and closing a second
// descriptor on the file would drop every fcntl lock this process holds on it (POSIX).
struct in_t {
  int   fd;
  off_t off = 0;
  bool  short_read = false;
  bool  raw(void *p, size_t n) {
    char *c = static_cast<char *>(p);
    while (n > 0) {
      ssize_t r = ::pread(fd, c, n, off);
      if (r > 0) off += r;
      if (r < 0) {
        if (errno == EINTR) continue;
        throw checkpoint_read_failure{"Failed to read a value"};
      }
      if (r == 0) {
        short_read = true;
        memset(c, 0, n);
        return false;
      }
      c += r;
      n -= (size_t)r;
    }
    return true;
  }
  template <typename T> bool pod(T &v) { return raw(&v, sizeof(T)); }
  bool str(std::string &v) {
    uint64_t n = 0;
    if (!pod(n)) return false;
    if (n == 0) return true;  // the reference leaves the target untouched
    if (n > (uint64_t(1) << 30)) {
      short_read = true;
      return false;
    }
    std::string t((size_t)n, '\0');
    if (!raw(&t[0], (size_t)n)) return false;
    v.swap(t);
    return true;
  }
  bool doubles(std::vector<double> &v, uint64_t limit) {
    uint64_t n = 0;
    if (!pod(n)) return false;
    if (n > limit) {
      short_read = true;
      return false;
    }
    std::vector<double> t((size_t)n);
    if (n && !raw(t.data(), (size_t)n * sizeof(double))) return false;
    v.swap(t);
    return true;
  }
};

constexpr size_t kRatehetImage = 32;  // sizeof(ratehet_opts_t) in the reference build (LP64)

void put_options(out_t &o, const cli_options_t &c) {
  o.str(c.msa_filename);
  o.str(c.tree_filename);
  o.str(c.prefix);
  o.str(c.prefix_dir);
  o.str(c.model_filename);
  o.str(c.freqs_filename);
  o.str(c.partition_filename);
  o.str(c.data_type);
  o.str(c.model_string);
  o.pod<uint64_t>(c.rate_cats.size());
  for (const auto &r : c.rate_cats) {
    unsigned char img[kRatehetImage];
    memset(img, 0, sizeof(img));
    int32_t  type = (int32_t)r.type, cat = (int32_t)r.rate_category_type;
    uint64_t n = r.rate_cats;
    uint8_t  ai = r.alpha_init ? 1 : 0;
    memcpy(img + 0, &type, 4);
    memcpy(img + 4, &cat, 4);
    memcpy(img + 8, &n, 8);
    memcpy(img + 16, &ai, 1);
    memcpy(img + 24, &r.alpha, 8);
    o.s.append(reinterpret_cast<const char *>(img), sizeof(img));
  }
  o.pod<uint64_t>(c.seed);
  o.pod<uint64_t>(c.min_roots);
  o.pod<uint64_t>(c.threads);
  o.pod(c.root_ratio);
  o.pod(c.abs_tolerance);
  o.pod(c.factor);
  o.pod(c.br_tolerance);
  o.pod(c.bfgs_tol);
  o.pod<uint8_t>(c.silent);
  o.pod<uint8_t>(c.exhaustive);
  o.pod<uint8_t>(c.echo);
  o.pod<uint8_t>(c.invariant_sites);
  o.pod<int32_t>(c.early_stop.raw());
  o.pod<int32_t>((int32_t)c.initial_root_strategy);
}

bool get_options(in_t &in, cli_options_t &c) {
  bool ok = in.str(c.msa_filename) && in.str(c.tree_filename) && in.str(c.prefix) && in.str(c.prefix_dir) &&
            in.str(c.model_filename) && in.str(c.freqs_filename) && in.str(c.partition_filename) &&
            in.str(c.data_type) && in.str(c.model_string);
  if (!ok) return false;
  uint64_t n = 0;
  if (!in.pod(n) || n > (1u << 20)) return false;
  std::vector<ratehet_opts_t> rc((size_t)n);
  for (auto &r : rc) {
    unsigned char img[kRatehetImage];
    if (!in.raw(img, sizeof(img))) return false;
    int32_t  type, cat;
    uint64_t cats;
    memcpy(&type, img + 0, 4);
    memcpy(&cat, img + 4, 4);
    memcpy(&cats, img + 8, 8);
    r.type = (param_type)type;
    r.rate_category_type = (rate_category)cat;
    r.rate_cats = (size_t)cats;
    r.alpha_init = img[16] != 0;
    memcpy(&r.alpha, img + 24, 8);
  }
  c.rate_cats.swap(rc);
  uint64_t seed, min_roots, threads;
  uint8_t  silent, exhaustive, echo, invariant;
  int32_t  early, strat;
  ok = in.pod(seed) && in.pod(min_roots) && in.pod(threads) && in.pod(c.root_ratio) && in.pod(c.abs_tolerance) &&
       in.pod(c.factor) && in.pod(c.br_tolerance) && in.pod(c.bfgs_tol) && in.pod(silent) && in.pod(exhaustive) &&
       in.pod(echo) && in.pod(invariant) && in.pod(early) && in.pod(strat);
  if (!ok) return false;
  c.seed = seed;
  c.min_roots = (size_t)min_roots;
  c.threads = (size_t)threads;
  c.silent = silent != 0;
  c.exhaustive = exhaustive != 0;
  c.echo = echo != 0;
  c.invariant_sites = invariant != 0;
  c.early_stop = initialized_flag_t::from_raw(early);
  c.initial_root_strategy = (initial_root_strategy_t)strat;
  return true;
}

constexpr uint32_t kWriteSuccessFlag = 1u << 0;

// header + success flag; throws checkpoint_read_success_failure when the flag is missing
void read_header(in_t &in, cli_options_t &c) {
  cli_options_t tmp;
  uint32_t      ff = 0;
  if (!get_options(in, tmp) || !in.pod(ff) || !(ff & kWriteSuccessFlag))
    throw checkpoint_read_success_failure{"The current read was unsuccessful due to an unsuccessful write flag"};
  c = std::move(tmp);
}

void append_all(int fd, const std::string &s, const char *what) {
  const char *p = s.data();
  size_t      n = s.size();
  while (n > 0) {
    ssize_t r = ::write(fd, p, n);
    if (r < 0) {
      if (errno == EINTR) continue;
      throw checkpoint_write_failure{what};
    }
    p += r;
    n -= (size_t)r;
  }
}

// whole-file write lock (a shared read lock on a read-only log), released (with an fsync) at scope
// exit (src/checkpoint.hpp:205-249)
class file_lock_t {
public:
  explicit file_lock_t(int fd, short type = F_WRLCK) : _fd{fcntl(fd, F_DUPFD, 0)} {
    memset(&_fl, 0, sizeof(_fl));
    _fl.l_type = type;
    _fl.l_whence = SEEK_SET;
    if (_fd == -1 || fcntl(_fd, F_SETLKW, &_fl) == -1) {
      if (_fd != -1) close(_fd);
      throw std::runtime_error("failed to obtain the lock");
    }
  }
  ~file_lock_t() {
    _fl.l_type = F_UNLCK;
    fcntl(_fd, F_SETLK, &_fl);
    fsync(_fd);
    close(_fd);
  }
  file_lock_t(const file_lock_t &) = delete;
  file_lock_t &operator=(const file_lock_t &) = delete;

private:
  int          _fd;
  struct flock _fl;
};

std::string serialise_record(const rd_result_t &r, const std::vector<partition_parameters_t> &params) {
  out_t o;
  o.pod<uint64_t>(r.root_id);
  o.pod(r.llh);
  o.pod(r.alpha);
  o.pod<uint32_t>(checkpoint_checksum(r));
  o.pod<uint64_t>(params.size());
  for (const auto &pp : params) {
    o.doubles(pp.subst_rates);
    o.doubles(pp.freqs);
    o.doubles(pp.gamma_alpha);
    o.doubles(pp.gamma_weights);
  }
  o.pod<uint32_t>(checkpoint_checksum(params));
  return o.s;
}

}  // namespace

uint32_t checkpoint_checksum(const rd_result_t &r) {
  // the struct image: {u64 root_id, f64 llh, f64 alpha}, no padding
  unsigned char img[24];
  uint64_t      id = r.root_id;
  memcpy(img, &id, 8);
  memcpy(img + 8, &r.llh, 8);
  memcpy(img + 16, &r.alpha, 8);
  adler_t s;
  s.bytes(img, sizeof(img));
  return s.value();
}

uint32_t checkpoint_checksum(const std::vector<partition_parameters_t> &params) {
  adler_t s;
  for (const auto &pp : params) checksum_params(s, pp);
  return s.value();
}

checkpoint_t::checkpoint_t() {}

checkpoint_t::checkpoint_t(const std::string &prefix) {
  _checkpoint_filename = prefix + ".ckp";
  _existing_results = (access(_checkpoint_filename.c_str(), F_OK) != -1);
  _file_descriptor = open(_checkpoint_filename.c_str(), O_RDWR | O_APPEND | O_CREAT, 0640);
  if (_file_descriptor == -1) throw std::runtime_error("Failed to open the checkpoint file");
}

checkpoint_t checkpoint_t::read_only(const std::string &prefix) {
  checkpoint_t c;
  c._checkpoint_filename = prefix + ".ckp";
  c._file_descriptor = open(c._checkpoint_filename.c_str(), O_RDONLY);
  if (c._file_descriptor == -1) throw std::runtime_error("no checkpoint " + c._checkpoint_filename);
  c._existing_results = true;
  c._read_only = true;
  return c;
}

checkpoint_t::~checkpoint_t() {
  if (_file_descriptor != -1) close(_file_descriptor);
}

checkpoint_t::checkpoint_t(checkpoint_t &&o) { *this = std::move(o); }

checkpoint_t &checkpoint_t::operator=(checkpoint_t &&o) {
  if (this == &o) return *this;
  if (_file_descriptor != -1) close(_file_descriptor);
  _file_descriptor = o._file_descriptor;
  o._file_descriptor = -1;
  _checkpoint_filename = std::move(o._checkpoint_filename);
  _existing_results = o._existing_results;
  _read_only = o._read_only;
  _records = std::move(o._records);
  return *this;
}

void checkpoint_t::clear() {
  std::lock_guard<std::mutex> lk(_mu);
  _records.clear();
}

void checkpoint_t::write(const rd_result_t &result, const std::vector<partition_parameters_t> &params) {
  std::lock_guard<std::mutex> lk(_mu);
  if (!on_disk()) {
    _records.emplace_back(result, params);
    return;
  }
  std::string bytes = serialise_record(result, params);
  file_lock_t lock(_file_descriptor);
  append_all(_file_descriptor, bytes, "Failed to write all data to the file");
}

void checkpoint_t::save_options(const cli_options_t &options) {
  if (!on_disk() || _existing_results) return;
  out_t o;
  put_options(o, options);
  o.pod<uint32_t>(kWriteSuccessFlag);
  std::lock_guard<std::mutex> lk(_mu);
  file_lock_t                 lock(_file_descriptor);
  append_all(_file_descriptor, o.s, "Failed to write the options to the checkpoint file");
}

void checkpoint_t::load_options(cli_options_t &options) {
  if (!on_disk() || !_existing_results) return;
  std::lock_guard<std::mutex> lk(_mu);
  file_lock_t                 lock(_file_descriptor);
  load_options_unlocked(options);
}

void checkpoint_t::load_options_unlocked(cli_options_t &options) {
  in_t in{_file_descriptor};
  read_header(in, options);
}

// every readable record, in file order; *damaged = the log ends in a record that fails its checksum
std::vector<checkpoint_t::record_t> checkpoint_t::scan(bool *damaged) {
  file_lock_t lock(_file_descriptor, _read_only ? F_RDLCK : F_WRLCK);
  return scan_unlocked(damaged);
}

// the caller holds _mu and the file lock
std::vector<checkpoint_t::record_t> checkpoint_t::scan_unlocked(bool *damaged) {
  std::vector<record_t> results;
  if (damaged) *damaged = false;
  struct stat st;
  if (fstat(_file_descriptor, &st) == -1) throw checkpoint_read_failure{"Failed to stat the checkpoint file"};
  const off_t   end = st.st_size;
  in_t          in{_file_descriptor};
  cli_options_t tmp;
  read_header(in, tmp);
  off_t pos = in.off;
  while (pos < end) {
    rd_result_t r{};
    uint64_t    id = 0;
    uint32_t    sum = 0;
    bool        ok = in.pod(id) && in.pod(r.llh) && in.pod(r.alpha) && in.pod(sum);
    r.root_id = (size_t)id;
    if (!ok || sum != checkpoint_checksum(r)) {
      if (damaged) *damaged = true;
      break;
    }
    uint64_t                            n = 0;
    std::vector<partition_parameters_t> params;
    const uint64_t                      limit = (uint64_t)(end - pos) / sizeof(double);
    ok = in.pod(n) && n <= (uint64_t)(end - pos);
    for (uint64_t i = 0; ok && i < n; ++i) {
      partition_parameters_t pp;
      ok = in.doubles(pp.subst_rates, limit) && in.doubles(pp.freqs, limit) &&
           in.doubles(pp.gamma_alpha, limit) && in.doubles(pp.gamma_weights, limit);
      if (ok) params.push_back(std::move(pp));
    }
    ok = ok && in.pod(sum);
    if (!ok || sum != checkpoint_checksum(params)) {
      if (damaged) *damaged = true;
      break;
    }
    results.emplace_back(r, std::move(params));
    pos = in.off;
  }
  return results;
}

std::vector<checkpoint_t::record_t> checkpoint_t::read_results() {
  std::lock_guard<std::mutex> lk(_mu);
  if (!on_disk()) return _records;
  return scan(nullptr);
}

std::vector<rd_result_t> checkpoint_t::current_progress() {
  std::vector<rd_result_t> r;
  for (auto &rec : read_results()) r.push_back(rec.first);
  return r;
}

std::vector<size_t> checkpoint_t::completed_indicies() {
  std::vector<size_t> r;
  for (auto &rec : read_results()) r.push_back(rec.first.root_id);
  return r;
}

bool checkpoint_t::needs_cleaning() {
  std::lock_guard<std::mutex> lk(_mu);
  if (!on_disk()) return false;
  bool damaged = false;
  scan(&damaged);
  return damaged;
}

void checkpoint_t::clean() {
  if (!on_disk() || !_existing_results) return;
  // ONE mutex and ONE file lock across read, rewrite and rename: a record appended by another
  // rank in between would otherwise be dropped
  std::lock_guard<std::mutex> lk(_mu);
  file_lock_t                 lock(_file_descriptor);
  cli_options_t               options;
  load_options_unlocked(options);
  auto        progress = scan_unlocked(nullptr);
  std::string backup = _checkpoint_filename + ".bak";
  int copy_fd = open(backup.c_str(), O_RDWR | O_CREAT | O_APPEND | O_EXCL, 0640);
  if (copy_fd == -1)
    throw std::runtime_error("Failed to open the new checkpoint when cleaning the checkpoint");
  try {
    out_t o;
    put_options(o, options);
    o.pod<uint32_t>(kWriteSuccessFlag);
    for (auto &rec : progress) o.s += serialise_record(rec.first, rec.second);
    append_all(copy_fd, o.s, "Failed to write the cleaned checkpoint");
  } catch (...) {
    close(copy_fd);
    unlink(backup.c_str());
    throw;
  }
  fsync(copy_fd);
  close(copy_fd);
  if (rename(backup.c_str(), _checkpoint_filename.c_str()) != 0)
    throw std::runtime_error("Failed to replace the checkpoint with its cleaned copy");
  // the descriptor still names the replaced inode: reopen
  close(_file_descriptor);
  _file_descriptor = open(_checkpoint_filename.c_str(), O_RDWR | O_APPEND | O_CREAT, 0640);
  if (_file_descriptor == -1) throw std::runtime_error{"Failed to reload the checkpoint file"};
}

void checkpoint_t::reload() {
  if (!on_disk()) return;
  close(_file_descriptor);
  _file_descriptor = open(_checkpoint_filename.c_str(), O_RDWR | O_APPEND | O_CREAT, 0640);
  if (_file_descriptor == -1) throw std::runtime_error{"Failed to reload the checkpoint file"};
}

int checkpoint_t::get_inode() {
  struct stat st;
  if (!on_disk() || fstat(_file_descriptor, &st) == -1)
    throw std::runtime_error{"There was an error getting the INODE of the checkpoint"};
  return (int)st.st_ino;
}
