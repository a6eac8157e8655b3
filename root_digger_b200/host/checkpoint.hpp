// checkpoint.hpp -- result log used by search()/exhaustive_search() (SURVEY 8f, row N4).
//
// The reference appends {root_id, llh, alpha} + the partition parameters of every
// finished start root / branch to "<prefix>.ckp" and rank 0 reads them all back
// (src/model.cpp:1107,1120,1215,1238); a restarted run skips the root ids already in
// the file (assign_indicies_by_rank_*, src/model.cpp:1899-1960).
//
// Two backings behind the reference's member names (src/checkpoint.hpp:251-301):
//   checkpoint_t()        in-memory log (what a library caller without a prefix gets);
//   checkpoint_t(prefix)  the reference's ON-DISK format, byte for byte, so that a run of
//                         this engine resumes from a checkpoint the reference wrote and
//                         vice versa.  File layout (native little-endian, LP64):
//
//     header   cli_options_t, field by field (src/checkpoint.cpp:61-91):
//                9 strings            u64 length + bytes (no terminator)
//                rate_cats            u64 count + count x 32-byte ratehet_opts_t images
//                                     {i32 type, i32 category type, u64 rate_cats,
//                                      u8 alpha_init, 7 pad, f64 alpha}
//                seed u64, min_roots u64, threads u64
//                root_ratio, abs_tolerance, factor, br_tolerance, bfgs_tol   f64
//                silent, exhaustive, echo, invariant_sites                  u8
//                early_stop i32, initial_root_strategy i32
//              u32 flags = 1 (CHECKPOINT_WRITE_SUCCESS_FLAG, src/checkpoint.hpp:20,110-115)
//     record*  rd_result_t {u64 root_id, f64 llh, f64 alpha} + u32 checksum
//              u64 n + n x partition_parameters_t {4 x (u64 len + len x f64)} + u32 checksum
//
//   The checksum is the reference's Adler-32 VARIANT (src/checkpoint.hpp:34-91), restated
//   in checkpoint.cpp with its two quirks: `b` is never reduced mod 65521 (it wraps at
//   2^32), and a partition_parameters_t runs one extra round over the 4 bytes of `a`
//   seeded with (a := b, b := 0) -- the tail of the reference's variadic overload set.
//   Writers take an fcntl write lock on the whole file (records of concurrent ranks never
//   interleave); a record whose checksum does not match ends the readable part of the log
//   ("resume with what we can", src/checkpoint.cpp:318-324) and makes needs_cleaning() true.
#ifndef RD_HOST_CHECKPOINT_HPP_
#define RD_HOST_CHECKPOINT_HPP_

#include "util.hpp"

#include <mutex>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

class checkpoint_write_failure : public std::runtime_error {
  using std::runtime_error::runtime_error;
};
class checkpoint_read_failure : public std::runtime_error {
  using std::runtime_error::runtime_error;
};
class checkpoint_read_success_failure : public checkpoint_read_failure {
  using checkpoint_read_failure::checkpoint_read_failure;
};

// the reference's checksum of one result / one parameter list (exposed for the tests)
uint32_t checkpoint_checksum(const rd_result_t &);
uint32_t checkpoint_checksum(const std::vector<partition_parameters_t> &);

class checkpoint_t {
public:
  typedef std::pair<rd_result_t, std::vector<partition_parameters_t>> record_t;

  checkpoint_t();                                    // in-memory
  explicit checkpoint_t(const std::string &prefix);  // "<prefix>.ckp", created if absent
  // an existing "<prefix>.ckp" opened for reading only (read_results under a shared lock); for
  // callers that only evaluate a log, possibly one they may not write (another user's run)
  static checkpoint_t read_only(const std::string &prefix);
  ~checkpoint_t();
  checkpoint_t(checkpoint_t &&);
  checkpoint_t &operator=(checkpoint_t &&);
  checkpoint_t(const checkpoint_t &) = delete;
  checkpoint_t &operator=(const checkpoint_t &) = delete;

  void write(const rd_result_t &result, const std::vector<partition_parameters_t> &params);
  std::vector<record_t>    read_results();
  std::vector<rd_result_t> current_progress();
  std::vector<size_t>      completed_indicies();

  void save_options(const cli_options_t &);  // only into a file that did not exist before
  void load_options(cli_options_t &);        // only from a file that did
  bool needs_cleaning();
  void clean();  // rewrite the readable prefix of a damaged log (rank 0 only in the reference)
  void reload();
  int  get_inode();
  bool existing_checkpoint() const { return _existing_results; }
  bool on_disk() const { return _file_descriptor != -1; }
  std::string get_filename() const { return _checkpoint_filename; }

  void clear();  // in-memory backing only

private:
  std::vector<record_t> scan(bool *damaged);
  std::vector<record_t> scan_unlocked(bool *damaged);  // caller holds _mu and the file lock
  void                  load_options_unlocked(cli_options_t &);

  std::string           _checkpoint_filename;
  int                   _file_descriptor = -1;
  bool                  _existing_results = false;
  bool                  _read_only = false;
  std::vector<record_t> _records;  // in-memory backing
  std::mutex            _mu;
};

#endif
