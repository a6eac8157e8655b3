// model.hpp -- model_t: the likelihood facade, root-location and parameter
// optimisers and the two search drivers of RootDigger, on the B200 engine.
//
// Same class surface as the reference's model_t (src/model.hpp:46-277): a user
// of the reference finds compute_lh, compute_lh_root, compute_dlh,
// optimize_alpha, optimize_root_location, search, exhaustive_search,
// initialize_partitions*, assign_indicies*, suggest_roots_*, with the same
// argument meaning and the same exceptions.  Underneath, every corax_* call of
// the reference is the rdk_* call of include/rdk.h, and the placement sweep /
// derivative evaluations may use the fused rdk entry points (same values).
#ifndef RD_HOST_MODEL_HPP_
#define RD_HOST_MODEL_HPP_

#include <rdk.h>

#include "checkpoint.hpp"
#include "msa.hpp"
#include "tree.hpp"
#include "optim.hpp"
#include "util.hpp"

#include <functional>
#include <random>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

struct invalid_empirical_frequencies_exception : public std::runtime_error {
  invalid_empirical_frequencies_exception(const char *m) : std::runtime_error(m) {}
};

model_params_t random_params(size_t size, uint64_t seed);

// how model_t's partitions are laid out over GPUs (new; SURVEY 8e).  The
// default is one unsharded partition per MSA partition on the current device.
struct shard_spec_t {
  unsigned long long site_offset = 0;  // first global site pattern held by this process
  unsigned long long global_sites = 0; // 0 = unsharded
  int                nranks = 1, rank = 0;
  const void        *comm_id = nullptr; // 128-byte id from rdk_comm_unique_id (rank 0), or nullptr
};

class model_t {
public:
  model_t(rooted_tree_t t, const std::vector<msa_t> &msa, const std::vector<ratehet_opts_t> &rate_cats,
          bool invariant_sites, uint64_t seed, bool early_stop, const shard_spec_t &shard = shard_spec_t());
  model_t(rooted_tree_t t, const std::vector<msa_t> &msa, size_t rate_cats, bool invariant_sites,
          uint64_t seed, bool early_stop)
      : model_t(std::move(t), msa, std::vector<ratehet_opts_t>(msa.size(), ratehet_opts_t{rate_cats}),
                invariant_sites, seed, early_stop) {}
  model_t(const model_t &) = delete;
  ~model_t();

  double compute_lh(const root_location_t &root_location);
  double compute_lh_root(const root_location_t &root);
  dlh_t  compute_dlh(const root_location_t &root_location);

  root_location_t                    optimize_alpha(const root_location_t &root, double atol);
  std::pair<root_location_t, double> optimize_root_location(size_t min_roots, double root_ratio);

  std::pair<root_location_t, double> search(size_t min_roots, double root_ratio, double atol, double pgtol,
                                            double brtol, double factor, checkpoint_t &);
  std::pair<root_location_t, double> exhaustive_search(double atol, double pgtol, double brtol,
                                                       double factor, checkpoint_t &);

  void initialize();
  void finalize();

  rooted_tree_t rooted_tree(const root_location_t &root) const;
  rooted_tree_t virtual_rooted_tree(const root_location_t &root) const;
  rooted_tree_t unrooted_tree() const;
  rooted_tree_t &tree() { return _tree; }

  void initialize_partitions(const std::vector<msa_t> &);
  void initialize_partitions_uniform_freqs(const std::vector<msa_t> &);

  std::string subst_string() const;

  std::vector<root_location_t> suggest_roots_random(size_t min, double ratio);
  std::vector<root_location_t> suggest_roots_lh(size_t min, double ratio);
  std::vector<root_location_t> suggest_roots_midpoint(size_t min, double ratio);
  std::vector<root_location_t> suggest_roots_modified_mad(size_t min, double ratio);

  std::vector<size_t> shuffle_root_indicies();
  std::vector<size_t> suggest_root_indicies_midpoint();
  std::vector<size_t> suggest_root_indicies_modified_mad();

  std::vector<double> compute_all_root_lh();
  // log-likelihood of every root placement at ratio 0.5 (the values
  // suggest_roots_lh ranks), and LWR = softmax of a log-likelihood vector
  // (exhaustive mode, src/model.cpp:1238-1258)
  std::vector<double>        sweep_root_lh();
  std::vector<double>        sweep_root_lh(size_t begin, size_t end);  // root ids [begin, end)
  static std::vector<double> lwr(const std::vector<double> &llh);

  void set_subst_rates(size_t, const model_params_t &);
  void set_freqs(size_t, const model_params_t &);
  void set_gamma_rates(size_t, const model_params_t &);
  void set_gamma_weights(size_t, model_params_t);

  void assign_indicies(const std::vector<size_t> &);
  void assign_indicies(size_t, size_t);
  void assign_indicies(size_t beg, size_t end, std::vector<size_t> idx);
  void assign_indicies();
  void assign_indicies_by_rank_search(size_t min_roots, double root_ratio, size_t rank, size_t num_tasks,
                                      checkpoint_t &checkpoint);
  void assign_indicies_by_rank_search(size_t min_roots, double root_ratio, size_t rank, size_t num_tasks,
                                      initial_root_strategy_t init_root, checkpoint_t &);
  void assign_indicies_by_rank_exhaustive(size_t rank, size_t num_tasks, checkpoint_t &);
  std::vector<size_t> assigned_indicies() const { return _assigned_idx; }

  // ---- B200-first addition: the per-partition terms of the last evaluation ------------------
  // compute_lh / compute_lh_root add the partitions' log-likelihoods in partition order; a run
  // that gives every GPU its own partitions (SURVEY 8e-3, BASELINE cfg4) needs the TERMS to
  // rebuild that same ordered sum across ranks (root_digger_b200.sharding.PartitionShardedModel).
  unsigned int sweep_chunks() const { return _sweep_chunks; }  // independent chunks of a directed sweep
  // outer iterations of search / exhaustive_search per root (the reference's loops run to 1e3,
  // src/model.cpp:1051,1171); a smaller cap bounds a benchmark sample, results are then not converged
  void   set_max_outer_iterations(size_t n) { _max_outer_iterations = n ? n : 1000; }
  size_t max_outer_iterations() const { return _max_outer_iterations; }
  const std::vector<double> &last_partition_lh() const { return _last_part_lh; }
  // ... and of the last sweep_root_lh: [partition][placement of the swept range]
  const std::vector<std::vector<double>> &last_sweep_partition_lh() const { return _last_sweep_part_lh; }

  // ---- partitions dealt to several processes (SURVEY 8e-3, BASELINE cfg4) ----------------------
  // This process holds the partitions global_index[0..local) of `global_partitions`.  Parameter
  // optimisation needs no exchange (each closure evaluates one partition, src/model.cpp:1544-1547);
  // every log-likelihood that the reference sums over partitions (:397,429 -- compute_lh,
  // compute_lh_root and with it compute_dlh / optimize_alpha, the placement sweep) is completed
  // through `exchange`: it receives this process's terms [local partition][count] and returns the
  // terms of ALL partitions [global partition][count]; they are then added in global partition
  // order, the order a single process uses, so search / exhaustive_search take the same decisions
  // on every rank and return the bits of a single-process run.  The model's random generator is
  // kept in step with a single process (one draw per GLOBAL partition in initialize_partitions*),
  // and the checkpoint records carry the parameters of ALL partitions (gathered the same way).
  typedef void (*partition_exchange_fn)(const double *local_terms, size_t local_partitions, size_t count,
                                        double *all_terms, void *user);
  void set_partition_exchange(const std::vector<size_t> &global_index, size_t global_partitions,
                              partition_exchange_fn exchange, void *user);
  bool partition_sharded() const { return _exchange != nullptr; }
  // state of the model's generator (std::minstd_rand: one integer), for callers that must put
  // several processes back in step after one of them failed half way through an initialisation
  uint64_t rng_state() const;
  void     set_rng_state(uint64_t state);
  void     discard_rng(unsigned long long draws) { _random_engine.discard(draws); }
  // the first local partition whose empirical frequencies have a zero entry, or -1 (loads the tips
  // of `msa`, the alignments initialize_partitions* will be given; draws nothing)
  int first_partition_without_empirical_freqs(const std::vector<msa_t> &msa);

  void move_root(const root_location_t &new_root);
  // use the fused engine entry points (rdk_sweep_root_placements) where the
  // reference loops over move_root + compute_lh_root; results are identical
  void set_fused(bool on) { _sweep_mode = on ? sweep_mode_t::directed : sweep_mode_t::sequential; }
  // how sweep_root_lh / suggest_roots_lh score the 2n-3 placements (identical values):
  //   sequential  the reference's loop, move_root + compute_lh_root per root (src/model.cpp:871-874)
  //   path        the same operations recorded into ONE rdk_sweep_root_placements call
  //   directed    one pre-order pass over directed CLVs (rooted_tree_t::generate_sweep_operations);
  //               leaves the tree rooted where it was
  enum class sweep_mode_t { sequential = 0, path = 1, directed = 2 };
  void         set_sweep_mode(sweep_mode_t m) { _sweep_mode = m; }
  sweep_mode_t sweep_mode() const { return _sweep_mode; }

  // The root-only evaluations of compute_dlh / optimize_alpha (two per slope, src/model.cpp:481-519;
  // five before the first decision, :679-693; one dyadic level of the sign-change search, :732-776)
  // go to the engine as ONE batch each (rdk_root_loglikelihood_multi) instead of one call, one
  // synchronisation -- and, on site shards, one all-reduce -- per evaluation.  Same values, same
  // decisions; off = the reference's call sequence (RD_BATCHED_PROBES=0 in the environment).
  void set_batched_probes(bool on) { _batched_probes = on; }
  bool batched_probes() const { return _batched_probes; }
  // what the position searches cost so far: fused batches issued, root-only evaluations inside
  // them, and root-only evaluations issued one by one (compute_lh_root included)
  struct probe_counters_t {
    unsigned long long fused_batches = 0, fused_evaluations = 0, single_evaluations = 0;
  };
  const probe_counters_t &probe_counters() const { return _probe_counters; }

  // ---- root placement support (DESIGN.md section 10) ------------------------------------------
  // RELL bootstrap proportions and one-sided KH / SH tests of every placement in a checkpoint:
  // each record's parameters are installed, the tree is rooted at (root_id, alpha) and one full
  // evaluation stores the unweighted per-pattern log-likelihoods; rdk_rell_support resamples them.
  // The model's parameters and root are put back afterwards; with keep_rows the rows stay on the
  // device, readable through site_lnl_rows, until the next call (otherwise their memory is freed).
  // On site shards (a communicator attached) every rank calls it with the same checkpoint,
  // replicates and seed and gets the bits of one GPU.  Each placement's branch is annotated with
  // BP, pKH, pSH.
  // With au_scales (thousandths; 2 to 32, strictly ascending, in [100, 10000]) the same call also
  // runs the multiscale bootstrap at those scales and fits the AU test per record, and computes the
  // expected likelihood weights (rdk_rell_support_ms; DESIGN.md section 10, items 6-8); the branches
  // then also carry pAU and ELW.
  // sampling chooses the resampling unit (DESIGN.md section 10, items 11-14): site (the above; each
  // partition resampled on its own), gene (the partitions themselves, with replacement) or gene_site
  // (partitions, then the sites of each drawn partition).  The gene modes need at least 2 partitions
  // and refuse au_scales; they also return each partition's fixed-point log-likelihood per record.
  enum class support_sampling_t { site, gene, gene_site };
  struct placement_support_t {
    std::vector<size_t>   root_id;
    std::vector<double>   alpha, llh, lnl_fixed, bp, p_kh, p_sh;
    std::vector<unsigned> bp_count, kh_count, sh_count;
    std::vector<unsigned long long> o_lo;  // O[r] as a two's-complement int128
    std::vector<long long>          o_hi;
    size_t                replicates = 0, best = 0;
    int                   exponent = 0;
    double                capture_ms = 0, counts_ms = 0, accumulate_ms = 0, statistics_ms = 0, resample_ms = 0;
    unsigned long long    device_bytes = 0;
    // AU mode only (empty otherwise): scale_count is [scale][record]
    std::vector<unsigned>           scales, scale_count, au_used;
    std::vector<double>             p_au, au_d, au_c, au_rss, elw;
    std::vector<unsigned long long> elw_fixed;
    double                          au_counts_ms = 0, au_accumulate_ms = 0, au_statistics_ms = 0;
    double                          positions_ms = 0;  // branch_support: the alpha searches
    // gene modes only (empty otherwise): [partition][record] O_i 2^-e and O_i as int128, and the
    // record of each partition's highest O_i (lowest index on ties)
    support_sampling_t              sampling = support_sampling_t::site;
    std::vector<double>             partition_lnl_fixed;
    std::vector<unsigned long long> partition_o_lo;
    std::vector<long long>          partition_o_hi;
    std::vector<unsigned>           partition_best;
    double                          gene_draws_ms = 0;
  };
  placement_support_t placement_support(checkpoint_t &checkpoint, size_t replicates, uint64_t seed,
                                        unsigned replicate_tile = 0, bool keep_rows = false,
                                        const std::vector<unsigned> &au_scales = {},
                                        support_sampling_t sampling = support_sampling_t::site);
  // The same statistics for EVERY branch at one set of parameters (DESIGN.md section 10, items 9-10):
  // the parameters of the checkpoint's best record (highest llh, lowest log index on ties) are
  // installed, root q is placed at a_q = optimize_alpha(root q at ratio 0.5, atol) (0.5 everywhere
  // with atol = 0) and record q of the statistics is the placement (q, a_q), for every root id q in
  // order.  One directed sweep scores all 2n - 3 placements and stores their rows.  Unlike
  // exhaustive mode, the substitution parameters are not re-optimised per branch.  alpha and llh
  // hold a_q and the log-likelihood at (q, a_q); positions_ms times the alpha searches, capture_ms
  // the sweep.  Every branch is annotated with BP, pKH, pSH (pAU, ELW in AU mode), LLH and alpha.
  // Refuses what placement_support refuses, and atol < 0.
  placement_support_t branch_support(checkpoint_t &checkpoint, size_t replicates, uint64_t seed, double atol,
                                     unsigned replicate_tile = 0, bool keep_rows = false,
                                     const std::vector<unsigned> &au_scales = {},
                                     support_sampling_t sampling = support_sampling_t::site);
  // the unweighted per-pattern log-likelihoods of the last placement_support / branch_support:
  // [record][pattern]
  std::vector<double> site_lnl_rows(size_t partition);

  // ---- marginal ancestral states (DESIGN.md section 11) ------------------------------------------
  // The posterior of every internal node of the tree rooted at `root` (its ratio included), at the
  // current parameters: one full traversal, then rdk_marginal_ancestral_states per partition.  Nodes
  // are the parents of the traversal's operations, in post-order (the root last).  The checkpoint form
  // installs the parameters and placement of the best record (highest llh, lowest log index on ties).
  // Both leave the parameters and the rooting as they found them.  Refuses models dealt to several
  // processes, a ratio outside [0, 1], and full_nodes that are not internal nodes of the rooted tree
  // or name a node twice.
  struct ancestral_options_t {
    std::vector<unsigned> full_nodes;      // CLV indices of the nodes whose full posterior is returned
    bool                  all_full = false;  // ... or every node; neither: the root
    unsigned              threads = 0;     // engine launch shape (rdk_ancestral_out_t): 0 = default
    unsigned              tile_sites = 0;
  };
  struct ancestral_states_t {
    struct partition_t {
      unsigned                   patterns = 0;
      std::vector<unsigned char> map_state;                  // [node][pattern], 0..3 = A, C, G, T
      std::vector<double>        map_prob, log_norm;         // [node][pattern]
      std::vector<double>        posterior;                  // [full node][pattern][4]
      std::vector<unsigned>      pattern_of_column;          // [column] -> pattern
      double                     ms = 0;                     // device time of the pass
      unsigned long long         device_bytes = 0;
      unsigned                   scratch = 0, tile_sites = 0;
    };
    std::vector<unsigned>                 clv_index;  // [node]
    std::vector<int>                      parent;     // [node]: position of the parent node, -1 for the root
    std::vector<std::vector<std::string>> clade;      // [node]: sorted tip labels below it
    std::vector<unsigned>                 full;       // positions of the nodes with full posteriors
    std::vector<rdk_operation_t>          ops;        // [node]: the post-order operation that computes it
    size_t                                root_id = 0;
    double                                ratio = 0.5;
    std::vector<partition_t>              partitions;
  };
  ancestral_states_t ancestral_states(const root_location_t &root, const ancestral_options_t &opts);
  ancestral_states_t ancestral_states(checkpoint_t &checkpoint, const ancestral_options_t &opts);
  const std::vector<unsigned> &pattern_of_column(size_t partition) const { return _pattern_of_column.at(partition); }

  rdk_partition_t *partition(size_t i) { return _partitions[i]; }
  size_t           partition_count() const { return _partitions.size(); }

private:
  // ---- root position on a branch ------------------------------------------------------------
  // log-likelihoods of the tree rooted at `ratios` on root's branch: ONE fused engine call per
  // partition when batched probes are on (rdk_root_loglikelihood_multi); compute_dlh and
  // optimize_alpha are rd::unit_segment_search_t (optim.hpp) over this
  std::vector<double> root_lh_on_branch(const root_location_t &root, const std::vector<double> &ratios);

  // ---- placement support, the parts placement_support and branch_support share ------------------
  void check_support_request(const std::string &who, size_t replicates, const std::vector<unsigned> &au_scales,
                             support_sampling_t sampling) const;
  void check_support_records(const std::string &who, const std::vector<checkpoint_t::record_t> &records) const;
  void install_record(const checkpoint_t::record_t &record);
  std::function<void()> support_restore_point(bool keep_rows);
  void reserve_support_rows(const std::string &who, unsigned rows);
  void resample_support(const std::string &who, placement_support_t &out, unsigned rows, size_t replicates,
                        uint64_t seed, unsigned replicate_tile, const std::vector<unsigned> &au_scales,
                        support_sampling_t sampling);
  void annotate_support(placement_support_t &out, const std::vector<root_location_t> &where);
  rooted_tree_t::sweep_schedule_t directed_sweep_schedule(size_t begin, size_t end, const std::vector<double> &ratio,
                                                          std::vector<unsigned int> &chunk_off) const;

  ancestral_states_t ancestral_states_here(const std::string &who, const root_location_t &root,
                                           const ancestral_options_t &opts);

  // ---- parameter plumbing ----------------------------------------------------------------------
  void set_subst_rates_random(size_t, const msa_t &);
  void set_subst_rates_uniform();
  void install_gamma_rates(size_t partition, double alpha, int mode);
  void set_gamma_rates(size_t);
  void update_invariant_sites(size_t);
  void set_tip_states(size_t, const msa_t &);
  void set_empirical_freqs(size_t);
  void set_empirical_freqs();
  void set_freqs_all_free(size_t, model_params_t);
  void set_model_params(const std::vector<partition_parameters_t> &);
  template <typename PerPartition> void for_each_partition_in_global_order(PerPartition &&body);
  void reset_to_defaults();  // rates 1/12, empirical frequencies (what every start begins from)
  std::vector<partition_parameters_t> fresh_parameters();
  std::vector<partition_parameters_t> parameters_of_all_partitions(const std::vector<partition_parameters_t> &mine);
  std::vector<partition_parameters_t> parameters_held_here(const std::vector<partition_parameters_t> &all) const;
  partition_parameters_t make_partition_parameters(size_t states, rate_category rc, size_t rate_cat_count);

  // ---- evaluation ------------------------------------------------------------------------------
  struct traversal_t {  // a full post-order schedule for one root placement
    std::vector<rdk_operation_t> ops;
    std::vector<unsigned int>    pmatrix_indices;
    std::vector<double>          branch_lengths;
  };
  traversal_t full_traversal(const root_location_t &rl);
  void   update_pmatrix_partition(size_t partition_index, const std::vector<unsigned int> &pmatrix_indices,
                                  const std::vector<double> &branch_lengths);
  double root_loglikelihood(size_t partition_index);
  double root_only_evaluation(const root_location_t &root);
  // sum over ALL partitions, in global partition order, of terms[local partition][0..count)
  std::vector<double> sum_over_partitions(const std::vector<std::vector<double>> &terms, size_t count);
  double              sum_over_partitions(const std::vector<double> &terms);
  double compute_lh_partition(size_t partition_index, const traversal_t &trav);
  void   optimize_params(std::vector<partition_parameters_t> &params, const root_location_t &rl,
                         double pgtol, double factor, bool optimize_gamma);
  std::pair<root_location_t, double> placement_of(const rd_result_t &result) const;
  void assign_rank_share(const std::vector<size_t> &work, size_t rank, size_t num_tasks);

  rooted_tree_t                          _tree;
  std::vector<rdk_partition_t *>         _partitions;
  std::vector<rate_category>             _rate_category_types;
  std::vector<double>                    _partition_weights;
  std::vector<model_params_t>            _rate_rates;
  std::vector<model_params_t>            _rate_weights;
  std::vector<bool>                      _rate_user_init;
  std::vector<std::vector<unsigned int>> _param_indicies;
  std::vector<size_t>                    _assigned_idx;
  std::minstd_rand                       _random_engine;
  bool                                   _invariant_sites;
  uint64_t                               _seed;
  bool                                   _early_stop;
  sweep_mode_t                           _sweep_mode = sweep_mode_t::directed;
  std::vector<double>                    _last_part_lh;
  std::vector<std::vector<double>>       _last_sweep_part_lh;
  unsigned int                           _sweep_extra = 0;   // spare directed-CLV buffers per sweep chunk
  unsigned int                           _sweep_chunks = 1;  // independent chunks of a directed sweep
  size_t                                 _max_outer_iterations = 1000;
  bool                                   _batched_probes = true;  // see set_batched_probes
  probe_counters_t                       _probe_counters;
  partition_exchange_fn                  _exchange = nullptr;     // see set_partition_exchange
  void                                  *_exchange_user = nullptr;
  unsigned                               _support_rows = 0;       // rows of the last placement_support
  std::vector<std::vector<unsigned>>     _pattern_of_column;     // per partition: [column] -> pattern
  std::vector<size_t>                    _global_index;           // global id of each local partition
  size_t                                 _global_partitions = 0;
  static constexpr unsigned int          _submodels = 1;
};

#endif
