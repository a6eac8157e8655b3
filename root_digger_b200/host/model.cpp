// model.cpp -- see model.hpp.  Members cite the reference code whose behaviour they reproduce
// (RootDigger src/model.cpp); quirks that change results are kept on purpose and named
// (SURVEY.md Appendix B).
//
// How this file is organised, and what it owes to the reference.
//   * The RESULT of RootDigger is the end point of two optimiser trajectories per candidate (model
//     parameters by L-BFGS-B, position on the branch by a bracketing search on the slope), so the
//     decisions taken along them -- which comparison, on which floating-point expression, in which
//     order -- are specified by the reference and reproduced here; tests/test_reference_sources.py
//     runs the reference's OWN src/model.cpp (compiled unchanged against compat/corax/corax.h) next
//     to this file and demands the same bits.
//   * The code that takes those decisions is this repository's: the optimisers are stand-alone
//     components (optim.hpp: slope_root_brent, lbfgsb_session_t, minimize_in_box) driven through
//     functors; every root-only evaluation on a branch goes through ONE primitive (probe_branch)
//     that hands the engine whole batches -- both evaluations of a slope, the five evaluations
//     optimize_alpha needs before its first decision, a whole dyadic level of its sign-change
//     search -- as one fused call, one synchronisation and (on site shards) one all-reduce; the
//     two search drivers share their bookkeeping; the placement sweep is a directed-CLV pass in
//     chunks; partitions may be sharded over GPUs (shard_spec_t) and report their terms.
#include "model.hpp"

#ifdef RD_BACKEND_ORACLE
#include "rdk_support.h"     // tests/oracle_shim: the placement-support entries over the CPU oracle
#include "rdk_support_au.h"  // ... and rdk_rell_support_ms
#include "rdk_sweep_rows.h"   // ... and the row capture of the placement sweep
#endif
#include "support_stats.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <exception>
#include <functional>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <numeric>
#include <sstream>

// src/model.cpp:87-93
model_params_t random_params(size_t size, uint64_t seed) {
  model_params_t                   mp(size);
  std::minstd_rand                 engine(seed);
  std::uniform_real_distribution<> dist(1e-4, 1.0);
  for (auto &f : mp) f = dist(engine);
  return mp;
}

static std::string engine_error() { return std::string(rdk_errmsg); }

// Partitions are driven concurrently from OpenMP threads (reference src/model.cpp:397,429,1935).
// An exception must not leave a parallel region (that terminates the process), and the engine's
// error message is thread-local: both are caught ON the failing thread and the first one (in
// partition order) is rethrown after the region.
template <typename Body>
static void for_each_partition(size_t n, bool dynamic, Body &&body) {
  std::vector<std::exception_ptr> errors(n);
  auto                            guarded = [&](size_t i) {
    try {
      body(i);
    } catch (...) {
      errors[i] = std::current_exception();
    }
  };
  if (n == 1) {
    guarded(0);  // the common case (cfg2 / cfg3 / cfg5): no thread team to wake per engine call
  } else if (dynamic) {
#pragma omp parallel for schedule(dynamic)
    for (size_t i = 0; i < n; ++i) guarded(i);
  } else {
#pragma omp parallel for
    for (size_t i = 0; i < n; ++i) guarded(i);
  }
  for (auto &e : errors)
    if (e) std::rethrow_exception(e);
}

// ---------------------------------------------------------------------------
// construction (src/model.cpp:99-182)
// ---------------------------------------------------------------------------
model_t::model_t(rooted_tree_t tree, const std::vector<msa_t> &msas,
                 const std::vector<ratehet_opts_t> &rate_cats, bool invariant_sites, uint64_t seed,
                 bool early_stop, const shard_spec_t &shard)
    : _invariant_sites{invariant_sites}, _seed{seed}, _early_stop{early_stop} {
  _random_engine = std::minstd_rand(_seed);
  _tree = std::move(tree);
  if (const char *env = std::getenv("RD_BATCHED_PROBES")) _batched_probes = std::atoi(env) != 0;
  if (rate_cats.size() < msas.size())
    throw std::invalid_argument("one rate heterogeneity option per partition is required");
  for (auto rc : rate_cats) {
    _rate_rates.emplace_back(rc.rate_cats, rc.alpha);
    _rate_weights.emplace_back(rc.rate_cats, 1.0 / rc.rate_cats);
    _rate_category_types.emplace_back(rc.rate_category_type);
    _rate_user_init.emplace_back(rc.alpha_init);
    _param_indicies.emplace_back(rc.rate_cats, 0);
  }
  for (auto &msa : msas)
    if (!msa.constiency_check(_tree.label_set()))
      throw std::invalid_argument("Taxa on the tree and in the MSA are inconsistient");

  for (size_t pi = 0; pi < msas.size(); ++pi) {
    auto &msa = msas[pi];
    if (msa.length() > static_cast<size_t>(std::numeric_limits<int>::max()))
      throw std::runtime_error("The length of the MSA is too large to safely cast");
    // the ARCH_* attributes of the reference select coraxlib CPU kernels; the
    // engine accepts and ignores them
    unsigned int attributes = RDK_ATTRIB_SITE_REPEATS | RDK_ATTRIB_NONREV;
    // on top of what the reference asks for (src/model.cpp:159-168): spare CLV / scale
    // buffers for the directed CLVs of the placement sweep (one per depth level) and three
    // spare P-matrices (rooted_tree_t::generate_sweep_operations); the engine allocates a
    // CLV on first use, so unused spares cost only their scale buffer
    // -- once per independent CHUNK of the sweep: a small partition fills the device only
    // when several chunks of placements are walked side by side (rdk_sweep_root_placements_chunks)
    _sweep_extra = _tree.sweep_depth_bound();
    if (pi == 0) {
      _sweep_chunks = 1;
      for (size_t q = 0; q < msas.size(); ++q) {
        // Site-sharded: the all-reduce adds the ranks' log-likelihoods slot by slot, so EVERY rank
        // must walk the placements in the same order, i.e. cut the sweep into the same chunks --
        // the count comes from the largest shard of the layout (a function of the global site
        // count and the number of ranks only), never from this rank's own site count.
        unsigned long long sites = msas[q].length();
        if (shard.global_sites && shard.nranks > 1) {
          const unsigned long long blocks = (shard.global_sites + RDK_SHARD_ALIGN - 1) / RDK_SHARD_ALIGN;
          const unsigned long long per = (blocks + (unsigned long long)shard.nranks - 1) / (unsigned long long)shard.nranks;
          sites = std::min<unsigned long long>(per * RDK_SHARD_ALIGN, shard.global_sites);
        }
        _sweep_chunks = std::max(_sweep_chunks, rdk_sweep_chunk_hint((unsigned int)sites,
                                                                     (unsigned int)_rate_rates[q].size()));
      }
      _sweep_chunks = std::min<unsigned int>(_sweep_chunks, RDK_SWEEP_MAX_CHUNKS);
    }
    rdk_partition_t *p = rdk_partition_create(
        _tree.tip_count(), _tree.branch_count() + _sweep_chunks * _sweep_extra, msa.states(), msa.length(),
        _submodels, _tree.branch_count() + 3, static_cast<unsigned int>(_rate_rates[pi].size()),
        _tree.branch_count() + _sweep_chunks * _sweep_extra, attributes);
    if (!p) throw std::runtime_error("partition could not be created: " + engine_error());
    _partitions.push_back(p);
#ifndef RD_BACKEND_ORACLE
    if (shard.global_sites) {
      if (msas.size() != 1) throw std::invalid_argument("site sharding supports a single MSA partition");
      if (rdk_partition_set_shard(p, shard.site_offset, shard.global_sites) != RDK_SUCCESS)
        throw std::runtime_error(engine_error());
      if (shard.comm_id && shard.nranks > 1 &&
          rdk_partition_attach_comm(p, shard.nranks, shard.rank, shard.comm_id) != RDK_SUCCESS)
        throw std::runtime_error(engine_error());
    }
#else
    (void)shard;
#endif
    _partition_weights.push_back(msa.total_weight());
    set_gamma_rates(pi);
  }
  assign_indicies();
}

model_t::~model_t() {
  for (auto p : _partitions)
    if (p) rdk_partition_destroy(p);
}

// ---------------------------------------------------------------------------
// parameter plumbing (reference src/model.cpp:184-355)
// ---------------------------------------------------------------------------
void model_t::set_subst_rates(size_t p, const model_params_t &mp) {
  rdk_set_subst_params(_partitions[p], 0, mp.data());
}

void model_t::set_subst_rates_random(size_t p, const msa_t &msa) {
  set_subst_rates(p, random_params(msa.states() * msa.states() - msa.states(), _random_engine()));
}

void model_t::set_subst_rates_uniform() {
  for (size_t p = 0; p < _partitions.size(); ++p) {
    const unsigned int states = _partitions[p]->states, off_diagonal = states * states - states;
    set_subst_rates(p, model_params_t(off_diagonal, 1.0 / off_diagonal));
  }
}

void model_t::set_gamma_weights(size_t p, model_params_t w) {
  double total = 0.0;
  for (double v : w) total += v;
  for (double &v : w) v /= total;
  rdk_set_category_weights(_partitions[p], w.data());
}

// discrete-Gamma category rates for shape `alpha` into the partition and into _rate_rates
void model_t::install_gamma_rates(size_t p, double alpha, int mode) {
  auto &rates = _rate_rates[p];
  rdk_compute_gamma_cats(alpha, (unsigned)rates.size(), rates.data(), mode);
  rdk_set_category_rates(_partitions[p], rates.data());
}

// Initial state of a partition: its category weights and the rates for shape 1.
// Appendix B-1: the reference initialises BOTH the mean- and the median-typed categories with
// the MEAN discretisation at alpha = 1 (src/model.cpp:238-245,256-263); free rates start at 1.
void model_t::set_gamma_rates(size_t p) {
  rdk_set_category_weights(_partitions[p], _rate_weights[p].data());
  if (_rate_category_types[p] == rate_category::FREE) {
    std::fill(_rate_rates[p].begin(), _rate_rates[p].end(), 1.0);
    rdk_set_category_rates(_partitions[p], _rate_rates[p].data());
    return;
  }
  install_gamma_rates(p, 1.0, RDK_GAMMA_RATES_MEAN);
}

// The shape the optimiser proposes.
// Appendix B-1: with a shape given, both category types use the MEDIAN discretisation
// (src/model.cpp:247-254,265-272).  Appendix B-2: proposed FREE rates are normalised into a
// temporary that is dropped -- the stored rates are what is (re)installed (:279-290), so free
// rates never move; only the free WEIGHTS are effective.
void model_t::set_gamma_rates(size_t p, const model_params_t &alpha) {
  if (_rate_category_types[p] == rate_category::FREE) {
    rdk_set_category_rates(_partitions[p], _rate_rates[p].data());
    return;
  }
  install_gamma_rates(p, alpha[0], RDK_GAMMA_RATES_MEDIAN);
}

void model_t::update_invariant_sites(size_t p) {
  if (_invariant_sites) {
    rdk_update_invariant_sites(_partitions[p]);
    return;
  }
  for (unsigned int m = 0; m < _submodels; ++m) rdk_update_invariant_sites_proportion(_partitions[p], m, 0.0);
}

// src/model.cpp:302-325: every alignment row goes to the tip of the same label
void model_t::set_tip_states(size_t p, const msa_t &msa) {
  const auto tip_of = _tree.label_map();
  for (int row = 0; row < msa.count(); ++row) {
    const auto hit = tip_of.find(msa.label(row));
    if (hit == tip_of.end())
      throw std::runtime_error(std::string("Could not find taxa ") + msa.label(row) + " in tree");
    if (rdk_set_tip_states(_partitions[p], hit->second, msa.map(), msa.sequence(row)) == RDK_FAILURE)
      throw std::runtime_error("failed to set tip " + std::to_string(row) + ": " + engine_error());
  }
  rdk_set_pattern_weights(_partitions[p], msa.weights());
}

// src/model.cpp:327-339: a state that never occurs makes the model degenerate -- refused
void model_t::set_empirical_freqs(size_t p) {
  rdk_partition_t *partition = _partitions[p];
  struct freed_t {
    double *v;
    ~freed_t() { free(v); }
  } emp{rdk_msa_empirical_frequencies(partition)};
  if (!emp.v) throw std::runtime_error("empirical frequencies failed: " + engine_error());
  if (std::any_of(emp.v, emp.v + partition->states, [](double f) { return f <= 0; }))
    throw invalid_empirical_frequencies_exception(
        "One of the state frequenices is zero while using emperical frequencies");
  rdk_set_frequencies(partition, 0, emp.v);
}

void model_t::set_empirical_freqs() {
  for (size_t p = 0; p < _partitions.size(); ++p) set_empirical_freqs(p);
}

void model_t::set_freqs(size_t p, const model_params_t &freqs) {
  if (std::any_of(freqs.begin(), freqs.end(), [](double f) { return f <= 0.0; }))
    throw std::runtime_error("Frequencies with 0 entries are not allowed");
  rdk_set_frequencies(_partitions[p], 0, freqs.data());
}

// Appendix B-4 (src/model.cpp:350-355): all four frequencies are free, renormalised on the way in
void model_t::set_freqs_all_free(size_t p, model_params_t freqs) {
  double total = 0.0;
  for (double v : freqs) total += v;
  for (double &v : freqs) v /= total;
  set_freqs(p, freqs);
}

void model_t::set_model_params(const std::vector<partition_parameters_t> &params) {
  for (size_t p = 0; p < params.size(); ++p) {
    set_subst_rates(p, params[p].subst_rates);
    set_freqs(p, params[p].freqs);
    set_gamma_rates(p, params[p].gamma_alpha);
    if (_rate_category_types[p] == rate_category::FREE) set_gamma_weights(p, params[p].gamma_weights);
  }
}

// Appendix B-9: every start begins from rates 1/12 and empirical frequencies
void model_t::reset_to_defaults() {
  set_subst_rates_uniform();
  set_empirical_freqs();
}

// src/model.cpp:979-1005: the optimiser's starting point for one partition; FREE weights are
// drawn from the model's generator (so the draw order over partitions is part of the result)
partition_parameters_t model_t::make_partition_parameters(size_t states, rate_category rc,
                                                          size_t rate_cat_count) {
  partition_parameters_t pp;
  const size_t           off_diagonal = states * states - states;
  pp.subst_rates.assign(off_diagonal, 1.0 / off_diagonal);
  pp.freqs.assign(states, 1.0 / states);
  if (rc == rate_category::FREE) {
    pp.gamma_alpha.assign(rate_cat_count, 1.0);
    pp.gamma_weights.resize(rate_cat_count);
    std::uniform_real_distribution<> unit(0.0, 1.0);
    for (auto &w : pp.gamma_weights) w = unit(_random_engine);
  } else {
    pp.gamma_alpha.assign(1, 1.0);
  }
  return pp;
}

std::vector<partition_parameters_t> model_t::fresh_parameters() {
  std::vector<partition_parameters_t> params;
  params.reserve(_partitions.size());
  for (size_t p = 0; p < _partitions.size(); ++p)
    params.push_back(
        make_partition_parameters(_partitions[p]->states, _rate_category_types[p], _partitions[p]->rate_cats));
  return params;
}

// The parameters of ALL partitions, in global order, for the checkpoint record of a start: on
// partition shards every rank contributes the blocks it fitted (12 rates, 4 frequencies, the Gamma
// shape) through the same exchange that completes the log-likelihood sums, so every rank's log
// holds complete records in the reference's format.
std::vector<partition_parameters_t> model_t::parameters_of_all_partitions(
    const std::vector<partition_parameters_t> &mine) {
  if (!_exchange) return mine;
  size_t rates = 0, freqs = 0, shape = 0;
  if (!mine.empty()) {
    rates = mine[0].subst_rates.size();
    freqs = mine[0].freqs.size();
    shape = mine[0].gamma_alpha.size();
  }
  const size_t                     width = rates + freqs + shape;
  std::vector<std::vector<double>> rows;
  for (const auto &pp : mine) {
    if (pp.subst_rates.size() != rates || pp.freqs.size() != freqs || pp.gamma_alpha.size() != shape ||
        !pp.gamma_weights.empty())
      throw std::logic_error("partition shards: parameter blocks of one shape per partition are expected");
    std::vector<double> row(pp.subst_rates);
    row.insert(row.end(), pp.freqs.begin(), pp.freqs.end());
    row.insert(row.end(), pp.gamma_alpha.begin(), pp.gamma_alpha.end());
    rows.push_back(std::move(row));
  }
  std::vector<double> local(rows.size() * width), all(_global_partitions * width, 0.0);
  for (size_t p = 0; p < rows.size(); ++p) std::copy(rows[p].begin(), rows[p].end(), local.begin() + (std::ptrdiff_t)(p * width));
  _exchange(local.data(), rows.size(), width, all.data(), _exchange_user);
  std::vector<partition_parameters_t> out(_global_partitions);
  for (size_t g = 0; g < _global_partitions; ++g) {
    const double *row = all.data() + g * width;
    out[g].subst_rates.assign(row, row + rates);
    out[g].freqs.assign(row + rates, row + rates + freqs);
    out[g].gamma_alpha.assign(row + rates + freqs, row + width);
  }
  return out;
}

// ... and back: the blocks of the partitions held here, out of a complete record
std::vector<partition_parameters_t> model_t::parameters_held_here(const std::vector<partition_parameters_t> &all) const {
  if (!_exchange || all.size() != _global_partitions) return all;
  std::vector<partition_parameters_t> mine;
  mine.reserve(_global_index.size());
  for (size_t g : _global_index) mine.push_back(all[g]);
  return mine;
}

// ---------------------------------------------------------------------------
// evaluation
// ---------------------------------------------------------------------------
model_t::traversal_t model_t::full_traversal(const root_location_t &rl) {
  traversal_t t;
  std::tie(t.ops, t.pmatrix_indices, t.branch_lengths) = _tree.generate_operations(rl);
  return t;
}

// src/model.cpp:357-370: the reference issues one corax_update_prob_matrices call per branch from
// an OpenMP loop; one call with all branches is the same thing for the engine (one kernel)
void model_t::update_pmatrix_partition(size_t pi, const std::vector<unsigned int> &pmatrix_indices,
                                       const std::vector<double> &branch_lengths) {
  if (pmatrix_indices.empty()) return;
  if (rdk_update_prob_matrices(_partitions[pi], _param_indicies[pi].data(), pmatrix_indices.data(),
                               branch_lengths.data(), (unsigned)pmatrix_indices.size()) == RDK_FAILURE)
    throw std::runtime_error(engine_error());  // the message of THIS thread
}

double model_t::root_loglikelihood(size_t pi) {
  return rdk_compute_root_loglikelihood(_partitions[pi], _tree.root_clv_index(), _tree.root_scaler_index(),
                                        _param_indicies[pi].data(), nullptr);
}

static double sum_in_order(const std::vector<double> &terms) {
  double total = 0.0;
  for (double v : terms) total += v;
  return total;
}

// ---- partitions dealt to several processes -------------------------------------------------
void model_t::set_partition_exchange(const std::vector<size_t> &global_index, size_t global_partitions,
                                     partition_exchange_fn exchange, void *user) {
  if (!exchange) {
    _exchange = nullptr;
    _exchange_user = nullptr;
    _global_index.clear();
    _global_partitions = 0;
    return;
  }
  if (global_index.size() != _partitions.size())
    throw std::invalid_argument("set_partition_exchange: one global index per local partition is required");
  for (size_t j = 0; j < global_index.size(); ++j)
    if (global_index[j] >= global_partitions || (j && global_index[j] <= global_index[j - 1]))
      throw std::invalid_argument("set_partition_exchange: global indices must be increasing and below the total");
  for (auto type : _rate_category_types)
    if (type == rate_category::FREE)
      throw std::invalid_argument("set_partition_exchange: free rate categories draw their start weights from the "
                                  "model's generator partition by partition and are not supported on shards");
  _global_index = global_index;
  _global_partitions = global_partitions;
  _exchange = exchange;
  _exchange_user = user;
}

std::vector<double> model_t::sum_over_partitions(const std::vector<std::vector<double>> &terms, size_t count) {
  std::vector<double> total(count, 0.0);
  if (!_exchange) {
    for (const auto &of_partition : terms)
      for (size_t i = 0; i < count; ++i) total[i] += of_partition[i];
    return total;
  }
  std::vector<double> local(terms.size() * count), all(_global_partitions * count, 0.0);
  for (size_t p = 0; p < terms.size(); ++p) std::copy(terms[p].begin(), terms[p].begin() + (std::ptrdiff_t)count,
                                                      local.begin() + (std::ptrdiff_t)(p * count));
  _exchange(local.data(), terms.size(), count, all.data(), _exchange_user);
  for (size_t g = 0; g < _global_partitions; ++g)
    for (size_t i = 0; i < count; ++i) total[i] += all[g * count + i];
  return total;
}

double model_t::sum_over_partitions(const std::vector<double> &terms) {
  if (!_exchange) return sum_in_order(terms);
  std::vector<std::vector<double>> as_rows;
  as_rows.reserve(terms.size());
  for (double v : terms) as_rows.push_back({v});
  return sum_over_partitions(as_rows, 1)[0];
}

uint64_t model_t::rng_state() const {
  std::ostringstream text;
  text << _random_engine;
  return std::stoull(text.str());
}

void model_t::set_rng_state(uint64_t state) { _random_engine.seed((std::minstd_rand::result_type)state); }

int model_t::first_partition_without_empirical_freqs(const std::vector<msa_t> &msa) {
  for (size_t p = 0; p < _partitions.size(); ++p) {
    set_tip_states(p, msa[p]);  // the frequencies are counted over the tips; setting them twice is harmless
    double *emp = rdk_msa_empirical_frequencies(_partitions[p]);
    if (!emp) throw std::runtime_error("empirical frequencies failed: " + engine_error());
    const bool degenerate = std::any_of(emp, emp + _partitions[p]->states, [](double f) { return f <= 0; });
    free(emp);
    if (degenerate) return (int)p;
  }
  return -1;
}

static void refuse_nan(double lh) {
  if (std::isnan(lh)) throw std::runtime_error("lh at root is not a number: " + std::to_string(lh));
}

// src/model.cpp:384-413.  The reference adds the partitions with an OpenMP reduction (:397) whose
// association order depends on the thread count; here the terms are added in partition order, so
// the result is the same on any host and on any number of GPUs.  (Appendix B-3: the P-matrices
// are refreshed on every call, the "changed" flags of the reference are always true.)
double model_t::compute_lh(const root_location_t &root_location) {
  const traversal_t trav = full_traversal(root_location);
  for (size_t p = 0; p < _partitions.size(); ++p)
    update_pmatrix_partition(p, trav.pmatrix_indices, trav.branch_lengths);
  std::vector<double> terms(_partitions.size(), 0.0);
  for_each_partition(_partitions.size(), false, [&](size_t p) {
    rdk_update_clvs(_partitions[p], trav.ops.data(), (unsigned)trav.ops.size());
    terms[p] = root_loglikelihood(p);
  });
  _last_part_lh = terms;
  return sum_over_partitions(terms);
}

// src/model.cpp:415-452: the two root branches and the root CLV only
double model_t::compute_lh_root(const root_location_t &root) {
  const double lh = root_only_evaluation(root);
  refuse_nan(lh);
  return lh;
}

// the tree re-rooted at `root` on the host, then, per partition: the two root P-matrices, the root
// CLV, the log-likelihood; summed over partitions.  NaN is the caller's to judge.
double model_t::root_only_evaluation(const root_location_t &root) {
  rdk_operation_t           op;
  std::vector<unsigned int> matrix_indices;
  std::vector<double>       branch_lengths;
  std::tie(op, matrix_indices, branch_lengths) = _tree.generate_derivative_operations(root);
  std::vector<double> terms(_partitions.size(), 0.0);
  for_each_partition(_partitions.size(), false, [&](size_t p) {
    update_pmatrix_partition(p, matrix_indices, branch_lengths);
    rdk_update_clvs(_partitions[p], &op, 1);
    terms[p] = root_loglikelihood(p);
  });
  _last_part_lh = terms;
  _probe_counters.single_evaluations++;
  return sum_over_partitions(terms);
}

// src/model.cpp:454-476: what the parameter optimiser evaluates, one partition at a time
double model_t::compute_lh_partition(size_t pi, const traversal_t &trav) {
  update_pmatrix_partition(pi, trav.pmatrix_indices, trav.branch_lengths);
  rdk_update_clvs(_partitions[pi], trav.ops.data(), (unsigned)trav.ops.size());
  const double lh = root_loglikelihood(pi);
  refuse_nan(lh);
  return lh;
}

// src/model.cpp:823-854: CLVs re-oriented along the path from the current root to the new one
void model_t::move_root(const root_location_t &new_root) {
  std::vector<rdk_operation_t> ops;
  std::vector<unsigned int>    pmatrix_indices;
  std::vector<double>          branch_lengths;
  std::tie(ops, pmatrix_indices, branch_lengths) = _tree.generate_root_update_operations(new_root);
  for (size_t p = 0; p < _partitions.size(); ++p) {
    if (rdk_update_prob_matrices(_partitions[p], _param_indicies[p].data(), pmatrix_indices.data(),
                                 branch_lengths.data(), (unsigned)pmatrix_indices.size()) == RDK_FAILURE)
      throw std::runtime_error(engine_error());
    rdk_update_clvs(_partitions[p], ops.data(), (unsigned)ops.size());
  }
}

// src/model.cpp:1737-1746
std::vector<double> model_t::compute_all_root_lh() {
  const auto &roots = _tree.roots();
  compute_lh(roots[0]);
  std::vector<double> lh;
  lh.reserve(roots.size());
  for (const auto &rl : roots) {
    move_root(rl);
    lh.push_back(compute_lh(rl));
  }
  return lh;
}

// ---------------------------------------------------------------------------
// position on the branch: slopes, the bracketing search, optimize_alpha
// ---------------------------------------------------------------------------
// Log-likelihood of the tree rooted on root's branch at each of `ratios`, the CLVs below the root
// being valid.  Batched: one rdk_root_loglikelihood_multi per partition for ALL ratios (the engine
// stages the 2 P-matrices of every candidate, evaluates them in one program and leaves the
// partition untouched).  Sequential: the reference's call sequence, one compute_lh_root each.
// Either way the host tree ends up rooted at the last ratio, as after the reference's calls, and
// NaN is reported by the CONSUMER of a value (rd::unit_segment_search_t), in consumption order --
// a batch may hold evaluations the decision never looks at.
std::vector<double> model_t::root_lh_on_branch(const root_location_t &root, const std::vector<double> &ratios) {
  std::vector<double> lh(ratios.size(), 0.0);
  if (ratios.empty()) return lh;
  root_location_t at{root};

  bool            fused = _batched_probes;
  rdk_operation_t root_op;
  std::vector<double> lengths;  // (child 1, child 2) per ratio
  if (fused) {
    lengths.reserve(2 * ratios.size());
    for (size_t i = 0; i < ratios.size(); ++i) {
      at.brlen_ratio = ratios[i];
      rdk_operation_t           op;
      std::vector<unsigned int> mi;
      std::vector<double>       bl;
      std::tie(op, mi, bl) = _tree.generate_derivative_operations(at);
      // one root operation serves the whole batch: the same branch must give the same operation
      if (i == 0)
        root_op = op;
      else if (std::memcmp(&op, &root_op, sizeof(op)) != 0)
        fused = false;
      lengths.insert(lengths.end(), bl.begin(), bl.end());
    }
  }
  if (!fused) {
    for (size_t i = 0; i < ratios.size(); ++i) {
      at.brlen_ratio = ratios[i];
      lh[i] = root_only_evaluation(at);
    }
    return lh;
  }

  std::vector<std::vector<double>> terms(_partitions.size(), std::vector<double>(ratios.size(), 0.0));
  for_each_partition(_partitions.size(), false, [&](size_t p) {
    if (rdk_root_loglikelihood_multi(_partitions[p], &root_op, _param_indicies[p].data(), _param_indicies[p].data(),
                                     lengths.data(), (unsigned)ratios.size(), terms[p].data()) == RDK_FAILURE)
      throw std::runtime_error(engine_error());
  });
  _probe_counters.fused_batches++;
  _probe_counters.fused_evaluations += ratios.size();
  lh = sum_over_partitions(terms, ratios.size());  // partition order, as compute_lh_root adds them
  _last_part_lh.resize(_partitions.size());
  for (size_t p = 0; p < _partitions.size(); ++p) _last_part_lh[p] = terms[p].back();
  return lh;
}

// compute_dlh (src/model.cpp:481-519) and optimize_alpha (:679-794) are rd::unit_segment_search_t
// (optim.hpp) on this branch: a batch of abscissae is a batch of root positions.
dlh_t model_t::compute_dlh(const root_location_t &root) {
  auto on_branch = rd::make_unit_segment_search(
      [&](const std::vector<double> &ratios) { return root_lh_on_branch(root, ratios); }, refuse_nan, _batched_probes);
  const auto s = on_branch.slope_at(root.brlen_ratio);
  return {s.value, s.slope};
}

root_location_t model_t::optimize_alpha(const root_location_t &root, double atol) {
  auto on_branch = rd::make_unit_segment_search(
      [&](const std::vector<double> &ratios) { return root_lh_on_branch(root, ratios); }, refuse_nan, _batched_probes);
  root_location_t best{root};
  best.brlen_ratio = on_branch.argmax(root.brlen_ratio, atol, std::to_string(root.edge->length));
  return best;
}

// src/model.cpp:796-821: the most likely placements of the sweep, each polished on its branch
// (Appendix B-6: the tolerance of that search is fixed at 1e-14 here)
std::pair<root_location_t, double> model_t::optimize_root_location(size_t min_roots, double root_ratio) {
  std::pair<root_location_t, double> best{root_location_t{}, -std::numeric_limits<double>::infinity()};
  for (auto &candidate : suggest_roots_lh(min_roots, root_ratio)) {
    move_root(candidate);
    candidate = optimize_alpha(candidate, 1e-14);
    const double lh = compute_lh_root(candidate);
    if (lh > best.second) best = {candidate, lh};
  }
  return best;
}

// ---------------------------------------------------------------------------
// candidate placements
// ---------------------------------------------------------------------------
static inline size_t shortlist_size(size_t candidates, double ratio, size_t at_least) {
  return std::max(static_cast<size_t>(candidates * ratio), at_least);
}

std::vector<root_location_t> model_t::suggest_roots_random(size_t min, double ratio) {
  auto roots = _tree.roots();
  std::shuffle(roots.begin(), roots.end(), _random_engine);
  roots.resize(shortlist_size(roots.size(), ratio, min));
  return roots;
}

// The directed sweep of the root ids [begin, end) from the current root, cut into _sweep_chunks
// ranges of consecutive root ids, each with its own spare buffers (and its own copy of the directed
// CLVs on the path to its first placement): independent programs the engine may walk side by side.
// `ratio` as rooted_tree_t::generate_sweep_operations takes it; chunk_off receives the chunk offsets.
rooted_tree_t::sweep_schedule_t model_t::directed_sweep_schedule(size_t begin, size_t end,
                                                                 const std::vector<double> &ratio,
                                                                 std::vector<unsigned int> &chunk_off) const {
  const size_t                    total = end - begin;
  const unsigned int              chunks = (unsigned int)std::max<size_t>(1, std::min<size_t>(_sweep_chunks, total / 8));
  rooted_tree_t::sweep_schedule_t sw;
  chunk_off.assign(1, 0u);
  for (unsigned int c = 0; c < chunks; ++c) {
    const size_t b0 = begin + total * c / chunks, b1 = begin + total * (c + 1) / chunks;
    auto part = _tree.generate_sweep_operations(b0, b1, _tree.tip_count() + _tree.branch_count() + c * _sweep_extra,
                                                (int)(_tree.branch_count() + c * _sweep_extra),
                                                _tree.branch_count(), _sweep_extra, ratio);
    const unsigned int pm_base = (unsigned int)sw.mi.size(), op_base = (unsigned int)sw.ops.size();
    sw.mi.insert(sw.mi.end(), part.mi.begin(), part.mi.end());
    sw.bl.insert(sw.bl.end(), part.bl.begin(), part.bl.end());
    sw.ops.insert(sw.ops.end(), part.ops.begin(), part.ops.end());
    for (size_t q = 1; q < part.pm_off.size(); ++q) sw.pm_off.push_back(pm_base + part.pm_off[q]);
    for (size_t q = 1; q < part.op_off.size(); ++q) sw.op_off.push_back(op_base + part.op_off[q]);
    sw.root_pos.insert(sw.root_pos.end(), part.root_pos.begin(), part.root_pos.end());
    chunk_off.push_back((unsigned int)sw.root_pos.size());
  }
  return sw;
}

// log-likelihood of every root placement at its stored ratio, in root-id order:
// what the loop at src/model.cpp:871-874 computes (move_root + compute_lh_root
// per root).  With the fused path the whole sweep is ONE engine call.
std::vector<double> model_t::sweep_root_lh() { return sweep_root_lh(0, _tree.roots().size()); }

// The same sweep restricted to the root ids [begin, end): the unit of work of one rank when
// the candidate roots are distributed over ranks the way exhaustive mode distributes them
// (src/model.cpp:1899-1907).  The CLVs must be valid for the current root (compute_lh); the
// first placement re-orients them along the path from there.
std::vector<double> model_t::sweep_root_lh(size_t begin, size_t end) {
  const auto &all_roots = _tree.roots();
  if (begin > end || end > all_roots.size()) throw std::invalid_argument("sweep_root_lh: bad root range");
  const std::vector<root_location_t> roots(all_roots.begin() + (std::ptrdiff_t)begin,
                                           all_roots.begin() + (std::ptrdiff_t)end);
  std::vector<double> lh(roots.size(), 0.0);
  _last_sweep_part_lh.assign(_partitions.size(), std::vector<double>(roots.size(), 0.0));
  if (roots.empty()) return lh;
  if (_sweep_mode == sweep_mode_t::sequential) {
    for (size_t r = 0; r < roots.size(); ++r) {
      move_root(roots[r]);
      lh[r] = compute_lh_root(roots[r]);
      for (size_t i = 0; i < _partitions.size(); ++i) _last_sweep_part_lh[i][r] = _last_part_lh[i];
    }
    return lh;
  }
  if (_sweep_mode == sweep_mode_t::directed) {
    // one pre-order pass over directed CLVs from the current root; same bits as the loop
    // above (tree.hpp), ~1 CLV operation + 1 root evaluation per placement, in chunks
    std::vector<unsigned int>       chunk_off;
    const rooted_tree_t::sweep_schedule_t sw = directed_sweep_schedule(begin, end, {}, chunk_off);
    const unsigned int              chunks = (unsigned int)chunk_off.size() - 1;
    std::vector<double> part(sw.root_pos.size());
    for (size_t i = 0; i < _partitions.size(); ++i) {
      int rc = rdk_sweep_root_placements_chunks(_partitions[i], (unsigned)sw.root_pos.size(),
                                                _param_indicies[i].data(), _param_indicies[i].data(),
                                                sw.pm_off.data(), sw.mi.data(), sw.bl.data(), sw.op_off.data(),
                                                sw.ops.data(), _tree.root_clv_index(), _tree.root_scaler_index(),
                                                RDK_SWEEP_KEEP_ROOT | RDK_SWEEP_DISCARD, chunks, chunk_off.data(), part.data());
      if (rc == RDK_FAILURE) throw std::runtime_error(engine_error());
      for (size_t q = 0; q < part.size(); ++q) {
        lh[sw.root_pos[q] - begin] += part[q];
        _last_sweep_part_lh[i][sw.root_pos[q] - begin] = part[q];
      }
    }
    if (_exchange) lh = sum_over_partitions(_last_sweep_part_lh, lh.size());
    for (double v : lh)
      if (std::isnan(v)) throw std::runtime_error("lh at root is not a number: " + std::to_string(v));
    return lh;
  }
  std::vector<unsigned int>    pm_off{0}, op_off{0}, mi;
  std::vector<double>          bl;
  std::vector<rdk_operation_t> ops;
  for (const auto &rl : roots) {
    auto mv = _tree.generate_root_update_operations(rl);
    mi.insert(mi.end(), std::get<1>(mv).begin(), std::get<1>(mv).end());
    bl.insert(bl.end(), std::get<2>(mv).begin(), std::get<2>(mv).end());
    ops.insert(ops.end(), std::get<0>(mv).begin(), std::get<0>(mv).end());
    auto dv = _tree.generate_derivative_operations(rl);
    mi.insert(mi.end(), std::get<1>(dv).begin(), std::get<1>(dv).end());
    bl.insert(bl.end(), std::get<2>(dv).begin(), std::get<2>(dv).end());
    ops.push_back(std::get<0>(dv));
    pm_off.push_back((unsigned)mi.size());
    op_off.push_back((unsigned)ops.size());
  }
  std::vector<double> part(roots.size());
  for (size_t i = 0; i < _partitions.size(); ++i) {
    int rc = rdk_sweep_root_placements(_partitions[i], (unsigned)roots.size(), _param_indicies[i].data(),
                                       _param_indicies[i].data(), pm_off.data(), mi.data(), bl.data(),
                                       op_off.data(), ops.data(), _tree.root_clv_index(),
                                       _tree.root_scaler_index(), part.data());
    if (rc == RDK_FAILURE) throw std::runtime_error(engine_error());
    for (size_t r = 0; r < roots.size(); ++r) {
      lh[r] += part[r];
      _last_sweep_part_lh[i][r] = part[r];
    }
  }
  if (_exchange) lh = sum_over_partitions(_last_sweep_part_lh, lh.size());
  for (double v : lh)
    if (std::isnan(v)) throw std::runtime_error("lh at root is not a number: " + std::to_string(v));
  return lh;
}

// src/model.cpp:865-889: the sweep's log-likelihoods rank the placements; the best
// max(ratio * N, min) come back, most likely first
std::vector<root_location_t> model_t::suggest_roots_lh(size_t min, double ratio) {
  const auto          lh = sweep_root_lh();
  const auto         &roots = _tree.roots();
  const size_t        keep = std::min(shortlist_size(roots.size(), ratio, min), roots.size());
  typedef std::pair<root_location_t, double> scored_t;
  std::vector<scored_t> scored;
  scored.reserve(roots.size());
  for (size_t r = 0; r < roots.size(); ++r) scored.emplace_back(roots[r], lh[r]);
  std::partial_sort(scored.begin(), scored.begin() + (std::ptrdiff_t)keep, scored.end(),
                    [](const scored_t &a, const scored_t &b) { return a.second > b.second; });
  std::vector<root_location_t> out;
  out.reserve(keep);
  for (size_t i = 0; i < keep; ++i) out.push_back(scored[i].first);
  return out;
}

std::vector<root_location_t> model_t::suggest_roots_midpoint(size_t min, double ratio) {
  auto ranked = _tree.rank_midpoints();
  ranked.resize(std::min(shortlist_size(ranked.size(), ratio, min), ranked.size()));
  return ranked;
}

std::vector<root_location_t> model_t::suggest_roots_modified_mad(size_t min, double ratio) {
  auto ranked = _tree.rank_modified_mad();
  ranked.resize(std::min(shortlist_size(ranked.size(), ratio, min), ranked.size()));
  return ranked;
}

static std::vector<size_t> ids_of(const std::vector<root_location_t> &placements) {
  std::vector<size_t> ids;
  ids.reserve(placements.size());
  for (const auto &rl : placements) ids.push_back(rl.id);
  return ids;
}

std::vector<size_t> model_t::shuffle_root_indicies() {
  std::vector<size_t> ids(_tree.root_count());
  std::iota(ids.begin(), ids.end(), 0);
  std::shuffle(ids.begin(), ids.end(), _random_engine);
  return ids;
}

std::vector<size_t> model_t::suggest_root_indicies_midpoint() { return ids_of(suggest_roots_midpoint(1, 1.0)); }

std::vector<size_t> model_t::suggest_root_indicies_modified_mad() {
  return ids_of(suggest_roots_modified_mad(1, 1.0));
}

// ---------------------------------------------------------------------------
// model parameters: L-BFGS-B in a box, one parameter block at a time
// ---------------------------------------------------------------------------
// src/model.cpp:1925-1984 with the four wrappers :1524-1735.  Per partition (the partitions are
// independent and run on their own threads): install the current values, then fit the 12 rates
// in [1e-4, 1e4], the 4 frequencies in [1e-4, 1 - 3e-4] (all free, renormalised on installation),
// and -- unless the user fixed it -- the Gamma shape in [0.2, 1e4] and, for free categories, the
// weights in [1e-4, 1].  Every objective evaluation is one full traversal of that partition: 13
// per gradient of the rates, which is what the lazily materialised evaluations of the engine are
// for (DESIGN 5.1b).
void model_t::optimize_params(std::vector<partition_parameters_t> &params, const root_location_t &rl,
                              double pgtol, double factor, bool optimize_gamma) {
  const traversal_t trav = full_traversal(rl);
  auto              box = [&](double lower, double upper) {
    rd::box_minimizer_options_t o;
    o.lower = lower;
    o.upper = upper;
    o.pgtol = pgtol;
    o.factr = factor;
    return o;
  };
  for_each_partition(_partitions.size(), true, [&](size_t p) {
    auto &mine = params[p];
    auto  fit = [&](model_params_t &block, const rd::box_minimizer_options_t &o, auto install) {
      rd::minimize_in_box(block, o, [&](const std::vector<double> &x) {
        install(x);
        return -compute_lh_partition(p, trav);
      });
    };
    const bool free_categories = _rate_category_types[p] == rate_category::FREE;
    set_subst_rates(p, mine.subst_rates);
    set_freqs_all_free(p, mine.freqs);
    set_gamma_rates(p, mine.gamma_alpha);
    if (free_categories) set_gamma_weights(p, mine.gamma_weights);

    fit(mine.subst_rates, box(1e-4, 1e4), [&](const model_params_t &x) { set_subst_rates(p, x); });
    fit(mine.freqs, box(1e-4, 1.0 - 1e-4 * 3), [&](const model_params_t &x) { set_freqs_all_free(p, x); });
    if (!optimize_gamma || _rate_user_init[p]) return;
    fit(mine.gamma_alpha, box(0.2, 10000.0), [&](const model_params_t &x) { set_gamma_rates(p, x); });
    if (free_categories)
      fit(mine.gamma_weights, box(1e-4, 1.0), [&](const model_params_t &x) { set_gamma_weights(p, x); });
  });
}

// ---------------------------------------------------------------------------
// search drivers
// ---------------------------------------------------------------------------
namespace {
struct placement_t {  // a root placement and its log-likelihood
  root_location_t where;
  double          lh = -std::numeric_limits<double>::infinity();
};
}  // namespace

// what rank 0 does once every rank is through (src/model.cpp:1119-1133, 1259-1269): the most
// likely record of the whole checkpoint, the first one on ties; all.size() when there is none
static size_t most_likely(const std::vector<checkpoint_t::record_t> &all) {
  size_t top = 0;
  for (size_t i = 1; i < all.size(); ++i)
    if (all[top].first.llh < all[i].first.llh) top = i;
  return top;
}

std::pair<root_location_t, double> model_t::placement_of(const rd_result_t &result) const {
  root_location_t where = _tree.root_location(result.root_id);
  where.brlen_ratio = result.alpha;
  return {where, result.llh};
}

// src/model.cpp:1008-1137.  Per assigned start: alternate "fit the parameters for this root" and
// "move the root to the best polished placement of a sweep" until the root stops moving (early
// stop), the likelihood stops changing, or it gets worse -- in which case the parameters of the
// previous round are put back.  One checkpoint record per start; the answer is the best record.
std::pair<root_location_t, double> model_t::search(size_t min_roots, double root_ratio, double atol,
                                                   double pgtol, double brtol, double factor,
                                                   checkpoint_t &checkpoint) {
  reset_to_defaults();
  for (size_t start : _assigned_idx) {
    root_location_t at = _tree.root_location(start);
    reset_to_defaults();
    auto        params = fresh_parameters();
    placement_t kept{at};

    for (size_t round = 0; round < _max_outer_iterations; ++round) {
      const auto before = params;
      optimize_params(params, at, pgtol, factor, true);
      const auto found = optimize_root_location(min_roots, root_ratio);
      if (found.second < kept.lh) {
        set_model_params(before);
        params = before;
        break;
      }
      const bool stayed = _early_stop && at.edge == found.first.edge &&
                          std::fabs(at.brlen_ratio - found.first.brlen_ratio) < brtol;
      const bool converged = std::fabs(found.second - kept.lh) < atol;
      kept = {found.first, found.second};
      if (stayed || converged) break;
      at = kept.where;
    }
    checkpoint.write({kept.where.id, kept.lh, kept.where.brlen_ratio}, parameters_of_all_partitions(params));
  }

  std::pair<root_location_t, double> best{root_location_t{}, -std::numeric_limits<double>::infinity()};
  const auto                         all = checkpoint.read_results();
  if (!all.empty()) {
    const auto &top = all[most_likely(all)];
    best = placement_of(top.first);
    set_model_params(parameters_held_here(top.second));
  }
  if (!_assigned_idx.empty()) move_root(best.first);
  return best;
}

// src/model.cpp:1139-1272.  Every assigned branch is optimised to convergence with the root held
// on it: fit the parameters (the Gamma shape only every 10th round, Appendix B-7), stop when a
// full evaluation no longer moves, else polish the position on the branch.  Then every record of
// the checkpoint is written onto the tree (LWR = softmax of the log-likelihoods, llh, ratio).
std::pair<root_location_t, double> model_t::exhaustive_search(double atol, double pgtol, double brtol,
                                                              double factor, checkpoint_t &checkpoint) {
  for (size_t branch : _assigned_idx) {
    root_location_t at = _tree.root_location(branch);
    reset_to_defaults();
    _tree.root_by(at);
    compute_lh(at);
    auto        params = fresh_parameters();
    placement_t kept{at};

    for (size_t round = 0; round < _max_outer_iterations; ++round) {
      optimize_params(params, at, pgtol, factor, round % 10 == 0);
      if (std::fabs(compute_lh(at) - kept.lh) < atol) break;
      const root_location_t polished = optimize_alpha(at, brtol);
      const double          lh = compute_lh_root(polished);
      const bool            stayed = _early_stop && std::fabs(at.brlen_ratio - polished.brlen_ratio) < brtol;
      const bool            small_gain = (lh - kept.lh) < atol;
      if (stayed || lh > kept.lh) kept = {polished, lh};
      if (stayed || small_gain) break;
      at = polished;
    }
    checkpoint.write({kept.where.id, kept.lh, kept.where.brlen_ratio}, parameters_of_all_partitions(params));
  }

  std::pair<root_location_t, double> best{root_location_t{}, -std::numeric_limits<double>::infinity()};
  const auto                         all = checkpoint.read_results();
  if (!all.empty()) {
    best = placement_of(all[most_likely(all)].first);
    std::vector<double> llh;
    llh.reserve(all.size());
    for (const auto &rec : all) llh.push_back(rec.first.llh);
    const auto weight = lwr(llh);
    for (size_t i = 0; i < all.size(); ++i) {
      const root_location_t rl = placement_of(all[i].first).first;
      _tree.annotate_branch(rl, "LWR", std::to_string(weight[i]));
      _tree.annotate_lh(rl, all[i].first.llh);
      _tree.annotate_ratio(rl, all[i].first.alpha);
    }
  }
  return best;
}

// ---------------------------------------------------------------------------
// root placement support (DESIGN.md section 10)
// ---------------------------------------------------------------------------
// what both support calls refuse before any work
void model_t::check_support_request(const std::string &who, size_t replicates,
                                    const std::vector<unsigned> &au_scales) const {
  if (_exchange)
    throw std::invalid_argument(who + ": a model whose partitions are dealt to several processes is not supported");
  if (replicates == 0 || replicates > (size_t(1) << 20))
    throw std::invalid_argument(who + ": replicates must be between 1 and 2^20");
  if (!au_scales.empty()) rd::check_au_scales(au_scales.data(), au_scales.size());
}

void model_t::check_support_records(const std::string &who, const std::vector<checkpoint_t::record_t> &records) const {
  if (records.empty()) throw std::invalid_argument(who + ": the checkpoint holds no records");
  if (records.size() > std::numeric_limits<unsigned>::max()) throw std::invalid_argument(who + ": too many records");
  for (size_t r = 0; r < records.size(); ++r) {
    const auto &rec = records[r];
    const std::string which = who + ": record " + std::to_string(r) + " (root id " +
                              std::to_string(rec.first.root_id) + ")";
    if (rec.first.root_id >= _tree.root_count()) throw std::invalid_argument(which + ": root id out of range");
    if (!(rec.first.alpha >= 0.0 && rec.first.alpha <= 1.0))
      throw std::invalid_argument(which + ": root position outside [0, 1]");
    if (rec.second.size() != _partitions.size())
      throw std::invalid_argument(which + ": " + std::to_string(rec.second.size()) + " parameter sets for " +
                                  std::to_string(_partitions.size()) + " partitions");
    for (size_t p = 0; p < _partitions.size(); ++p) {
      const auto    &pp = rec.second[p];
      const size_t   states = _partitions[p]->states, cats = _partitions[p]->rate_cats;
      const bool     free_rates = _rate_category_types[p] == rate_category::FREE;
      if (pp.subst_rates.size() != states * states - states || pp.freqs.size() != states ||
          pp.gamma_alpha.size() != (free_rates ? cats : 1) || (free_rates && pp.gamma_weights.size() != cats))
        throw std::invalid_argument(which + ": the parameters of partition " + std::to_string(p) +
                                    " do not match the model");
    }
  }
}

// installed as optimize_params installs them: a record holds the optimiser's variables, whose
// frequencies are normalised on the way in (set_model_params would take them as they are)
void model_t::install_record(const checkpoint_t::record_t &record) {
  for (size_t p = 0; p < _partitions.size(); ++p) {
    const auto &pp = record.second[p];
    set_subst_rates(p, pp.subst_rates);
    set_freqs_all_free(p, pp.freqs);
    set_gamma_rates(p, pp.gamma_alpha);
    if (_rate_category_types[p] == rate_category::FREE) set_gamma_weights(p, pp.gamma_weights);
  }
}

// what is put back after a support call: the installed parameters and the rooting (and the row
// matrix is freed unless keep_rows)
std::function<void()> model_t::support_restore_point(bool keep_rows) {
  struct installed_t {
    std::vector<double> subst, freqs, rates, weights, rate_rates;
  };
  std::vector<installed_t> installed(_partitions.size());
  for (size_t p = 0; p < _partitions.size(); ++p) {
    const rdk_partition_t *part = _partitions[p];
    const size_t           states = part->states;
    installed[p].subst.assign(part->subst_params[0], part->subst_params[0] + states * states - states);
    installed[p].freqs.assign(part->frequencies[0], part->frequencies[0] + states);
    installed[p].rates.assign(part->rates, part->rates + part->rate_cats);
    installed[p].weights.assign(part->rate_weights, part->rate_weights + part->rate_cats);
    installed[p].rate_rates = _rate_rates[p];
  }
  const bool            was_rooted = _tree.rooted();
  const root_location_t was_root = _tree.root_location();
  return [this, installed, was_rooted, was_root, keep_rows]() {
    if (!keep_rows) {
      for (size_t p = 0; p < _partitions.size(); ++p) rdk_partition_set_site_lnl_rows(_partitions[p], 0);
      _support_rows = 0;
    }
    for (size_t p = 0; p < _partitions.size(); ++p) {
      rdk_set_subst_params(_partitions[p], 0, installed[p].subst.data());
      rdk_set_frequencies(_partitions[p], 0, installed[p].freqs.data());
      rdk_set_category_rates(_partitions[p], installed[p].rates.data());
      rdk_set_category_weights(_partitions[p], installed[p].weights.data());
      _rate_rates[p] = installed[p].rate_rates;
    }
    if (was_rooted) {
      _tree.root_by(was_root);
      compute_lh(was_root);  // the CLVs of the previous rooting, for root-only evaluations
    } else {
      _tree.unroot();
    }
  };
}

void model_t::reserve_support_rows(const std::string &who, unsigned rows) {
  for (size_t p = 0; p < _partitions.size(); ++p)
    if (rdk_partition_set_site_lnl_rows(_partitions[p], rows) != RDK_SUCCESS)
      throw std::runtime_error(who + ": " + engine_error());
  _support_rows = rows;
}

// the statistics of DESIGN.md section 10, items 2-8, over rows 0..rows-1 of the partitions' site
// matrices (rdk_rell_support, or rdk_rell_support_ms in AU mode)
void model_t::resample_support(const std::string &who, placement_support_t &out, unsigned rows, size_t replicates,
                               uint64_t seed, unsigned replicate_tile, const std::vector<unsigned> &au_scales) {
  const bool            au = !au_scales.empty();
  std::vector<unsigned> global_index(_partitions.size());
  std::iota(global_index.begin(), global_index.end(), 0u);
  out.replicates = replicates;
  out.lnl_fixed.resize(rows);
  out.bp_count.resize(rows);
  out.kh_count.resize(rows);
  out.sh_count.resize(rows);
  out.o_lo.resize(rows);
  out.o_hi.resize(rows);
  rdk_rell_out_t rell;
  memset(&rell, 0, sizeof(rell));
  rell.replicate_tile = replicate_tile;
  rell.lnl_fixed = out.lnl_fixed.data();
  rell.bp_count = out.bp_count.data();
  rell.kh_count = out.kh_count.data();
  rell.sh_count = out.sh_count.data();
  rell.o_lo = out.o_lo.data();
  rell.o_hi = out.o_hi.data();
  if (au) {
    out.scales = au_scales;
    out.scale_count.resize(au_scales.size() * rows);
    out.elw_fixed.resize(rows);
    rdk_rell_ms_out_t ms;
    memset(&ms, 0, sizeof(ms));
    ms.scales = out.scales.data();
    ms.n_scales = (unsigned)out.scales.size();
    ms.scale_count = out.scale_count.data();
    ms.elw_fixed = out.elw_fixed.data();
    if (rdk_rell_support_ms(_partitions.data(), (unsigned)_partitions.size(), global_index.data(), rows, replicates,
                            seed, &rell, &ms) != RDK_SUCCESS)
      throw std::runtime_error(who + ": " + engine_error());
    out.au_counts_ms = ms.ms[0];
    out.au_accumulate_ms = ms.ms[1];
    out.au_statistics_ms = ms.ms[2];
  } else if (rdk_rell_support(_partitions.data(), (unsigned)_partitions.size(), global_index.data(), rows,
                              replicates, seed, &rell) != RDK_SUCCESS) {
    throw std::runtime_error(who + ": " + engine_error());
  }
  out.best = rell.best;
  out.exponent = rell.exponent;
  out.counts_ms = rell.ms[0];
  out.accumulate_ms = rell.ms[1];
  out.statistics_ms = rell.ms[2];
  out.resample_ms = rell.ms[3];
  out.device_bytes = rell.device_bytes;
}

// the per-record values the counts stand for, and the branch annotations: record r is the placement
// on where[r]'s branch
void model_t::annotate_support(placement_support_t &out, const std::vector<root_location_t> &where) {
  const bool   au = !out.scales.empty();
  const size_t rows = where.size();
  const double B = (double)out.replicates;
  for (size_t r = 0; r < rows; ++r) {
    out.bp.push_back(out.bp_count[r] / B);
    out.p_kh.push_back(out.kh_count[r] / B);
    out.p_sh.push_back(out.sh_count[r] / B);
    _tree.annotate_branch(where[r], "BP", std::to_string(out.bp[r]));
    _tree.annotate_branch(where[r], "pKH", std::to_string(out.p_kh[r]));
    _tree.annotate_branch(where[r], "pSH", std::to_string(out.p_sh[r]));
    if (au) {
      std::vector<unsigned> count(out.scales.size());
      for (size_t k = 0; k < count.size(); ++k) count[k] = out.scale_count[k * rows + r];
      const rd::au_fit_t fit = rd::au_fit(count.data(), out.scales.data(), count.size(), out.replicates);
      out.p_au.push_back(fit.p_au);
      out.au_d.push_back(fit.d);
      out.au_c.push_back(fit.c);
      out.au_rss.push_back(fit.rss);
      out.au_used.push_back(fit.used);
      out.elw.push_back(ldexp((double)out.elw_fixed[r], -40) / B);
      _tree.annotate_branch(where[r], "pAU", std::to_string(fit.p_au));
      _tree.annotate_branch(where[r], "ELW", std::to_string(out.elw[r]));
    }
  }
}

model_t::placement_support_t model_t::placement_support(checkpoint_t &checkpoint, size_t replicates, uint64_t seed,
                                                        unsigned replicate_tile, bool keep_rows,
                                                        const std::vector<unsigned> &au_scales) {
  const std::string who = "placement_support";
  check_support_request(who, replicates, au_scales);
  const auto records = checkpoint.read_results();
  check_support_records(who, records);

  auto           restore = support_restore_point(keep_rows);
  const unsigned rows = (unsigned)records.size();
  reserve_support_rows(who, rows);

  placement_support_t out;
  try {
    const auto t0 = std::chrono::steady_clock::now();
    for (unsigned r = 0; r < rows; ++r) {
      install_record(records[r]);
      const root_location_t rl = placement_of(records[r].first).first;
      _tree.root_by(rl);
      const traversal_t trav = full_traversal(rl);
      for (size_t p = 0; p < _partitions.size(); ++p) {
        update_pmatrix_partition(p, trav.pmatrix_indices, trav.branch_lengths);
        rdk_update_clvs(_partitions[p], trav.ops.data(), (unsigned)trav.ops.size());
        const double lh = rdk_compute_root_loglikelihood_row(_partitions[p], _tree.root_clv_index(),
                                                             _tree.root_scaler_index(), r);
        if (std::isnan(lh))
          throw std::runtime_error("placement_support: record " + std::to_string(r) + ": " + engine_error());
      }
    }
    out.capture_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    resample_support(who, out, rows, replicates, seed, replicate_tile, au_scales);
  } catch (...) {
    restore();
    throw;
  }
  restore();

  std::vector<root_location_t> where;
  for (unsigned r = 0; r < rows; ++r) {
    out.root_id.push_back(records[r].first.root_id);
    out.alpha.push_back(records[r].first.alpha);
    out.llh.push_back(records[r].first.llh);
    where.push_back(placement_of(records[r].first).first);
  }
  annotate_support(out, where);
  return out;
}

model_t::placement_support_t model_t::branch_support(checkpoint_t &checkpoint, size_t replicates, uint64_t seed,
                                                     double atol, unsigned replicate_tile, bool keep_rows,
                                                     const std::vector<unsigned> &au_scales) {
  const std::string who = "branch_support";
  check_support_request(who, replicates, au_scales);
  if (!(atol >= 0.0 && atol <= std::numeric_limits<double>::max()))
    throw std::invalid_argument(who + ": atol must be finite and non-negative");
  const auto records = checkpoint.read_results();
  check_support_records(who, records);
  size_t best = 0;  // highest llh, lowest log index on ties
  for (size_t r = 1; r < records.size(); ++r)
    if (records[r].first.llh > records[best].first.llh) best = r;

  auto           restore = support_restore_point(keep_rows);
  const size_t   n_roots = _tree.root_count();
  const unsigned rows = (unsigned)n_roots;
  reserve_support_rows(who, rows);

  placement_support_t out;
  std::vector<double> alpha(n_roots, 0.5), llh(n_roots, 0.0);
  try {
    install_record(records[best]);
    const root_location_t at = placement_of(records[best].first).first;
    for (size_t q = 0; !_tree.can_root_by(at) && q < n_roots; ++q)  // an unrooted tree: root it elsewhere first
      if (_tree.can_root_by(_tree.root_location(q))) _tree.root_by(_tree.root_location(q));
    compute_lh(at);
    // a_q: the position optimize_root_location would polish root q to, from ratio 0.5
    const auto t0 = std::chrono::steady_clock::now();
    if (atol > 0.0) {
      for (size_t q = 0; q < n_roots; ++q) {
        const root_location_t rl = _tree.root_location(q);
        move_root(rl);
        alpha[q] = optimize_alpha(rl, atol).brlen_ratio;
      }
    }
    const auto t1 = std::chrono::steady_clock::now();
    out.positions_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    compute_lh(at);  // the sweep starts from valid CLVs of one rooting

    // one directed sweep over every placement (q, a_q) that also stores the rows, in sweep order;
    // then the rows are put in root-id order, the order the statistics index records by
    const auto t2 = std::chrono::steady_clock::now();
    std::vector<unsigned int>       chunk_off;
    const rooted_tree_t::sweep_schedule_t sw = directed_sweep_schedule(0, n_roots, alpha, chunk_off);
    std::vector<unsigned int> order(n_roots);
    for (size_t q = 0; q < sw.root_pos.size(); ++q) order[sw.root_pos[q]] = (unsigned)q;
    std::vector<double> part(sw.root_pos.size());
    for (size_t i = 0; i < _partitions.size(); ++i) {
      if (rdk_sweep_root_placements_chunks(_partitions[i], (unsigned)sw.root_pos.size(), _param_indicies[i].data(),
                                           _param_indicies[i].data(), sw.pm_off.data(), sw.mi.data(), sw.bl.data(),
                                           sw.op_off.data(), sw.ops.data(), _tree.root_clv_index(),
                                           _tree.root_scaler_index(),
                                           RDK_SWEEP_KEEP_ROOT | RDK_SWEEP_DISCARD | RDK_SWEEP_ROWS,
                                           (unsigned)chunk_off.size() - 1, chunk_off.data(),
                                           part.data()) == RDK_FAILURE ||
          rdk_partition_permute_site_lnl_rows(_partitions[i], rows, order.data()) == RDK_FAILURE)
        throw std::runtime_error(who + ": " + engine_error());
      for (size_t q = 0; q < part.size(); ++q) llh[sw.root_pos[q]] += part[q];
    }
    out.capture_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t2).count();
    for (double v : llh)
      if (std::isnan(v)) throw std::runtime_error(who + ": lh at root is not a number");
    resample_support(who, out, rows, replicates, seed, replicate_tile, au_scales);
  } catch (...) {
    restore();
    throw;
  }
  restore();

  std::vector<root_location_t> where;
  for (size_t q = 0; q < n_roots; ++q) {
    out.root_id.push_back(q);
    where.push_back(_tree.root_location(q));
  }
  out.alpha = alpha;
  out.llh = llh;
  annotate_support(out, where);
  for (size_t q = 0; q < n_roots; ++q) {
    _tree.annotate_lh(where[q], llh[q]);
    _tree.annotate_ratio(where[q], alpha[q]);
  }
  return out;
}

std::vector<double> model_t::site_lnl_rows(size_t partition) {
  if (partition >= _partitions.size()) throw std::invalid_argument("site_lnl_rows: partition out of range");
  std::vector<double> out((size_t)_support_rows * _partitions[partition]->sites);
  if (_support_rows &&
      rdk_partition_get_site_lnl_rows(_partitions[partition], 0, _support_rows, out.data()) != RDK_SUCCESS)
    throw std::runtime_error("site_lnl_rows: " + engine_error());
  return out;
}

// LWR_i = exp(llh_i - max) / sum_j exp(llh_j - max) (src/model.cpp:1238-1253)
std::vector<double> model_t::lwr(const std::vector<double> &llh) {
  double top = -std::numeric_limits<double>::infinity();
  for (double v : llh) top = std::max(v, top);
  double mass = 0;
  for (double v : llh) mass += exp(v - top);
  std::vector<double> out;
  out.reserve(llh.size());
  for (double v : llh) out.push_back(exp(v - top) / mass);
  return out;
}

void model_t::initialize() { compute_lh(_tree.root_location(0)); }
void model_t::finalize() { _tree.unroot(); }

rooted_tree_t model_t::rooted_tree(const root_location_t &root) const {
  rooted_tree_t t(_tree);
  t.root_by((unsigned)root.id);
  return t;
}
rooted_tree_t model_t::virtual_rooted_tree(const root_location_t &root) const {
  rooted_tree_t t = rooted_tree(root);
  t.unroot();
  return t;
}
rooted_tree_t model_t::unrooted_tree() const {
  rooted_tree_t t(_tree);
  t.unroot();
  return t;
}

// src/model.cpp:1297-1321: tips, invariant sites, frequencies, random start rates (Appendix B-10:
// one draw of the model's generator per partition, in partition order).  On partition shards the
// draws of the partitions held elsewhere are skipped, so that every process leaves with the
// generator a single process would have -- the random start order of a search depends on it.
template <typename PerPartition>
void model_t::for_each_partition_in_global_order(PerPartition &&body) {
  if (!_exchange) {
    for (size_t p = 0; p < _partitions.size(); ++p) body(p);
    return;
  }
  size_t local = 0;
  for (size_t g = 0; g < _global_partitions; ++g) {
    if (local < _global_index.size() && _global_index[local] == g)
      body(local++);
    else
      _random_engine.discard(1);
  }
}

void model_t::initialize_partitions(const std::vector<msa_t> &msa) {
  for_each_partition_in_global_order([&](size_t p) {
    set_tip_states(p, msa[p]);
    update_invariant_sites(p);
    set_empirical_freqs(p);
    set_subst_rates_random(p, msa[p]);
  });
}

void model_t::initialize_partitions_uniform_freqs(const std::vector<msa_t> &msa) {
  for_each_partition_in_global_order([&](size_t p) {
    set_tip_states(p, msa[p]);
    update_invariant_sites(p);
    const unsigned int states = _partitions[p]->states;
    set_freqs(p, model_params_t(states, 1.0 / (double)states));
    set_subst_rates_random(p, msa[p]);
    set_gamma_rates(p);
  });
}

// "{{r0,...,r11},{...}}": the rates of every partition, six decimals
std::string model_t::subst_string() const {
  std::ostringstream text;
  text << "{";
  for (size_t p = 0; p < _partitions.size(); ++p) {
    const auto  *part = _partitions[p];
    const size_t n = part->states * part->states - part->states;
    text << (p ? ",{" : "{");
    for (size_t i = 0; i < n; ++i) text << (i ? "," : "") << std::to_string(part->subst_params[0][i]);
    text << "}";
  }
  text << "}";
  return text.str();
}

// ---------------------------------------------------------------------------
// work assignment (src/model.cpp:1761-1911)
// ---------------------------------------------------------------------------
void model_t::assign_indicies(const std::vector<size_t> &idx) { _assigned_idx = idx; }

void model_t::assign_indicies(size_t begin, size_t end) {
  _assigned_idx.resize(end - begin);
  std::iota(_assigned_idx.begin(), _assigned_idx.end(), begin);
}

void model_t::assign_indicies() { assign_indicies(0, _tree.root_count()); }

void model_t::assign_indicies(size_t beg, size_t end, std::vector<size_t> idx) {
  _assigned_idx.assign(idx.begin() + (std::ptrdiff_t)beg, idx.begin() + (std::ptrdiff_t)end);
}

// rank r of n takes the r-th of n contiguous shares of `work`, the first |work| mod n shares one
// item longer (src/model.cpp:1843-1849,1899-1907; sharding.plan_root_shards is the same rule)
void model_t::assign_rank_share(const std::vector<size_t> &work, size_t rank, size_t num_tasks) {
  const size_t share = work.size() / num_tasks, longer = work.size() % num_tasks;
  const size_t beg = share * rank + std::min(longer, rank);
  const size_t end = share * (rank + 1) + std::min(longer, rank + 1);
  assign_indicies(beg, end, work);
}

void model_t::assign_indicies_by_rank_search(size_t min_roots, double root_ratio, size_t rank,
                                             size_t num_tasks, checkpoint_t &checkpoint) {
  assign_indicies_by_rank_search(min_roots, root_ratio, rank, num_tasks, initial_root_strategy_t::random,
                                 checkpoint);
}

// the starts of a search: the first max(ratio * N, min) roots of the chosen ranking, minus what
// the checkpoint already holds, dealt to the ranks
void model_t::assign_indicies_by_rank_search(size_t min_roots, double root_ratio, size_t rank,
                                             size_t num_tasks, initial_root_strategy_t init_root,
                                             checkpoint_t &checkpoint) {
  auto                done = checkpoint.completed_indicies();
  std::vector<size_t> order;
  switch (init_root) {
  case initial_root_strategy_t::random: order = shuffle_root_indicies(); break;
  case initial_root_strategy_t::midpoint: order = suggest_root_indicies_midpoint(); break;
  case initial_root_strategy_t::modified_mad: order = suggest_root_indicies_modified_mad(); break;
  default: throw std::runtime_error{"The initial root strategy was not recognized"};
  }
  const size_t wanted = std::min(std::max(static_cast<size_t>(_tree.root_count() * root_ratio), min_roots),
                                 _tree.root_count());
  if (wanted < done.size())
    throw std::runtime_error{"There are too many results in the checkpoint for this search. Is the "
                             "checkpoint corrupted?"};
  std::sort(done.begin(), done.end());
  std::vector<size_t> open;
  for (size_t id : order)
    if (!std::binary_search(done.begin(), done.end(), id)) open.push_back(id);
  // the reference cuts the shares from `wanted - done` items of the open list, not from all of it
  open.resize(std::min(open.size(), wanted - done.size()));
  assign_rank_share(open, rank, num_tasks);
}

// exhaustive mode: every root id the checkpoint does not hold yet, in id order, dealt to the ranks
void model_t::assign_indicies_by_rank_exhaustive(size_t rank, size_t num_tasks, checkpoint_t &checkpoint) {
  const auto done = checkpoint.current_progress();
  if (_tree.root_count() < done.size())
    throw std::runtime_error{"There are too many results in the checkpoint for this tree, are you "
                             "sure the checkpoint matches?"};
  std::vector<char> seen(_tree.root_count(), 0);
  for (const auto &r : done)
    if (r.root_id < seen.size()) seen[r.root_id] = 1;
  std::vector<size_t> open;
  for (size_t id = 0; id < seen.size(); ++id)
    if (!seen[id]) open.push_back(id);
  assign_rank_share(open, rank, num_tasks);
}
