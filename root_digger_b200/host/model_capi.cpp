// model_capi.cpp -- C wrappers around model_t for ctypes (tests, bench, the
// Python multi-GPU launcher).  Return 1 on success, 0 on failure with the
// message available from rdh_last_error() (exceptions never cross the boundary).
#include "model.hpp"
#include "support_stats.hpp"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>

extern "C" const char *rdh_last_error(void);
void                   rdh_set_error(const std::string &s);

namespace {
struct holder_t {
  std::vector<msa_t>       msa;
  std::unique_ptr<model_t> model;
  checkpoint_t             checkpoint;
};
holder_t &H(void *h) { return *reinterpret_cast<holder_t *>(h); }
}  // namespace

#define RDH_TRY(body)                                                                              \
  try {                                                                                            \
    body                                                                                           \
  } catch (const std::exception &e) {                                                              \
    rdh_set_error(e.what());                                                                       \
    return 0;                                                                                      \
  }

// partitions: `n_parts` column ranges [part_begin[i], part_end[i]) of the given
// alignment (n_parts == 0: one partition with every column).  Sharding: this
// process holds global site patterns [site_offset, site_offset + local) of
// `global_sites` (0 = unsharded); comm_id = 128-byte NCCL id or NULL.
extern "C" void *rdh_model_create(void *tree, int n_taxa, const char **labels, const char **seqs,
                                  int compress, unsigned rate_cats, int invariant_sites,
                                  unsigned long long seed, int early_stop, int n_parts,
                                  const unsigned long long *part_begin,
                                  const unsigned long long *part_end,
                                  unsigned long long site_offset, unsigned long long global_sites,
                                  int nranks, int rank, const void *comm_id) {
  try {
    auto                     h = std::make_unique<holder_t>();
    std::vector<std::string> l(labels, labels + n_taxa), s(seqs, seqs + n_taxa);
    if (n_parts <= 0) {
      h->msa.emplace_back(l, s, rdk_map_nt, 4u, compress != 0);
    } else {
      msa_t whole(l, s, rdk_map_nt, 4u, false);
      for (int i = 0; i < n_parts; ++i) {
        h->msa.emplace_back(whole, (size_t)part_begin[i], (size_t)part_end[i]);
        if (compress) h->msa.back().compress();
      }
    }
    shard_spec_t shard;
    shard.site_offset = site_offset;
    shard.global_sites = global_sites;
    shard.nranks = nranks;
    shard.rank = rank;
    shard.comm_id = comm_id;
    rooted_tree_t t(*reinterpret_cast<rooted_tree_t *>(tree));
    h->model = std::make_unique<model_t>(std::move(t), h->msa,
                                         std::vector<ratehet_opts_t>(h->msa.size(), ratehet_opts_t{rate_cats}),
                                         invariant_sites != 0, (uint64_t)seed, early_stop != 0, shard);
    return h.release();
  } catch (const std::exception &e) {
    rdh_set_error(e.what());
    return nullptr;
  }
}

// The ingest path of the reference's main (src/main.cpp:513-560): alignment file
// (PHYLIP or FASTA), optional RAxML-NG partition file; with a partition file the
// alignment is loaded uncompressed, split, every partition compressed on its own,
// and the rate categories come from the partition file's model strings (0 -> 1).
extern "C" void *rdh_model_create_from_files(void *tree, const char *msa_path, const char *partition_path,
                                             unsigned rate_cats, int invariant_sites,
                                             unsigned long long seed, int early_stop) {
  try {
    auto                        h = std::make_unique<holder_t>();
    std::vector<ratehet_opts_t> cats;
    if (!partition_path || !*partition_path) {
      h->msa.emplace_back(std::string(msa_path), rdk_map_nt, 4u, true);
      cats.emplace_back(ratehet_opts_t{rate_cats});
    } else {
      msa_t whole(std::string(msa_path), rdk_map_nt, 4u, false);
      auto  infos = parse_partition_file(partition_path);
      if (infos.empty()) throw std::runtime_error("the partition file names no partition");
      h->msa = whole.partition(infos);
      for (auto &p : infos) {
        ratehet_opts_t r = p.model.ratehet_opts;
        if (r.rate_cats == 0) r.rate_cats = 1;
        cats.push_back(r);
      }
    }
    for (auto &m : h->msa) m.valid_data();
    rooted_tree_t t(*reinterpret_cast<rooted_tree_t *>(tree));
    h->model = std::make_unique<model_t>(std::move(t), h->msa, cats, invariant_sites != 0, (uint64_t)seed,
                                         early_stop != 0, shard_spec_t{});
    return h.release();
  } catch (const std::exception &e) {
    rdh_set_error(e.what());
    return nullptr;
  }
}

extern "C" unsigned rdh_model_partition_count(void *h) { return (unsigned)H(h).msa.size(); }

namespace {
const char *ptype(param_type t) {
  switch (t) {
    case param_type::emperical: return "emperical";
    case param_type::estimate: return "estimate";
    case param_type::equal: return "equal";
    default: return "user";
  }
}
}  // namespace

// parse partition-file text; one line per partition:
//   model_name|partition_name|b-e,b-e|subst|freq|invar_present|invar|invar_prop|ratehet|cat_type|rate_cats|alpha_init|alpha|asc
// malloc'd (free with rdh_free); NULL + rdh_last_error() when the text does not parse
extern "C" char *rdh_partition_describe(const char *text) {
  try {
    std::string out;
    for (auto &p : parse_partition_text(text)) {
      char buf[256];
      out += p.model_name + "|" + p.partition_name + "|";
      for (size_t i = 0; i < p.parts.size(); ++i)
        out += (i ? "," : "") + std::to_string(p.parts[i].first) + "-" + std::to_string(p.parts[i].second);
      const auto &m = p.model;
      const char *cat = m.ratehet_opts.rate_category_type == rate_category::MEDIAN ? "median"
                        : m.ratehet_opts.rate_category_type == rate_category::FREE ? "free"
                                                                                    : "mean";
      const char *asc = m.asc_opts.type == asc_bias_type::lewis  ? "lewis"
                        : m.asc_opts.type == asc_bias_type::fels ? "fels"
                        : m.asc_opts.type == asc_bias_type::stam ? "stam"
                                                                  : "none";
      snprintf(buf, sizeof(buf), "|%s|%s|%d|%s|%.17g|%s|%s|%zu|%d|%.17g|%s\n", m.subst_str.c_str(),
               ptype(m.freq_opts.type), m.invar_opts.present ? 1 : 0, ptype(m.invar_opts.type),
               m.invar_opts.user_prop, ptype(m.ratehet_opts.type), cat, m.ratehet_opts.rate_cats,
               m.ratehet_opts.alpha_init ? 1 : 0, m.ratehet_opts.alpha, asc);
      out += buf;
    }
    char *r = (char *)malloc(out.size() + 1);
    memcpy(r, out.c_str(), out.size() + 1);
    return r;
  } catch (const std::exception &e) {
    rdh_set_error(e.what());
    return nullptr;
  }
}

// pattern counts of the partitions of an alignment file (test/src/msa.cpp:236-283)
extern "C" int rdh_msa_partition_lengths(const char *msa_path, const char *partition_text, int compress_first,
                                         unsigned *out, unsigned cap) {
  RDH_TRY({
    msa_t whole(std::string(msa_path), rdk_map_nt, 4u, compress_first != 0);
    auto  parts = whole.partition(parse_partition_text(partition_text));
    if (parts.size() > cap) throw std::runtime_error("output buffer too small");
    for (size_t i = 0; i < parts.size(); ++i) out[i] = parts[i].length();
    return (int)parts.size() + 1;
  })
}

extern "C" void rdh_model_destroy(void *h) { delete reinterpret_cast<holder_t *>(h); }

extern "C" unsigned rdh_model_sites(void *h, unsigned part) { return H(h).msa[part].length(); }
extern "C" unsigned rdh_model_root_count(void *h) { return (unsigned)H(h).model->tree().root_count(); }
extern "C" unsigned rdh_model_sweep_chunks(void *h) { return H(h).model->sweep_chunks(); }
extern "C" void rdh_model_set_max_outer_iterations(void *h, unsigned n) { H(h).model->set_max_outer_iterations(n); }

extern "C" int rdh_model_initialize_partitions(void *h, int uniform_freqs) {
  RDH_TRY({
    if (uniform_freqs)
      H(h).model->initialize_partitions_uniform_freqs(H(h).msa);
    else
      H(h).model->initialize_partitions(H(h).msa);
    return 1;
  })
}

extern "C" int rdh_model_set_fused(void *h, int on) {
  H(h).model->set_fused(on != 0);
  return 1;
}

// root-only evaluations of compute_dlh / optimize_alpha as fused batches (default) or one by one
extern "C" int rdh_model_set_batched_probes(void *h, int on) {
  H(h).model->set_batched_probes(on != 0);
  return 1;
}
extern "C" int rdh_model_batched_probes(void *h) { return H(h).model->batched_probes() ? 1 : 0; }
// out[0..3) = fused batches, root-only evaluations inside them, root-only evaluations issued singly
extern "C" void rdh_model_probe_counters(void *h, unsigned long long *out) {
  const auto &c = H(h).model->probe_counters();
  out[0] = c.fused_batches;
  out[1] = c.fused_evaluations;
  out[2] = c.single_evaluations;
}

// partitions dealt to several processes (model_t::set_partition_exchange): this process holds the
// partitions global_index[0..n_local) of global_partitions; `exchange` completes every sum over
// partitions (NULL detaches)
extern "C" int rdh_model_set_partition_exchange(void *h, const unsigned *global_index, unsigned n_local,
                                                unsigned global_partitions,
                                                model_t::partition_exchange_fn exchange, void *user) {
  RDH_TRY({
    std::vector<size_t> idx(global_index, global_index + n_local);
    H(h).model->set_partition_exchange(idx, global_partitions, exchange, user);
    return 1;
  })
}
extern "C" unsigned long long rdh_model_rng_state(void *h) { return H(h).model->rng_state(); }
extern "C" void rdh_model_set_rng_state(void *h, unsigned long long state) { H(h).model->set_rng_state(state); }
extern "C" void rdh_model_discard_rng(void *h, unsigned long long draws) { H(h).model->discard_rng(draws); }
// first local partition whose empirical frequencies have a zero entry: -1 none, -2 error
extern "C" int rdh_model_first_partition_without_empirical_freqs(void *h) {
  try {
    return H(h).model->first_partition_without_empirical_freqs(H(h).msa);
  } catch (const std::exception &e) {
    rdh_set_error(e.what());
    return -2;
  }
}

// 0 = sequential (the reference's loop), 1 = path (same operations, one engine call),
// 2 = directed (one pre-order pass over directed CLVs); identical values
extern "C" int rdh_model_set_sweep_mode(void *h, int mode) {
  RDH_TRY({
    if (mode < 0 || mode > 2) throw std::invalid_argument("sweep mode must be 0, 1 or 2");
    H(h).model->set_sweep_mode(static_cast<model_t::sweep_mode_t>(mode));
    return 1;
  })
}

extern "C" int rdh_model_set_params(void *h, unsigned part, const double *rates12, const double *freqs4,
                                    const double *alpha) {
  RDH_TRY({
    if (rates12) H(h).model->set_subst_rates(part, model_params_t(rates12, rates12 + 12));
    if (freqs4) H(h).model->set_freqs(part, model_params_t(freqs4, freqs4 + 4));
    if (alpha) H(h).model->set_gamma_rates(part, model_params_t(alpha, alpha + 1));
    return 1;
  })
}

static root_location_t RL(void *h, unsigned id, double ratio) {
  auto rl = H(h).model->tree().root_location((size_t)id);
  rl.brlen_ratio = ratio;
  return rl;
}

extern "C" int rdh_model_compute_lh(void *h, unsigned id, double ratio, double *out) {
  RDH_TRY({
    *out = H(h).model->compute_lh(RL(h, id, ratio));
    return 1;
  })
}
extern "C" int rdh_model_compute_lh_root(void *h, unsigned id, double ratio, double *out) {
  RDH_TRY({
    *out = H(h).model->compute_lh_root(RL(h, id, ratio));
    return 1;
  })
}
extern "C" int rdh_model_compute_dlh(void *h, unsigned id, double ratio, double *lh, double *dlh) {
  RDH_TRY({
    auto d = H(h).model->compute_dlh(RL(h, id, ratio));
    *lh = d.lh;
    *dlh = d.dlh;
    return 1;
  })
}
extern "C" int rdh_model_move_root(void *h, unsigned id, double ratio) {
  RDH_TRY({
    H(h).model->move_root(RL(h, id, ratio));
    return 1;
  })
}
extern "C" int rdh_model_optimize_alpha(void *h, unsigned id, double ratio, double atol, double *out) {
  RDH_TRY({
    *out = H(h).model->optimize_alpha(RL(h, id, ratio), atol).brlen_ratio;
    return 1;
  })
}
extern "C" int rdh_model_optimize_root_location(void *h, unsigned min_roots, double root_ratio,
                                                unsigned *id, double *alpha, double *lh) {
  RDH_TRY({
    auto r = H(h).model->optimize_root_location(min_roots, root_ratio);
    *id = (unsigned)r.first.id;
    *alpha = r.first.brlen_ratio;
    *lh = r.second;
    return 1;
  })
}
extern "C" int rdh_model_sweep_root_lh(void *h, double *out) {
  RDH_TRY({
    auto v = H(h).model->sweep_root_lh();
    for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
    return 1;
  })
}
extern "C" int rdh_model_sweep_root_lh_range(void *h, unsigned begin, unsigned end, double *out) {
  RDH_TRY({
    auto v = H(h).model->sweep_root_lh(begin, end);
    for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
    return 1;
  })
}
// per-partition terms of the last compute_lh / compute_lh_root (out: partition_count doubles) and of
// the last sweep (part: the partition; out: one double per placement of the swept range)
extern "C" int rdh_model_last_partition_lh(void *h, double *out, unsigned cap) {
  RDH_TRY({
    const auto &v = H(h).model->last_partition_lh();
    if (v.size() > cap) throw std::runtime_error("output buffer too small");
    for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
    return 1;
  })
}
extern "C" int rdh_model_last_sweep_partition_lh(void *h, unsigned part, double *out, unsigned cap) {
  RDH_TRY({
    const auto &m = H(h).model->last_sweep_partition_lh();
    if (part >= m.size()) throw std::runtime_error("no such partition in the last sweep");
    if (m[part].size() > cap) throw std::runtime_error("output buffer too small");
    for (size_t i = 0; i < m[part].size(); ++i) out[i] = m[part][i];
    return 1;
  })
}
extern "C" int rdh_model_compute_all_root_lh(void *h, double *out) {
  RDH_TRY({
    auto v = H(h).model->compute_all_root_lh();
    for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
    return 1;
  })
}

// Back the model's result log by the reference's on-disk checkpoint "<prefix>.ckp"
// (NULL: back to the in-memory log).  A file that already holds results makes the next
// search / exhaustive_search RESUME: root ids found in it are skipped
// (assign_indicies_by_rank_*, reference src/model.cpp:1899-1960).
extern "C" int rdh_model_set_checkpoint(void *h, const char *prefix) {
  RDH_TRY({
    H(h).checkpoint = prefix ? checkpoint_t(std::string(prefix)) : checkpoint_t();
    if (prefix && !H(h).checkpoint.existing_checkpoint()) {
      cli_options_t o;
      o.prefix = prefix;
      H(h).checkpoint.save_options(o);
    }
    return 1;
  })
}

// Work assignment against the model's result log (reference src/model.cpp:1899-1960): the root
// ids this rank still has to do.  mode 0: search (min_roots / root_ratio / init_strategy as in
// rdh_model_search), mode 1: exhaustive.  The ids are copied to out (capacity cap).
extern "C" int rdh_model_assign_indicies(void *h, int mode, unsigned min_roots, double root_ratio, unsigned rank,
                                         unsigned num_tasks, int init_strategy, unsigned *out, unsigned cap,
                                         unsigned *n_out) {
  RDH_TRY({
    auto &m = *H(h).model;
    if (mode == 0) {
      auto strat = init_strategy == 0   ? initial_root_strategy_t::random
                   : init_strategy == 1 ? initial_root_strategy_t::midpoint
                                        : initial_root_strategy_t::modified_mad;
      m.assign_indicies_by_rank_search(min_roots, root_ratio, rank, num_tasks, strat, H(h).checkpoint);
    } else {
      m.assign_indicies_by_rank_exhaustive(rank, num_tasks, H(h).checkpoint);
    }
    auto idx = m.assigned_indicies();
    if (idx.size() > cap) throw std::runtime_error("output buffer too small");
    for (size_t i = 0; i < idx.size(); ++i) out[i] = (unsigned)idx[i];
    *n_out = (unsigned)idx.size();
    return 1;
  })
}

// init_strategy: 0 random, 1 midpoint, 2 modified MAD
extern "C" int rdh_model_search(void *h, unsigned min_roots, double root_ratio, double atol, double pgtol,
                                double brtol, double factor, int init_strategy, unsigned rank,
                                unsigned num_tasks, unsigned *id, double *alpha, double *lh) {
  RDH_TRY({
    auto &m = *H(h).model;
    H(h).checkpoint.clear();
    auto strat = init_strategy == 0   ? initial_root_strategy_t::random
                 : init_strategy == 1 ? initial_root_strategy_t::midpoint
                                      : initial_root_strategy_t::modified_mad;
    m.assign_indicies_by_rank_search(min_roots, root_ratio, rank, num_tasks, strat, H(h).checkpoint);
    auto r = m.search(min_roots, root_ratio, atol, pgtol, brtol, factor, H(h).checkpoint);
    *id = (unsigned)r.first.id;
    *alpha = r.first.brlen_ratio;
    *lh = r.second;
    return 1;
  })
}

// exhaustive mode over this rank's slice of the root ids; per-root results are
// written to ids/llh/alpha (capacity `cap`), n_out receives their number
extern "C" int rdh_model_exhaustive_search(void *h, double atol, double pgtol, double brtol, double factor,
                                           unsigned rank, unsigned num_tasks, unsigned *ids, double *llh,
                                           double *alpha, unsigned cap, unsigned *n_out) {
  RDH_TRY({
    auto &m = *H(h).model;
    H(h).checkpoint.clear();
    m.assign_indicies_by_rank_exhaustive(rank, num_tasks, H(h).checkpoint);
    m.exhaustive_search(atol, pgtol, brtol, factor, H(h).checkpoint);
    auto res = H(h).checkpoint.current_progress();
    if (res.size() > cap) throw std::runtime_error("output buffers too small");
    for (size_t i = 0; i < res.size(); ++i) {
      ids[i] = (unsigned)res[i].root_id;
      llh[i] = res[i].llh;
      alpha[i] = res[i].alpha;
    }
    *n_out = (unsigned)res.size();
    return 1;
  })
}

// the per-record outputs every support entry fills (capacity cap), and info[0..5]
static void copy_support(const model_t::placement_support_t &res, unsigned cap, unsigned long long *root_id,
                         double *alpha, double *llh, double *lnl_fixed, unsigned long long *o_lo, long long *o_hi,
                         unsigned *bp_count, unsigned *kh_count, unsigned *sh_count, int *exponent, unsigned *best,
                         double *info, unsigned *n_out) {
  const size_t n = res.root_id.size();
  if (n > cap) throw std::runtime_error("output buffers too small");
  for (size_t i = 0; i < n; ++i) {
    root_id[i] = res.root_id[i];
    alpha[i] = res.alpha[i];
    llh[i] = res.llh[i];
    lnl_fixed[i] = res.lnl_fixed[i];
    if (o_lo) o_lo[i] = res.o_lo[i];
    if (o_hi) o_hi[i] = res.o_hi[i];
    bp_count[i] = res.bp_count[i];
    kh_count[i] = res.kh_count[i];
    sh_count[i] = res.sh_count[i];
  }
  *exponent = res.exponent;
  *best = (unsigned)res.best;
  info[0] = res.capture_ms;
  info[1] = res.counts_ms;
  info[2] = res.accumulate_ms;
  info[3] = res.statistics_ms;
  info[4] = res.resample_ms;
  info[5] = (double)res.device_bytes;
  *n_out = (unsigned)n;
}

// the AU-mode outputs (scale_count is [scale][cap]) and info[6..8]
static void copy_support_au(const model_t::placement_support_t &res, unsigned cap, unsigned *scale_count,
                            double *p_au, double *au_d, double *au_c, double *au_rss, unsigned *au_used, double *elw,
                            unsigned long long *elw_fixed, double *info) {
  const size_t n = res.root_id.size();
  for (size_t i = 0; i < n; ++i) {
    for (size_t k = 0; k < res.scales.size(); ++k) scale_count[k * cap + i] = res.scale_count[k * n + i];
    p_au[i] = res.p_au[i];
    au_d[i] = res.au_d[i];
    au_c[i] = res.au_c[i];
    au_rss[i] = res.au_rss[i];
    au_used[i] = res.au_used[i];
    elw[i] = res.elw[i];
    elw_fixed[i] = res.elw_fixed[i];
  }
  info[6] = res.au_counts_ms;
  info[7] = res.au_accumulate_ms;
  info[8] = res.au_statistics_ms;
}

// the body of rdh_model_placement_support and rdh_model_placement_support_au
static model_t::placement_support_t placement_support_into(
    void *h, const char *checkpoint_prefix, unsigned long long replicates, unsigned long long seed,
    unsigned replicate_tile, int keep_rows, unsigned cap, unsigned long long *root_id, double *alpha, double *llh,
    double *lnl_fixed, unsigned long long *o_lo, long long *o_hi, unsigned *bp_count, unsigned *kh_count,
    unsigned *sh_count, int *exponent, unsigned *best, double *info, unsigned *n_out,
    const std::vector<unsigned> &au_scales) {
  checkpoint_t  external;
  checkpoint_t &ckp = checkpoint_prefix ? (external = checkpoint_t::read_only(checkpoint_prefix)) : H(h).checkpoint;
  const size_t  records = ckp.read_results().size();
  if (records > cap) {
    *n_out = (unsigned)records;
    throw std::runtime_error("output buffers too small: " + std::to_string(records) + " records");
  }
  auto res = H(h).model->placement_support(ckp, replicates, seed, replicate_tile, keep_rows != 0, au_scales);
  copy_support(res, cap, root_id, alpha, llh, lnl_fixed, o_lo, o_hi, bp_count, kh_count, sh_count, exponent, best,
               info, n_out);
  return res;
}

// RELL bootstrap proportions and one-sided KH / SH tests of every placement recorded in
// "<checkpoint_prefix>.ckp" (opened read-only; NULL: the model's own result log), B = replicates in
// [1, 2^20] (model_t::placement_support; DESIGN.md section 10).  Per record, in log order (capacity
// cap): root id, alpha and llh as recorded, the fixed-point log-likelihood, O as a two's-complement
// int128 (o_lo, o_hi; may be NULL) and the integer counts (bp / p_KH / p_SH = count / replicates).
// A log of more than cap records fails before any work, with n_out = its record count.  info
// receives {capture ms, counts ms, accumulation ms, statistics ms, whole resampling ms, device
// bytes}; replicate_tile 0 = the engine's choice; keep_rows != 0 keeps the per-pattern rows for
// rdh_model_site_lnl_rows (otherwise their device memory is freed on return).
extern "C" int rdh_model_placement_support(void *h, const char *checkpoint_prefix, unsigned long long replicates,
                                           unsigned long long seed, unsigned replicate_tile, int keep_rows,
                                           unsigned cap, unsigned long long *root_id, double *alpha, double *llh,
                                           double *lnl_fixed, unsigned long long *o_lo, long long *o_hi,
                                           unsigned *bp_count, unsigned *kh_count, unsigned *sh_count, int *exponent,
                                           unsigned *best, double *info, unsigned *n_out) {
  RDH_TRY({
    placement_support_into(h, checkpoint_prefix, replicates, seed, replicate_tile, keep_rows, cap, root_id, alpha,
                           llh, lnl_fixed, o_lo, o_hi, bp_count, kh_count, sh_count, exponent, best, info, n_out, {});
    return 1;
  })
}

// rdh_model_placement_support plus the AU test and the expected likelihood weights (DESIGN.md
// section 10, items 6-8) from a multiscale bootstrap at n_scales scales in thousandths (2 to 32,
// strictly ascending, in [100, 10000]).  Per record (capacity cap): scale_count[k * cap + r] = #b whose
// argmax at scale k is r, p_au, the fit's d, c and weighted residual sum of squares, the number of
// scales it used, elw and its fixed-point sum elw_fixed (elw = elw_fixed 2^-40 / replicates).  info
// receives the six values of rdh_model_placement_support, then {multiscale counts ms, multiscale
// accumulation ms, statistics + ELW ms}.  Refuses before any work as rdh_model_placement_support does.
extern "C" int rdh_model_placement_support_au(void *h, const char *checkpoint_prefix, unsigned long long replicates,
                                              unsigned long long seed, unsigned replicate_tile, int keep_rows,
                                              unsigned n_scales, const unsigned *scales, unsigned cap,
                                              unsigned long long *root_id, double *alpha, double *llh,
                                              double *lnl_fixed, unsigned long long *o_lo, long long *o_hi,
                                              unsigned *bp_count, unsigned *kh_count, unsigned *sh_count,
                                              unsigned *scale_count, double *p_au, double *au_d, double *au_c,
                                              double *au_rss, unsigned *au_used, double *elw,
                                              unsigned long long *elw_fixed, int *exponent, unsigned *best,
                                              double *info, unsigned *n_out) {
  RDH_TRY({
    if (!scales) throw std::invalid_argument("AU scales: none given");
    const std::vector<unsigned> au(scales, scales + n_scales);
    rd::check_au_scales(au.data(), au.size());
    const auto res = placement_support_into(h, checkpoint_prefix, replicates, seed, replicate_tile, keep_rows, cap,
                                            root_id, alpha, llh, lnl_fixed, o_lo, o_hi, bp_count, kh_count, sh_count,
                                            exponent, best, info, n_out, au);
    copy_support_au(res, cap, scale_count, p_au, au_d, au_c, au_rss, au_used, elw, elw_fixed, info);
    return 1;
  })
}

// The support statistics of EVERY branch at the parameters of the best record of
// "<checkpoint_prefix>.ckp" (opened read-only; NULL: the model's own result log), with root q at
// a_q = optimize_alpha(q at 0.5, atol) (atol = 0: 0.5) -- model_t::branch_support, DESIGN.md section 10,
// items 9-10.  One record per root id, in root-id order (capacity cap >= the model's root count):
// root id, a_q, the log-likelihood at (q, a_q) and the outputs of rdh_model_placement_support.
// n_scales = 0: the plain statistics, and scales and the AU outputs may be NULL; otherwise as
// rdh_model_placement_support_au.  info receives the nine values of rdh_model_placement_support_au
// (zeros for the AU timings in plain mode), then the alpha searches' ms.
extern "C" int rdh_model_branch_support(void *h, const char *checkpoint_prefix, unsigned long long replicates,
                                        unsigned long long seed, double atol, unsigned replicate_tile, int keep_rows,
                                        unsigned n_scales, const unsigned *scales, unsigned cap,
                                        unsigned long long *root_id, double *alpha, double *llh, double *lnl_fixed,
                                        unsigned long long *o_lo, long long *o_hi, unsigned *bp_count,
                                        unsigned *kh_count, unsigned *sh_count, unsigned *scale_count, double *p_au,
                                        double *au_d, double *au_c, double *au_rss, unsigned *au_used, double *elw,
                                        unsigned long long *elw_fixed, int *exponent, unsigned *best, double *info,
                                        unsigned *n_out) {
  RDH_TRY({
    std::vector<unsigned> au;
    if (n_scales) {
      if (!scales) throw std::invalid_argument("AU scales: none given");
      au.assign(scales, scales + n_scales);
      rd::check_au_scales(au.data(), au.size());
    }
    const size_t roots = H(h).model->tree().root_count();
    if (roots > cap) {
      *n_out = (unsigned)roots;
      throw std::runtime_error("output buffers too small: " + std::to_string(roots) + " branches");
    }
    checkpoint_t  external;
    checkpoint_t &ckp = checkpoint_prefix ? (external = checkpoint_t::read_only(checkpoint_prefix)) : H(h).checkpoint;
    const auto    res = H(h).model->branch_support(ckp, replicates, seed, atol, replicate_tile, keep_rows != 0, au);
    copy_support(res, cap, root_id, alpha, llh, lnl_fixed, o_lo, o_hi, bp_count, kh_count, sh_count, exponent, best,
                 info, n_out);
    info[6] = info[7] = info[8] = 0.0;
    if (n_scales) copy_support_au(res, cap, scale_count, p_au, au_d, au_c, au_rss, au_used, elw, elw_fixed, info);
    info[9] = res.positions_ms;
    return 1;
  })
}

// the AU fit of one record alone (model_t::placement_support in AU mode; DESIGN.md section 10, item 7):
// counts[k] of B replicates at scales[k] (thousandths) -> out = {p_AU, d, c, rss}, used = the number of
// scales with 0 < count < B
extern "C" int rdh_placement_au_fit(const unsigned *counts, unsigned n_scales, const unsigned *scales,
                                    unsigned long long B, double *out, unsigned *used) {
  RDH_TRY({
    if (!counts || !scales) throw std::invalid_argument("AU fit: null counts or scales");
    rd::check_au_scales(scales, n_scales);
    if (B == 0) throw std::invalid_argument("AU fit: no replicates");
    for (unsigned k = 0; k < n_scales; ++k)
      if (counts[k] > B) throw std::invalid_argument("AU fit: a count exceeds the replicates");
    const rd::au_fit_t fit = rd::au_fit(counts, scales, n_scales, B);
    out[0] = fit.p_au;
    out[1] = fit.d;
    out[2] = fit.c;
    out[3] = fit.rss;
    *used = fit.used;
    return 1;
  })
}

// the unweighted per-pattern log-likelihoods of the last placement support, [record][pattern] of
// partition `part` (capacity cap doubles), and the partition's pattern weights (capacity
// weights_cap); n_out = records * patterns
extern "C" int rdh_model_site_lnl_rows(void *h, unsigned part, double *out, unsigned long long cap,
                                       unsigned *weights, unsigned weights_cap, unsigned long long *n_out) {
  RDH_TRY({
    if (part >= H(h).msa.size()) throw std::invalid_argument("partition out of range");
    const auto rows = H(h).model->site_lnl_rows(part);
    const auto &msa = H(h).msa[part];
    if (rows.size() > cap || msa.length() > weights_cap) throw std::runtime_error("output buffers too small");
    std::memcpy(out, rows.data(), sizeof(double) * rows.size());
    std::memcpy(weights, msa.weights(), sizeof(unsigned) * msa.length());
    *n_out = rows.size();
    return 1;
  })
}

extern "C" int rdh_model_lwr(const double *llh, unsigned n, double *out) {
  auto w = model_t::lwr(std::vector<double>(llh, llh + n));
  for (unsigned i = 0; i < n; ++i) out[i] = w[i];
  return 1;
}

extern "C" char *rdh_model_newick(void *h, int annotations) {
  try {
    std::string s = H(h).model->tree().newick(annotations != 0);
    char       *out = (char *)malloc(s.size() + 1);
    std::memcpy(out, s.c_str(), s.size() + 1);
    return out;
  } catch (const std::exception &e) {
    rdh_set_error(e.what());
    return nullptr;
  }
}

extern "C" int rdh_model_get_params(void *h, unsigned part, double *rates12, double *freqs4,
                                    double *cat_rates) {
  auto p = H(h).model->partition(part);
  for (int i = 0; i < 12; ++i) rates12[i] = p->subst_params[0][i];
  for (int i = 0; i < 4; ++i) freqs4[i] = p->frequencies[0][i];
  for (unsigned k = 0; k < p->rate_cats; ++k) cat_rates[k] = p->rates[k];
  return 1;
}

extern "C" void *rdh_model_partition(void *h, unsigned part) { return H(h).model->partition(part); }
