/*
 * rdk.h -- C ABI of the B200-native RootDigger likelihood engine.
 *
 * Drop-in boundary: the subset of coraxlib's C API that RootDigger's model_t
 * calls (SURVEY.md section 8b).  Every entry point below names the reference
 * call site it replaces (paths relative to the RootDigger tree).  Signatures
 * are plain C: pointers, sizes, ints, doubles.  No torch types, no C++ types,
 * no exceptions cross this boundary.
 *
 * Error convention (as the corax call sites expect, src/model.cpp:439,849):
 * functions returning int give RDK_SUCCESS / RDK_FAILURE and set
 * rdk_errno / rdk_errmsg; rdk_compute_root_loglikelihood reports through its
 * return value (NaN on a device error, -inf for a zero-likelihood site).
 *
 * Execution model: every partition owns a CUDA stream.  P-matrix updates and
 * CLV operations are *recorded* and executed, in order, at the next call
 * that needs a result (root log-likelihood, a getter, a setter that changes an
 * input they depend on, or rdk_partition_flush).  Semantics are exactly those
 * of executing each call eagerly.
 *
 * There is no CPU fallback: if no CUDA device is usable,
 * rdk_partition_create fails.
 */
#ifndef RDK_H_
#define RDK_H_

#ifdef __cplusplus
extern "C" {
#endif

#define RDK_SUCCESS 1
#define RDK_FAILURE 0

#define RDK_SCALE_BUFFER_NONE (-1)

#define RDK_GAMMA_RATES_MEAN 0
#define RDK_GAMMA_RATES_MEDIAN 1

/* attributes accepted by rdk_partition_create (src/model.cpp:145-157).  The
 * ARCH_* and SITE_REPEATS bits select CPU code paths in coraxlib; they are
 * accepted and ignored.  NONREV is required (the engine implements the
 * non-reversible model only). */
#define RDK_ATTRIB_ARCH_CPU 0u
#define RDK_ATTRIB_ARCH_SSE (1u << 0)
#define RDK_ATTRIB_ARCH_AVX (1u << 1)
#define RDK_ATTRIB_ARCH_AVX2 (1u << 2)
#define RDK_ATTRIB_SITE_REPEATS (1u << 10)
#define RDK_ATTRIB_NONREV (1u << 11)

/* error codes in rdk_errno */
#define RDK_ERROR_NONE 0
#define RDK_ERROR_PARAM 1
#define RDK_ERROR_CUDA 2
#define RDK_ERROR_MEM 3
#define RDK_ERROR_TIP_DATA 4
#define RDK_ERROR_COMM 5

typedef unsigned long long rdk_state_t; /* corax_state_t */

/* corax_operation_t: the 8 fields filled at src/tree.cpp:401-410 */
typedef struct rdk_operation {
  unsigned int parent_clv_index;
  int          parent_scaler_index;
  unsigned int child1_clv_index;
  unsigned int child1_matrix_index;
  int          child1_scaler_index;
  unsigned int child2_clv_index;
  unsigned int child2_matrix_index;
  int          child2_scaler_index;
} rdk_operation_t;

/* corax_partition_t: the leading fields are public because model_t reads
 * them directly (states: src/model.cpp:330,1043,1315,1750; rate_cats: :1045,
 * :1166; subst_params[0][0..11]: :1330-1331).  Host mirrors are kept in sync
 * by the setters.  Everything device-side is behind `engine`. */
typedef struct rdk_partition {
  unsigned int tips;
  unsigned int clv_buffers;
  unsigned int states;
  unsigned int sites; /* sites resident on THIS device (the local shard) */
  unsigned int rate_matrices;
  unsigned int prob_matrices;
  unsigned int rate_cats;
  unsigned int scale_buffers;
  unsigned int attributes;

  double      **subst_params;    /* [rate_matrices][12]  host mirror */
  double      **frequencies;     /* [rate_matrices][4]   host mirror */
  double       *rates;           /* [rate_cats]          host mirror */
  double       *rate_weights;    /* [rate_cats]          host mirror */
  double       *prop_invar;      /* [rate_matrices]      host mirror */
  unsigned int *pattern_weights; /* [sites]              host mirror */

  void *engine; /* opaque */
} rdk_partition_t;

/* thread-local error channel: replaces corax_errno / corax_errmsg
 * (src/model.cpp:439,849; src/msa.cpp:628-629) */
int        *rdk_errno_location(void);
char       *rdk_errmsg_location(void);
#define rdk_errno (*rdk_errno_location())
#define rdk_errmsg (rdk_errmsg_location())

/* corax_map_nt (used through msa_t::map(), src/model.cpp:312) */
extern const rdk_state_t rdk_map_nt[256];

/* ---- device selection (new; one process per GPU picks its device) ------- */
int rdk_device_count(void);
int rdk_set_device(int device); /* affects partitions created afterwards by
                                   the calling thread */

/* ---- partition life cycle ------------------------------------------------ */
/* replaces corax_partition_create, src/model.cpp:159-168 */
rdk_partition_t *rdk_partition_create(unsigned int tips,
                                      unsigned int clv_buffers,
                                      unsigned int states,
                                      unsigned int sites,
                                      unsigned int rate_matrices,
                                      unsigned int prob_matrices,
                                      unsigned int rate_cats,
                                      unsigned int scale_buffers,
                                      unsigned int attributes);
/* replaces corax_partition_destroy, src/model.cpp:180 */
void rdk_partition_destroy(rdk_partition_t *partition);

/* ---- inputs -------------------------------------------------------------- */
/* replaces corax_set_tip_states, src/model.cpp:310-313 */
int rdk_set_tip_states(rdk_partition_t *partition, unsigned int tip_index,
                       const rdk_state_t *map, const char *sequence);
/* replaces corax_set_pattern_weights, src/model.cpp:324 */
void rdk_set_pattern_weights(rdk_partition_t *partition,
                             const unsigned int *pattern_weights);
/* replaces corax_set_subst_params, src/model.cpp:185 */
void rdk_set_subst_params(rdk_partition_t *partition,
                          unsigned int params_index, const double *params);
/* replaces corax_set_frequencies, src/model.cpp:337,347 */
void rdk_set_frequencies(rdk_partition_t *partition, unsigned int params_index,
                         const double *frequencies);
/* replaces corax_set_category_rates, src/model.cpp:244,253,262,271,276,289 */
void rdk_set_category_rates(rdk_partition_t *partition, const double *rates);
/* replaces corax_set_category_weights, src/model.cpp:205,209 */
void rdk_set_category_weights(rdk_partition_t *partition,
                              const double *rate_weights);
/* replaces corax_update_invariant_sites, src/model.cpp:294 */
int rdk_update_invariant_sites(rdk_partition_t *partition);
/* replaces corax_update_invariant_sites_proportion, src/model.cpp:297 */
int rdk_update_invariant_sites_proportion(rdk_partition_t *partition,
                                          unsigned int params_index,
                                          double prop_invar);

/* ---- the hot path -------------------------------------------------------- */
/* replaces corax_update_prob_matrices, src/model.cpp:367,432,842.
 * Re-entrant for distinct matrix indices of one partition (it is called from
 * an OpenMP loop at src/model.cpp:362-369). */
int rdk_update_prob_matrices(rdk_partition_t *partition,
                             const unsigned int *params_indices,
                             const unsigned int *matrix_indices,
                             const double *branch_lengths,
                             unsigned int count);
/* replaces corax_update_clvs, src/model.cpp:402,440,461,851 */
void rdk_update_clvs(rdk_partition_t *partition,
                     const rdk_operation_t *operations, unsigned int count);
/* replaces corax_compute_root_loglikelihood, src/model.cpp:406,441,466.
 * persite_lnl may be NULL; otherwise receives `sites` weighted per-site
 * log-likelihoods.  With a communicator attached (below) the return value is
 * the log-likelihood over ALL shards. */
double rdk_compute_root_loglikelihood(rdk_partition_t *partition,
                                      unsigned int clv_index,
                                      int scaler_index,
                                      const unsigned int *freqs_indices,
                                      double *persite_lnl);

/* ---- host-side model utilities ------------------------------------------- */
/* replaces corax_compute_gamma_cats, src/model.cpp:239,248,257,266 */
int rdk_compute_gamma_cats(double alpha, unsigned int categories,
                           double *output_rates, int rates_mode);
/* replaces corax_msa_empirical_frequencies, src/model.cpp:329 (result is
 * malloc'd; the caller frees it with free(), src/model.cpp:338).  With a
 * communicator attached the counts are summed over all shards. */
double *rdk_msa_empirical_frequencies(rdk_partition_t *partition);

/* ---- fused extensions (new; same results as the call sequences named) ---- */
/* One root-only evaluation per candidate without touching partition state:
 * for b in [0,count): logL of the tree rooted by `root_op` with the two root
 * branches at lengths branch_lengths[2b], branch_lengths[2b+1].  Equivalent to
 * count x { update_prob_matrices(2) ; update_clvs(root_op) ;
 * compute_root_loglikelihood } = model_t::compute_lh_root, src/model.cpp:415-452,
 * as used by compute_dlh (:481-519) and brents (:606-676), except that the
 * root CLV, root scaler and the two P-matrices are left unmodified. */
int rdk_root_loglikelihood_multi(rdk_partition_t *partition,
                                 const rdk_operation_t *root_op,
                                 const unsigned int *params_indices,
                                 const unsigned int *freqs_indices,
                                 const double *branch_lengths,
                                 unsigned int count, double *out_lnl);

/* The placement sweep of model_t::suggest_roots_lh (src/model.cpp:865-889):
 * for each placement p, in order: update_prob_matrices(pmatrix entries
 * [pm_offsets[p], pm_offsets[p+1])) ; update_clvs(ops [op_offsets[p],
 * op_offsets[p+1])) ; out_lnl[p] = compute_root_loglikelihood(root_clv_index,
 * root_scaler_index).  The caller concatenates what move_root (:823-854) and
 * compute_lh_root (:415-452) would have passed.  Partition state afterwards is
 * the state after the last placement. */
int rdk_sweep_root_placements(rdk_partition_t *partition,
                              unsigned int placements,
                              const unsigned int *params_indices,
                              const unsigned int *freqs_indices,
                              const unsigned int *pm_offsets,
                              const unsigned int *matrix_indices,
                              const double *branch_lengths,
                              const unsigned int *op_offsets,
                              const rdk_operation_t *operations,
                              unsigned int root_clv_index,
                              int root_scaler_index, double *out_lnl);

/* The same sweep with options.  RDK_SWEEP_KEEP_ROOT: the LAST operation of a
 * placement, when its parent is (root_clv_index, root_scaler_index), is only
 * evaluated -- the root CLV and root scale buffer are not stored, so partition
 * state seen through them is what it was before the call (log-likelihoods are
 * unchanged: the root CLV is consumed in registers).  This is what the
 * directed-CLV sweep (rooted_tree_t::generate_sweep_operations in the host
 * mirror) uses: one pre-order pass over spare CLV buffers scores all 2n-3
 * placements with ~1 CLV operation + 1 root evaluation each instead of a
 * re-orientation path per placement. */
#define RDK_SWEEP_KEEP_ROOT 1u
/* RDK_SWEEP_DISCARD: the content, after the call, of every CLV and scale buffer that the
 * operations of this call write is UNDEFINED (they are scratch: the spare directed-CLV
 * buffers of the directed sweep).  The engine then keeps a value in registers instead of
 * storing it whenever no later operation of the sweep reads it back from memory.  The
 * log-likelihoods are unchanged. */
#define RDK_SWEEP_DISCARD 2u
/* RDK_SWEEP_ROWS: the evaluation of placement q also stores every pattern's UNWEIGHTED
 * log-likelihood (the value rdk_compute_root_loglikelihood_row stores, before the pattern weight)
 * into row q of the partition's site matrix, which rdk_partition_set_site_lnl_rows must have
 * reserved with at least `placements` rows (the call fails before any work otherwise).  On a site
 * shard the rows hold the local patterns.  out_lnl is unchanged, bit for bit.  Combines with the
 * other flags and with rdk_sweep_root_placements_chunks. */
#define RDK_SWEEP_ROWS 4u
/* If a sweep fails, none of its evaluations stays recorded: no later call runs one.  The engine
 * may already have run the batches before the failing one, so the buffers the call's operations
 * write have undefined content afterwards. */
int rdk_sweep_root_placements_ex(rdk_partition_t *partition,
                                 unsigned int placements,
                                 const unsigned int *params_indices,
                                 const unsigned int *freqs_indices,
                                 const unsigned int *pm_offsets,
                                 const unsigned int *matrix_indices,
                                 const double *branch_lengths,
                                 const unsigned int *op_offsets,
                                 const rdk_operation_t *operations,
                                 unsigned int root_clv_index,
                                 int root_scaler_index, unsigned int flags,
                                 double *out_lnl);

/* The same sweep cut into n_chunks INDEPENDENT chunks of consecutive placements
 * (chunk c = placements [chunk_offsets[c], chunk_offsets[c+1]), chunk_offsets[0] = 0,
 * chunk_offsets[n_chunks] = placements).  Contract: no chunk reads a CLV or scale
 * buffer that another chunk writes (rooted_tree_t::generate_sweep_operations gives
 * every chunk its own spare buffers and re-derives the directed CLVs on the path to
 * its first placement); with RDK_SWEEP_KEEP_ROOT the root buffers are not written
 * either.  The engine may then walk the chunks SIDE BY SIDE -- (site range) x (chunk)
 * warps in one launch -- which is what fills the device when the shard is small (a
 * 12.5k-site shard has one warp iteration per warp: one long latency-bound chain);
 * otherwise it runs them in order.  Results are those of rdk_sweep_root_placements_ex
 * on the same arrays, bit for bit.
 * Site-sharded partitions (rdk_partition_attach_comm): the ranks' values are added
 * slot by slot, so -- as for every sweep call -- all ranks must pass the SAME
 * placements in the SAME order: derive the chunk count from the layout (the largest
 * shard), not from the local site count (model_t and bench.py do). */
int rdk_sweep_root_placements_chunks(rdk_partition_t *partition,
                                     unsigned int placements,
                                     const unsigned int *params_indices,
                                     const unsigned int *freqs_indices,
                                     const unsigned int *pm_offsets,
                                     const unsigned int *matrix_indices,
                                     const double *branch_lengths,
                                     const unsigned int *op_offsets,
                                     const rdk_operation_t *operations,
                                     unsigned int root_clv_index,
                                     int root_scaler_index, unsigned int flags,
                                     unsigned int n_chunks,
                                     const unsigned int *chunk_offsets,
                                     double *out_lnl);
/* how many chunks a sweep over a shard of `sites` patterns x `rate_cats` categories
 * should be cut into to fill the current device (1: the shard fills it alone);
 * at most RDK_SWEEP_MAX_CHUNKS */
#define RDK_SWEEP_MAX_CHUNKS 16u
unsigned int rdk_sweep_chunk_hint(unsigned int sites, unsigned int rate_cats);

/* ---- site sharding across GPUs (new; SURVEY 8e) --------------------------- */
/* A partition holds a contiguous range of the alignment's site patterns.
 * site_offset must be a multiple of RDK_SHARD_ALIGN unless it is 0; the
 * reduction tree is defined over the GLOBAL site index, so the result does not
 * depend on the number of shards. */
#define RDK_SHARD_ALIGN 256u
#define RDK_COMM_ID_BYTES 128
int rdk_partition_set_shard(rdk_partition_t *partition,
                            unsigned long long site_offset,
                            unsigned long long global_sites);
/* NCCL bootstrap: rank 0 calls rdk_comm_unique_id and ships the 128 bytes to
 * the other ranks by any means (torch.distributed broadcast, MPI_Bcast as at
 * src/main.cpp:324, a file); then every rank attaches. */
int rdk_comm_unique_id(void *id_out);
int rdk_partition_attach_comm(rdk_partition_t *partition, int nranks, int rank,
                              const void *id);

/* ---- plumbing / introspection (new) --------------------------------------- */
int rdk_partition_flush(rdk_partition_t *partition); /* launch recorded work */
int rdk_partition_sync(rdk_partition_t *partition);  /* flush + stream sync  */
/* adopt a caller-owned cudaStream_t (e.g. torch's current stream) */
int rdk_partition_set_stream(rdk_partition_t *partition, void *cuda_stream);
void *rdk_partition_stream(rdk_partition_t *partition);
/* read back device state (tips are expanded to 0/1 vectors) */
int rdk_get_clv(rdk_partition_t *partition, unsigned int clv_index,
                double *out /* sites*rate_cats*4 */);
int rdk_get_scale_buffer(rdk_partition_t *partition, int scaler_index,
                         unsigned int *out /* sites */);
int rdk_get_pmatrix(rdk_partition_t *partition, unsigned int matrix_index,
                    double *out /* rate_cats*16 */);

typedef struct rdk_stats {
  unsigned long long kernel_launches;   /* all kernels launched by the engine */
  unsigned long long program_launches;  /* CLV/log-likelihood program kernels */
  unsigned long long pmatrix_launches;
  unsigned long long reduce_launches;
  unsigned long long clv_ops;           /* CLV operations executed            */
  unsigned long long root_evals;        /* root log-likelihood evaluations    */
  unsigned long long pmatrices;         /* branch P-matrix sets built         */
  unsigned long long algorithmic_bytes; /* SURVEY 8d accounting, this shard   */
  unsigned long long h2d_bytes;
  unsigned long long d2h_bytes;
  unsigned long long device_bytes;      /* currently allocated                */
  unsigned long long program_time_ns;   /* device time of the program kernels,
                                           CUDA events on the partition's
                                           stream; 0 unless timing is enabled */
  unsigned long long program_timed;     /* launches included in program_time_ns */
  unsigned long long instructions;      /* program instructions launched (operations + the
                                           register loads the lowering inserted)           */
  unsigned long long stores_elided;     /* CLV stores dropped because nothing reads them back */
  unsigned long long lazy_evaluations;  /* full evaluations that kept CLVs in registers only  */
  unsigned long long materializations;  /* kept programs replayed with all their stores       */
  unsigned long long host_record_ns;    /* host wall time: recording P-matrix updates / operations */
  unsigned long long host_lower_ns;     /* ... lowering, pointer translation, enqueueing launches   */
  unsigned long long host_wait_ns;      /* ... waiting for the device at the result synchronisation */
  unsigned long long grouped_programs;  /* programs run as subtree groups + a joining program (rdk_partition_set_subtree_groups) */
  unsigned long long programs_reused;   /* programs whose lowering was taken from the previous traversal of the same structure */
} rdk_stats_t;
void rdk_partition_stats(rdk_partition_t *partition, rdk_stats_t *out);
void rdk_partition_reset_stats(rdk_partition_t *partition);
/* Bracket every program-kernel launch with CUDA events on the partition's
 * stream; rdk_partition_stats then reports their summed device time. */
int rdk_partition_set_timing(rdk_partition_t *partition, int enabled);
/* tuning knobs (0 = engine default): program-kernel CTAs per SM, threads */
int rdk_partition_set_launch_config(rdk_partition_t *partition,
                                    int ctas_per_sm, int threads_per_cta,
                                    int elems_per_thread);
/* Lazily materialised evaluations (default on; RDK_LAZY=0 in the environment turns them off for
 * partitions created afterwards).  A full traversal whose only requested result is the root
 * log-likelihood -- rdk_update_clvs of >= 16 operations followed by
 * rdk_compute_root_loglikelihood(..., persite_lnl = NULL) on the CLV the last operation produces,
 * i.e. compute_lh_partition inside the BFGS closures (src/model.cpp:455-476, 1488-1502) -- stores
 * only the CLVs it reads back itself, from the second such traversal in a row onwards (a single
 * compute_lh before a sweep or a root move would only have to be replayed).  The engine keeps the operations and replays them with all
 * their stores before anything reads such a CLV (the next traversal overwriting all of them drops
 * the kept program instead).  Results and observable partition state are those of eager
 * execution, bit for bit. */
int rdk_partition_set_lazy(rdk_partition_t *partition, int enabled);
/* Subtree groups.  On a small shard the walk of a long traversal is bound by the latency of one
 * instruction, so the engine runs disjoint subtrees of the recorded operations side by side
 * (groups, one per blockIdx.y, as the chunks of a placement sweep) and then the operations that
 * join them -- when its launch cost model says that is faster, and only for programs that are
 * plainly forests (csrc/rdk_lower.hpp).  Every operation computes the same value from the same
 * operands as in array order (corax_update_clvs, src/model.cpp:402): results are identical bit
 * for bit.  groups = 0: the engine decides (default; RDK_SUBTREE_GROUPS in the environment sets
 * the value for partitions created afterwards), 1: never, 2..16: always that many groups where
 * the program allows it (tests, experiments). */
int rdk_partition_set_subtree_groups(rdk_partition_t *partition, int groups);
/* accepted and ignored (round-1 kernels had two tail rules); results never depended on it */
int rdk_partition_set_tail_mode(rdk_partition_t *partition, int mode);
const char *rdk_version(void);
/* Introspection of the lowering (csrc/rdk_lower.hpp), pure host code: `n_ops` recorded
 * operations of 10 ints each {parent clv, parent scaler, child1 clv, child2 clv, child1
 * scaler, child2 scaler, P slot 1, P slot 2, flags (1 store, 2 evaluate, 4 evaluate the
 * stored CLV child1), eval slot} -> instructions of 10 ints each {flags, parent, parent
 * scaler, child1, child1 scaler, child2, P slot 1, P slot 2, eval slot, child2 scaler}.  Returns the
 * number of instructions, -1 if out_cap is too small. */
int rdk_debug_lower_program(unsigned int tips, unsigned int n_ops, const int *ops,
                            unsigned int n_chunks, const unsigned int *chunk_off,
                            int discard_writes, const unsigned char *scratch_clv,
                            unsigned int n_scratch_clv, int *out, unsigned int out_cap,
                            unsigned int *out_chunk_off);

/* The subtree-group rearrangement, lowered: the instructions of the groups (out_group_off:
 * groups + 1 offsets), then those of the joining program; *n_group_instr = instructions of all
 * groups, *n_total_instr = all instructions written.  `cap` = largest subtree dealt as a whole.
 * Returns the number of groups (0: the program keeps its order), -1 if out_cap is too small. */
int rdk_debug_lower_grouped(unsigned int tips, unsigned int n_ops, const int *ops,
                            unsigned int n_groups, unsigned int cap, int discard_writes, int *out,
                            unsigned int out_cap, unsigned int *out_group_off,
                            unsigned int *n_group_instr, unsigned int *n_total_instr);

/* What the engine decides for a program (operations as above) on a shard of `sites` patterns x
 * `rate_cats` categories on a device of `sm_count` SMs (0: 148): the number of subtree groups
 * (0: one program in array order), the operations of the longest group and of the joining program.
 * Pure host code. */
int rdk_debug_choose_subtree_groups(unsigned int tips, unsigned int n_ops, const int *ops,
                                    unsigned int sites, unsigned int rate_cats, int sm_count,
                                    unsigned int *longest, unsigned int *n_join);

/* ---- root placement support (new; DESIGN.md section 10) ------------------- */
/* Reserve a device matrix of `rows` x (local patterns) doubles that
 * rdk_compute_root_loglikelihood_row fills (rows = 0 frees it). */
int rdk_partition_set_site_lnl_rows(rdk_partition_t *partition, unsigned int rows);
/* rdk_compute_root_loglikelihood, same value bit for bit, that also stores every pattern's
 * UNWEIGHTED log-likelihood (the value before the pattern weight is applied) into row `row`. */
double rdk_compute_root_loglikelihood_row(rdk_partition_t *partition, unsigned int clv_index,
                                          int scaler_index, unsigned int row);
/* copy rows [first, first + count) of that matrix to out ([count][local patterns]) */
int rdk_partition_get_site_lnl_rows(rdk_partition_t *partition, unsigned int first,
                                    unsigned int count, double *out);

/* reorder the first `count` rows of that matrix on the device: row r afterwards holds what row
 * order[r] held before (order is a permutation of 0..count-1).  A placement sweep captures rows in
 * its own placement order; this puts them in the order the statistics below index records by. */
int rdk_partition_permute_site_lnl_rows(rdk_partition_t *partition, unsigned int count,
                                        const unsigned int *order);

/* RELL bootstrap proportions and one-sided KH / SH tests over `rows` records whose per-pattern
 * log-likelihoods L are rows 0..rows-1 of the site matrices of n partitions (all on one device),
 * or of ONE site shard with a communicator attached (every rank makes the same call and gets the
 * bits of one GPU); global_index[i] is partition i's global index (it keys the random draws).
 * Fixed point q = rint(L * 2^exponent), exponent = 52 - frexp exponent of max |L|; replicate b
 * draws, per partition g, N_g = sum of its weights sites with Philox4x64-10 keyed
 * {seed, (g << 32) | b}; Z[b][r] = sum c * q and O[r] = sum w * q are exact (int128).
 * Caller-owned arrays have `rows` entries. */
typedef struct rdk_rell_out_t {
  unsigned int        replicate_tile; /* in: replicates per counts tile, 0 = engine default */
  int                 exponent;       /* out: e */
  unsigned int        best;           /* out: argmax_r O[r], lowest index on ties */
  unsigned int        bad_row;        /* out on failure: a record with a non-finite L, or ~0u */
  double             *lnl_fixed;      /* out: O[r] * 2^-e rounded once */
  unsigned long long *o_lo;           /* out (optional): O[r] as two's-complement int128, low word */
  long long          *o_hi;           /* ... high word */
  unsigned int       *bp_count;       /* out: #b whose argmax_r Z[b][r] is r */
  unsigned int       *kh_count;       /* out: #b passing the centred KH test against best */
  unsigned int       *sh_count;       /* out: #b passing the SH test */
  double              ms[4];          /* out: device time of counts, accumulation, statistics, all */
  unsigned long long  device_bytes;   /* out: device memory the call allocated (freed on return) */
} rdk_rell_out_t;
int rdk_rell_support(rdk_partition_t *const *partitions, unsigned int n,
                     const unsigned int *global_index, unsigned int rows,
                     unsigned long long replicates, unsigned long long seed, rdk_rell_out_t *out);

/* The multiscale RELL bootstrap of the AU test and expected likelihood weights (DESIGN.md section 10,
 * items 6-8), on top of everything rdk_rell_support computes (it fills *out the same way).  At scale s
 * (thousandths) replicate b draws max(1, (s N_g + 500) / 1000) sites of partition g with the Philox
 * counter's second word s - 1000 (mod 2^64), so scale 1000 is the draws of rdk_rell_support and its
 * column is bp_count.  Scales are strictly ascending, in [100, 10000], 2 to 32 of them. */
typedef struct rdk_rell_ms_out_t {
  const unsigned int *scales;      /* in: n_scales scales in thousandths */
  unsigned int        n_scales;    /* in */
  unsigned int       *scale_count; /* out: [n_scales][rows], #b whose argmax_r Z_k[b][r] is r */
  unsigned long long *elw_fixed;   /* out: [rows], sum_b floor(u_b[r] 2^40 / sum_r' u_b[r']) */
  double              ms[3];       /* out: device time of multiscale counts, accumulation, statistics + ELW */
} rdk_rell_ms_out_t;
int rdk_rell_support_ms(rdk_partition_t *const *partitions, unsigned int n,
                        const unsigned int *global_index, unsigned int rows,
                        unsigned long long replicates, unsigned long long seed, rdk_rell_out_t *out,
                        rdk_rell_ms_out_t *ms);

/* Gene and gene-then-site resampling of n >= 2 whole partitions (DESIGN.md section 10, items
 * 11-14), with everything rdk_rell_support computes (it fills *out the same way).  Replicate b draws
 * n partitions with replacement, draw j = word j of Philox4x64-10 keyed {seed, b} from the counter
 * {0, 0, 1, 0} picking partition (x_j n) >> 64; m[b][i] = how often it drew partition i.
 * RDK_RELL_GENE: Z[b][r] = sum_i m[b][i] O_i[r].  RDK_RELL_GENE_SITE: replicate b takes the first
 * m[b][i] N_i draws of rdk_rell_support's stream of partition i (m = 1: exactly its draws).  O_i is
 * O over partition i alone (O = sum_i O_i).  Refuses site shards, n * max_i N_i >= 2^32 and
 * replicates outside [1, 2^20]. */
#define RDK_RELL_GENE      1u
#define RDK_RELL_GENE_SITE 2u
typedef struct rdk_rell_gene_out_t {
  unsigned int        sampling;            /* in: RDK_RELL_GENE or RDK_RELL_GENE_SITE */
  double             *partition_lnl_fixed; /* out: [n][rows], O_i[r] * 2^-e rounded once */
  unsigned long long *o_lo;                /* out (optional): [n][rows] O_i[r] as int128, low word */
  long long          *o_hi;                /* ... high word */
  double              draws_ms;            /* out: device time of the gene draws (out->ms has the rest) */
} rdk_rell_gene_out_t;
int rdk_rell_support_genes(rdk_partition_t *const *partitions, unsigned int n,
                           const unsigned int *global_index, unsigned int rows,
                           unsigned long long replicates, unsigned long long seed, rdk_rell_out_t *out,
                           rdk_rell_gene_out_t *genes);

/* ---- marginal ancestral states (new; DESIGN.md section 11) ----------------- */
/* The posterior of every internal node of the rooted tree whose post-order operations are
 * ops[0..count) -- those of the last full traversal: node i is ops[i].parent_clv_index, the root is
 * the parent of ops[count - 1], whose state has the prior pi.  One pre-order pass over outside vectors
 * (smaller subtree first: at most ceil(log2 count) + 2 CLV-sized scratch buffers) from the stored child
 * CLVs, their scalers and the P-matrices of the operations; recorded P-matrix updates are run and a
 * kept lazy program is materialised first.  The patterns are walked in tiles, so the device holds the
 * outputs and scratch of one tile at a time.  full_ops must not repeat an operation.  On a site shard the outputs hold the local patterns.
 * Arrays are caller-owned; patterns = the partition's `sites`. */
typedef struct rdk_ancestral_out_t {
  const unsigned int *full_ops;     /* in: positions i of the nodes whose full posterior is wanted */
  unsigned int        n_full;       /* in */
  unsigned int        threads;      /* in: threads per block, a multiple of 32 up to 256 (0: 256) */
  unsigned int        tile_sites;   /* in: patterns per pass (0: as many as keep the outputs and scratch of a
                                       pass within 512 MiB); out: the tile used */
  unsigned char      *map_state;    /* out: [count][patterns], argmax of the posterior, lowest state on ties */
  double             *map_prob;     /* out: [count][patterns], its posterior */
  double             *posterior;    /* out: [n_full][patterns][4] */
  double             *log_norm;     /* out (optional): [count][patterns], log of the normaliser + scalers */
  double              ms;           /* out: device time of the pass */
  unsigned long long  device_bytes; /* out: device memory the call allocated (freed on return) */
  unsigned int        scratch;      /* out: outside-vector buffers the pass used */
} rdk_ancestral_out_t;
int rdk_marginal_ancestral_states(rdk_partition_t *partition, const rdk_operation_t *ops, unsigned int count,
                                  const unsigned int *freqs_indices, rdk_ancestral_out_t *out);

#ifdef __cplusplus
}
#endif
#endif
