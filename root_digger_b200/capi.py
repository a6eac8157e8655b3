"""ctypes binding of the C ABI (include/rdk.h) and of the host scheduler.

This is plumbing for tests, bench.py and Python callers; the product is the
shared library.  Loading fails loudly when the CUDA library has not been built:
there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from . import _build

RDK_SUCCESS = 1
RDK_SCALE_BUFFER_NONE = -1
RDK_ATTRIB_SITE_REPEATS = 1 << 10
RDK_ATTRIB_NONREV = 1 << 11
RDK_GAMMA_RATES_MEAN = 0
RDK_GAMMA_RATES_MEDIAN = 1
RDK_SHARD_ALIGN = 256
RDK_SWEEP_KEEP_ROOT = 1
RDK_SWEEP_DISCARD = 2
RDK_SWEEP_ROWS = 4
# the scales of the AU test's multiscale bootstrap that CONSEL and IQ-TREE use by default
AU_SCALES = (0.5, 0.6, 0.7, 0.8, 0.9, 1.0, 1.1, 1.2, 1.3, 1.4)


def au_thousandths(scales) -> list:
    """AU scales -> integers in thousandths (what the host and the engine take); ValueError when a
    scale is not a multiple of 0.001.  Order, range and count are checked by the host."""
    out = []
    for s in scales:
        t = round(float(s) * 1000)
        if abs(float(s) * 1000 - t) > 1e-6:
            raise ValueError("AU scale %r is not a multiple of 0.001" % (s,))
        if t <= 0:
            raise ValueError("AU scale %r is not positive" % (s,))
        out.append(t)
    return out


class Operation(C.Structure):
    """rdk_operation_t / corax_operation_t"""
    _fields_ = [
        ("parent_clv_index", C.c_uint),
        ("parent_scaler_index", C.c_int),
        ("child1_clv_index", C.c_uint),
        ("child1_matrix_index", C.c_uint),
        ("child1_scaler_index", C.c_int),
        ("child2_clv_index", C.c_uint),
        ("child2_matrix_index", C.c_uint),
        ("child2_scaler_index", C.c_int),
    ]

    def astuple(self):
        return tuple(getattr(self, f[0]) for f in self._fields_)


class PartitionStruct(C.Structure):
    """public prefix of rdk_partition_t"""
    _fields_ = [
        ("tips", C.c_uint), ("clv_buffers", C.c_uint), ("states", C.c_uint), ("sites", C.c_uint),
        ("rate_matrices", C.c_uint), ("prob_matrices", C.c_uint), ("rate_cats", C.c_uint),
        ("scale_buffers", C.c_uint), ("attributes", C.c_uint),
        ("subst_params", C.POINTER(C.POINTER(C.c_double))),
        ("frequencies", C.POINTER(C.POINTER(C.c_double))),
        ("rates", C.POINTER(C.c_double)),
        ("rate_weights", C.POINTER(C.c_double)),
        ("prop_invar", C.POINTER(C.c_double)),
        ("pattern_weights", C.POINTER(C.c_uint)),
        ("engine", C.c_void_p),
    ]


class Stats(C.Structure):
    _fields_ = [(n, C.c_ulonglong) for n in (
        "kernel_launches", "program_launches", "pmatrix_launches", "reduce_launches", "clv_ops",
        "root_evals", "pmatrices", "algorithmic_bytes", "h2d_bytes", "d2h_bytes", "device_bytes",
        "program_time_ns", "program_timed", "instructions", "stores_elided", "lazy_evaluations",
        "materializations", "host_record_ns", "host_lower_ns", "host_wait_ns", "grouped_programs", "programs_reused")]

    def asdict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class AncestralOut(C.Structure):  # rdk_ancestral_out_t
    _fields_ = [("full_ops", C.POINTER(C.c_uint)), ("n_full", C.c_uint), ("threads", C.c_uint),
                ("tile_sites", C.c_uint), ("map_state", C.POINTER(C.c_ubyte)), ("map_prob", C.POINTER(C.c_double)),
                ("posterior", C.POINTER(C.c_double)), ("log_norm", C.POINTER(C.c_double)), ("ms", C.c_double),
                ("device_bytes", C.c_ulonglong), ("scratch", C.c_uint)]


_dp = C.POINTER(C.c_double)
_up = C.POINTER(C.c_uint)
_pp = C.POINTER(PartitionStruct)

_engine_lib = None
_host_lib = None


def _ptr(a, t):
    return a.ctypes.data_as(t)


def engine_lib_path() -> Path:
    import os
    # another build of the same ABI, e.g. the parent commit's, to compare outputs (bench.py --dump-outputs)
    override = os.environ.get("RDK_ENGINE_LIB")
    return Path(override) if override else _build.LIBDIR / "librdk_b200.so"


def load_engine() -> C.CDLL:
    """dlopen lib/librdk_b200.so (building it when nvcc is available)."""
    global _engine_lib
    if _engine_lib is not None:
        return _engine_lib
    path = engine_lib_path()
    if not path.exists():
        _build.build_engine()
    if not path.exists():
        raise RuntimeError(f"{path} is missing: build the CUDA engine first (no CPU fallback exists)")
    L = C.CDLL(str(path), mode=C.RTLD_GLOBAL)
    L.rdk_errno_location.restype = C.POINTER(C.c_int)
    L.rdk_errmsg_location.restype = C.c_char_p
    L.rdk_version.restype = C.c_char_p
    L.rdk_partition_create.restype = _pp
    L.rdk_partition_create.argtypes = [C.c_uint] * 9
    L.rdk_partition_destroy.argtypes = [_pp]
    L.rdk_partition_destroy.restype = None
    L.rdk_set_tip_states.argtypes = [_pp, C.c_uint, C.c_void_p, C.c_char_p]
    L.rdk_set_pattern_weights.argtypes = [_pp, _up]
    L.rdk_set_pattern_weights.restype = None
    L.rdk_set_subst_params.argtypes = [_pp, C.c_uint, _dp]
    L.rdk_set_subst_params.restype = None
    L.rdk_set_frequencies.argtypes = [_pp, C.c_uint, _dp]
    L.rdk_set_frequencies.restype = None
    L.rdk_set_category_rates.argtypes = [_pp, _dp]
    L.rdk_set_category_rates.restype = None
    L.rdk_set_category_weights.argtypes = [_pp, _dp]
    L.rdk_set_category_weights.restype = None
    L.rdk_update_invariant_sites.argtypes = [_pp]
    L.rdk_update_invariant_sites_proportion.argtypes = [_pp, C.c_uint, C.c_double]
    L.rdk_update_prob_matrices.argtypes = [_pp, _up, _up, _dp, C.c_uint]
    L.rdk_update_clvs.argtypes = [_pp, C.POINTER(Operation), C.c_uint]
    L.rdk_update_clvs.restype = None
    L.rdk_compute_root_loglikelihood.argtypes = [_pp, C.c_uint, C.c_int, _up, _dp]
    L.rdk_compute_root_loglikelihood.restype = C.c_double
    L.rdk_compute_gamma_cats.argtypes = [C.c_double, C.c_uint, _dp, C.c_int]
    L.rdk_msa_empirical_frequencies.argtypes = [_pp]
    L.rdk_msa_empirical_frequencies.restype = C.c_void_p
    L.rdk_root_loglikelihood_multi.argtypes = [_pp, C.POINTER(Operation), _up, _up, _dp, C.c_uint, _dp]
    L.rdk_sweep_root_placements.argtypes = [_pp, C.c_uint, _up, _up, _up, _up, _dp, _up,
                                            C.POINTER(Operation), C.c_uint, C.c_int, _dp]
    L.rdk_sweep_root_placements_ex.argtypes = [_pp, C.c_uint, _up, _up, _up, _up, _dp, _up,
                                               C.POINTER(Operation), C.c_uint, C.c_int, C.c_uint, _dp]
    L.rdk_sweep_root_placements_chunks.argtypes = [_pp, C.c_uint, _up, _up, _up, _up, _dp, _up,
                                                   C.POINTER(Operation), C.c_uint, C.c_int, C.c_uint, C.c_uint, _up,
                                                   _dp]
    L.rdk_sweep_chunk_hint.argtypes = [C.c_uint, C.c_uint]
    L.rdk_sweep_chunk_hint.restype = C.c_uint
    L.rdk_partition_set_shard.argtypes = [_pp, C.c_ulonglong, C.c_ulonglong]
    L.rdk_comm_unique_id.argtypes = [C.c_void_p]
    L.rdk_partition_attach_comm.argtypes = [_pp, C.c_int, C.c_int, C.c_void_p]
    L.rdk_partition_flush.argtypes = [_pp]
    L.rdk_partition_sync.argtypes = [_pp]
    L.rdk_partition_set_stream.argtypes = [_pp, C.c_void_p]
    L.rdk_partition_stream.argtypes = [_pp]
    L.rdk_partition_stream.restype = C.c_void_p
    L.rdk_get_clv.argtypes = [_pp, C.c_uint, _dp]
    L.rdk_get_scale_buffer.argtypes = [_pp, C.c_int, _up]
    L.rdk_get_pmatrix.argtypes = [_pp, C.c_uint, _dp]
    L.rdk_partition_stats.argtypes = [_pp, C.POINTER(Stats)]
    L.rdk_partition_stats.restype = None
    L.rdk_partition_reset_stats.argtypes = [_pp]
    L.rdk_partition_reset_stats.restype = None
    L.rdk_partition_set_launch_config.argtypes = [_pp, C.c_int, C.c_int, C.c_int]
    L.rdk_partition_set_timing.argtypes = [_pp, C.c_int]
    L.rdk_partition_set_tail_mode.argtypes = [_pp, C.c_int]
    L.rdk_partition_set_lazy.argtypes = [_pp, C.c_int]
    L.rdk_partition_set_subtree_groups.argtypes = [_pp, C.c_int]
    L.rdk_set_device.argtypes = [C.c_int]
    L.rdk_partition_set_site_lnl_rows.argtypes = [_pp, C.c_uint]
    L.rdk_compute_root_loglikelihood_row.argtypes = [_pp, C.c_uint, C.c_int, C.c_uint]
    L.rdk_compute_root_loglikelihood_row.restype = C.c_double
    L.rdk_partition_get_site_lnl_rows.argtypes = [_pp, C.c_uint, C.c_uint, _dp]
    L.rdk_partition_permute_site_lnl_rows.argtypes = [_pp, C.c_uint, _up]
    L.rdk_marginal_ancestral_states.argtypes = [_pp, C.POINTER(Operation), C.c_uint, _up, C.POINTER(AncestralOut)]
    _engine_lib = L
    return L


class EngineError(RuntimeError):
    pass


def _err(L) -> str:
    return L.rdk_errmsg_location().decode(errors="replace")


def ops_array(ops) -> C.Array:
    """list of 8-tuples / Operation -> ctypes array"""
    arr = (Operation * max(1, len(ops)))()
    for i, o in enumerate(ops):
        if isinstance(o, Operation):
            arr[i] = o
        else:
            arr[i] = Operation(*o)
    return arr


def gamma_cats(alpha: float, k: int, mode: int = RDK_GAMMA_RATES_MEAN) -> np.ndarray:
    L = load_engine()
    out = np.zeros(k)
    if L.rdk_compute_gamma_cats(alpha, k, _ptr(out, _dp), mode) != RDK_SUCCESS:
        raise EngineError(_err(L))
    return out


class Partition:
    """One rdk_partition_t (a site shard resident on one GPU)."""

    def __init__(self, tips: int, sites: int, rate_cats: int = 4, *, clv_buffers: int | None = None,
                 prob_matrices: int | None = None, scale_buffers: int | None = None,
                 attributes: int = RDK_ATTRIB_NONREV | RDK_ATTRIB_SITE_REPEATS, device: int | None = None):
        self.L = load_engine()
        if device is not None:
            if self.L.rdk_set_device(device) != RDK_SUCCESS:
                raise EngineError(_err(self.L))
        branches = 2 * tips - 2
        self.tips, self.sites, self.K = tips, sites, rate_cats
        self.clv_buffers = branches if clv_buffers is None else clv_buffers
        self.prob_matrices = branches if prob_matrices is None else prob_matrices
        self.scale_buffers = branches if scale_buffers is None else scale_buffers
        self.p = self.L.rdk_partition_create(tips, self.clv_buffers, 4, sites, 1, self.prob_matrices,
                                             rate_cats, self.scale_buffers, attributes)
        if not self.p:
            raise EngineError("rdk_partition_create failed: " + _err(self.L))
        self._zeros = (C.c_uint * max(1, rate_cats))()

    def close(self):
        if getattr(self, "p", None):
            self.L.rdk_partition_destroy(self.p)
            self.p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- inputs
    def set_tip_states(self, tip: int, seq: bytes):
        assert len(seq) >= self.sites
        rc = self.L.rdk_set_tip_states(self.p, tip, C.addressof(C.c_ulonglong.in_dll(self.L, "rdk_map_nt")), seq)
        if rc != RDK_SUCCESS:
            raise EngineError(_err(self.L))

    def set_pattern_weights(self, w):
        w = np.ascontiguousarray(w, dtype=np.uint32)
        self.L.rdk_set_pattern_weights(self.p, _ptr(w, _up))

    def set_subst_params(self, r):
        r = np.ascontiguousarray(r, dtype=np.float64)
        self.L.rdk_set_subst_params(self.p, 0, _ptr(r, _dp))

    def set_frequencies(self, f):
        f = np.ascontiguousarray(f, dtype=np.float64)
        self.L.rdk_set_frequencies(self.p, 0, _ptr(f, _dp))

    def set_category_rates(self, r):
        r = np.ascontiguousarray(r, dtype=np.float64)
        self.L.rdk_set_category_rates(self.p, _ptr(r, _dp))

    def set_category_weights(self, w):
        w = np.ascontiguousarray(w, dtype=np.float64)
        self.L.rdk_set_category_weights(self.p, _ptr(w, _dp))

    # ---- hot path
    def update_prob_matrices(self, matrix_indices, branch_lengths):
        mi = np.ascontiguousarray(matrix_indices, dtype=np.uint32)
        bl = np.ascontiguousarray(branch_lengths, dtype=np.float64)
        rc = self.L.rdk_update_prob_matrices(self.p, self._zeros, _ptr(mi, _up), _ptr(bl, _dp), len(mi))
        if rc != RDK_SUCCESS:
            raise EngineError(_err(self.L))

    def update_clvs(self, ops):
        arr = ops if isinstance(ops, C.Array) else ops_array(ops)
        n = len(ops)
        self.L.rdk_errno_location()[0] = 0
        self.L.rdk_update_clvs(self.p, arr, n)
        if self.L.rdk_errno_location()[0] != 0:
            raise EngineError(_err(self.L))

    def root_loglikelihood(self, clv_index: int, scaler_index: int, persite: bool = False):
        ps = np.zeros(self.sites) if persite else None
        v = self.L.rdk_compute_root_loglikelihood(self.p, clv_index, scaler_index, self._zeros,
                                                  _ptr(ps, _dp) if persite else None)
        if persite:
            return v, ps
        return v

    def set_site_lnl_rows(self, rows: int):
        """reserve `rows` device rows of unweighted per-pattern log-likelihoods"""
        if self.L.rdk_partition_set_site_lnl_rows(self.p, rows) != 1:
            raise EngineError(_err(self.L))

    def root_loglikelihood_row(self, clv_index: int, scaler_index: int, row: int) -> float:
        """root_loglikelihood (same bits) that also stores the unweighted per-pattern values in `row`"""
        v = self.L.rdk_compute_root_loglikelihood_row(self.p, clv_index, scaler_index, row)
        if np.isnan(v):
            raise EngineError(_err(self.L))
        return v

    def site_lnl_rows(self, first: int, count: int) -> np.ndarray:
        out = np.zeros((count, self.sites))
        if self.L.rdk_partition_get_site_lnl_rows(self.p, first, count, _ptr(out, _dp)) != 1:
            raise EngineError(_err(self.L))
        return out

    def permute_site_lnl_rows(self, order):
        """row r afterwards holds what row order[r] held (order: a permutation of 0..len(order)-1)"""
        o = np.ascontiguousarray(order, dtype=np.uint32)
        if self.L.rdk_partition_permute_site_lnl_rows(self.p, len(o), _ptr(o, _up)) != 1:
            raise EngineError(_err(self.L))

    def marginal_ancestral_states(self, ops, full_ops=(), threads: int = 0, tile_sites: int = 0) -> dict:
        """rdk_marginal_ancestral_states over the post-order operations `ops` of the last full traversal:
        map_state (0..3) and map_prob, log_norm [op][pattern], posterior [len(full_ops)][pattern][4], and
        ms, device_bytes, scratch, tile_sites"""
        arr = ops if isinstance(ops, C.Array) else ops_array(ops)
        n, S = len(ops), self.sites
        full = np.ascontiguousarray(list(full_ops), dtype=np.uint32)
        ms_, mp, ln = np.zeros((n, S), dtype=np.uint8), np.zeros((n, S)), np.zeros((n, S))
        post = np.zeros((max(1, len(full)), S, 4))
        out = AncestralOut(_ptr(full, _up) if len(full) else None, len(full), threads, tile_sites,
                           _ptr(ms_, C.POINTER(C.c_ubyte)), _ptr(mp, _dp), _ptr(post, _dp), _ptr(ln, _dp))
        if not self.L.rdk_marginal_ancestral_states(self.p, arr, n, self._zeros, C.byref(out)):
            raise EngineError(_err(self.L))
        return {"map_state": ms_, "map_prob": mp, "log_norm": ln, "posterior": post[:len(full)], "ms": out.ms,
                "device_bytes": int(out.device_bytes), "scratch": int(out.scratch), "tile_sites": int(out.tile_sites)}

    def root_loglikelihood_multi(self, root_op, branch_length_pairs):
        bl = np.ascontiguousarray(branch_length_pairs, dtype=np.float64).reshape(-1)
        n = len(bl) // 2
        out = np.zeros(n)
        op = root_op if isinstance(root_op, Operation) else Operation(*root_op)
        rc = self.L.rdk_root_loglikelihood_multi(self.p, C.byref(op), self._zeros, self._zeros, _ptr(bl, _dp), n,
                                                 _ptr(out, _dp))
        if rc != RDK_SUCCESS:
            raise EngineError(_err(self.L))
        return out

    def sweep_root_placements(self, pm_offsets, matrix_indices, branch_lengths, op_offsets, ops,
                              root_clv_index: int, root_scaler_index: int, flags: int = 0, chunk_offsets=None):
        pmo = np.ascontiguousarray(pm_offsets, dtype=np.uint32)
        mi = np.ascontiguousarray(matrix_indices, dtype=np.uint32)
        bl = np.ascontiguousarray(branch_lengths, dtype=np.float64)
        opo = np.ascontiguousarray(op_offsets, dtype=np.uint32)
        arr = ops if isinstance(ops, C.Array) else ops_array(ops)
        n = len(pmo) - 1
        out = np.zeros(n)
        if chunk_offsets is None:
            rc = self.L.rdk_sweep_root_placements_ex(self.p, n, self._zeros, self._zeros, _ptr(pmo, _up),
                                                     _ptr(mi, _up), _ptr(bl, _dp), _ptr(opo, _up), arr,
                                                     root_clv_index, root_scaler_index, flags, _ptr(out, _dp))
        else:  # independent chunks of consecutive placements (rdk.h): the engine may walk them side by side
            co = np.ascontiguousarray(chunk_offsets, dtype=np.uint32)
            rc = self.L.rdk_sweep_root_placements_chunks(self.p, n, self._zeros, self._zeros, _ptr(pmo, _up),
                                                         _ptr(mi, _up), _ptr(bl, _dp), _ptr(opo, _up), arr,
                                                         root_clv_index, root_scaler_index, flags, len(co) - 1,
                                                         _ptr(co, _up), _ptr(out, _dp))
        if rc != RDK_SUCCESS:
            raise EngineError(_err(self.L))
        return out

    def empirical_frequencies(self) -> np.ndarray:
        ptr = self.L.rdk_msa_empirical_frequencies(self.p)
        if not ptr:
            raise EngineError(_err(self.L))
        out = np.array(C.cast(ptr, _dp)[0:4])
        libc = C.CDLL(None)
        libc.free.argtypes = [C.c_void_p]
        libc.free(ptr)
        return out

    # ---- sharding
    def set_shard(self, site_offset: int, global_sites: int):
        if self.L.rdk_partition_set_shard(self.p, site_offset, global_sites) != RDK_SUCCESS:
            raise EngineError(_err(self.L))

    def attach_comm(self, nranks: int, rank: int, unique_id: bytes):
        buf = C.create_string_buffer(unique_id, 128)
        if self.L.rdk_partition_attach_comm(self.p, nranks, rank, buf) != RDK_SUCCESS:
            raise EngineError(_err(self.L))

    # ---- plumbing
    def flush(self):
        if self.L.rdk_partition_flush(self.p) != RDK_SUCCESS:
            raise EngineError(_err(self.L))

    def sync(self):
        if self.L.rdk_partition_sync(self.p) != RDK_SUCCESS:
            raise EngineError(_err(self.L))

    def set_stream(self, cuda_stream: int):
        if self.L.rdk_partition_set_stream(self.p, C.c_void_p(cuda_stream)) != RDK_SUCCESS:
            raise EngineError(_err(self.L))

    def set_launch_config(self, ctas_per_sm=0, threads=0, elems=0):
        if self.L.rdk_partition_set_launch_config(self.p, ctas_per_sm, threads, elems) != RDK_SUCCESS:
            raise EngineError(_err(self.L))

    def set_lazy(self, enabled: bool):
        """rdk_partition_set_lazy: lazily materialised full evaluations on / off"""
        if self.L.rdk_partition_set_lazy(self.p, 1 if enabled else 0) != RDK_SUCCESS:
            raise EngineError(_err(self.L))

    def set_subtree_groups(self, groups: int = 0):
        """rdk_partition_set_subtree_groups: 0 = the engine decides, 1 = never, n = always n groups"""
        if self.L.rdk_partition_set_subtree_groups(self.p, int(groups)) != RDK_SUCCESS:
            raise EngineError(_err(self.L))

    def set_tail_mode(self, mode: int = 0):
        if self.L.rdk_partition_set_tail_mode(self.p, mode) != RDK_SUCCESS:
            raise EngineError(_err(self.L))

    def set_timing(self, on: bool = True):
        if self.L.rdk_partition_set_timing(self.p, 1 if on else 0) != RDK_SUCCESS:
            raise EngineError(_err(self.L))

    def get_clv(self, idx: int) -> np.ndarray:
        out = np.zeros(self.sites * self.K * 4)
        if self.L.rdk_get_clv(self.p, idx, _ptr(out, _dp)) != RDK_SUCCESS:
            raise EngineError(_err(self.L))
        return out.reshape(self.sites, self.K, 4)

    def get_scaler(self, idx: int) -> np.ndarray:
        out = np.zeros(self.sites, dtype=np.uint32)
        if self.L.rdk_get_scale_buffer(self.p, idx, _ptr(out, _up)) != RDK_SUCCESS:
            raise EngineError(_err(self.L))
        return out

    def get_pmatrix(self, idx: int) -> np.ndarray:
        out = np.zeros(self.K * 16)
        if self.L.rdk_get_pmatrix(self.p, idx, _ptr(out, _dp)) != RDK_SUCCESS:
            raise EngineError(_err(self.L))
        return out.reshape(self.K, 4, 4)

    def stats(self) -> dict:
        s = Stats()
        self.L.rdk_partition_stats(self.p, C.byref(s))
        return s.asdict()

    def reset_stats(self):
        self.L.rdk_partition_reset_stats(self.p)


def sweep_chunk_hint(sites: int, rate_cats: int) -> int:
    """rdk_sweep_chunk_hint: independent chunks a directed sweep over such a shard should be cut into"""
    return int(load_engine().rdk_sweep_chunk_hint(sites, rate_cats))


def comm_unique_id() -> bytes:
    L = load_engine()
    buf = C.create_string_buffer(128)
    if L.rdk_comm_unique_id(buf) != RDK_SUCCESS:
        raise EngineError(_err(L))
    return buf.raw


# ---------------------------------------------------------------------------
# host traversal scheduler (rooted_tree_t mirror)
# ---------------------------------------------------------------------------
def load_tree_lib(path: Path | None = None) -> C.CDLL:
    global _host_lib
    if path is None and _host_lib is not None:
        return _host_lib
    if path is None:
        path = _build.LIBDIR / "librd_host.so"
        if not path.exists():
            _build.build_host()
    L = C.CDLL(str(path))
    vp = C.c_void_p
    L.rdh_last_error.restype = C.c_char_p
    L.rdh_tree_from_newick.restype = vp
    L.rdh_tree_from_newick.argtypes = [C.c_char_p]
    L.rdh_tree_from_file.restype = vp
    L.rdh_tree_from_file.argtypes = [C.c_char_p]
    L.rdh_tree_copy.restype = vp
    L.rdh_tree_copy.argtypes = [vp]
    L.rdh_tree_destroy.argtypes = [vp]
    L.rdh_tree_destroy.restype = None
    for f in ("tip_count", "inner_count", "branch_count", "root_count", "root_clv_index"):
        getattr(L, "rdh_tree_" + f).argtypes = [vp]
        getattr(L, "rdh_tree_" + f).restype = C.c_uint
    for f in ("root_scaler_index", "rooted", "sanity_check", "unroot"):
        getattr(L, "rdh_tree_" + f).argtypes = [vp]
        getattr(L, "rdh_tree_" + f).restype = C.c_int
    L.rdh_tree_root_info.argtypes = [vp, C.c_uint, _dp, C.POINTER(C.c_int), C.c_char_p, C.c_uint]
    L.rdh_tree_root_id_by_label.argtypes = [vp, C.c_char_p]
    L.rdh_tree_tip_index.argtypes = [vp, C.c_char_p]
    L.rdh_tree_tip_label.argtypes = [vp, C.c_uint, C.c_char_p, C.c_uint]
    sig = [vp, C.c_uint, C.c_double, C.POINTER(Operation), C.c_uint, _up, _up, _dp, C.c_uint, _up]
    L.rdh_tree_generate_operations.argtypes = sig
    L.rdh_tree_generate_root_update_operations.argtypes = sig
    L.rdh_tree_generate_derivative_operations.argtypes = [vp, C.c_uint, C.c_double, C.POINTER(Operation), _up, _dp]
    L.rdh_tree_root_by.argtypes = [vp, C.c_uint, C.c_double]
    L.rdh_tree_sweep_depth_bound.argtypes = [vp]
    L.rdh_tree_sweep_depth_bound.restype = C.c_uint
    L.rdh_tree_generate_sweep_operations.argtypes = [vp, C.c_uint, C.c_uint, C.c_uint, C.c_int, C.c_uint, C.c_uint,
                                                     _up, _up, _up, _up, C.c_uint, _up, _dp, C.c_uint,
                                                     C.POINTER(Operation), C.c_uint]
    L.rdh_tree_newick.argtypes = [vp, C.c_int]
    L.rdh_tree_newick.restype = vp
    L.rdh_free.argtypes = [vp]
    L.rdh_free.restype = None
    L.rdh_tree_annotate_branch.argtypes = [vp, C.c_uint, C.c_char_p, C.c_char_p]
    L.rdh_tree_annotate_lwr.argtypes = [vp, C.c_uint, C.c_double, C.c_double, C.c_double]
    L.rdh_tree_rank_roots.argtypes = [vp, C.c_int, _up, C.c_uint]
    if path == _build.LIBDIR / "librd_host.so":
        _host_lib = L
    return L


class RootedTree:
    """rooted_tree_t through the C wrappers (reference src/tree.hpp:54-201)."""

    def __init__(self, newick: str | None = None, *, path: str | None = None, lib: C.CDLL | None = None, _h=None):
        self.L = lib or load_tree_lib()
        if _h is not None:
            self.h = _h
        elif newick is not None:
            self.h = self.L.rdh_tree_from_newick(newick.encode())
        else:
            self.h = self.L.rdh_tree_from_file(str(path).encode())
        if not self.h:
            raise ValueError("tree could not be parsed: " + self.L.rdh_last_error().decode())
        self.h = C.c_void_p(self.h)
        n = self.tip_count
        self._cap = 2 * n + 2
        self._ops = (Operation * self._cap)()
        self._pm = (C.c_uint * self._cap)()
        self._br = (C.c_double * self._cap)()

    def close(self):
        if getattr(self, "h", None):
            self.L.rdh_tree_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def copy(self) -> "RootedTree":
        h = self.L.rdh_tree_copy(self.h)
        if not h:
            raise RuntimeError(self.L.rdh_last_error().decode())
        return RootedTree(lib=self.L, _h=h)

    tip_count = property(lambda s: s.L.rdh_tree_tip_count(s.h))
    inner_count = property(lambda s: s.L.rdh_tree_inner_count(s.h))
    branch_count = property(lambda s: s.L.rdh_tree_branch_count(s.h))
    root_count = property(lambda s: s.L.rdh_tree_root_count(s.h))
    root_clv_index = property(lambda s: s.L.rdh_tree_root_clv_index(s.h))
    root_scaler_index = property(lambda s: s.L.rdh_tree_root_scaler_index(s.h))
    rooted = property(lambda s: bool(s.L.rdh_tree_rooted(s.h)))

    def sanity_check(self) -> bool:
        return bool(self.L.rdh_tree_sanity_check(self.h))

    def root_info(self, rid: int):
        br = C.c_double()
        internal = C.c_int()
        label = C.create_string_buffer(256)
        if not self.L.rdh_tree_root_info(self.h, rid, C.byref(br), C.byref(internal), label, 256):
            raise IndexError(self.L.rdh_last_error().decode())
        return br.value, bool(internal.value), label.value.decode()

    def root_id(self, label: str) -> int:
        r = self.L.rdh_tree_root_id_by_label(self.h, label.encode())
        if r < 0:
            raise KeyError(label)
        return r

    def tip_index(self, label: str) -> int:
        return self.L.rdh_tree_tip_index(self.h, label.encode())

    def tip_label(self, index: int) -> str:
        buf = C.create_string_buffer(256)
        if not self.L.rdh_tree_tip_label(self.h, index, buf, 256):
            raise IndexError(index)
        return buf.value.decode()

    def _bundle(self, fn, rid, ratio):
        no, npm = C.c_uint(), C.c_uint()
        if not fn(self.h, rid, ratio, self._ops, self._cap, C.byref(no), self._pm, self._br, self._cap, C.byref(npm)):
            raise RuntimeError(self.L.rdh_last_error().decode())
        ops = [Operation(*self._ops[i].astuple()) for i in range(no.value)]
        pm = np.array(self._pm[: npm.value], dtype=np.uint32)
        br = np.array(self._br[: npm.value], dtype=np.float64)
        return ops, pm, br

    def generate_operations(self, rid: int, ratio: float = 0.5):
        return self._bundle(self.L.rdh_tree_generate_operations, rid, ratio)

    def generate_root_update_operations(self, rid: int, ratio: float = 0.5):
        return self._bundle(self.L.rdh_tree_generate_root_update_operations, rid, ratio)

    def generate_derivative_operations(self, rid: int, ratio: float = 0.5):
        op = Operation()
        pm = (C.c_uint * 2)()
        br = (C.c_double * 2)()
        if not self.L.rdh_tree_generate_derivative_operations(self.h, rid, ratio, C.byref(op), pm, br):
            raise RuntimeError(self.L.rdh_last_error().decode())
        return op, np.array(pm[:], dtype=np.uint32), np.array(br[:], dtype=np.float64)

    sweep_depth_bound = property(lambda s: s.L.rdh_tree_sweep_depth_bound(s.h))

    def sweep_layout(self, chunks: int = 1):
        """buffer counts and first spare indices of a partition that can run the directed sweep in
        `chunks` independent chunks: dict(clv_buffers, scale_buffers, prob_matrices, clv0, scaler0, pm0,
        extra, chunks)"""
        n, br, extra = self.tip_count, self.branch_count, self.sweep_depth_bound
        return dict(clv_buffers=br + chunks * extra, scale_buffers=br + chunks * extra, prob_matrices=br + 3,
                    clv0=n + br, scaler0=br, pm0=br, extra=extra, chunks=chunks)

    def generate_chunked_sweep_operations(self, begin: int | None = None, end: int | None = None, layout=None):
        """the directed sweep of root positions [begin, end) cut into layout["chunks"] independent chunks,
        each on its own spare buffers (model_t::sweep_root_lh does the same).  Returns
        (pm_off, mi, bl, op_off, ops, root_pos, chunk_offsets): the arguments of
        Partition.sweep_root_placements(..., chunk_offsets=...)."""
        lay = layout or self.sweep_layout()
        begin = 0 if begin is None else begin
        end = self.root_count if end is None else end
        total = end - begin
        chunks = max(1, min(lay.get("chunks", 1), total // 8))
        pm_off, op_off, mi, bl, ops, pos, coff = [0], [0], [], [], [], [], [0]
        for c in range(chunks):
            b0, b1 = begin + total * c // chunks, begin + total * (c + 1) // chunks
            sub = dict(lay, clv0=lay["clv0"] + c * lay["extra"], scaler0=lay["scaler0"] + c * lay["extra"])
            p_off, p_mi, p_bl, o_off, p_ops, p_pos = self.generate_sweep_operations(b0, b1, layout=sub)
            pm_off += [len(mi) + int(x) for x in p_off[1:]]
            op_off += [len(ops) + int(x) for x in o_off[1:]]
            mi += p_mi.tolist()
            bl += p_bl.tolist()
            ops += p_ops
            pos += p_pos.tolist()
            coff.append(len(pos))
        return (np.array(pm_off, dtype=np.uint32), np.array(mi, dtype=np.uint32), np.array(bl, dtype=np.float64),
                np.array(op_off, dtype=np.uint32), ops, np.array(pos, dtype=np.int64), np.array(coff, dtype=np.uint32))

    def generate_sweep_operations(self, begin: int | None = None, end: int | None = None, layout=None):
        """rooted_tree_t::generate_sweep_operations from the CURRENT root: the directed-CLV sweep of
        root positions [begin, end).  Returns (pm_off, mi, bl, op_off, ops, root_pos): the arguments of
        Partition.sweep_root_placements + the root position each placement scores."""
        lay = layout or self.sweep_layout()
        nroots = self.root_count
        begin = 0 if begin is None else begin
        end = nroots if end is None else end
        pcap = nroots + 1
        cap = 8 * self.tip_count + 16
        pm_off, op_off, pos = (C.c_uint * pcap)(), (C.c_uint * pcap)(), (C.c_uint * pcap)()
        pm, br, ops = (C.c_uint * cap)(), (C.c_double * cap)(), (Operation * cap)()
        npl = C.c_uint()
        if not self.L.rdh_tree_generate_sweep_operations(self.h, begin, end, lay["clv0"], lay["scaler0"], lay["pm0"],
                                                         lay["extra"], C.byref(npl), pm_off, op_off, pos, nroots,
                                                         pm, br, cap, ops, cap):
            raise RuntimeError(self.L.rdh_last_error().decode())
        q = npl.value
        npm, nops = pm_off[q], op_off[q]
        return (np.array(pm_off[: q + 1], dtype=np.uint32), np.array(pm[:npm], dtype=np.uint32),
                np.array(br[:npm], dtype=np.float64), np.array(op_off[: q + 1], dtype=np.uint32),
                [Operation(*ops[i].astuple()) for i in range(nops)], np.array(pos[:q], dtype=np.int64))

    def root_by(self, rid: int, ratio: float = 0.5):
        if not self.L.rdh_tree_root_by(self.h, rid, ratio):
            raise RuntimeError(self.L.rdh_last_error().decode())

    def unroot(self):
        if not self.L.rdh_tree_unroot(self.h):
            raise RuntimeError(self.L.rdh_last_error().decode())

    def newick(self, annotations: bool = True) -> str:
        p = self.L.rdh_tree_newick(self.h, 1 if annotations else 0)
        if not p:
            raise RuntimeError(self.L.rdh_last_error().decode())
        s = C.string_at(p).decode()
        self.L.rdh_free(p)
        return s

    def annotate_branch(self, rid: int, key: str, value: str):
        self.L.rdh_tree_annotate_branch(self.h, rid, key.encode(), value.encode())

    def annotate_lwr(self, rid: int, ratio: float, lwr: float, llh: float):
        self.L.rdh_tree_annotate_lwr(self.h, rid, ratio, lwr, llh)

    def rank_roots(self, which: str = "modified_mad"):
        n = self.root_count
        ids = (C.c_uint * n)()
        if not self.L.rdh_tree_rank_roots(self.h, 0 if which == "midpoint" else 1, ids, n):
            raise RuntimeError(self.L.rdh_last_error().decode())
        return list(ids)


# ---------------------------------------------------------------------------
# model_t mirror (host C++) through the C wrappers
# ---------------------------------------------------------------------------
# the optimiser components of host/optim.hpp, driven alone (host/optim_capi.cpp)
# ---------------------------------------------------------------------------
_SLOPE_FN = C.CFUNCTYPE(None, C.c_double, _dp, _dp, C.c_void_p)
_OBJECTIVE_FN = C.CFUNCTYPE(C.c_double, _dp, C.c_int, C.c_void_p)


def slope_root(fn, lo: float, hi: float, x_tolerance: float = 1e-12, lib: C.CDLL | None = None):
    """rd::slope_root_brent: the root of the slope of `fn` between lo and hi, where fn(x) ->
    (value, slope) and the slopes at lo and hi have opposite signs (model_t::optimize_alpha's
    bracketing search, reference src/model.cpp:606-676).  Returns (x, value, slope, probes)."""
    L = lib or load_tree_lib()
    L.rdh_optim_slope_root.argtypes = [_SLOPE_FN, C.c_void_p, C.c_double, C.c_double, C.c_double, _dp, _up]

    def thunk(x, value, slope, _user):
        v, s = fn(x)
        value[0], slope[0] = v, s

    out = (C.c_double * 3)()
    probes = C.c_uint(0)
    if not L.rdh_optim_slope_root(_SLOPE_FN(thunk), None, lo, hi, x_tolerance, out, C.byref(probes)):
        raise RuntimeError(L.rdh_last_error().decode())
    return out[0], out[1], out[2], probes.value


_BATCH_FN = C.CFUNCTYPE(None, _dp, C.c_int, _dp, C.c_void_p)


def _batch_thunk(fn, log):
    def thunk(xs, n, out, _user):
        batch = [xs[i] for i in range(n)]
        log.append(batch)
        for i, x in enumerate(batch):
            out[i] = fn(x)
    return _BATCH_FN(thunk)


def argmax_on_segment(fn, x_now: float, atol: float, look_ahead: bool = True, lib: C.CDLL | None = None):
    """rd::unit_segment_search_t::argmax: the best position on [0, 1] by the sign of the slope of
    `fn` (model_t::optimize_alpha without the tree, reference src/model.cpp:679-794), evaluations
    handed over in batches (look_ahead) or one slope at a time.  Returns (x, [batches of abscissae])."""
    L = lib or load_tree_lib()
    L.rdh_optim_argmax_on_segment.argtypes = [_BATCH_FN, C.c_void_p, C.c_double, C.c_double, C.c_int, _dp, _up]
    log = []
    best = C.c_double(0.0)
    if not L.rdh_optim_argmax_on_segment(_batch_thunk(fn, log), None, x_now, atol, 1 if look_ahead else 0,
                                         C.byref(best), None):
        raise RuntimeError(L.rdh_last_error().decode())
    return best.value, log


def slope_on_segment(fn, x: float, lib: C.CDLL | None = None):
    """the forward-difference slope model_t::compute_dlh takes (src/model.cpp:481-519) -> (value, slope)"""
    L = lib or load_tree_lib()
    L.rdh_optim_slope_on_segment.argtypes = [_BATCH_FN, C.c_void_p, C.c_double, _dp]
    out = (C.c_double * 2)()
    if not L.rdh_optim_slope_on_segment(_batch_thunk(fn, []), None, x, out):
        raise RuntimeError(L.rdh_last_error().decode())
    return out[0], out[1]


def minimize_in_box(fn, x0, lower: float, upper: float, pgtol: float = 1e-7, factr: float = 1e4,
                    lib: C.CDLL | None = None):
    """rd::minimize_in_box: L-BFGS-B with forward-difference gradients inside [lower, upper]^n
    (model_t::optimize_params, reference src/model.cpp:1430-1522).  Returns (x, f_end, evaluations);
    x is the final point when it is not worse than x0, else x0."""
    L = lib or load_tree_lib()
    L.rdh_optim_minimize_in_box.argtypes = [_OBJECTIVE_FN, C.c_void_p, _dp, C.c_int, C.c_double, C.c_double,
                                            C.c_double, C.c_double, _dp, _up]
    x = np.array(x0, dtype=np.float64)

    def thunk(ptr, n, _user):
        return float(fn(np.ctypeslib.as_array(ptr, shape=(n,)).copy()))

    f_end = C.c_double(0.0)
    calls = C.c_uint(0)
    if not L.rdh_optim_minimize_in_box(_OBJECTIVE_FN(thunk), None, _ptr(x, _dp), len(x), lower, upper, pgtol,
                                       factr, C.byref(f_end), C.byref(calls)):
        raise RuntimeError(L.rdh_last_error().decode())
    return x, f_end.value, calls.value


# ---------------------------------------------------------------------------
def _bind_model(L: C.CDLL):
    if getattr(L, "_rdh_model_bound", False):
        return
    vp = C.c_void_p
    ull = C.c_ulonglong
    L.rdh_model_create.restype = vp
    L.rdh_model_create.argtypes = [vp, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.c_int, C.c_uint,
                                   C.c_int, ull, C.c_int, C.c_int, C.POINTER(ull), C.POINTER(ull), ull, ull,
                                   C.c_int, C.c_int, vp]
    L.rdh_model_destroy.argtypes = [vp]
    L.rdh_model_destroy.restype = None
    L.rdh_model_create_from_files.restype = vp
    L.rdh_model_create_from_files.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_uint, C.c_int, ull, C.c_int]
    L.rdh_model_partition_count.argtypes = [vp]
    L.rdh_model_partition_count.restype = C.c_uint
    L.rdh_partition_describe.argtypes = [C.c_char_p]
    L.rdh_partition_describe.restype = vp
    L.rdh_msa_partition_lengths.argtypes = [C.c_char_p, C.c_char_p, C.c_int, _up, C.c_uint]
    L.rdh_model_sites.argtypes = [vp, C.c_uint]
    L.rdh_model_sites.restype = C.c_uint
    L.rdh_model_root_count.argtypes = [vp]
    L.rdh_model_root_count.restype = C.c_uint
    L.rdh_model_initialize_partitions.argtypes = [vp, C.c_int]
    L.rdh_model_set_fused.argtypes = [vp, C.c_int]
    L.rdh_model_set_sweep_mode.argtypes = [vp, C.c_int]
    L.rdh_model_set_batched_probes.argtypes = [vp, C.c_int]
    L.rdh_model_batched_probes.argtypes = [vp]
    L.rdh_model_set_params.argtypes = [vp, C.c_uint, _dp, _dp, _dp]
    L.rdh_model_compute_lh.argtypes = [vp, C.c_uint, C.c_double, _dp]
    L.rdh_model_compute_lh_root.argtypes = [vp, C.c_uint, C.c_double, _dp]
    L.rdh_model_compute_dlh.argtypes = [vp, C.c_uint, C.c_double, _dp, _dp]
    L.rdh_model_move_root.argtypes = [vp, C.c_uint, C.c_double]
    L.rdh_model_optimize_alpha.argtypes = [vp, C.c_uint, C.c_double, C.c_double, _dp]
    L.rdh_model_optimize_root_location.argtypes = [vp, C.c_uint, C.c_double, _up, _dp, _dp]
    L.rdh_model_sweep_root_lh.argtypes = [vp, _dp]
    L.rdh_model_sweep_root_lh_range.argtypes = [vp, C.c_uint, C.c_uint, _dp]
    L.rdh_model_compute_all_root_lh.argtypes = [vp, _dp]
    L.rdh_model_search.argtypes = [vp, C.c_uint, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                   C.c_int, C.c_uint, C.c_uint, _up, _dp, _dp]
    L.rdh_model_exhaustive_search.argtypes = [vp, C.c_double, C.c_double, C.c_double, C.c_double, C.c_uint,
                                              C.c_uint, _up, _dp, _dp, C.c_uint, _up]
    L.rdh_model_lwr.argtypes = [_dp, C.c_uint, _dp]
    L.rdh_model_newick.argtypes = [vp, C.c_int]
    L.rdh_model_newick.restype = vp
    L.rdh_model_get_params.argtypes = [vp, C.c_uint, _dp, _dp, _dp]
    L.rdh_model_partition.argtypes = [vp, C.c_uint]
    L.rdh_model_partition.restype = vp
    L.rdh_model_set_checkpoint.argtypes = [vp, C.c_char_p]
    L.rdh_model_sweep_chunks.argtypes = [vp]
    L.rdh_model_sweep_chunks.restype = C.c_uint
    L.rdh_model_set_max_outer_iterations.argtypes = [vp, C.c_uint]
    L.rdh_model_set_max_outer_iterations.restype = None
    L.rdh_model_last_partition_lh.argtypes = [vp, _dp, C.c_uint]
    L.rdh_model_last_sweep_partition_lh.argtypes = [vp, C.c_uint, _dp, C.c_uint]
    L.rdh_model_placement_support.argtypes = [vp, C.c_char_p, ull, ull, C.c_uint, C.c_int, C.c_uint, C.POINTER(ull),
                                              _dp, _dp, _dp, C.POINTER(ull), C.POINTER(C.c_longlong), _up, _up, _up,
                                              C.POINTER(C.c_int), _up, _dp, _up]
    L.rdh_model_placement_support_au.argtypes = [vp, C.c_char_p, ull, ull, C.c_uint, C.c_int, C.c_uint, _up,
                                                 C.c_uint, C.POINTER(ull), _dp, _dp, _dp, C.POINTER(ull),
                                                 C.POINTER(C.c_longlong), _up, _up, _up, _up, _dp, _dp, _dp, _dp,
                                                 _up, _dp, C.POINTER(ull), C.POINTER(C.c_int), _up, _dp, _up]
    L.rdh_model_branch_support.argtypes = [vp, C.c_char_p, ull, ull, C.c_double, C.c_uint, C.c_int, C.c_uint, _up,
                                           C.c_uint, C.POINTER(ull), _dp, _dp, _dp, C.POINTER(ull),
                                           C.POINTER(C.c_longlong), _up, _up, _up, _up, _dp, _dp, _dp, _dp, _up, _dp,
                                           C.POINTER(ull), C.POINTER(C.c_int), _up, _dp, _up]
    gene_outputs = [_dp, C.POINTER(ull), C.POINTER(C.c_longlong), _up, C.POINTER(C.c_int), _up, _dp, _up]
    L.rdh_model_placement_support_genes.argtypes = [vp, C.c_char_p, ull, ull, C.c_uint, C.c_int, C.c_uint, C.c_uint,
                                                    C.POINTER(ull), _dp, _dp, _dp, C.POINTER(ull),
                                                    C.POINTER(C.c_longlong), _up, _up, _up] + gene_outputs
    L.rdh_model_branch_support_genes.argtypes = [vp, C.c_char_p, ull, ull, C.c_double, C.c_uint, C.c_int, C.c_uint,
                                                 C.c_uint, C.POINTER(ull), _dp, _dp, _dp, C.POINTER(ull),
                                                 C.POINTER(C.c_longlong), _up, _up, _up] + gene_outputs
    L.rdh_placement_au_fit.argtypes = [_up, C.c_uint, _up, ull, _dp, _up]
    L.rdh_model_site_lnl_rows.argtypes = [vp, C.c_uint, _dp, ull, _up, C.c_uint, C.POINTER(ull)]
    L.rdh_model_assign_indicies.argtypes = [vp, C.c_int, C.c_uint, C.c_double, C.c_uint, C.c_uint, C.c_int, _up,
                                            C.c_uint, _up]
    L.rdh_model_ancestral_states.argtypes = [vp, C.c_uint, C.c_double, C.c_char_p, C.c_int, C.c_uint, _up, C.c_uint,
                                             C.c_uint, _up, _up]
    L.rdh_model_ancestral_nodes.argtypes = [vp, C.c_uint, C.c_uint, _up, C.POINTER(C.c_int), _up, C.POINTER(ull), _dp,
                                            C.POINTER(C.c_int)]
    L.rdh_model_ancestral_clade.argtypes = [vp, C.c_uint]
    L.rdh_model_ancestral_clade.restype = vp
    L.rdh_model_ancestral_partition.argtypes = [vp, C.c_uint, ull, ull, C.POINTER(C.c_ubyte), _dp, _dp, _dp, _dp]
    L.rdh_model_pattern_of_column.argtypes = [vp, C.c_uint, _up, C.c_uint, _up]
    L._rdh_model_bound = True


def _bind_checkpoint(L: C.CDLL):
    if getattr(L, "_rdh_ckp_bound", False):
        return
    vp, ull = C.c_void_p, C.c_ulonglong
    ullp = C.POINTER(ull)
    opts = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, ullp, C.c_uint, ull, ull, ull, C.c_int, C.c_int, C.c_int]
    L.rdh_ckp_open.restype = vp
    L.rdh_ckp_open.argtypes = [C.c_char_p]
    L.rdh_ckp_close.argtypes = [vp]
    L.rdh_ckp_close.restype = None
    L.rdh_ckp_existing.argtypes = [vp]
    L.rdh_ckp_filename.argtypes = [vp, C.c_char_p, C.c_uint]
    L.rdh_ckp_save_options.argtypes = [vp] + opts
    L.rdh_ckp_load_options.argtypes = [vp] + opts + [C.c_char_p, C.c_uint, ullp, _up]
    L.rdh_ckp_write.argtypes = [vp, ull, C.c_double, C.c_double, C.c_uint, _dp, _dp, _dp, _dp, C.c_uint]
    L.rdh_ckp_read.argtypes = [vp, C.c_uint, ullp, _dp, _dp, _up, _up]
    L.rdh_ckp_read_params.argtypes = [vp, C.c_uint, C.c_uint, _dp, _dp, _dp, _dp, C.c_uint]
    L.rdh_ckp_completed.argtypes = [vp, C.c_uint, ullp, _up]
    L.rdh_ckp_needs_cleaning.argtypes = [vp]
    L.rdh_ckp_clean.argtypes = [vp]
    L.rdh_ckp_checksum_result.argtypes = [ull, C.c_double, C.c_double]
    L.rdh_ckp_checksum_result.restype = C.c_uint
    L.rdh_ckp_checksum_params.argtypes = [C.c_uint, _dp, _dp, _dp, _dp, C.c_uint]
    L.rdh_ckp_checksum_params.restype = C.c_uint
    L._rdh_ckp_bound = True


class Checkpoint:
    """checkpoint_t (reference src/checkpoint.hpp:251-301): the "<prefix>.ckp" result log in the
    reference's on-disk format (prefix=None: the in-memory log)."""

    OPTION_DEFAULTS = dict(msa="", tree="", prefix="", model_string="", rate_cats=(1,), seed=0, min_roots=1,
                           threads=0, exhaustive=False, early_stop=0, strategy=2)

    def __init__(self, prefix: str | None, lib: C.CDLL | None = None):
        self.L = lib or load_tree_lib()
        _bind_checkpoint(self.L)
        self.h = self.L.rdh_ckp_open(prefix.encode() if prefix is not None else None)
        if not self.h:
            raise RuntimeError("checkpoint_t could not be opened: " + self.L.rdh_last_error().decode())
        self.h = C.c_void_p(self.h)

    def close(self):
        if getattr(self, "h", None):
            self.L.rdh_ckp_close(self.h)
            self.h = None

    __del__ = close

    def _check(self, rc):
        if rc == 0:
            raise RuntimeError(self.L.rdh_last_error().decode())
        return rc

    @property
    def existing(self) -> bool:
        return bool(self.L.rdh_ckp_existing(self.h))

    @property
    def filename(self) -> str:
        buf = C.create_string_buffer(4096)
        self._check(self.L.rdh_ckp_filename(self.h, buf, 4096))
        return buf.value.decode()

    def _opts(self, kw):
        o = dict(self.OPTION_DEFAULTS)
        o.update(kw)
        rc = (C.c_ulonglong * max(1, len(o["rate_cats"])))(*o["rate_cats"])
        return [o["msa"].encode(), o["tree"].encode(), o["prefix"].encode(), o["model_string"].encode(), rc,
                len(o["rate_cats"]), o["seed"], o["min_roots"], o["threads"], int(o["exhaustive"]),
                int(o["early_stop"]), int(o["strategy"])]

    def save_options(self, **kw):
        self._check(self.L.rdh_ckp_save_options(self.h, *self._opts(kw)))

    def load_options(self, **kw) -> dict:
        """stored options vs the given ones: {"equal": bool, "msa": str, "seed": int, "n_rate_cats": int}"""
        buf = C.create_string_buffer(4096)
        seed, nrc = C.c_ulonglong(), C.c_uint()
        rc = self._check(self.L.rdh_ckp_load_options(self.h, *self._opts(kw), buf, 4096, C.byref(seed), C.byref(nrc)))
        return {"equal": rc == 2, "msa": buf.value.decode(), "seed": seed.value, "n_rate_cats": nrc.value}

    @staticmethod
    def _flat(params, K):
        n = len(params)
        rates = np.ascontiguousarray([p["rates"] for p in params], dtype=np.float64).reshape(n, 12) if n else np.zeros((0, 12))
        freqs = np.ascontiguousarray([p["freqs"] for p in params], dtype=np.float64).reshape(n, 4) if n else np.zeros((0, 4))
        alpha = np.ascontiguousarray([p["alpha"] for p in params], dtype=np.float64).reshape(n) if n else np.zeros(0)
        w = np.ascontiguousarray([p["weights"] for p in params], dtype=np.float64).reshape(n, K) if n else np.zeros((0, K))
        return n, rates, freqs, alpha, w

    def write(self, root_id: int, llh: float, alpha: float, params=(), K: int = 4):
        n, r, f, a, w = self._flat(list(params), K)
        self._check(self.L.rdh_ckp_write(self.h, root_id, llh, alpha, n, _ptr(r, _dp), _ptr(f, _dp), _ptr(a, _dp),
                                         _ptr(w, _dp), K))

    def read_results(self):
        cap = 1 << 16
        ids = np.zeros(cap, dtype=np.uint64)
        llh, alpha = np.zeros(cap), np.zeros(cap)
        nparts = np.zeros(cap, dtype=np.uint32)
        got = C.c_uint()
        self._check(self.L.rdh_ckp_read(self.h, cap, _ptr(ids, C.POINTER(C.c_ulonglong)), _ptr(llh, _dp),
                                        _ptr(alpha, _dp), _ptr(nparts, _up), C.byref(got)))
        k = min(got.value, cap)
        return [(int(ids[i]), float(llh[i]), float(alpha[i]), int(nparts[i])) for i in range(k)]

    def read_params(self, index: int, part: int = 0, K: int = 4) -> dict:
        r, f, w = np.zeros(12), np.zeros(4), np.zeros(K)
        a = C.c_double()
        self._check(self.L.rdh_ckp_read_params(self.h, index, part, _ptr(r, _dp), _ptr(f, _dp), C.byref(a),
                                               _ptr(w, _dp), K))
        return {"rates": r, "freqs": f, "alpha": a.value, "weights": w}

    def completed_indicies(self):
        cap = 1 << 16
        ids = np.zeros(cap, dtype=np.uint64)
        got = C.c_uint()
        self._check(self.L.rdh_ckp_completed(self.h, cap, _ptr(ids, C.POINTER(C.c_ulonglong)), C.byref(got)))
        return [int(x) for x in ids[:min(got.value, cap)]]

    def needs_cleaning(self) -> bool:
        rc = self.L.rdh_ckp_needs_cleaning(self.h)
        if rc < 0:
            raise RuntimeError(self.L.rdh_last_error().decode())
        return rc == 1

    def clean(self):
        self._check(self.L.rdh_ckp_clean(self.h))

    def checksum_result(self, root_id, llh, alpha) -> int:
        return self.L.rdh_ckp_checksum_result(root_id, llh, alpha)

    def checksum_params(self, params, K: int = 4) -> int:
        n, r, f, a, w = self._flat(list(params), K)
        return self.L.rdh_ckp_checksum_params(n, _ptr(r, _dp), _ptr(f, _dp), _ptr(a, _dp), _ptr(w, _dp), K)


def parse_partitions(text: str, lib: C.CDLL | None = None) -> list:
    """RAxML-NG partition-file text -> list of dicts (host/partition_file.cpp; reference
    parse_partition_info / parse_model_info, src/msa.cpp:364-493).  Raises ValueError when the
    text does not parse."""
    L = lib or load_tree_lib()
    _bind_model(L)
    r = L.rdh_partition_describe(text.encode())
    if not r:
        raise ValueError(L.rdh_last_error().decode())
    out = []
    try:
        for line in C.string_at(r).decode().splitlines():
            f = line.split("|")
            out.append({"model_name": f[0], "partition_name": f[1],
                        "parts": [tuple(int(x) for x in rg.split("-")) for rg in f[2].split(",")],
                        "subst": f[3], "freq": f[4], "invar_present": f[5] == "1", "invar": f[6],
                        "invar_prop": float(f[7]), "ratehet": f[8], "cat_type": f[9], "rate_cats": int(f[10]),
                        "alpha_init": f[11] == "1", "alpha": float(f[12]), "asc": f[13]})
    finally:
        L.rdh_free(C.c_void_p(r))
    return out


def msa_partition_lengths(msa_path: str, partition_text: str, compress_first: bool = True,
                          lib: C.CDLL | None = None) -> list:
    """pattern counts of msa_t::partition() on an alignment file (reference test/src/msa.cpp:236-283)"""
    L = lib or load_tree_lib()
    _bind_model(L)
    out = (C.c_uint * 64)()
    rc = L.rdh_msa_partition_lengths(str(msa_path).encode(), partition_text.encode(), 1 if compress_first else 0,
                                     out, 64)
    if not rc:
        raise ValueError(L.rdh_last_error().decode())
    return [int(out[i]) for i in range(rc - 1)]


def write_state_file(result: dict, path, fasta_path=None) -> None:
    """Write the result of Model.ancestral_states as IQ-TREE's .state table, one line per node with a
    full posterior (in the order of result["full"]) and alignment column: the node ("Node<CLV index>"),
    the site, the MAP state and the posterior of A, C, G, T (5 decimals).  With one partition the header
    is "Node Site State p_A p_C p_G p_T" and Site is the alignment column, from 1.  With several
    partitions a "Part" column (the partition, from 1) follows Node, as in IQ-TREE's partitioned output,
    and Site counts from 1 within the partition, over its columns in the order of its ranges (a
    partition "1-100, 301-400" has sites 1-200; site 101 is alignment column 301).  Fields are
    tab-separated.  Also writes the root's MAP sequence as FASTA (">root", 60 columns per line, the
    partitions' columns in the same order) to fasta_path (default: path with the suffix .fasta)."""
    path = Path(path)
    nodes, full = result["nodes"], result["full"]
    parts = result["pattern_of_column"]
    several = len(parts) > 1
    lines = ["Node\tPart\tSite\tState\tp_A\tp_C\tp_G\tp_T" if several else "Node\tSite\tState\tp_A\tp_C\tp_G\tp_T"]
    for f, node in enumerate(full.tolist()):
        name = "Node%d" % nodes[node]
        for part, cols in enumerate(parts):
            post = result["posterior"][part][f]
            state = result["map_state"][part][node]
            lead = "%s\t%d\t" % (name, part + 1) if several else name + "\t"
            for site, p in enumerate(cols.tolist(), start=1):
                q = post[p]
                lines.append("%s%d\t%s\t%.5f\t%.5f\t%.5f\t%.5f" % (lead, site, chr(state[p]), q[0], q[1], q[2], q[3]))
    root = len(nodes) - 1
    seq = "".join(bytes(result["map_state"][part][root][cols]).decode() for part, cols in enumerate(parts))
    path.write_text("\n".join(lines) + "\n")
    fasta = Path(fasta_path) if fasta_path is not None else path.with_suffix(".fasta")
    fasta.write_text(">root\n" + "".join(seq[i:i + 60] + "\n" for i in range(0, len(seq), 60)))


class Model:
    """model_t (reference src/model.hpp:46-277) on the engine the host library was linked against."""

    STRATEGY = {"random": 0, "midpoint": 1, "modified_mad": 2}

    def __init__(self, tree: RootedTree, alignment: dict, rate_cats: int = 4, *, compress: bool = False,
                 invariant_sites: bool = False, seed: int = 1, early_stop: bool = False, partitions=None,
                 site_offset: int = 0, global_sites: int = 0, nranks: int = 1, rank: int = 0,
                 comm_id: bytes | None = None):
        self.L = tree.L
        _bind_model(self.L)
        labels = list(alignment)
        n = len(labels)
        la = (C.c_char_p * n)(*[l.encode() for l in labels])
        sa = (C.c_char_p * n)(*[alignment[l] if isinstance(alignment[l], bytes) else alignment[l].encode()
                                for l in labels])
        nparts = 0 if not partitions else len(partitions)
        pb = (C.c_ulonglong * max(1, nparts))(*([p[0] for p in partitions] if partitions else [0]))
        pe = (C.c_ulonglong * max(1, nparts))(*([p[1] for p in partitions] if partitions else [0]))
        cid = C.create_string_buffer(comm_id, 128) if comm_id else None
        self.h = self.L.rdh_model_create(tree.h, n, la, sa, 1 if compress else 0, rate_cats,
                                         1 if invariant_sites else 0, seed, 1 if early_stop else 0, nparts, pb, pe,
                                         site_offset, global_sites, nranks, rank, cid)
        if not self.h:
            raise RuntimeError("model_t could not be created: " + self.L.rdh_last_error().decode())
        self.h = C.c_void_p(self.h)
        self.K = rate_cats
        self.root_count = self.L.rdh_model_root_count(self.h)

    @classmethod
    def from_files(cls, tree: RootedTree, msa_path, partition_path=None, rate_cats: int = 4, *,
                   invariant_sites: bool = False, seed: int = 1, early_stop: bool = False) -> "Model":
        """the reference's ingest path (src/main.cpp:513-560): PHYLIP/FASTA alignment + optional
        RAxML-NG partition file (rate categories then come from the partition file)"""
        self = cls.__new__(cls)
        self.L = tree.L
        _bind_model(self.L)
        h = self.L.rdh_model_create_from_files(tree.h, str(msa_path).encode(),
                                               str(partition_path).encode() if partition_path else None,
                                               rate_cats, 1 if invariant_sites else 0, seed, 1 if early_stop else 0)
        if not h:
            raise RuntimeError("model_t could not be created: " + self.L.rdh_last_error().decode())
        self.h = C.c_void_p(h)
        self.K = rate_cats
        self.root_count = self.L.rdh_model_root_count(self.h)
        return self

    @property
    def partition_count(self) -> int:
        return int(self.L.rdh_model_partition_count(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.L.rdh_model_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if not rc:
            raise RuntimeError(self.L.rdh_last_error().decode())

    def sites(self, part: int = 0) -> int:
        return self.L.rdh_model_sites(self.h, part)

    def initialize_partitions(self, uniform_freqs: bool = False):
        self._check(self.L.rdh_model_initialize_partitions(self.h, 1 if uniform_freqs else 0))

    def set_fused(self, on: bool):
        self.L.rdh_model_set_fused(self.h, 1 if on else 0)

    def set_batched_probes(self, on: bool):
        """root-only evaluations of compute_dlh / optimize_alpha go to the engine as one fused batch
        (default; RD_BATCHED_PROBES=0 in the environment turns it off) or one call each, as the
        reference issues them (src/model.cpp:481-519, 679-794).  Same values either way."""
        self.L.rdh_model_set_batched_probes(self.h, 1 if on else 0)

    @property
    def batched_probes(self) -> bool:
        return bool(self.L.rdh_model_batched_probes(self.h))

    def probe_counters(self) -> dict:
        """root-only evaluations so far: fused batches, evaluations inside them, evaluations issued singly"""
        out = (C.c_ulonglong * 3)()
        self.L.rdh_model_probe_counters.argtypes = [C.c_void_p, C.POINTER(C.c_ulonglong)]
        self.L.rdh_model_probe_counters.restype = None
        self.L.rdh_model_probe_counters(self.h, out)
        return {"fused_batches": int(out[0]), "fused_evaluations": int(out[1]), "single_evaluations": int(out[2])}

    SWEEP_SEQUENTIAL, SWEEP_PATH, SWEEP_DIRECTED = 0, 1, 2

    def set_sweep_mode(self, mode: int):
        """how sweep_root_lh scores the placements (identical values): 0 the reference's
        move_root + compute_lh_root loop, 1 the same operations in one engine call, 2 (default)
        one pre-order pass over directed CLVs"""
        self._check(self.L.rdh_model_set_sweep_mode(self.h, mode))

    def set_params(self, rates=None, freqs=None, alpha=None, part: int = 0):
        r = np.ascontiguousarray(rates, dtype=np.float64) if rates is not None else None
        f = np.ascontiguousarray(freqs, dtype=np.float64) if freqs is not None else None
        a = np.array([alpha], dtype=np.float64) if alpha is not None else None
        self._check(self.L.rdh_model_set_params(self.h, part, _ptr(r, _dp) if r is not None else None,
                                                _ptr(f, _dp) if f is not None else None,
                                                _ptr(a, _dp) if a is not None else None))

    def get_params(self, part: int = 0):
        r, f, c = np.zeros(12), np.zeros(4), np.zeros(self.K)
        self.L.rdh_model_get_params(self.h, part, _ptr(r, _dp), _ptr(f, _dp), _ptr(c, _dp))
        return r, f, c

    def compute_lh(self, rid: int, ratio: float = 0.5) -> float:
        out = C.c_double()
        self._check(self.L.rdh_model_compute_lh(self.h, rid, ratio, C.byref(out)))
        return out.value

    def compute_lh_root(self, rid: int, ratio: float = 0.5) -> float:
        out = C.c_double()
        self._check(self.L.rdh_model_compute_lh_root(self.h, rid, ratio, C.byref(out)))
        return out.value

    def compute_dlh(self, rid: int, ratio: float = 0.5):
        lh, dlh = C.c_double(), C.c_double()
        self._check(self.L.rdh_model_compute_dlh(self.h, rid, ratio, C.byref(lh), C.byref(dlh)))
        return lh.value, dlh.value

    def move_root(self, rid: int, ratio: float = 0.5):
        self._check(self.L.rdh_model_move_root(self.h, rid, ratio))

    def optimize_alpha(self, rid: int, ratio: float = 0.5, atol: float = 1e-7) -> float:
        out = C.c_double()
        self._check(self.L.rdh_model_optimize_alpha(self.h, rid, ratio, atol, C.byref(out)))
        return out.value

    def optimize_root_location(self, min_roots: int = 1, root_ratio: float = 0.05):
        rid, alpha, lh = C.c_uint(), C.c_double(), C.c_double()
        self._check(self.L.rdh_model_optimize_root_location(self.h, min_roots, root_ratio, C.byref(rid),
                                                            C.byref(alpha), C.byref(lh)))
        return rid.value, alpha.value, lh.value

    def sweep_root_lh(self, begin: int | None = None, end: int | None = None) -> np.ndarray:
        """log-likelihood of every root placement (root-id order); with begin/end only of the
        root ids [begin, end) -- one rank's share when the roots are distributed over GPUs"""
        if begin is None and end is None:
            out = np.zeros(self.root_count)
            self._check(self.L.rdh_model_sweep_root_lh(self.h, _ptr(out, _dp)))
            return out
        begin = 0 if begin is None else begin
        end = self.root_count if end is None else end
        out = np.zeros(max(0, end - begin))
        self._check(self.L.rdh_model_sweep_root_lh_range(self.h, begin, end, _ptr(out, _dp)))
        return out

    def compute_all_root_lh(self) -> np.ndarray:
        out = np.zeros(self.root_count)
        self._check(self.L.rdh_model_compute_all_root_lh(self.h, _ptr(out, _dp)))
        return out

    def search(self, min_roots=1, root_ratio=0.01, atol=1e-7, pgtol=1e-7, brtol=1e-12, factor=1e4,
               strategy="modified_mad", rank=0, num_tasks=1):
        rid, alpha, lh = C.c_uint(), C.c_double(), C.c_double()
        self._check(self.L.rdh_model_search(self.h, min_roots, root_ratio, atol, pgtol, brtol, factor,
                                            self.STRATEGY[strategy], rank, num_tasks, C.byref(rid), C.byref(alpha),
                                            C.byref(lh)))
        return rid.value, alpha.value, lh.value

    def exhaustive_search(self, atol=1e-7, pgtol=1e-7, brtol=1e-12, factor=1e4, rank=0, num_tasks=1):
        n = self.root_count
        ids = np.zeros(n, dtype=np.uint32)
        llh, alpha = np.zeros(n), np.zeros(n)
        got = C.c_uint()
        self._check(self.L.rdh_model_exhaustive_search(self.h, atol, pgtol, brtol, factor, rank, num_tasks,
                                                       _ptr(ids, _up), _ptr(llh, _dp), _ptr(alpha, _dp), n,
                                                       C.byref(got)))
        k = got.value
        return ids[:k].copy(), llh[:k].copy(), alpha[:k].copy()

    def set_checkpoint(self, prefix: str | None):
        """log search / exhaustive_search results to "<prefix>.ckp" (the reference's on-disk format);
        a file that already holds results makes the next run resume from it"""
        self._check(self.L.rdh_model_set_checkpoint(self.h, prefix.encode() if prefix is not None else None))

    def set_max_outer_iterations(self, n: int):
        """cap the outer iterations of search / exhaustive_search per root (0 = the reference's 1000)"""
        self.L.rdh_model_set_max_outer_iterations(self.h, int(n))

    @property
    def sweep_chunks(self) -> int:
        """independent chunks the directed sweep is cut into (the same on every rank of a site-sharded run)"""
        return int(self.L.rdh_model_sweep_chunks(self.h))

    def last_partition_lh(self) -> np.ndarray:
        """the per-partition terms of the last compute_lh / compute_lh_root, in partition order"""
        out = np.zeros(self.partition_count)
        self._check(self.L.rdh_model_last_partition_lh(self.h, _ptr(out, _dp), len(out)))
        return out

    def last_sweep_partition_lh(self, placements: int | None = None) -> np.ndarray:
        """[partition][placement] terms of the last sweep_root_lh"""
        n = self.root_count if placements is None else placements
        out = np.zeros((self.partition_count, n))
        for p in range(self.partition_count):
            row = np.zeros(n)
            self._check(self.L.rdh_model_last_sweep_partition_lh(self.h, p, _ptr(row, _dp), n))
            out[p] = row
        return out

    def assign_indicies(self, mode: str = "exhaustive", min_roots: int = 1, root_ratio: float = 0.0, rank: int = 0,
                        num_tasks: int = 1, strategy: str = "modified_mad"):
        """assign_indicies_by_rank_search / _exhaustive against the model's result log
        (reference src/model.cpp:1899-1960): the root ids this rank still has to do"""
        out = np.zeros(self.root_count, dtype=np.uint32)
        got = C.c_uint()
        self._check(self.L.rdh_model_assign_indicies(self.h, 0 if mode == "search" else 1, min_roots, root_ratio,
                                                     rank, num_tasks, self.STRATEGY[strategy], _ptr(out, _up),
                                                     len(out), C.byref(got)))
        return out[:got.value].tolist()

    SAMPLING = {"gene": 1, "gene_site": 2}

    def _gene_sampling(self, who, sampling, au_scales):
        """the C code of a gene mode, or None for site resampling"""
        if sampling == "site":
            return None
        if sampling not in self.SAMPLING:
            raise ValueError("%s: unknown sampling %r (site, gene or gene_site)" % (who, sampling))
        if au_scales is not None:
            raise ValueError("%s: the AU test and ELW (au_scales) are not available with gene sampling" % who)
        return self.SAMPLING[sampling]

    def _support_genes(self, call, cap, args, retry):
        """one gene-mode support entry (placement or branch) and its result dict"""
        G = self.partition_count
        ull = C.POINTER(C.c_ulonglong)
        for attempt in range(2):
            ids = np.zeros(cap, dtype=np.uint64)
            alpha, llh, fixed = np.zeros(cap), np.zeros(cap), np.zeros(cap)
            o_lo, o_hi = np.zeros(cap, dtype=np.uint64), np.zeros(cap, dtype=np.int64)
            bp, kh, sh = (np.zeros(cap, dtype=np.uint32) for _ in range(3))
            p_fixed = np.zeros((G, cap))
            p_lo, p_hi = np.zeros((G, cap), dtype=np.uint64), np.zeros((G, cap), dtype=np.int64)
            p_best = np.zeros(G, dtype=np.uint32)
            exponent, best, got = C.c_int(), C.c_uint(), C.c_uint()
            info = np.zeros(8)
            rc = call(*args, cap, _ptr(ids, ull), _ptr(alpha, _dp), _ptr(llh, _dp), _ptr(fixed, _dp), _ptr(o_lo, ull),
                      _ptr(o_hi, C.POINTER(C.c_longlong)), _ptr(bp, _up), _ptr(kh, _up), _ptr(sh, _up),
                      _ptr(p_fixed, _dp), _ptr(p_lo, ull), _ptr(p_hi, C.POINTER(C.c_longlong)), _ptr(p_best, _up),
                      C.byref(exponent), C.byref(best), _ptr(info, _dp), C.byref(got))
            if rc or attempt or not retry or got.value <= cap:
                break
            cap = got.value  # the log holds more records than the first buffers: nothing was computed
        self._check(rc)
        n = got.value
        B = float(args[2])
        O = [(int(h) << 64) | int(l) for l, h in zip(o_lo[:n], o_hi[:n])]
        return {"root_id": ids[:n].copy(), "alpha": alpha[:n].copy(), "llh": llh[:n].copy(),
                "lnl_fixed": fixed[:n].copy(), "O": O, "bp_count": bp[:n].copy(), "kh_count": kh[:n].copy(),
                "sh_count": sh[:n].copy(), "bp": bp[:n] / B, "p_kh": kh[:n] / B, "p_sh": sh[:n] / B,
                "exponent": exponent.value, "best": best.value, "replicates": int(args[2]),
                "capture_ms": info[0], "counts_ms": info[1], "accumulate_ms": info[2], "statistics_ms": info[3],
                "resample_ms": info[4], "device_bytes": int(info[5]), "gene_draws_ms": info[6],
                "positions_ms": info[7], "partition_llh": p_fixed[:, :n].copy(),
                "partition_O": [[(int(h) << 64) | int(l) for l, h in zip(p_lo[i, :n], p_hi[i, :n])] for i in range(G)],
                "partition_best": p_best.copy()}

    def placement_support(self, checkpoint_prefix: str | None = None, replicates: int = 10000, seed: int = 0,
                          replicate_tile: int = 0, keep_rows: bool = False, au_scales=None,
                          sampling: str = "site") -> dict:
        """RELL bootstrap proportions and one-sided KH / SH tests of every placement recorded in
        "<checkpoint_prefix>.ckp" (opened read-only; None: the model's own result log, e.g. of
        exhaustive_search), from `replicates` (1..2^20) resamplings of the sites, each partition on
        its own (DESIGN.md section 10).  Per record, in log order: root_id, alpha, llh (as recorded),
        lnl_fixed, O (the exact fixed-point sum, Python ints), bp, p_kh, p_sh and their integer
        counts; also exponent, best (record index), replicates and the timings.  The model's
        parameters and root are unchanged afterwards; the tree's branches carry BP, pKH and pSH in
        newick(True).  keep_rows keeps the per-pattern rows for site_lnl_rows.  On site shards
        every rank calls it with the same arguments and gets the same result.

        au_scales (e.g. AU_SCALES: multiples of 0.001, 2 to 32 of them, strictly ascending, in
        [0.1, 10]) adds Shimodaira's approximately unbiased test from a multiscale bootstrap (the
        replicates drawn at scale s have s times as many sites) and Strimmer & Rambaut's expected
        likelihood weights (DESIGN.md section 10, items 6-8): scales, scale_counts [scale][record]
        (the column of scale 1 is bp_count), p_au, the fit's au_d, au_c, au_rss and au_used (scales
        with 0 < count < replicates), elw and elw_fixed (elw = elw_fixed 2^-40 / replicates), and
        au_counts_ms, au_accumulate_ms, au_statistics_ms; the branches also carry pAU and ELW.  The
        fit is the two-parameter model of Shimodaira (2002) without the iterated threshold
        refinement of CONSEL and IQ-TREE, so p_au may differ from theirs.

        sampling chooses what a replicate resamples (DESIGN.md section 10, items 11-14): "site" (the
        above), "gene" (the model's partitions, with replacement) or "gene_site" (partitions, then
        the sites of each drawn partition, as Gadagkar, Rosenberg & Kumar 2005).  The gene modes need
        at least 2 partitions and refuse au_scales; the counts come from the chosen resampling, and
        the result adds sampling, partition_llh [partition][record] (O_i 2^-exponent, the gene-wise
        log-likelihoods), partition_O (Python ints), partition_best (each partition's record of the
        highest log-likelihood) and gene_draws_ms."""
        mode = self._gene_sampling("placement_support", sampling, au_scales)
        if mode is not None:
            prefix = checkpoint_prefix.encode() if checkpoint_prefix is not None else None
            args = (self.h, prefix, int(replicates), int(seed) & ((1 << 64) - 1), int(replicate_tile),
                    1 if keep_rows else 0, mode)
            out = self._support_genes(self.L.rdh_model_placement_support_genes, 128, args, retry=True)
            del out["positions_ms"]
            self._support_rows = len(out["root_id"]) if keep_rows else 0
            out["sampling"] = sampling
            return out
        if au_scales is not None:
            return self._placement_support_au(checkpoint_prefix, replicates, seed, replicate_tile, keep_rows,
                                              au_thousandths(au_scales))
        prefix = checkpoint_prefix.encode() if checkpoint_prefix is not None else None
        cap = 128
        for attempt in range(2):
            ids = np.zeros(cap, dtype=np.uint64)
            alpha, llh, fixed = np.zeros(cap), np.zeros(cap), np.zeros(cap)
            o_lo, o_hi = np.zeros(cap, dtype=np.uint64), np.zeros(cap, dtype=np.int64)
            bp, kh, sh = (np.zeros(cap, dtype=np.uint32) for _ in range(3))
            exponent, best, got = C.c_int(), C.c_uint(), C.c_uint()
            info = np.zeros(6)
            rc = self.L.rdh_model_placement_support(
                self.h, prefix, int(replicates), int(seed) & ((1 << 64) - 1), int(replicate_tile),
                1 if keep_rows else 0, cap, _ptr(ids, C.POINTER(C.c_ulonglong)), _ptr(alpha, _dp), _ptr(llh, _dp),
                _ptr(fixed, _dp), _ptr(o_lo, C.POINTER(C.c_ulonglong)), _ptr(o_hi, C.POINTER(C.c_longlong)),
                _ptr(bp, _up), _ptr(kh, _up), _ptr(sh, _up), C.byref(exponent), C.byref(best), _ptr(info, _dp),
                C.byref(got))
            if rc or attempt or got.value <= cap:
                break
            cap = got.value  # the log holds more records than the first buffers: nothing was computed
        self._check(rc)
        n = got.value
        self._support_rows = n if keep_rows else 0
        B = float(replicates)
        O = [(int(h) << 64) | int(l) for l, h in zip(o_lo[:n], o_hi[:n])]
        return {"root_id": ids[:n].copy(), "alpha": alpha[:n].copy(), "llh": llh[:n].copy(),
                "lnl_fixed": fixed[:n].copy(), "O": O, "bp_count": bp[:n].copy(), "kh_count": kh[:n].copy(),
                "sh_count": sh[:n].copy(), "bp": bp[:n] / B, "p_kh": kh[:n] / B, "p_sh": sh[:n] / B,
                "exponent": exponent.value, "best": best.value, "replicates": int(replicates),
                "capture_ms": info[0], "counts_ms": info[1], "accumulate_ms": info[2], "statistics_ms": info[3],
                "resample_ms": info[4], "device_bytes": int(info[5])}

    def _placement_support_au(self, checkpoint_prefix, replicates, seed, replicate_tile, keep_rows, scales):
        prefix = checkpoint_prefix.encode() if checkpoint_prefix is not None else None
        sc = np.ascontiguousarray(scales, dtype=np.uint32)
        K, cap = len(sc), 128
        ull = C.POINTER(C.c_ulonglong)
        for attempt in range(2):
            ids = np.zeros(cap, dtype=np.uint64)
            alpha, llh, fixed = np.zeros(cap), np.zeros(cap), np.zeros(cap)
            o_lo, o_hi = np.zeros(cap, dtype=np.uint64), np.zeros(cap, dtype=np.int64)
            bp, kh, sh, used = (np.zeros(cap, dtype=np.uint32) for _ in range(4))
            counts = np.zeros((max(1, K), cap), dtype=np.uint32)
            p_au, d, c, rss, elw = (np.zeros(cap) for _ in range(5))
            elw_fixed = np.zeros(cap, dtype=np.uint64)
            exponent, best, got = C.c_int(), C.c_uint(), C.c_uint()
            info = np.zeros(9)
            rc = self.L.rdh_model_placement_support_au(
                self.h, prefix, int(replicates), int(seed) & ((1 << 64) - 1), int(replicate_tile),
                1 if keep_rows else 0, K, _ptr(sc, _up), cap, _ptr(ids, ull), _ptr(alpha, _dp), _ptr(llh, _dp),
                _ptr(fixed, _dp), _ptr(o_lo, ull), _ptr(o_hi, C.POINTER(C.c_longlong)), _ptr(bp, _up),
                _ptr(kh, _up), _ptr(sh, _up), _ptr(counts, _up), _ptr(p_au, _dp), _ptr(d, _dp), _ptr(c, _dp),
                _ptr(rss, _dp), _ptr(used, _up), _ptr(elw, _dp), _ptr(elw_fixed, ull), C.byref(exponent),
                C.byref(best), _ptr(info, _dp), C.byref(got))
            if rc or attempt or got.value <= cap:
                break
            cap = got.value
        self._check(rc)
        n = got.value
        self._support_rows = n if keep_rows else 0
        B = float(replicates)
        O = [(int(h) << 64) | int(l) for l, h in zip(o_lo[:n], o_hi[:n])]
        return {"root_id": ids[:n].copy(), "alpha": alpha[:n].copy(), "llh": llh[:n].copy(),
                "lnl_fixed": fixed[:n].copy(), "O": O, "bp_count": bp[:n].copy(), "kh_count": kh[:n].copy(),
                "sh_count": sh[:n].copy(), "bp": bp[:n] / B, "p_kh": kh[:n] / B, "p_sh": sh[:n] / B,
                "exponent": exponent.value, "best": best.value, "replicates": int(replicates),
                "capture_ms": info[0], "counts_ms": info[1], "accumulate_ms": info[2], "statistics_ms": info[3],
                "resample_ms": info[4], "device_bytes": int(info[5]),
                "scales": sc / 1000.0, "scale_counts": counts[:, :n].copy(), "p_au": p_au[:n].copy(),
                "au_d": d[:n].copy(), "au_c": c[:n].copy(), "au_rss": rss[:n].copy(), "au_used": used[:n].copy(),
                "elw": elw[:n].copy(), "elw_fixed": elw_fixed[:n].copy(), "au_counts_ms": info[6],
                "au_accumulate_ms": info[7], "au_statistics_ms": info[8]}

    def branch_support(self, checkpoint_prefix: str | None = None, replicates: int = 10000, seed: int = 0,
                       atol: float = 1e-14, replicate_tile: int = 0, keep_rows: bool = False, au_scales=None,
                       sampling: str = "site") -> dict:
        """The statistics of placement_support for EVERY branch, at one set of parameters (DESIGN.md
        section 10, items 9-10): the parameters of the best record of "<checkpoint_prefix>.ckp" (None:
        the model's own result log; highest llh, lowest log index on ties) are installed, root q is
        put at a_q, its best position on its branch (optimize_alpha from 0.5 with tolerance atol, as
        optimize_root_location polishes a candidate; atol = 0: 0.5 everywhere, the placements
        suggest_roots_lh ranks), and record q is the placement (q, a_q), for every root id q in
        order.  The substitution parameters are NOT re-optimised per branch, as exhaustive mode does.
        Returns the keys of placement_support (with or without au_scales): root_id = 0..root_count-1,
        alpha = a_q, llh = the log-likelihood at (q, a_q); plus positions_ms (the alpha searches).
        capture_ms is the one placement sweep that scores all branches and stores their rows.  Every
        branch carries BP, pKH, pSH (pAU, ELW) and its LLH and alpha in newick(True).  sampling is
        placement_support's: "gene" and "gene_site" add the same per-partition keys."""
        prefix = checkpoint_prefix.encode() if checkpoint_prefix is not None else None
        mode = self._gene_sampling("branch_support", sampling, au_scales)
        if mode is not None:
            args = (self.h, prefix, int(replicates), int(seed) & ((1 << 64) - 1), float(atol), int(replicate_tile),
                    1 if keep_rows else 0, mode)
            out = self._support_genes(self.L.rdh_model_branch_support_genes, self.root_count, args, retry=False)
            self._support_rows = len(out["root_id"]) if keep_rows else 0
            out["sampling"] = sampling
            return out
        sc = np.ascontiguousarray(au_thousandths(au_scales) if au_scales is not None else [], dtype=np.uint32)
        K, n = len(sc), self.root_count
        ull = C.POINTER(C.c_ulonglong)
        ids = np.zeros(n, dtype=np.uint64)
        alpha, llh, fixed = np.zeros(n), np.zeros(n), np.zeros(n)
        o_lo, o_hi = np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.int64)
        bp, kh, sh, used = (np.zeros(n, dtype=np.uint32) for _ in range(4))
        counts = np.zeros((max(1, K), n), dtype=np.uint32)
        p_au, d, c, rss, elw = (np.zeros(n) for _ in range(5))
        elw_fixed = np.zeros(n, dtype=np.uint64)
        exponent, best, got = C.c_int(), C.c_uint(), C.c_uint()
        info = np.zeros(10)
        self._check(self.L.rdh_model_branch_support(
            self.h, prefix, int(replicates), int(seed) & ((1 << 64) - 1), float(atol), int(replicate_tile),
            1 if keep_rows else 0, K, _ptr(sc, _up) if K else None, n, _ptr(ids, ull), _ptr(alpha, _dp),
            _ptr(llh, _dp), _ptr(fixed, _dp), _ptr(o_lo, ull), _ptr(o_hi, C.POINTER(C.c_longlong)), _ptr(bp, _up),
            _ptr(kh, _up), _ptr(sh, _up), _ptr(counts, _up), _ptr(p_au, _dp), _ptr(d, _dp), _ptr(c, _dp),
            _ptr(rss, _dp), _ptr(used, _up), _ptr(elw, _dp), _ptr(elw_fixed, ull), C.byref(exponent), C.byref(best),
            _ptr(info, _dp), C.byref(got)))
        n = got.value
        self._support_rows = n if keep_rows else 0
        B = float(replicates)
        O = [(int(h) << 64) | int(l) for l, h in zip(o_lo[:n], o_hi[:n])]
        out = {"root_id": ids[:n].copy(), "alpha": alpha[:n].copy(), "llh": llh[:n].copy(),
               "lnl_fixed": fixed[:n].copy(), "O": O, "bp_count": bp[:n].copy(), "kh_count": kh[:n].copy(),
               "sh_count": sh[:n].copy(), "bp": bp[:n] / B, "p_kh": kh[:n] / B, "p_sh": sh[:n] / B,
               "exponent": exponent.value, "best": best.value, "replicates": int(replicates),
               "capture_ms": info[0], "counts_ms": info[1], "accumulate_ms": info[2], "statistics_ms": info[3],
               "resample_ms": info[4], "device_bytes": int(info[5]), "positions_ms": info[9]}
        if K:
            out.update({"scales": sc / 1000.0, "scale_counts": counts[:, :n].copy(), "p_au": p_au[:n].copy(),
                        "au_d": d[:n].copy(), "au_c": c[:n].copy(), "au_rss": rss[:n].copy(),
                        "au_used": used[:n].copy(), "elw": elw[:n].copy(), "elw_fixed": elw_fixed[:n].copy(),
                        "au_counts_ms": info[6], "au_accumulate_ms": info[7], "au_statistics_ms": info[8]})
        return out

    def site_lnl_rows(self, part: int = 0):
        """(rows [record][pattern], pattern weights) of partition `part` from the last
        placement_support(..., keep_rows=True) or branch_support(..., keep_rows=True)"""
        P = self.sites(part)
        rows = getattr(self, "_support_rows", 0)
        buf = np.zeros(max(1, rows * P))
        w = np.zeros(max(1, P), dtype=np.uint32)
        n = C.c_ulonglong()
        self._check(self.L.rdh_model_site_lnl_rows(self.h, part, _ptr(buf, _dp), len(buf), _ptr(w, _up), len(w),
                                                   C.byref(n)))
        return buf[:n.value].reshape(rows, P), w[:P].copy()

    def lwr(self, llh) -> np.ndarray:
        llh = np.ascontiguousarray(llh, dtype=np.float64)
        out = np.zeros(len(llh))
        self.L.rdh_model_lwr(_ptr(llh, _dp), len(llh), _ptr(out, _dp))
        return out

    def pattern_of_column(self, part: int = 0) -> np.ndarray:
        """the pattern every column of partition `part` was compressed into (a partition's columns in
        the order of its ranges)"""
        n = C.c_uint()
        self.L.rdh_model_pattern_of_column(self.h, part, None, 0, C.byref(n))
        out = np.zeros(max(1, n.value), dtype=np.uint32)
        self._check(self.L.rdh_model_pattern_of_column(self.h, part, _ptr(out, _up), n.value, C.byref(n)))
        return out[:n.value].copy()

    def ancestral_states(self, root_id: int | None = None, ratio: float | None = None,
                         checkpoint_prefix: str | None = None, full_nodes="root", threads: int = 0,
                         tile_sites: int = 0) -> dict:
        """Marginal ancestral states of the rooted tree (DESIGN.md section 11): the posterior of every
        internal node's state, with the root's prior pi, at the model's parameters and root position.

        root_id / ratio: the placement (ratio 0.5 if not given).  checkpoint_prefix: instead, the
        parameters and placement of the best record of "<checkpoint_prefix>.ckp" (highest llh, lowest
        log index on ties).  Parameters and rooting are left as they were.  full_nodes: "root", "all" or
        distinct CLV indices of the nodes whose full posterior is returned.  threads / tile_sites: the
        engine's launch shape (threads per block, patterns per pass; 0 = its default), which does not
        change any result.  Keys: nodes (CLV indices in post-order, the root last), parent (position of
        the parent node, -1 at the root), clade (sorted tip labels below each node), full (positions of
        the nodes in `posterior`), ops (each node's post-order operation, the 8 fields of
        rdk_operation_t), root_id, ratio, and per partition (lists): map_state (bytes of ACGT,
        [node][pattern]), map_prob, posterior ([full node][pattern][4]), log_norm, pattern_of_column,
        ms (device time of the pass), device_bytes, tile_sites."""
        if checkpoint_prefix is not None and (root_id is not None or ratio is not None):
            raise ValueError("ancestral_states: give a placement or a checkpoint, not both")
        if checkpoint_prefix is None and root_id is None:
            raise ValueError("ancestral_states: give root_id (and ratio) or checkpoint_prefix")
        full = np.zeros(1, dtype=np.uint32)
        if isinstance(full_nodes, str):
            if full_nodes not in ("root", "all"):
                raise ValueError("ancestral_states: full_nodes is 'root', 'all' or a list of CLV indices")
            nf = 0 if full_nodes == "root" else 0xFFFFFFFF
        else:
            full = np.ascontiguousarray(list(full_nodes), dtype=np.uint32)
            nf = len(full)
        n_nodes, n_full = C.c_uint(), C.c_uint()
        self._check(self.L.rdh_model_ancestral_states(
            self.h, int(root_id or 0), float(0.5 if ratio is None else ratio),
            checkpoint_prefix.encode() if checkpoint_prefix is not None else None,
            1 if checkpoint_prefix is not None else 0, nf, _ptr(full, _up) if len(full) else None, int(threads),
            int(tile_sites), C.byref(n_nodes), C.byref(n_full)))
        n, nf = n_nodes.value, n_full.value
        nodes = np.zeros(n, dtype=np.uint32)
        parent = np.zeros(n, dtype=np.int32)
        pos = np.zeros(max(1, nf), dtype=np.uint32)
        ops = np.zeros((n, 8), dtype=np.int32)
        rid, rr = C.c_ulonglong(), C.c_double()
        self._check(self.L.rdh_model_ancestral_nodes(self.h, n, nf, _ptr(nodes, _up), _ptr(parent, C.POINTER(C.c_int)),
                                                     _ptr(pos, _up), C.byref(rid), C.byref(rr),
                                                     _ptr(ops, C.POINTER(C.c_int))))
        clade = []
        for i in range(n):
            p = self.L.rdh_model_ancestral_clade(self.h, i)
            if not p:
                raise RuntimeError(self.L.rdh_last_error().decode())
            text = C.string_at(p).decode()
            self.L.rdh_free(p)
            clade.append(text.split("\n") if text else [])
        out = {"nodes": nodes, "parent": parent, "clade": clade, "full": pos[:nf].copy(), "ops": ops,
               "root_id": int(rid.value), "ratio": float(rr.value), "map_state": [], "map_prob": [], "posterior": [],
               "log_norm": [], "pattern_of_column": [], "ms": [], "device_bytes": [], "tile_sites": []}
        acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
        for part in range(self.partition_count):
            P = self.sites(part)
            ms_ = np.zeros((n, P), dtype=np.uint8)
            mp, ln = np.zeros((n, P)), np.zeros((n, P))
            post = np.zeros((nf, P, 4))
            info = np.zeros(4)
            self._check(self.L.rdh_model_ancestral_partition(
                self.h, part, n * P, nf * P * 4, _ptr(ms_, C.POINTER(C.c_ubyte)), _ptr(mp, _dp),
                _ptr(post, _dp) if post.size else None, _ptr(ln, _dp), _ptr(info, _dp)))
            out["map_state"].append(acgt[ms_])
            out["map_prob"].append(mp)
            out["posterior"].append(post)
            out["log_norm"].append(ln)
            out["pattern_of_column"].append(self.pattern_of_column(part))
            out["ms"].append(float(info[0]))
            out["device_bytes"].append(int(info[1]))
            out["tile_sites"].append(int(info[3]))
        return out

    def newick(self, annotations: bool = True) -> str:
        p = self.L.rdh_model_newick(self.h, 1 if annotations else 0)
        if not p:
            raise RuntimeError(self.L.rdh_last_error().decode())
        s = C.string_at(p).decode()
        self.L.rdh_free(p)
        return s
