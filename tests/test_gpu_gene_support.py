"""Gene and gene-then-site resampling of root placement support on the CUDA engine (DESIGN.md section
10, items 11-14): the engine host against the oracle-backed host (which tests/test_gene_support_cpu.py
checks against the restated definition), against that restatement on a 500-taxon tree in 8
partitions, under other replicate tiles, and the bound rdk_rell_support_genes refuses."""
import ctypes as C

import numpy as np
import pytest

import gene_reference
from root_digger_b200 import capi, synth
from test_branch_support_cpu import search_log
from test_gene_support_cpu import CASES, COUNT_KEYS, parts_of
from test_gpu_support import RellOut, libs, model  # noqa: F401  (libs is a fixture)
from test_support_cpu import write_records

pytestmark = pytest.mark.gpu

GENE_KEYS = ("partition_llh", "partition_best") + COUNT_KEYS + ("lnl_fixed", "root_id")


def same_bits(a, b):
    assert a["exponent"] == b["exponent"] and a["best"] == b["best"] and a["O"] == b["O"]
    assert a["partition_O"] == b["partition_O"]
    for key in GENE_KEYS:
        assert a[key].tobytes() == b[key].tobytes(), key


def against_reference(m, res, B, seed, sampling):
    rows = [m.site_lnl_rows(p) for p in range(m.partition_count)]
    ref = gene_reference.support([r for r, _ in rows], [w for _, w in rows], B, seed, sampling)
    assert res["exponent"] == ref["exponent"] and res["best"] == ref["best"] and res["O"] == ref["O"]
    for key in COUNT_KEYS + ("partition_best",):
        assert res[key].tolist() == ref[key], key
    assert res["partition_O"] == ref["partition_O"]
    assert res["partition_llh"].tolist() == ref["partition_llh"]


@pytest.mark.parametrize("sampling", ["gene", "gene_site"])
@pytest.mark.parametrize("name,K,G", CASES)
def test_engine_matches_the_oracle_host(libs, tmp_path, name, K, G, sampling):  # noqa: F811
    ms = [model(lib, name, K, parts_of(name, G)) for lib in libs]
    write_records(libs[0], tmp_path / "s", ms[0], range(ms[0].root_count))
    res = [m.placement_support(str(tmp_path / "s"), replicates=300, seed=77, sampling=sampling) for m in ms]
    same_bits(*res)
    search_log(libs[0], tmp_path / "b", ms[0])
    res = [m.branch_support(str(tmp_path / "b"), replicates=300, seed=78, atol=1e-6, sampling=sampling) for m in ms]
    same_bits(*res)
    for m in ms:
        m.close()


def test_a_500_taxon_tree_in_8_partitions(libs, tmp_path):  # noqa: F811
    top = synth.random_tree(500, 11)
    rates, freqs = synth.random_params(12)
    aln = synth.simulate_alignment(top, 20000, 13, rates, freqs, capi.gamma_cats(0.8, 4))
    parts = [(i * 2500, (i + 1) * 2500) for i in range(8)]
    m = capi.Model(capi.RootedTree(synth.to_newick(top), lib=libs[0]), aln, rate_cats=4, compress=True, seed=1,
                   partitions=parts)
    m.initialize_partitions(uniform_freqs=False)
    assert m.root_count == 997 and m.partition_count == 8
    B, seed = 2000, 2024
    search_log(libs[0], tmp_path / "s", m)
    write_records(libs[0], tmp_path / "big", m, range(0, m.root_count, 3), seed=5)
    for sampling in ("gene", "gene_site"):
        res = m.branch_support(str(tmp_path / "s"), replicates=B, seed=seed, keep_rows=True, sampling=sampling)
        against_reference(m, res, B, seed, sampling)
        res = m.placement_support(str(tmp_path / "big"), replicates=B, seed=seed, keep_rows=True,
                                  sampling=sampling)
        against_reference(m, res, B, seed, sampling)
    m.close()


def test_replicate_tiles_change_no_bit_and_site_mode_is_unchanged(libs, tmp_path):  # noqa: F811
    m = model(libs[0], "101.phy", 4, parts_of("101.phy", 16))
    write_records(libs[0], tmp_path / "s", m, range(m.root_count))
    s = str(tmp_path / "s")
    site = m.placement_support(s, replicates=500, seed=3)
    for sampling in ("gene", "gene_site"):
        base = m.placement_support(s, replicates=500, seed=3, sampling=sampling)
        for tile in (1, 7, 0):
            same_bits(base, m.placement_support(s, replicates=500, seed=3, replicate_tile=tile, sampling=sampling))
    again = m.placement_support(s, replicates=500, seed=3)
    for key in COUNT_KEYS + ("lnl_fixed",):
        assert site[key].tobytes() == again[key].tobytes(), key
    assert site["O"] == again["O"] and site["best"] == again["best"]
    m.close()


class RellGeneOut(C.Structure):
    _fields_ = [("sampling", C.c_uint), ("partition_lnl_fixed", C.POINTER(C.c_double)),
                ("o_lo", C.POINTER(C.c_ulonglong)), ("o_hi", C.POINTER(C.c_longlong)), ("draws_ms", C.c_double)]


def test_what_the_engine_entry_refuses():
    """n N_max >= 2^32 (item 14), one partition, an unknown mode; the same partitions are accepted
    below the bound"""
    from cases import Case, compute_lh
    L = capi.load_engine()
    L.rdk_rell_support_genes.argtypes = [C.POINTER(C.c_void_p), C.c_uint, C.POINTER(C.c_uint), C.c_uint,
                                         C.c_ulonglong, C.c_ulonglong, C.POINTER(RellOut), C.POINTER(RellGeneOut)]
    case = Case(24, 3000, 4, seed=6, data="evolved", weights="random")
    gs = []
    for _ in range(2):
        g = capi.Partition(case.n, case.S, case.K, device=0)
        case.setup(g)
        g.set_site_lnl_rows(2)
        for r, rid in enumerate((0, 5)):
            compute_lh(g, case.full_schedule(rid, 0.4), case.root_clv, case.root_scaler)
            g.root_loglikelihood_row(case.root_clv, case.root_scaler, r)
        gs.append(g)
    arrays = [np.zeros(2), np.zeros(2, dtype=np.uint64), np.zeros(2, dtype=np.int64)] + \
             [np.zeros(2, dtype=np.uint32) for _ in range(3)]
    out = RellOut(0, 0, 0, 0, *(a.ctypes.data_as(t) for a, t in zip(arrays, (
        C.POINTER(C.c_double), C.POINTER(C.c_ulonglong), C.POINTER(C.c_longlong), C.POINTER(C.c_uint),
        C.POINTER(C.c_uint), C.POINTER(C.c_uint)))))
    fixed = np.zeros(4)
    parts = (C.c_void_p * 2)(*(C.cast(g.p, C.c_void_p).value for g in gs))

    def call(sampling, n=2):
        genes = RellGeneOut(sampling, fixed.ctypes.data_as(C.POINTER(C.c_double)))
        return L.rdk_rell_support_genes(parts, n, None, 2, 100, 9, C.byref(out), C.byref(genes))

    assert call(capi.Model.SAMPLING["gene"]) == 1, capi._err(L)
    assert call(capi.Model.SAMPLING["gene_site"]) == 1, capi._err(L)
    assert call(3) != 1 and "unknown sampling mode" in capi._err(L)
    assert call(1, n=1) != 1 and "at least 2" in capi._err(L)
    w = np.full(case.S, 1, dtype=np.uint32)
    w[0] = (1 << 31) - case.S + 1  # N = 2^31: 2 partitions x 2^31 = 2^32
    gs[1].set_pattern_weights(w)
    assert call(1) != 1 and "2^32" in capi._err(L)
    w[0] -= 1
    gs[1].set_pattern_weights(w)
    assert call(1) == 1, capi._err(L)
    for g in gs:
        g.close()
