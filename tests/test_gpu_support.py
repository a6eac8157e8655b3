"""Root placement support on the CUDA engine (DESIGN.md section 10): the per-pattern rows and every
integer the statistics are made of, against the oracle-backed model_t (which tests/test_support_cpu.py
checks against the restated definition) and against that restatement at 500 taxa x 20 000 sites."""
import ctypes as C

import numpy as np
import pytest

import fixtures
import oracle_build
import oracle_capi
import rell_reference
from root_digger_b200 import capi, synth
from test_support_cpu import thirds, write_records

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def libs():
    oracle_capi.load_oracle().rdo_set_default_mode(oracle_capi.MODE_ENGINE)
    return capi.load_tree_lib(), capi.load_tree_lib(oracle_build.build_host_on_oracle())


def model(lib, name, K, partitions=None):
    fx = fixtures.load(name)
    m = capi.Model(capi.RootedTree(path=str(fx["tree_path"]), lib=lib), fx["alignment"], rate_cats=K, compress=True,
                   seed=7, partitions=partitions)
    m.initialize_partitions(uniform_freqs=False)
    return m


def same(a, b):
    assert a["exponent"] == b["exponent"] and a["best"] == b["best"]
    for key in ("root_id", "bp_count", "kh_count", "sh_count"):
        assert np.array_equal(a[key], b[key]), key
    assert a["lnl_fixed"].tobytes() == b["lnl_fixed"].tobytes()


@pytest.mark.parametrize("name,K,parts", [("10.fasta", 1, False), ("10.fasta", 4, True), ("101.phy", 4, False),
                                          ("101.phy", 1, True)])
def test_engine_matches_the_oracle_host(libs, tmp_path, name, K, parts):
    ms = [model(lib, name, K, thirds(name) if parts else None) for lib in libs]
    write_records(libs[0], tmp_path / "s", ms[0], range(ms[0].root_count))
    res = [m.placement_support(str(tmp_path / "s"), replicates=300, seed=77, keep_rows=True) for m in ms]
    same(*res)
    for p in range(ms[0].partition_count):
        (ra, wa), (rb, wb) = ms[0].site_lnl_rows(p), ms[1].site_lnl_rows(p)
        assert ra.tobytes() == rb.tobytes() and np.array_equal(wa, wb)


def test_rows_are_the_unweighted_persite_values():
    """rdk_compute_root_loglikelihood_row returns the bits of rdk_compute_root_loglikelihood, and
    dmul(row, w) is its persite_lnl, on the engine; the row is the oracle's value with weights 1"""
    from cases import Case, compute_lh
    case = Case(24, 3000, 4, seed=5, data="evolved", weights="random")
    g = capi.Partition(case.n, case.S, case.K, device=0)
    o = oracle_capi.OraclePartition(case.n, case.S, case.K)
    case.setup(g)
    case.setup(o)
    sched = case.full_schedule(0, 0.5)
    lw, pw = compute_lh(g, sched, case.root_clv, case.root_scaler, persite=True)
    g.set_site_lnl_rows(3)
    assert g.root_loglikelihood_row(case.root_clv, case.root_scaler, 2) == lw
    row = g.site_lnl_rows(2, 1)[0]
    assert np.array_equal(row * case.weights.astype(np.float64), pw)
    compute_lh(o, sched, case.root_clv, case.root_scaler, mode=oracle_capi.MODE_ENGINE)
    o.set_pattern_weights(np.ones(case.S, dtype=np.uint32))
    _, L = o.root_loglikelihood(case.root_clv, case.root_scaler, persite=True, mode=oracle_capi.MODE_ENGINE)
    assert row.tobytes() == L.tobytes()
    g.close()


def test_launch_shapes_and_replicate_tiles_change_no_bit(libs, tmp_path):
    m = model(libs[0], "101.phy", 4)
    write_records(libs[0], tmp_path / "s", m, range(m.root_count))
    L = capi.load_engine()
    part = C.c_void_p(m.L.rdh_model_partition(m.h, 0))
    L.rdk_partition_set_launch_config.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.rdk_partition_set_subtree_groups.argtypes = [C.c_void_p, C.c_int]
    base = m.placement_support(str(tmp_path / "s"), replicates=500, seed=3, keep_rows=True)
    rows = m.site_lnl_rows(0)[0]
    for elems, groups, tile in ((1, 1, 7), (4, 4, 64), (4, 0, 499), (1, 0, 1)):
        assert L.rdk_partition_set_launch_config(part, 0, 0, elems) == 1
        assert L.rdk_partition_set_subtree_groups(part, groups) == 1
        other = m.placement_support(str(tmp_path / "s"), replicates=500, seed=3, replicate_tile=tile, keep_rows=True)
        same(base, other)
        assert m.site_lnl_rows(0)[0].tobytes() == rows.tobytes()


def test_all_placements_of_a_500_taxon_tree(libs, tmp_path):
    """500 taxa x 20 000 sites, all 997 placements: the engine against the restated definition"""
    top = synth.random_tree(500, 11)
    rates, freqs = synth.random_params(12)
    aln = synth.simulate_alignment(top, 20000, 13, rates, freqs, capi.gamma_cats(0.8, 4))
    m = capi.Model(capi.RootedTree(synth.to_newick(top), lib=libs[0]), aln, rate_cats=4, compress=True, seed=1)
    m.initialize_partitions(uniform_freqs=False)
    assert m.root_count == 997
    write_records(libs[0], tmp_path / "big", m, range(m.root_count), seed=5)
    B, seed = 40, 2024
    res = m.placement_support(str(tmp_path / "big"), replicates=B, seed=seed, keep_rows=True)
    rows, w = m.site_lnl_rows(0)
    ref = rell_reference.support([rows], [w], B, seed)
    assert res["exponent"] == ref["exponent"] and res["best"] == ref["best"]
    for key in ("bp_count", "kh_count", "sh_count"):
        assert res[key].tolist() == ref[key], key
    assert res["lnl_fixed"].tolist() == ref["lnl_fixed"] and res["O"] == ref["O"]
    # a subset of the records against the oracle-backed host: rows (bits), e, O and the counts
    oracle = capi.Model(capi.RootedTree(synth.to_newick(top), lib=libs[1]), aln, rate_cats=4, compress=True, seed=1)
    oracle.initialize_partitions(uniform_freqs=False)
    write_records(libs[0], tmp_path / "few", m, [0, 311, 996], seed=6)
    a, b = (x.placement_support(str(tmp_path / "few"), replicates=B, seed=seed, keep_rows=True) for x in (m, oracle))
    same(a, b)
    assert a["O"] == b["O"]
    assert m.site_lnl_rows(0)[0].tobytes() == oracle.site_lnl_rows(0)[0].tobytes()


class RellOut(C.Structure):
    _fields_ = [("replicate_tile", C.c_uint), ("exponent", C.c_int), ("best", C.c_uint), ("bad_row", C.c_uint),
                ("lnl_fixed", C.POINTER(C.c_double)), ("o_lo", C.POINTER(C.c_ulonglong)),
                ("o_hi", C.POINTER(C.c_longlong)), ("bp_count", C.POINTER(C.c_uint)),
                ("kh_count", C.POINTER(C.c_uint)), ("sh_count", C.POINTER(C.c_uint)), ("ms", C.c_double * 4),
                ("device_bytes", C.c_ulonglong)]


def test_exchanges_on_a_one_rank_communicator():
    """the site-shard path of rdk_rell_support (offset prefix, all-reduce max, limb all-reduces of Z
    and O) on a communicator of one rank returns the bits of the unsharded path"""
    from cases import Case, compute_lh
    case = Case(24, 3000, 4, seed=6, data="evolved", weights="random")
    L = capi.load_engine()
    L.rdk_rell_support.argtypes = [C.POINTER(C.c_void_p), C.c_uint, C.POINTER(C.c_uint), C.c_uint, C.c_ulonglong,
                                   C.c_ulonglong, C.POINTER(RellOut)]
    got = []
    for sharded in (False, True):
        g = capi.Partition(case.n, case.S, case.K, device=0)
        case.setup(g)
        if sharded:
            g.set_shard(0, case.S)
            g.attach_comm(1, 0, capi.comm_unique_id())
        g.set_site_lnl_rows(3)
        for r, rid in enumerate((0, 5, 9)):
            compute_lh(g, case.full_schedule(rid, 0.4), case.root_clv, case.root_scaler)
            g.root_loglikelihood_row(case.root_clv, case.root_scaler, r)
        arrays = [np.zeros(3), np.zeros(3, dtype=np.uint64), np.zeros(3, dtype=np.int64)] + \
                 [np.zeros(3, dtype=np.uint32) for _ in range(3)]
        out = RellOut(0, 0, 0, 0, *(a.ctypes.data_as(t) for a, t in zip(arrays, (
            C.POINTER(C.c_double), C.POINTER(C.c_ulonglong), C.POINTER(C.c_longlong), C.POINTER(C.c_uint),
            C.POINTER(C.c_uint), C.POINTER(C.c_uint)))))
        parts = (C.c_void_p * 1)(C.cast(g.p, C.c_void_p).value)
        assert L.rdk_rell_support(parts, 1, None, 3, 400, 11, C.byref(out)) == 1, capi._err(L)
        got.append((out.exponent, out.best, [a.tobytes() for a in arrays], g.site_lnl_rows(0, 3).tobytes()))
        g.close()
    assert got[0] == got[1]
