"""The AU test and expected likelihood weights of root placement support on the CUDA engine (DESIGN.md
section 10, items 6-8): the multiscale counts, elw_fixed and p_AU against the oracle-backed model_t
(which tests/test_au_cpu.py checks against the restated definition), against that restatement at
500 taxa x 20 000 sites, under other launch shapes and replicate tiles, and on a one-rank communicator."""
import ctypes as C

import numpy as np
import pytest

import au_reference
from root_digger_b200 import capi, synth
from test_gpu_support import RellOut, libs, model  # noqa: F401  (libs is a fixture)
from test_support_cpu import thirds, write_records

pytestmark = pytest.mark.gpu

SCALES = capi.au_thousandths(capi.AU_SCALES)
AU_KEYS = ("scale_counts", "elw_fixed", "p_au", "au_d", "au_c", "au_rss", "au_used", "elw")
PLAIN_KEYS = ("root_id", "bp_count", "kh_count", "sh_count", "lnl_fixed")


def same_bits(a, b):
    assert a["exponent"] == b["exponent"] and a["best"] == b["best"] and a["O"] == b["O"]
    for key in PLAIN_KEYS + AU_KEYS:
        assert a[key].tobytes() == b[key].tobytes(), key


@pytest.mark.parametrize("name,K,parts", [("10.fasta", 1, False), ("10.fasta", 4, True), ("101.phy", 4, False),
                                          ("101.phy", 1, True)])
def test_engine_matches_the_oracle_host(libs, tmp_path, name, K, parts):  # noqa: F811
    ms = [model(lib, name, K, thirds(name) if parts else None) for lib in libs]
    write_records(libs[0], tmp_path / "s", ms[0], range(ms[0].root_count))
    res = [m.placement_support(str(tmp_path / "s"), replicates=300, seed=77, au_scales=capi.AU_SCALES) for m in ms]
    same_bits(*res)
    plain = ms[0].placement_support(str(tmp_path / "s"), replicates=300, seed=77)
    for key in PLAIN_KEYS:
        assert plain[key].tobytes() == res[0][key].tobytes(), key
    assert res[0]["scale_counts"][SCALES.index(1000)].tobytes() == plain["bp_count"].tobytes()


def test_all_placements_of_a_500_taxon_tree(libs, tmp_path):  # noqa: F811
    top = synth.random_tree(500, 11)
    rates, freqs = synth.random_params(12)
    aln = synth.simulate_alignment(top, 20000, 13, rates, freqs, capi.gamma_cats(0.8, 4))
    m = capi.Model(capi.RootedTree(synth.to_newick(top), lib=libs[0]), aln, rate_cats=4, compress=True, seed=1)
    m.initialize_partitions(uniform_freqs=False)
    assert m.root_count == 997
    write_records(libs[0], tmp_path / "big", m, range(m.root_count), seed=5)
    B, seed = 40, 2024
    res = m.placement_support(str(tmp_path / "big"), replicates=B, seed=seed, keep_rows=True, au_scales=capi.AU_SCALES)
    rows, w = m.site_lnl_rows(0)
    ref = au_reference.support([rows], [w], B, seed, SCALES)
    assert res["scale_counts"].tolist() == ref["scale_count"]
    assert res["elw_fixed"].tolist() == ref["elw_fixed"]
    assert res["au_used"].tolist() == ref["au_used"]
    for key in ("p_au", "au_d", "au_c", "au_rss"):
        assert np.allclose(res[key], ref[key], rtol=0, atol=1e-12), key


def test_launch_shapes_and_replicate_tiles_change_no_bit(libs, tmp_path):  # noqa: F811
    m = model(libs[0], "101.phy", 4)
    write_records(libs[0], tmp_path / "s", m, range(m.root_count))
    L = capi.load_engine()
    part = C.c_void_p(m.L.rdh_model_partition(m.h, 0))
    L.rdk_partition_set_launch_config.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.rdk_partition_set_subtree_groups.argtypes = [C.c_void_p, C.c_int]
    base = m.placement_support(str(tmp_path / "s"), replicates=500, seed=3, au_scales=capi.AU_SCALES)
    for elems, groups, tile in ((1, 1, 7), (4, 4, 64), (4, 0, 499), (1, 0, 1)):
        assert L.rdk_partition_set_launch_config(part, 0, 0, elems) == 1
        assert L.rdk_partition_set_subtree_groups(part, groups) == 1
        other = m.placement_support(str(tmp_path / "s"), replicates=500, seed=3, replicate_tile=tile,
                                    au_scales=capi.AU_SCALES)
        same_bits(base, other)


class RellMsOut(C.Structure):
    _fields_ = [("scales", C.POINTER(C.c_uint)), ("n_scales", C.c_uint), ("scale_count", C.POINTER(C.c_uint)),
                ("elw_fixed", C.POINTER(C.c_ulonglong)), ("ms", C.c_double * 3)]


def test_exchanges_on_a_one_rank_communicator():
    """the site-shard path of rdk_rell_support_ms (the limb all-reduce of Z_k per scale) on a
    communicator of one rank returns the bits of the unsharded path; the entry refuses bad scales"""
    from cases import Case, compute_lh
    case = Case(24, 3000, 4, seed=6, data="evolved", weights="random")
    L = capi.load_engine()
    L.rdk_rell_support_ms.argtypes = [C.POINTER(C.c_void_p), C.c_uint, C.POINTER(C.c_uint), C.c_uint, C.c_ulonglong,
                                      C.c_ulonglong, C.POINTER(RellOut), C.POINTER(RellMsOut)]
    scales = np.array([400, 700, 1000, 1600, 2500], dtype=np.uint32)
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
        counts, elw = np.zeros((len(scales), 3), dtype=np.uint32), np.zeros(3, dtype=np.uint64)
        ms = RellMsOut(scales.ctypes.data_as(C.POINTER(C.c_uint)), len(scales), counts.ctypes.data_as(C.POINTER(C.c_uint)),
                       elw.ctypes.data_as(C.POINTER(C.c_ulonglong)))
        parts = (C.c_void_p * 1)(C.cast(g.p, C.c_void_p).value)
        assert L.rdk_rell_support_ms(parts, 1, None, 3, 400, 11, C.byref(out), C.byref(ms)) == 1, capi._err(L)
        assert (counts.sum(axis=1) == 400).all() and counts[2].tobytes() == arrays[3].tobytes()
        got.append((out.exponent, out.best, [a.tobytes() for a in arrays], counts.tobytes(), elw.tobytes()))
        if not sharded:
            for bad in ([1000, 900], [1000], [50, 1000], [1000, 10001]):
                b = np.array(bad, dtype=np.uint32)
                ms_bad = RellMsOut(b.ctypes.data_as(C.POINTER(C.c_uint)), len(b),
                                   counts.ctypes.data_as(C.POINTER(C.c_uint)), elw.ctypes.data_as(C.POINTER(C.c_ulonglong)))
                assert L.rdk_rell_support_ms(parts, 1, None, 3, 400, 11, C.byref(out), C.byref(ms_bad)) != 1
            assert L.rdk_rell_support_ms(parts, 1, None, 3, 400, 11, C.byref(out), None) != 1
        g.close()
    assert got[0] == got[1]
