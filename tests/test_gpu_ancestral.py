"""Marginal ancestral states on the CUDA engine (DESIGN.md section 11): bit for bit the oracle-backed
host's map_state, map_prob, posterior and log_norm on the fixtures at K = 1, 3, 4, 8, at two launch
shapes (threads per block, patterns per tile), with lazy evaluation on (after a run of traversals) and
off; a kept lazy program materialised by the call itself; at 500 taxa x 20 000 sites the numpy
restatement and the identity; the scratch bound of the pass; a one-rank communicator."""
import math

import numpy as np
import pytest

import ancestral_reference as ref
from cases import Case, compute_lh
from root_digger_b200 import capi
from test_ancestral_cpu import rel
from test_gpu_support import libs, model  # noqa: F401  (libs is a fixture)

pytestmark = pytest.mark.gpu

KEYS = ("map_state", "map_prob", "posterior", "log_norm")


def same(a, b):
    assert a["nodes"].tolist() == b["nodes"].tolist()
    for key in KEYS:
        for pa, pb in zip(a[key], b[key]):
            assert pa.tobytes() == pb.tobytes(), key


@pytest.mark.parametrize("shape", [(0, 0), (64, 100)])  # (threads per block, patterns per tile): defaults, small
@pytest.mark.parametrize("lazy", ["1", "0"])
@pytest.mark.parametrize("name,K,rid,ratio", [("10.fasta", 1, 3, 0.3), ("10.fasta", 3, 0, 1.0), ("101.phy", 4, 57, 0.8),
                                              ("101.phy", 8, 120, 0.0)])
def test_engine_matches_the_oracle_host(libs, monkeypatch, name, K, rid, ratio, lazy, shape):  # noqa: F811
    monkeypatch.setenv("RDK_LAZY", lazy)
    ms = [model(lib, name, K) for lib in libs]
    out = []
    for m in ms:
        for r in range(4):  # a run of full traversals: lazily kept programs on the engine
            m.compute_lh(r, 0.5)
        out.append(m.ancestral_states(rid, ratio, full_nodes="all", threads=shape[0], tile_sites=shape[1]))
    same(out[0], out[1])
    if shape[1]:
        assert out[0]["tile_sites"][0] == min(shape[1], ms[0].sites(0))


def test_the_call_materialises_a_kept_program_and_gives_the_eager_bits():
    # on the ABI: the second full traversal in a row keeps its CLVs in registers only; the pass reads
    # them, so the engine replays the kept program first
    case = Case(120, 900, 4, seed=41, data="ambiguous")
    lazy, eager = (capi.Partition(case.n, case.S, case.K) for _ in range(2))
    for part in (lazy, eager):
        case.setup(part)
    eager.set_lazy(False)
    sched = case.full_schedule(9, 0.35)
    for _ in range(2):
        for part in (lazy, eager):
            compute_lh(part, sched, case.root_clv, case.root_scaler)
    before = lazy.stats()
    assert before["lazy_evaluations"] >= 1
    n = len(sched[0])
    got = [p.marginal_ancestral_states(sched[0], full_ops=range(n), threads=t, tile_sites=ts)
           for p, t, ts in ((lazy, 0, 0), (eager, 0, 0), (eager, 96, 128))]
    assert lazy.stats()["materializations"] == before["materializations"] + 1
    for g in got[1:]:
        for key in KEYS:
            assert got[0][key].tobytes() == g[key].tobytes(), key
    assert got[2]["tile_sites"] == 128
    with pytest.raises(capi.EngineError, match="listed twice"):
        eager.marginal_ancestral_states(sched[0], full_ops=[n - 1, n - 1])
    with pytest.raises(capi.EngineError, match="threads"):
        eager.marginal_ancestral_states(sched[0], threads=48)


def test_checkpoint_form_matches_the_oracle_host(libs, tmp_path):  # noqa: F811
    from test_branch_support_cpu import search_log
    ms = [model(lib, "101.phy", 4) for lib in libs]
    search_log(libs[1], tmp_path / "s", ms[1])
    same(*[m.ancestral_states(checkpoint_prefix=str(tmp_path / "s")) for m in ms])


def test_full_size_against_the_restatement_and_the_scratch_bound():
    case = Case(500, 20000, 4, seed=11)
    m = capi.Model(case.tree, {l: s for l, s in case.aln.items()}, rate_cats=4, compress=False, seed=3)
    m.initialize_partitions()
    m.set_params(rates=case.rates, freqs=case.freqs, alpha=0.7)
    rid = 123
    m.compute_lh(rid, 0.4)
    res = m.ancestral_states(rid, 0.4, full_nodes="all")
    n = len(res["nodes"])
    S = m.sites(0)
    assert res["ms"][0] > 0
    # at most ceil(log2 n) + 2 outside vectors besides the outputs
    outputs = n * S * (1 + 8 + 8) + 32 * n * S
    nodes_table = n * 128
    bound = (math.ceil(math.log2(n)) + 2) * (S * 4 * 32 + 4 * S) + outputs + nodes_table + 7 * 256
    assert res["device_bytes"][0] <= bound
    # the restatement, from the engine's own P-matrices and 0/1 tips
    import ctypes as C
    ops = [tuple(int(x) for x in o) for o in res["ops"]]
    eng = capi.load_engine()
    ptr = C.cast(m.L.rdh_model_partition(m.h, 0), C.POINTER(capi.PartitionStruct))
    P, tips = {}, {}
    for op in ops:
        for c, mi in ((op[2], op[3]), (op[5], op[6])):
            buf = np.zeros(4 * 16)
            assert eng.rdk_get_pmatrix(ptr, mi, buf.ctypes.data_as(C.POINTER(C.c_double)))
            P[mi] = buf.reshape(4, 4, 4)
            if c < 500:
                t = np.zeros(S * 16)
                assert eng.rdk_get_clv(ptr, c, t.ctypes.data_as(C.POINTER(C.c_double)))
                tips[c] = t.reshape(S, 4, 4)
    pstruct = ptr.contents
    pi = np.array([pstruct.frequencies[0][i] for i in range(4)])
    w = np.array([pstruct.rate_weights[k] for k in range(4)])
    r = ref.marginal(ops, P, tips, pi, w)
    assert rel(res["posterior"][0], r["posterior"]) < 1e-12
    assert rel(res["log_norm"][0], r["log_norm"], 1.0) < 1e-12
    ln = res["log_norm"][0]
    assert rel(ln, np.broadcast_to(ln[-1], ln.shape), 1.0) < 1e-12
    lh = m.compute_lh(rid, 0.4)
    assert abs(float(ln[-1].sum()) - lh) <= 1e-12 * abs(lh)


def test_a_one_rank_communicator_returns_the_unsharded_bits():
    import gpu_multi_worker as base
    case = base.build_case()
    got = []
    for sharded in (False, True):
        kw = dict(site_offset=0, global_sites=base.SITES, nranks=1, rank=0, comm_id=capi.comm_unique_id()) \
            if sharded else {}
        m = capi.Model(capi.RootedTree(case.newick), case.aln, base.K, **kw)
        m.initialize_partitions()
        got.append(m.ancestral_states(3, 0.4, full_nodes="all"))
        m.close()
    same(got[0], got[1])
