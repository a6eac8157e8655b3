"""Branch support on the CUDA engine (DESIGN.md section 10, items 9-10).

ABI: rows the placement sweep stores with RDK_SWEEP_ROWS are, byte for byte, the rows
rdk_compute_root_loglikelihood_row stores after a full traversal at the same placement, and the
oracle's ENGINE-mode rows; the flag changes no returned log-likelihood.  Model: the engine's
branch_support equals the oracle-backed host's, and the engine's placement_support on the equivalent
checkpoint; a one-rank communicator returns the bits of the unsharded path."""
import numpy as np
import pytest

import oracle_capi
from cases import Case, compute_lh
from root_digger_b200 import capi
from test_branch_support_cpu import AU_KEYS, CASES, PLAIN_KEYS, same, search_log, write_log
from test_gpu_support import libs, model  # noqa: F401  (libs is a fixture)
from test_support_cpu import thirds

pytestmark = pytest.mark.gpu

SWEEP = capi.RDK_SWEEP_KEEP_ROOT | capi.RDK_SWEEP_DISCARD


def with_ratios(sched, tree, ratio):
    """the sweep schedule with placement q's root half-branches at ratio[root_pos[q]] (child 1, the
    root location's edge, takes ratio * length, as rooted_tree_t::generate_derivative_operations)"""
    pm_off, mi, bl, *rest = sched
    pos = rest[2]
    bl = bl.copy()
    for q, rid in enumerate(pos.tolist()):
        length = tree.root_info(rid)[0]
        bl[pm_off[q + 1] - 2] = length * ratio[rid]
        bl[pm_off[q + 1] - 1] = length * (1 - ratio[rid])
    return (pm_off, mi, bl, *rest)


@pytest.mark.parametrize("mode", ["unchunked", "chunks", "batches"])
@pytest.mark.parametrize("n,S,K,data", [(150, 700, 4, "iid"), (300, 129, 2, "iid"), (80, 1200, 3, "ambiguous")])
def test_sweep_rows_are_the_rows_of_full_evaluations(monkeypatch, n, S, K, data, mode):
    case = Case(n, S, K, seed=29 + n, data=data, weights="random")
    chunks = 1 if mode == "unchunked" else 4
    if mode == "batches":
        monkeypatch.setenv("RDK_SWEEP_MAX_SLOTS", "7")  # several batches: row of slot s = first placement + s
    lay = case.tree.sweep_layout(chunks)
    kw = dict(clv_buffers=lay["clv_buffers"], scale_buffers=lay["scale_buffers"], prob_matrices=lay["prob_matrices"])
    g = capi.Partition(case.n, case.S, case.K, **kw)
    case.setup(g)
    R = case.tree.root_count
    rng = np.random.default_rng(n)
    ratio = np.where(np.arange(R) % 2 == 0, 0.5, rng.uniform(0.05, 0.95, R))
    start = R // 3
    compute_lh(g, case.full_schedule(start, 0.4), case.root_clv, case.root_scaler)
    *sw, pos, coff = with_ratios(case.tree.generate_chunked_sweep_operations(layout=lay), case.tree, ratio)
    assert sorted(pos.tolist()) == list(range(R))
    co = coff if mode != "unchunked" else None
    plain = g.sweep_root_placements(*sw, case.root_clv, case.root_scaler, flags=SWEEP, chunk_offsets=co)
    with pytest.raises(capi.EngineError, match="site rows"):
        g.sweep_root_placements(*sw, case.root_clv, case.root_scaler, flags=SWEEP | capi.RDK_SWEEP_ROWS,
                                chunk_offsets=co)
    g.set_site_lnl_rows(R)
    got = g.sweep_root_placements(*sw, case.root_clv, case.root_scaler, flags=SWEEP | capi.RDK_SWEEP_ROWS,
                                  chunk_offsets=co)
    assert got.tobytes() == plain.tobytes()
    rows = g.site_lnl_rows(0, R)
    g.close()

    ref = capi.Partition(case.n, case.S, case.K)
    case.setup(ref)
    ref.set_site_lnl_rows(1)
    o = oracle_capi.OraclePartition(case.n, case.S, case.K)
    case.setup(o)
    o.set_pattern_weights(np.ones(case.S, dtype=np.uint32))
    for q, rid in enumerate(pos.tolist()):
        ops, pm, br = case.full_schedule(rid, ratio[rid])
        ref.update_prob_matrices(pm, br)
        ref.update_clvs(ops)
        lh = ref.root_loglikelihood_row(case.root_clv, case.root_scaler, 0)
        assert lh == got[q], (q, rid)
        assert rows[q].tobytes() == ref.site_lnl_rows(0, 1)[0].tobytes(), (q, rid)
        if q % 9 == 0:
            _, want = compute_lh(o, (ops, pm, br), case.root_clv, case.root_scaler, persite=True,
                                 mode=oracle_capi.MODE_ENGINE)
            assert rows[q].tobytes() == want.tobytes(), (q, rid)
    ref.close()


def test_rows_are_put_in_any_order():
    case = Case(24, 3000, 4, seed=5, data="evolved", weights="random")
    g = capi.Partition(case.n, case.S, case.K)
    case.setup(g)
    g.set_site_lnl_rows(6)
    for r in range(6):
        compute_lh(g, case.full_schedule(r, 0.3), case.root_clv, case.root_scaler)
        g.root_loglikelihood_row(case.root_clv, case.root_scaler, r)
    before = g.site_lnl_rows(0, 6)
    order = [3, 0, 1, 5, 4, 2]
    g.permute_site_lnl_rows(order)
    assert g.site_lnl_rows(0, 6).tobytes() == before[order].tobytes()
    with pytest.raises(capi.EngineError, match="permutation"):
        g.permute_site_lnl_rows([0, 0, 1])
    g.close()


@pytest.mark.parametrize("au", [False, True])
@pytest.mark.parametrize("name,K,parts,atol", CASES)
def test_engine_matches_the_oracle_host_and_its_own_placement_support(libs, tmp_path, name, K, parts, atol, au):  # noqa: F811
    ms = [model(lib, name, K, thirds(name) if parts else None) for lib in libs]
    best = search_log(libs[0], tmp_path / "s", ms[0])
    scales = capi.AU_SCALES if au else None
    keys = PLAIN_KEYS + ("root_id", "alpha", "llh") + (AU_KEYS if au else ())
    res = [m.branch_support(str(tmp_path / "s"), replicates=300, seed=71, atol=atol, keep_rows=True,
                            au_scales=scales) for m in ms]
    same(res[0], res[1], keys)
    rows = [ms[0].site_lnl_rows(p) for p in range(ms[0].partition_count)]
    for p in range(ms[0].partition_count):
        (ra, wa), (rb, wb) = rows[p], ms[1].site_lnl_rows(p)
        assert ra.tobytes() == rb.tobytes() and np.array_equal(wa, wb)
    # item 10 on the engine
    R = ms[0].root_count
    write_log(libs[0], tmp_path / "eq", ms[0], [(q, 0.0, res[0]["alpha"][q], best[3]) for q in range(R)])
    eq = ms[0].placement_support(str(tmp_path / "eq"), replicates=300, seed=71, keep_rows=True, au_scales=scales)
    same(res[0], eq, PLAIN_KEYS + (AU_KEYS if au else ()))
    for p in range(ms[0].partition_count):
        assert rows[p][0].tobytes() == ms[0].site_lnl_rows(p)[0].tobytes()
    for m in ms:
        m.close()


def test_a_one_rank_communicator_returns_the_unsharded_bits(tmp_path):
    import gpu_multi_worker as base
    case = base.build_case()
    got = []
    for sharded in (False, True):
        kw = dict(site_offset=0, global_sites=base.SITES, nranks=1, rank=0, comm_id=capi.comm_unique_id()) \
            if sharded else {}
        m = capi.Model(capi.RootedTree(case.newick), case.aln, base.K, **kw)
        m.initialize_partitions()
        if not sharded:
            search_log(capi.load_tree_lib(), tmp_path / "s", m)
        res = m.branch_support(str(tmp_path / "s"), replicates=200, seed=4, keep_rows=True, au_scales=capi.AU_SCALES)
        got.append((res, m.site_lnl_rows(0)[0].tobytes()))
        m.close()
    same(got[0][0], got[1][0], PLAIN_KEYS + ("alpha", "llh") + AU_KEYS)
    assert got[0][1] == got[1][1]
