"""Root placement support (RELL bootstrap proportions, KH and SH tests; DESIGN.md section 10) on the
ORACLE-backed model_t: the integer counts against the numpy / Python-int restatement of the
definition (tests/rell_reference.py), its invariants, the checkpoints it reads and what it refuses."""
import ctypes as C

import numpy as np
import pytest

import fixtures
import oracle_build
import oracle_capi
import rell_reference
from root_digger_b200 import capi


@pytest.fixture(scope="module")
def lib():
    oracle_capi.load_oracle().rdo_set_default_mode(oracle_capi.MODE_ENGINE)
    return capi.load_tree_lib(oracle_build.build_host_on_oracle())


def make_model(lib, name="10.fasta", K=1, partitions=None):
    fx = fixtures.load(name)
    tree = capi.RootedTree(path=str(fx["tree_path"]), lib=lib)
    m = capi.Model(tree, fx["alignment"], rate_cats=K, compress=True, seed=7, partitions=partitions)
    m.initialize_partitions(uniform_freqs=False)
    return m


def thirds(name):
    n = len(next(iter(fixtures.load(name)["alignment"].values())))
    return [(0, n // 3), (n // 3, 2 * n // 3), (2 * n // 3, n)]


def write_records(lib, prefix, m, roots, seed=1):
    """one record per root id, with its own parameters per partition"""
    rng = np.random.default_rng(seed)
    ckp = capi.Checkpoint(str(prefix), lib=lib)
    ckp.save_options(prefix=str(prefix))
    for rid in roots:
        params = []
        for _ in range(m.partition_count):
            f = rng.uniform(0.5, 1.5, 4)
            params.append({"rates": rng.uniform(0.2, 2.0, 12), "freqs": f / f.sum(),
                           "alpha": float(rng.uniform(0.3, 3.0)), "weights": np.full(m.K, 1.0 / m.K)})
        ckp.write(int(rid), -1000.0 - rid, float(rng.uniform(0.0, 1.0)), params, K=m.K)
    ckp.close()


def reference(m, res, replicates, seed):
    rows, weights = zip(*(m.site_lnl_rows(p) for p in range(m.partition_count)))
    return rows, weights, rell_reference.support(list(rows), list(weights), replicates, seed)


def assert_same(res, ref):
    assert res["exponent"] == ref["exponent"]
    assert res["best"] == ref["best"]
    for key in ("bp_count", "kh_count", "sh_count"):
        assert res[key].tolist() == ref[key], key
    assert res["lnl_fixed"].tolist() == ref["lnl_fixed"]
    assert res["O"] == ref["O"]


@pytest.mark.parametrize("name,K,parts", [("10.fasta", 1, False), ("10.fasta", 4, True), ("101.phy", 4, False),
                                          ("101.phy", 1, True)])
def test_counts_match_the_restated_definition(lib, tmp_path, name, K, parts):
    m = make_model(lib, name, K, thirds(name) if parts else None)
    roots = range(m.root_count) if m.root_count < 40 else range(0, m.root_count, 7)
    write_records(lib, tmp_path / "s", m, roots)
    B, seed = 48, 0xC0FFEE1234
    res = m.placement_support(str(tmp_path / "s"), replicates=B, seed=seed, keep_rows=True)
    assert res["root_id"].tolist() == list(roots)
    rows, weights, ref = reference(m, res, B, seed)
    assert_same(res, ref)
    assert res["bp_count"].sum() == B
    assert res["kh_count"][res["best"]] == B and res["sh_count"][res["best"]] == B
    assert np.allclose(res["bp"] * B, res["bp_count"])
    # lnl_fixed is the full log-likelihood of the record up to the grid
    total = sum((L * w).sum(axis=1) for L, w in zip(rows, weights))
    assert np.allclose(res["lnl_fixed"], total, rtol=1e-12, atol=0)


def test_same_seed_same_counts_other_seed_other_counts(lib, tmp_path):
    m = make_model(lib, "10.fasta", 4)
    write_records(lib, tmp_path / "s", m, range(m.root_count))
    a = m.placement_support(str(tmp_path / "s"), replicates=200, seed=1)
    b = m.placement_support(str(tmp_path / "s"), replicates=200, seed=1)
    c = m.placement_support(str(tmp_path / "s"), replicates=200, seed=2)
    for key in ("bp_count", "kh_count", "sh_count", "lnl_fixed"):
        assert np.array_equal(a[key], b[key])
    assert any(not np.array_equal(a[k], c[k]) for k in ("bp_count", "kh_count", "sh_count"))
    assert np.array_equal(a["lnl_fixed"], c["lnl_fixed"])


def test_rows_times_weights_are_the_persite_values_of_the_oracle():
    """the unweighted row is what the weighted per-site value is made of: dmul(L, w) == persite"""
    from cases import Case, compute_lh
    case = Case(12, 700, 4, seed=3, data="evolved", weights="random")
    o = oracle_capi.OraclePartition(case.n, case.S, case.K)
    case.setup(o)
    sched = case.full_schedule(0, 0.5)
    lw, pw = compute_lh(o, sched, case.root_clv, case.root_scaler, persite=True, mode=oracle_capi.MODE_ENGINE)
    o.set_pattern_weights(np.ones(case.S, dtype=np.uint32))
    _, L = o.root_loglikelihood(case.root_clv, case.root_scaler, persite=True, mode=oracle_capi.MODE_ENGINE)
    assert np.array_equal(L * case.weights.astype(np.float64), pw)


def test_checkpoint_of_exhaustive_search(lib, tmp_path):
    m = make_model(lib, "10.fasta", 1)
    m.set_checkpoint(str(tmp_path / "x"))
    m.set_max_outer_iterations(1)
    ids, llh, _ = m.exhaustive_search(1e-3, 1e-3, 1e-3, 1e12, rank=0, num_tasks=4)
    res = m.placement_support(str(tmp_path / "x"), replicates=64, seed=9, keep_rows=True)
    assert res["root_id"].tolist() == ids.tolist() and np.array_equal(res["llh"], llh)
    # the recorded log-likelihood is the model's, on the fixed-point grid
    assert np.allclose(res["lnl_fixed"], llh, rtol=1e-9, atol=0)
    _, _, ref = reference(m, res, 64, 9)
    assert_same(res, ref)
    # the model's own log (None) is the same checkpoint here
    again = m.placement_support(None, replicates=64, seed=9, keep_rows=True)
    assert np.array_equal(again["bp_count"], res["bp_count"])
    nwk = m.newick(True)
    assert "BP=" in nwk and "pKH=" in nwk and "pSH=" in nwk


def test_parameters_and_root_are_put_back(lib, tmp_path):
    m = make_model(lib, "10.fasta", 4)
    write_records(lib, tmp_path / "s", m, range(m.root_count))
    m.set_params(alpha=0.77)
    lh = m.compute_lh(5, 0.3)
    before = m.get_params()
    nwk = m.newick(False)
    m.placement_support(str(tmp_path / "s"), replicates=16, seed=4)
    for a, b in zip(before, m.get_params()):
        assert np.array_equal(a, b)
    assert m.newick(False) == nwk
    assert m.compute_lh_root(5, 0.3) == lh and m.compute_lh(5, 0.3) == lh


def test_refusals(lib, tmp_path):
    m = make_model(lib, "10.fasta", 1)
    empty = capi.Checkpoint(str(tmp_path / "empty"), lib=lib)
    empty.save_options(prefix="empty")
    empty.close()
    with pytest.raises(RuntimeError, match="no records"):
        m.placement_support(str(tmp_path / "empty"), replicates=10)
    with pytest.raises(RuntimeError, match="no checkpoint"):
        m.placement_support(str(tmp_path / "absent"), replicates=10)
    write_records(lib, tmp_path / "s", m, range(3))
    for B in (0, (1 << 20) + 1):
        with pytest.raises(RuntimeError, match="replicates"):
            m.placement_support(str(tmp_path / "s"), replicates=B)
    write_records(lib, tmp_path / "far", m, [m.root_count])
    with pytest.raises(RuntimeError, match="root id out of range"):
        m.placement_support(str(tmp_path / "far"), replicates=10)
    three = make_model(lib, "10.fasta", 1, thirds("10.fasta"))
    write_records(lib, tmp_path / "three", three, range(3))
    with pytest.raises(RuntimeError, match="parameter sets"):
        m.placement_support(str(tmp_path / "three"), replicates=10)
    k4 = make_model(lib, "10.fasta", 4)
    write_records(lib, tmp_path / "ok", k4, range(3))
    # a partition-sharded model is refused
    fn_t = C.CFUNCTYPE(None, C.POINTER(C.c_double), C.c_size_t, C.c_size_t, C.POINTER(C.c_double), C.c_void_p)

    def exchange(local, n_local, count, all_terms, _user):
        C.memmove(all_terms, local, 8 * n_local * count)

    fn = fn_t(exchange)
    lib.rdh_model_set_partition_exchange.argtypes = [C.c_void_p, C.POINTER(C.c_uint), C.c_uint, C.c_uint, fn_t,
                                                     C.c_void_p]
    idx = (C.c_uint * 1)(0)
    assert lib.rdh_model_set_partition_exchange(k4.h, idx, 1, 1, fn, None)
    with pytest.raises(RuntimeError, match="several processes"):
        k4.placement_support(str(tmp_path / "ok"), replicates=10)
    lib.rdh_model_set_partition_exchange(k4.h, None, 0, 0, C.cast(None, fn_t), None)


def test_read_only_log_all_records_and_rows_freed(lib, tmp_path):
    """a log the user may not write is read; more records than the first output buffers hold; the
    rows are freed on return unless kept"""
    import os
    import stat
    m = make_model(lib, "101.phy", 1)
    write_records(lib, tmp_path / "ro", m, range(m.root_count))
    path = str(tmp_path / "ro") + ".ckp"
    before = open(path, "rb").read()
    os.chmod(path, stat.S_IRUSR)
    os.chmod(tmp_path, stat.S_IRUSR | stat.S_IXUSR)
    try:
        res = m.placement_support(str(tmp_path / "ro"), replicates=8, seed=2, keep_rows=True)
        rows, _ = m.site_lnl_rows(0)
        again = m.placement_support(str(tmp_path / "ro"), replicates=8, seed=2)
    finally:
        os.chmod(tmp_path, stat.S_IRWXU)
        os.chmod(path, stat.S_IRUSR | stat.S_IWUSR)
    assert open(path, "rb").read() == before
    assert res["root_id"].tolist() == list(range(m.root_count)) and rows.shape[0] == m.root_count
    assert np.array_equal(res["bp_count"], again["bp_count"]) and res["O"] == again["O"]
    assert m.site_lnl_rows(0)[0].shape[0] == 0
