"""Branch support (DESIGN.md section 10, items 9-10) on the ORACLE-backed model_t: the support
statistics of every branch at the parameters of a checkpoint's best record, with each root at its
best position on its branch.  Pinned by item 10 -- placement_support on a checkpoint of one record per
root id q, at (q, a_q) with the best record's parameters, returns the same bits -- and by the
restatements of the statistics (tests/rell_reference.py, tests/au_reference.py) on the kept rows."""
import numpy as np
import pytest

import au_reference
import rell_reference
from root_digger_b200 import capi
from test_support_cpu import lib, make_model, thirds  # noqa: F401  (lib is a fixture)

SCALES = capi.au_thousandths(capi.AU_SCALES)
PLAIN_KEYS = ("O", "exponent", "best", "bp_count", "kh_count", "sh_count", "lnl_fixed")
AU_KEYS = ("scale_counts", "elw_fixed", "p_au", "au_d", "au_c", "au_rss", "au_used")


def random_params(m, rng):
    out = []
    for _ in range(m.partition_count):
        f = rng.uniform(0.5, 1.5, 4)
        out.append({"rates": rng.uniform(0.2, 2.0, 12), "freqs": f / f.sum(), "alpha": float(rng.uniform(0.3, 3.0)),
                    "weights": np.full(m.K, 1.0 / m.K)})
    return out


def write_log(lib, prefix, m, records):  # noqa: F811
    """records: (root id, llh, alpha, parameters per partition)"""
    ckp = capi.Checkpoint(str(prefix), lib=lib)
    ckp.save_options(prefix=str(prefix))
    for rid, llh, alpha, params in records:
        ckp.write(int(rid), float(llh), float(alpha), params, K=m.K)
    ckp.close()


def search_log(lib, prefix, m, seed=5):  # noqa: F811
    """a search-mode-like log: a few records on neighbouring branches, each with its own parameters;
    the best (highest llh) is returned with the log"""
    rng = np.random.default_rng(seed)
    recs = [(rid, -1000.0 - rid, float(rng.uniform(0.1, 0.9)), random_params(m, rng)) for rid in (4, 2, 3, 6)]
    write_log(lib, prefix, m, recs)
    return max(recs, key=lambda r: r[1])


def install(m, params):
    """the best record's parameters, installed as model_t::install_record installs them"""
    for p, pp in enumerate(params):
        f = np.asarray(pp["freqs"], dtype=np.float64)
        total = 0.0
        for v in f.tolist():
            total += v
        m.set_params(rates=pp["rates"], freqs=f / total, alpha=pp["alpha"], part=p)


def same(a, b, keys):
    for k in keys:
        if k == "O" or isinstance(a[k], (int, float)):
            assert a[k] == b[k], k
        else:
            assert np.asarray(a[k]).tobytes() == np.asarray(b[k]).tobytes(), k


def rows_of(m):
    return [m.site_lnl_rows(p) for p in range(m.partition_count)]


CASES = [("10.fasta", 1, False, 1e-14), ("10.fasta", 4, True, 1e-14), ("101.phy", 4, False, 1e-6)]


@pytest.mark.parametrize("au", [False, True])
@pytest.mark.parametrize("name,K,parts,atol", CASES)
def test_branch_support_equals_placement_support_on_the_equivalent_log(lib, tmp_path, name, K, parts, atol, au):  # noqa: F811
    m = make_model(lib, name, K, thirds(name) if parts else None)
    best = search_log(lib, tmp_path / "s", m)
    B, seed = 40, 0xBADC0FFEE
    scales = capi.AU_SCALES if au else None
    res = m.branch_support(str(tmp_path / "s"), replicates=B, seed=seed, atol=atol, keep_rows=True, au_scales=scales)
    R = m.root_count
    assert res["root_id"].tolist() == list(range(R))
    assert ((res["alpha"] >= 0) & (res["alpha"] <= 1)).all() and (res["alpha"] != 0.5).any()
    assert res["positions_ms"] >= 0 and res["capture_ms"] >= 0
    rows = rows_of(m)
    # the restated statistics on the kept rows
    L, W = [r for r, _ in rows], [w for _, w in rows]
    ref = rell_reference.support(L, W, B, seed)
    assert res["best"] == ref["best"] and res["exponent"] == ref["exponent"] and res["O"] == ref["O"]
    for key in ("bp_count", "kh_count", "sh_count"):
        assert res[key].tolist() == ref[key], key
    assert res["lnl_fixed"].tolist() == ref["lnl_fixed"]
    if au:
        ref = au_reference.support(L, W, B, seed, SCALES)
        assert res["scale_counts"].tolist() == ref["scale_count"]
        assert res["elw_fixed"].tolist() == ref["elw_fixed"]
        assert res["au_used"].tolist() == ref["au_used"]
    # item 10: the equivalent checkpoint through placement_support, every key and every row
    write_log(lib, tmp_path / "eq", m, [(q, 0.0, res["alpha"][q], best[3]) for q in range(R)])
    eq = m.placement_support(str(tmp_path / "eq"), replicates=B, seed=seed, keep_rows=True, au_scales=scales)
    same(res, eq, PLAIN_KEYS + (AU_KEYS if au else ()))
    assert np.array_equal(res["alpha"], eq["alpha"])
    for (a, wa), (b, wb) in zip(rows, rows_of(m)):
        assert a.tobytes() == b.tobytes() and np.array_equal(wa, wb)
    # llh: the sweep's log-likelihood at (q, a_q) is compute_lh_root there, bit for bit
    install(m, best[3])
    m.compute_lh(best[0], best[2])
    for q in range(0, R, max(1, R // 25)):
        m.move_root(q, res["alpha"][q])
        assert m.compute_lh_root(q, res["alpha"][q]) == res["llh"][q], q
    # the whole log-likelihood up to the fixed-point grid
    assert np.allclose(res["lnl_fixed"], res["llh"], rtol=1e-12, atol=0)


def test_without_a_position_search_the_placements_are_those_suggest_roots_lh_ranks(lib, tmp_path):  # noqa: F811
    m = make_model(lib, "10.fasta", 4, thirds("10.fasta"))
    best = search_log(lib, tmp_path / "s", m)
    res = m.branch_support(str(tmp_path / "s"), replicates=16, seed=3, atol=0.0)
    assert (res["alpha"] == 0.5).all()
    assert res["positions_ms"] < 50.0  # no search at all
    install(m, best[3])
    m.compute_lh(best[0], best[2])
    assert res["llh"].tobytes() == m.sweep_root_lh().tobytes()


def test_every_branch_is_annotated_and_the_model_is_unchanged(lib, tmp_path):  # noqa: F811
    m = make_model(lib, "10.fasta", 4)
    search_log(lib, tmp_path / "s", m)
    rid, ratio = 5, 0.3
    before = m.compute_lh(rid, ratio)
    params = [m.get_params(p) for p in range(m.partition_count)]
    res = m.branch_support(str(tmp_path / "s"), replicates=32, seed=1, au_scales=capi.AU_SCALES)
    nwk = m.newick(True)
    R = m.root_count
    for key in ("BP=", "pKH=", "pSH=", "pAU=", "ELW=", "LLH=", "alpha="):
        # a branch is written once per end point it is annotated on; every branch carries every key
        assert nwk.count(key) >= R, key
    for p, (r, f, c) in enumerate(params):
        r2, f2, c2 = m.get_params(p)
        assert r.tobytes() == r2.tobytes() and f.tobytes() == f2.tobytes() and c.tobytes() == c2.tobytes()
    assert m.compute_lh(rid, ratio) == before
    assert res["bp_count"].sum() == 32


def test_the_best_record_is_the_first_of_equal_log_likelihoods(lib, tmp_path):  # noqa: F811
    m = make_model(lib, "10.fasta", 1)
    rng = np.random.default_rng(11)
    a, b, c = (random_params(m, rng) for _ in range(3))
    write_log(lib, tmp_path / "tie", m, [(1, -1100.0, 0.2, c), (3, -1000.0, 0.4, a), (6, -1000.0, 0.7, b)])
    write_log(lib, tmp_path / "a", m, [(3, -1000.0, 0.4, a)])
    write_log(lib, tmp_path / "b", m, [(6, -1000.0, 0.7, b)])
    kw = dict(replicates=24, seed=2, atol=1e-10)
    tie, first, second = (m.branch_support(str(tmp_path / x), **kw) for x in ("tie", "a", "b"))
    same(tie, first, PLAIN_KEYS + ("alpha", "llh"))
    assert tie["llh"].tobytes() != second["llh"].tobytes()


def test_what_branch_support_refuses(lib, tmp_path):  # noqa: F811
    m = make_model(lib, "10.fasta", 1)
    search_log(lib, tmp_path / "s", m)
    s = str(tmp_path / "s")
    with pytest.raises(RuntimeError, match="replicates"):
        m.branch_support(s, replicates=0)
    with pytest.raises(RuntimeError, match="replicates"):
        m.branch_support(s, replicates=(1 << 20) + 1)
    with pytest.raises(RuntimeError, match="atol"):
        m.branch_support(s, replicates=8, atol=-1e-9)
    with pytest.raises(RuntimeError, match="atol"):
        m.branch_support(s, replicates=8, atol=float("nan"))
    with pytest.raises(RuntimeError, match="scale"):
        m.branch_support(s, replicates=8, au_scales=(1.0, 0.5))
    write_log(lib, tmp_path / "empty", m, [])
    with pytest.raises(RuntimeError, match="no records"):
        m.branch_support(str(tmp_path / "empty"), replicates=8)
    rng = np.random.default_rng(0)
    write_log(lib, tmp_path / "far", m, [(m.root_count + 3, -1.0, 0.5, random_params(m, rng))])
    with pytest.raises(RuntimeError, match="root id out of range"):
        m.branch_support(str(tmp_path / "far"), replicates=8)
    write_log(lib, tmp_path / "pos", m, [(2, -1.0, 1.5, random_params(m, rng))])
    with pytest.raises(RuntimeError, match="outside"):
        m.branch_support(str(tmp_path / "pos"), replicates=8)
    m3 = make_model(lib, "10.fasta", 1, thirds("10.fasta"))
    with pytest.raises(RuntimeError, match="parameter sets"):
        m3.branch_support(s, replicates=8)
    # nothing was left behind by the refusals
    assert m.branch_support(s, replicates=8)["bp_count"].sum() == 8


def test_a_model_dealt_to_several_processes_is_refused(lib, tmp_path):  # noqa: F811
    import ctypes as C
    m = make_model(lib, "10.fasta", 4)
    search_log(lib, tmp_path / "s", m)
    fn_t = C.CFUNCTYPE(None, C.POINTER(C.c_double), C.c_size_t, C.c_size_t, C.POINTER(C.c_double), C.c_void_p)

    def exchange(local, n_local, count, all_terms, _user):
        C.memmove(all_terms, local, 8 * n_local * count)

    fn = fn_t(exchange)
    lib.rdh_model_set_partition_exchange.argtypes = [C.c_void_p, C.POINTER(C.c_uint), C.c_uint, C.c_uint, fn_t,
                                                     C.c_void_p]
    idx = (C.c_uint * 1)(0)
    assert lib.rdh_model_set_partition_exchange(m.h, idx, 1, 1, fn, None)
    with pytest.raises(RuntimeError, match="several processes"):
        m.branch_support(str(tmp_path / "s"), replicates=10)
    lib.rdh_model_set_partition_exchange(m.h, None, 0, 0, C.cast(None, fn_t), None)
