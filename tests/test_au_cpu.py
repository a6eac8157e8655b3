"""The AU test and expected likelihood weights of root placement support (DESIGN.md section 10, items
6-8) on the ORACLE-backed model_t: the multiscale counts and ELW against the numpy / Python restatement
(tests/au_reference.py), the fit's edge cases through rdh_placement_au_fit, rd_exp and AS241 against
the standard library and scipy, and what AU mode refuses."""
import ctypes as C
import math

import numpy as np
import pytest

import au_reference
from root_digger_b200 import capi
from test_support_cpu import lib, make_model, thirds, write_records  # noqa: F401  (lib is a fixture)

SCALES = capi.au_thousandths(capi.AU_SCALES)


@pytest.mark.parametrize("name,K,parts", [("10.fasta", 1, False), ("10.fasta", 4, True), ("101.phy", 4, False),
                                          ("101.phy", 1, True)])
def test_au_and_elw_match_the_restated_definition(lib, tmp_path, name, K, parts):  # noqa: F811
    m = make_model(lib, name, K, thirds(name) if parts else None)
    roots = range(m.root_count) if m.root_count < 40 else range(0, m.root_count, 7)
    write_records(lib, tmp_path / "s", m, roots)
    B, seed = 48, 0xC0FFEE1234
    plain = m.placement_support(str(tmp_path / "s"), replicates=B, seed=seed)
    nwk_plain = m.newick(True)
    res = m.placement_support(str(tmp_path / "s"), replicates=B, seed=seed, keep_rows=True,
                              au_scales=capi.AU_SCALES)
    rows, weights = zip(*(m.site_lnl_rows(p) for p in range(m.partition_count)))
    ref = au_reference.support(list(rows), list(weights), B, seed, SCALES)
    assert res["scale_counts"].tolist() == ref["scale_count"]
    assert res["elw_fixed"].tolist() == ref["elw_fixed"]
    for key in ("p_au", "au_d", "au_c", "au_rss"):
        assert np.allclose(res[key], ref[key], rtol=0, atol=1e-12), key
    assert res["au_used"].tolist() == ref["au_used"]
    # the unit scale is today's bootstrap; everything else is the plain call's
    assert res["scale_counts"][SCALES.index(1000)].tolist() == res["bp_count"].tolist()
    for key in ("bp_count", "kh_count", "sh_count", "lnl_fixed", "root_id"):
        assert res[key].tobytes() == plain[key].tobytes(), key
    assert res["O"] == plain["O"] and res["exponent"] == plain["exponent"] and res["best"] == plain["best"]
    assert set(plain) < set(res)
    assert np.array_equal(res["scales"], np.array(capi.AU_SCALES))
    assert (res["scale_counts"].sum(axis=1) == B).all()
    R = len(res["elw"])
    assert abs(res["elw"].sum() - 1.0) <= R * 2.0 ** -40
    assert np.array_equal(res["elw"], np.ldexp(res["elw_fixed"].astype(np.float64), -40) / B)
    nwk = m.newick(True)
    assert "pAU=" in nwk and "ELW=" in nwk
    assert "pAU=" not in nwk_plain and "ELW=" not in nwk_plain


def test_rd_exp_is_within_one_ulp_of_exp():
    assert au_reference.rd_exp(0.0) == 1.0 and au_reference.rd_exp(-0.0) == 1.0
    for x in np.linspace(-40.0, 0.0, 200001).tolist() + [-2.0 ** -29, -0.34657359027997264, -1.0397207708399179]:
        assert abs(au_reference.rd_exp(x) - math.exp(x)) <= math.ulp(math.exp(x)), x


def test_as241_matches_scipy():
    """AS241 against scipy's ndtri (itself accurate to a few ulp): the largest relative difference over
    this grid is 1.02e-15, at p = 0.8628"""
    from scipy.special import ndtri
    p = np.concatenate([np.linspace(1e-6, 1 - 1e-6, 20001), np.logspace(-300, -1, 500),
                        1.0 - np.logspace(-15, -1, 200), [0.075, 0.925]])
    assert au_reference.ppnd16(0.5) == 0.0
    for v in p.tolist():
        want = float(ndtri(v))
        assert abs(au_reference.ppnd16(v) - want) <= 2e-15 * abs(want), v


def au_fit(lib, counts, scales=SCALES, B=1000):  # noqa: F811
    counts = np.ascontiguousarray(counts, dtype=np.uint32)
    sc = np.ascontiguousarray(scales, dtype=np.uint32)
    out, used = np.zeros(4), C.c_uint()
    capi._bind_model(lib)
    if not lib.rdh_placement_au_fit(counts.ctypes.data_as(capi._up), len(sc), sc.ctypes.data_as(capi._up), B,
                                    out.ctypes.data_as(capi._dp), C.byref(used)):
        raise RuntimeError(lib.rdh_last_error().decode())
    return out, used.value


def test_fit_edge_cases(lib):  # noqa: F811
    K = len(SCALES)
    out, used = au_fit(lib, [0] * K)
    assert out.tolist() == [0.0, 0.0, 0.0, 0.0] and used == 0
    out, used = au_fit(lib, [1000] * K)
    assert out.tolist() == [1.0, 0.0, 0.0, 0.0] and used == 0
    one = [0] * 6 + [300] + [1000] * 3
    out, used = au_fit(lib, one)
    assert used == 1 and out[0] == sum(one) / (K * 1000) and out[1:].tolist() == [0.0, 0.0, 0.0]
    # counts of 1 - Phi(d a + c / a) at a large B give back d, c and p_AU = Phi(c - d)
    from scipy.special import ndtr
    B, d, c = 1 << 20, 0.8, 0.3
    a = np.sqrt(np.array(SCALES) / 1000.0)
    counts = np.rint(B * (1.0 - ndtr(d * a + c / a))).astype(np.int64)
    out, used = au_fit(lib, counts, B=B)
    assert used == K
    assert abs(out[1] - d) < 2e-3 and abs(out[2] - c) < 2e-3
    assert abs(out[0] - float(ndtr(c - d))) < 1e-3
    ref = au_reference.au_fit(counts.tolist(), SCALES, B)
    assert np.allclose(out, [ref["p_au"], ref["d"], ref["c"], ref["rss"]], rtol=0, atol=1e-12)


def test_refusals(lib, tmp_path):  # noqa: F811
    m = make_model(lib, "10.fasta", 1)
    write_records(lib, tmp_path / "s", m, range(3))
    prefix = str(tmp_path / "s")
    for scales, match in (([1.0, 0.5], "ascending"), ([0.5, 0.5, 1.0], "ascending"), ([0.05, 1.0], "outside"),
                          ([1.0, 10.5], "outside"), ([1.0], "2 to 32"), ([0.1 + 0.01 * i for i in range(33)], "2 to 32")):
        with pytest.raises(RuntimeError, match=match):
            m.placement_support(prefix, replicates=10, au_scales=scales)
    for scales in ([0.5, 1.0005], [0.5, 0.12345]):
        with pytest.raises(ValueError, match="multiple of 0.001"):
            m.placement_support(prefix, replicates=10, au_scales=scales)
    with pytest.raises(RuntimeError, match="ascending"):
        au_fit(lib, [1, 2], scales=[1000, 900])
    with pytest.raises(RuntimeError, match="2 to 32"):
        au_fit(lib, [1], scales=[1000])
