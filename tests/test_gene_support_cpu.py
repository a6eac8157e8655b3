"""Gene and gene-then-site resampling of root placement support (DESIGN.md section 10, items 11-14) on
the ORACLE-backed model_t: placement_support and branch_support in both gene modes against the numpy /
Python-int restatement (tests/gene_reference.py), their invariants against site mode, and what the
gene modes refuse."""
import numpy as np
import pytest

import gene_reference
from test_branch_support_cpu import search_log
from test_support_cpu import lib, make_model, thirds, write_records  # noqa: F401  (lib is a fixture)

PLAIN_KEYS = ("O", "exponent", "best", "lnl_fixed")
COUNT_KEYS = ("bp_count", "kh_count", "sh_count")


def parts_of(name, G):
    if G == 3:
        return thirds(name)
    import fixtures
    n = len(next(iter(fixtures.load(name)["alignment"].values())))
    return [(i * n // G, (i + 1) * n // G) for i in range(G)]


# 10.fasta in thirds (K = 4), 101.phy in thirds (K = 1), 101.phy in 16 partitions (K = 4)
CASES = [("10.fasta", 4, 3), ("101.phy", 1, 3), ("101.phy", 4, 16)]


def check_against_reference(m, res, B, seed, sampling):
    rows = [m.site_lnl_rows(p) for p in range(m.partition_count)]
    ref = gene_reference.support([r for r, _ in rows], [w for _, w in rows], B, seed, sampling)
    assert res["exponent"] == ref["exponent"] and res["best"] == ref["best"] and res["O"] == ref["O"]
    assert res["lnl_fixed"].tolist() == ref["lnl_fixed"]
    for key in COUNT_KEYS:
        assert res[key].tolist() == ref[key], key
    assert res["partition_O"] == ref["partition_O"]
    assert res["partition_llh"].tolist() == ref["partition_llh"]
    assert res["partition_best"].tolist() == ref["partition_best"]
    return ref


@pytest.mark.parametrize("sampling", ["gene", "gene_site"])
@pytest.mark.parametrize("name,K,G", CASES)
def test_placement_support_matches_the_restated_definition(lib, tmp_path, name, K, G, sampling):  # noqa: F811
    m = make_model(lib, name, K, parts_of(name, G))
    roots = range(m.root_count) if m.root_count < 40 else range(0, m.root_count, 7)
    write_records(lib, tmp_path / "s", m, roots)
    B, seed = 48, 0xC0FFEE1234
    site = m.placement_support(str(tmp_path / "s"), replicates=B, seed=seed)
    res = m.placement_support(str(tmp_path / "s"), replicates=B, seed=seed, keep_rows=True, sampling=sampling)
    assert res["sampling"] == sampling
    ref = check_against_reference(m, res, B, seed, sampling)
    if G == 16:  # partitions drawn more than once and not at all
        assert (ref["m"] > 1).any() and (ref["m"] == 0).any()
    # O is the sum of the gene-wise O_i, and everything but the counts is site mode's
    assert [sum(col) for col in zip(*res["partition_O"])] == res["O"]
    for key in PLAIN_KEYS:
        assert (res[key] == site[key]) if key != "lnl_fixed" else res[key].tobytes() == site[key].tobytes(), key
    assert res["bp_count"].sum() == B
    assert res["kh_count"][res["best"]] == B and res["sh_count"][res["best"]] == B
    nwk = m.newick(True)
    assert "BP=" in nwk and "pKH=" in nwk and "pSH=" in nwk


@pytest.mark.parametrize("sampling", ["gene", "gene_site"])
@pytest.mark.parametrize("name,K,G", CASES)
def test_branch_support_matches_the_restated_definition(lib, tmp_path, name, K, G, sampling):  # noqa: F811
    m = make_model(lib, name, K, parts_of(name, G))
    search_log(lib, tmp_path / "s", m)
    B, seed = 40, 0xBADC0FFEE
    site = m.branch_support(str(tmp_path / "s"), replicates=B, seed=seed, atol=1e-6)
    res = m.branch_support(str(tmp_path / "s"), replicates=B, seed=seed, atol=1e-6, keep_rows=True,
                           sampling=sampling)
    check_against_reference(m, res, B, seed, sampling)
    for key in PLAIN_KEYS + ("alpha", "llh"):
        assert (res[key] == site[key]) if key in ("O", "exponent", "best") else \
            res[key].tobytes() == site[key].tobytes(), key
    assert res["root_id"].tolist() == list(range(m.root_count))
    nwk = m.newick(True)
    for key in ("BP=", "pKH=", "pSH=", "LLH="):
        assert nwk.count(key) >= m.root_count, key


def test_site_mode_is_unchanged_by_a_gene_call(lib, tmp_path):  # noqa: F811
    m = make_model(lib, "10.fasta", 4, thirds("10.fasta"))
    write_records(lib, tmp_path / "s", m, range(m.root_count))
    kw = dict(replicates=64, seed=5)
    before = m.placement_support(str(tmp_path / "s"), **kw)
    m.placement_support(str(tmp_path / "s"), sampling="gene_site", **kw)
    after = m.placement_support(str(tmp_path / "s"), **kw)
    assert set(before) == set(after) and "sampling" not in before
    for key, v in before.items():
        if key.endswith("_ms"):  # timings
            continue
        assert v.tobytes() == after[key].tobytes() if isinstance(v, np.ndarray) else v == after[key], key


def test_same_seed_same_counts_other_seed_or_mode_other_counts(lib, tmp_path):  # noqa: F811
    m = make_model(lib, "101.phy", 1, parts_of("101.phy", 16))
    write_records(lib, tmp_path / "s", m, range(0, m.root_count, 5))
    s = str(tmp_path / "s")

    def counts(**kw):
        r = m.placement_support(s, replicates=200, **kw)
        return np.concatenate([r[k] for k in COUNT_KEYS])

    a, b = counts(seed=1, sampling="gene"), counts(seed=1, sampling="gene")
    assert np.array_equal(a, b)
    assert not np.array_equal(a, counts(seed=2, sampling="gene"))
    assert not np.array_equal(a, counts(seed=1, sampling="gene_site"))
    assert not np.array_equal(counts(seed=1, sampling="gene_site"), counts(seed=1))


@pytest.mark.parametrize("call", ["placement_support", "branch_support"])
def test_parameters_and_root_are_put_back_and_rows_freed(lib, tmp_path, call):  # noqa: F811
    m = make_model(lib, "10.fasta", 4, thirds("10.fasta"))
    write_records(lib, tmp_path / "s", m, range(m.root_count))
    m.set_params(alpha=0.77)
    lh = m.compute_lh(5, 0.3)
    before = [m.get_params(p) for p in range(m.partition_count)]
    nwk = m.newick(False)
    getattr(m, call)(str(tmp_path / "s"), replicates=16, seed=4, sampling="gene")
    for p, params in enumerate(before):
        for a, b in zip(params, m.get_params(p)):
            assert a.tobytes() == b.tobytes()
    assert m.newick(False) == nwk
    assert m.compute_lh_root(5, 0.3) == lh and m.compute_lh(5, 0.3) == lh
    assert m.site_lnl_rows(0)[0].shape[0] == 0


def test_refusals(lib, tmp_path):  # noqa: F811
    one = make_model(lib, "10.fasta", 1)
    write_records(lib, tmp_path / "one", one, range(3))
    for call in ("placement_support", "branch_support"):
        with pytest.raises(RuntimeError, match=call + ": gene sampling needs at least 2 partitions"):
            getattr(one, call)(str(tmp_path / "one"), replicates=10, sampling="gene")
    m = make_model(lib, "10.fasta", 1, thirds("10.fasta"))
    write_records(lib, tmp_path / "s", m, range(3))
    s = str(tmp_path / "s")
    for call in ("placement_support", "branch_support"):
        with pytest.raises(ValueError, match=call + ": the AU test and ELW"):
            getattr(m, call)(s, replicates=10, sampling="gene_site", au_scales=(0.5, 1.0))
        with pytest.raises(ValueError, match=call + ": unknown sampling"):
            getattr(m, call)(s, replicates=10, sampling="genes")
        with pytest.raises(RuntimeError, match="replicates"):
            getattr(m, call)(s, replicates=0, sampling="gene")
    # the C entries refuse an unknown mode code
    with pytest.raises(RuntimeError, match="unknown sampling mode 3"):
        m._check(m.L.rdh_model_placement_support_genes(m.h, s.encode(), 10, 1, 0, 0, 3, 8, *([None] * 17)))
    # nothing was left behind by the refusals
    assert m.placement_support(s, replicates=8, sampling="gene")["bp_count"].sum() == 8
