"""Marginal ancestral states (DESIGN.md section 11) on the ORACLE-backed model_t: against the numpy
restatement (tests/ancestral_reference.py) and brute-force enumeration, the identity between every
node's normaliser and the site log-likelihood, the model state around the call, the checkpoint form,
the refusals, the .state file and the column map."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

import ancestral_reference as ref
import fixtures
import oracle_capi
from root_digger_b200 import capi
from test_support_cpu import lib, make_model, thirds  # noqa: F401  (lib is a fixture)


def placed(m, rid, ratio, **kw):
    """ancestral_states at (rid, ratio) on a model rooted there: the call puts the rooting back, so the
    oracle partition then holds the P-matrices and tip CLVs the call used"""
    m.compute_lh(rid, ratio)
    return m.ancestral_states(rid, ratio, **kw)


def inputs(m, res, part=0):
    """the operations of an ancestral_states result (see placed), and its P-matrices and tip CLVs"""
    ops = [tuple(int(x) for x in o) for o in res["ops"]]
    p = C.cast(m.L.rdh_model_partition(m.h, part), C.POINTER(oracle_capi.OraclePartitionStruct)).contents
    S, K = p.sites, p.rate_cats
    P = {}
    tips = {}
    for op in ops:
        for c, mi in ((op[2], op[3]), (op[5], op[6])):
            P[mi] = np.ctypeslib.as_array(p.pmatrix[mi], shape=(K * 16,)).reshape(K, 4, 4).copy()
            if c < p.tips:
                tips[c] = np.ctypeslib.as_array(p.clv[c], shape=(S * K * 4,)).reshape(S, K, 4).copy()
    pi = np.ctypeslib.as_array(p.frequencies[0], shape=(4,)).copy()
    w = np.ctypeslib.as_array(p.rate_weights, shape=(K,)).copy()
    weights = np.ctypeslib.as_array(p.pattern_weights, shape=(S,)).copy()
    return ops, P, tips, pi, w, weights


def tree_of(name, lib):  # noqa: F811
    return capi.RootedTree(path=str(fixtures.load(name)["tree_path"]), lib=lib)


def rel(a, b, floor=1e-300):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), floor))


@pytest.mark.parametrize("name,K,rid,ratio", [("10.fasta", 1, 3, 0.3), ("10.fasta", 4, 0, 0.5), ("101.phy", 4, 57, 0.8),
                                              ("101.phy", 1, 120, 0.0)])
def test_the_host_equals_the_restatement_and_the_identity_holds(lib, name, K, rid, ratio):  # noqa: F811
    m = make_model(lib, name, K)
    res = placed(m, rid, ratio, full_nodes="all")
    ops, P, tips, pi, w, weights = inputs(m, res)
    assert res["nodes"].tolist() == [o[0] for o in ops]
    r = ref.marginal(ops, P, tips, pi, w)
    assert rel(res["posterior"][0], r["posterior"]) < 1e-13
    assert rel(res["log_norm"][0], r["log_norm"], 1.0) < 1e-13  # log(Z) ~ 0 where a pattern is all gaps
    assert rel(res["map_prob"][0], r["map_prob"]) < 1e-13
    # MAP states agree wherever the top two posteriors are not within rounding of each other
    srt = np.sort(r["posterior"], axis=2)
    clear = srt[:, :, 3] - srt[:, :, 2] > 1e-12
    assert np.array_equal(np.frombuffer(b"ACGT", np.uint8)[r["map_state"]][clear], res["map_state"][0][clear])
    # identity: every node's normaliser is the site log-likelihood of the rooted tree
    ln = res["log_norm"][0]
    assert rel(ln, np.broadcast_to(ln[-1], ln.shape), 1.0) < 1e-12
    lh = m.compute_lh(rid, ratio)
    assert abs(float(np.dot(ln[-1], weights)) - lh) <= 1e-12 * abs(lh)
    assert np.allclose(res["posterior"][0].sum(axis=2), 1.0, atol=1e-14)


SMALL = "((a:0.1,b:0.2):0.05,((c:0.3,d:0.1):0.2,(e:0.15,f:0.25):0.1):0.1);"
SMALL_ALN = {"a": "ACGTTGCAAN", "b": "ACGTAGCTRA", "c": "AGGTTCCAAA", "d": "ACCTTGCAYA", "e": "TCGTTGGAAA",
             "f": "ACGATGCAAC"}


SMALL_PARTS = [(0, 4), (4, 10)]
GOLDEN_ROOT = 5


def small_model(lib, K, partitions=None):  # noqa: F811
    m = capi.Model(capi.RootedTree(SMALL, lib=lib), SMALL_ALN, rate_cats=K, compress=True, seed=3,
                   partitions=partitions)
    m.initialize_partitions(uniform_freqs=False)
    for p in range(m.partition_count):
        m.set_params(rates=np.linspace(0.3, 2.1, 12), freqs=np.array([0.1, 0.2, 0.3, 0.4]), alpha=0.7, part=p)
    return m


@pytest.mark.parametrize("K", [1, 4])
@pytest.mark.parametrize("ratio", [0.0, 0.3, 1.0])
def test_the_posteriors_are_those_of_enumerating_every_assignment(lib, K, ratio):  # noqa: F811
    m = small_model(lib, K)
    for rid in range(m.root_count):
        res = placed(m, rid, ratio, full_nodes="all")
        ops, P, tips, pi, w, _ = inputs(m, res)
        bf = ref.brute_force(ops, P, tips, pi, w)
        assert np.max(np.abs(res["posterior"][0] - bf)) < 1e-12


def test_model_state_is_unchanged_and_the_checkpoint_form_is_the_plain_call(lib, tmp_path):  # noqa: F811
    from test_branch_support_cpu import install, search_log
    m = make_model(lib, "101.phy", 4)
    before = m.compute_lh(5, 0.4)
    m.ancestral_states(40, 0.2, full_nodes="all")
    after = m.compute_lh(5, 0.4)
    assert np.float64(before).tobytes() == np.float64(after).tobytes()
    best = search_log(lib, tmp_path / "s", m)
    got = m.ancestral_states(checkpoint_prefix=str(tmp_path / "s"), full_nodes="all")
    assert np.float64(m.compute_lh(5, 0.4)).tobytes() == np.float64(before).tobytes()
    rid, _llh, alpha, params = best
    install(m, params)
    want = m.ancestral_states(rid, alpha, full_nodes="all")
    assert got["root_id"] == rid and got["ratio"] == alpha
    for key in ("map_state", "map_prob", "posterior", "log_norm"):
        assert got[key][0].tobytes() == want[key][0].tobytes(), key


def test_what_ancestral_states_refuses(lib):  # noqa: F811
    m = make_model(lib, "10.fasta", 1)
    with pytest.raises(RuntimeError, match="outside"):
        m.ancestral_states(2, 1.5)
    with pytest.raises(RuntimeError, match="not an internal node"):
        m.ancestral_states(2, 0.5, full_nodes=[3])
    v = int(m.ancestral_states(2, 0.5)["nodes"][0])
    with pytest.raises(RuntimeError, match="listed twice"):
        m.ancestral_states(2, 0.5, full_nodes=[v, v])
    with pytest.raises(ValueError):
        m.ancestral_states(full_nodes="root")

    def exchange(local, n_local, count, all_terms, _user):
        for i in range(n_local * count):
            all_terms[i] = local[i]

    fn = C.CFUNCTYPE(None, C.POINTER(C.c_double), C.c_size_t, C.c_size_t, C.POINTER(C.c_double), C.c_void_p)(exchange)
    gi = (C.c_uint * 1)(0)
    assert m.L.rdh_model_set_partition_exchange(m.h, gi, 1, 1, fn, None)
    with pytest.raises(RuntimeError, match="several processes"):
        m.ancestral_states(2, 0.5)


def test_columns_map_to_their_patterns_and_the_state_file(lib, tmp_path):  # noqa: F811
    fx = fixtures.load("10.fasta")
    aln = fx["alignment"]
    m = make_model(lib, "10.fasta", 4)
    cols = m.pattern_of_column(0)
    L = len(next(iter(aln.values())))
    assert len(cols) == L and cols.max() + 1 == m.sites(0)
    res = m.ancestral_states(4, 0.5)
    seqs = [aln[t] for t in sorted(aln)]
    # identical columns share a pattern, and the expanded root sequence has one state per column
    for c in range(0, L, 37):
        same = [d for d in range(L) if all(s[d].upper() == s[c].upper() for s in seqs)]
        assert len(set(cols[same].tolist())) == 1
    capi.write_state_file(res, tmp_path / "a.state")
    lines = (tmp_path / "a.state").read_text().splitlines()
    assert lines[0] == "Node\tSite\tState\tp_A\tp_C\tp_G\tp_T"
    assert len(lines) == 1 + L
    node = "Node%d" % res["nodes"][-1]
    f = lines[1].split("\t")
    p0 = res["posterior"][0][0][cols[0]]
    assert f[0] == node and f[1] == "1" and f[2] == "ACGT"[int(np.argmax(p0))]
    assert [float(x) for x in f[3:]] == [float("%.5f" % x) for x in p0]
    fasta = (tmp_path / "a.fasta").read_text().splitlines()
    assert fasta[0] == ">root" and "".join(fasta[1:]) == "".join(l.split("\t")[2] for l in lines[1:])


def test_a_partition_file_maps_columns_in_range_order(lib, tmp_path):  # noqa: F811
    fx = fixtures.load("10.fasta")
    L = len(next(iter(fx["alignment"].values())))
    part = tmp_path / "p.txt"
    part.write_text("DNA, one = 1-%d, %d-%d\nDNA, two = %d-%d\n" % (L // 4, L // 2 + 1, L, L // 4 + 1, L // 2))
    tree = tree_of("10.fasta", lib)
    m = capi.Model.from_files(tree, fx["tree_path"].parent / "10.fasta", part, rate_cats=1)
    m.initialize_partitions()
    seqs = [fx["alignment"][t] for t in sorted(fx["alignment"])]
    one = list(range(L // 4)) + list(range(L // 2, L))
    cols = m.pattern_of_column(0)
    assert len(cols) == len(one) and len(m.pattern_of_column(1)) == L // 2 - L // 4
    for i, c in enumerate(one[:: 23]):
        i = one.index(c)
        same = [j for j, d in enumerate(one) if all(s[d].upper() == s[c].upper() for s in seqs)]
        assert set(cols[same].tolist()) == {cols[i]}
    res = m.ancestral_states(2, 0.5)
    capi.write_state_file(res, tmp_path / "b.state")
    lines = (tmp_path / "b.state").read_text().splitlines()
    assert lines[0] == "Node\tPart\tSite\tState\tp_A\tp_C\tp_G\tp_T" and len(lines) == 1 + L
    # partition 1's site i is its i-th column in range order; partition 2 follows, numbered from 1
    n1 = len(one)
    for i in (0, L // 4 - 1, L // 4, n1 - 1):
        f = lines[1 + i].split("\t")
        q = res["posterior"][0][0][cols[i]]
        assert f[1:3] == ["1", str(i + 1)] and [float(x) for x in f[4:]] == [float("%.5f" % x) for x in q]
    assert lines[1 + n1].split("\t")[1:3] == ["2", "1"]


def test_the_state_file_is_the_golden_one(lib, tmp_path):  # noqa: F811
    here = Path(__file__).resolve().parent / "golden"
    for name, parts, full in (("ancestral_small", None, "all"), ("ancestral_small_parts", SMALL_PARTS, "root")):
        res = small_model(lib, 4, parts).ancestral_states(GOLDEN_ROOT, 0.3, full_nodes=full)
        capi.write_state_file(res, tmp_path / (name + ".state"))
        for ext in (".state", ".fasta"):
            assert (tmp_path / (name + ext)).read_bytes() == (here / (name + ext)).read_bytes(), name + ext


def sides(res, i, taxa):
    """node i of a result, named by the three taxon sets on its sides (unrooted: root-independent)"""
    kids = [j for j in range(len(res["nodes"])) if res["parent"][j] == i]
    below = set().union(*[set(res["clade"][j]) for j in kids]) if kids else set()
    out = [frozenset(res["clade"][j]) for j in kids] + [frozenset([t]) for t in res["clade"][i] if t not in below]
    out.append(frozenset(taxa - set(res["clade"][i])))
    return frozenset(out)


@pytest.mark.parametrize("name", ["10.fasta", "small"])
def test_pulley_principle_every_node_has_one_posterior_at_every_placement(lib, name):  # noqa: F811
    # all rates 1 and pi = 1/4 (the reference's own test set-up, test/src/model.cpp:367-387): the model is
    # reversible, so a node's posterior does not depend on where the root is
    m = small_model(lib, 1) if name == "small" else make_model(lib, name, 1)
    m.set_params(rates=np.ones(12), freqs=np.full(4, 0.25), alpha=1.0)
    seen = {}
    for rid in range(m.root_count):
        res = m.ancestral_states(rid, 0.5, full_nodes="all")
        taxa = set(res["clade"][-1])
        for i in range(len(res["nodes"]) - 1):  # the root sits on a branch: not a node of the unrooted tree
            key = sides(res, i, taxa)
            assert len(key) == 3
            post = res["posterior"][0][i]
            if key in seen:
                assert np.max(np.abs(post - seen[key])) < 1e-12
            else:
                seen[key] = post
    assert len(seen) == len(res["nodes"]) - 1  # every unrooted inner node, each seen from every placement
