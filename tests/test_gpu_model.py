"""GPU parity at the model_t level: the host C++ (search, Brent, L-BFGS-B drivers)
compiled against the CUDA engine vs. the same sources compiled against the CPU
oracle in ENGINE arithmetic.  Because every likelihood evaluation is bit-identical,
the whole optimiser trajectory is: chosen root branch, optimised alpha, LWR
ranking and final log-likelihood must be IDENTICAL (north_star)."""
import numpy as np
import pytest

import fixtures
import oracle_capi
import oracle_build
from root_digger_b200 import capi, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def libs():
    oracle_capi.load_oracle().rdo_set_default_mode(oracle_capi.MODE_ENGINE)
    return capi.load_tree_lib(), capi.load_tree_lib(oracle_build.build_host_on_oracle())


def pair(libs, name="10.fasta", K=4, uniform=True, seed=4242):
    fx = fixtures.load(name)
    out = []
    for lib in libs:
        tree = capi.RootedTree(path=str(fx["tree_path"]), lib=lib)
        m = capi.Model(tree, fx["alignment"], rate_cats=K, compress=True, invariant_sites=True, seed=seed)
        m.initialize_partitions(uniform_freqs=uniform)
        out.append(m)
    return out


def synthetic_pair(libs, n=24, S=3000, K=4, seed=9):
    top = synth.random_tree(n, seed)
    rates, freqs = synth.random_params(seed + 1)
    aln = synth.simulate_alignment(top, S, seed + 2, rates, freqs, capi.gamma_cats(0.8, K))
    out = []
    for lib in libs:
        tree = capi.RootedTree(synth.to_newick(top), lib=lib)
        m = capi.Model(tree, aln, rate_cats=K, compress=True, seed=seed)
        m.initialize_partitions(uniform_freqs=False)
        out.append(m)
    return out


def bits(x):
    return np.asarray(x, dtype=np.float64).view(np.uint64)


@pytest.mark.parametrize("K", [1, 4])
def test_likelihood_facade_is_bit_identical(libs, K):
    g, o = pair(libs, K=K)
    assert g.sites() == o.sites() == 991
    for rid in range(g.root_count):
        a, b = g.compute_lh(rid, 0.3), o.compute_lh(rid, 0.3)
        assert a.hex() == b.hex()
        assert g.compute_lh_root(rid, 0.8).hex() == o.compute_lh_root(rid, 0.8).hex()
        assert [v.hex() for v in g.compute_dlh(rid, 0.5)] == [v.hex() for v in o.compute_dlh(rid, 0.5)]
    # reference invariants on the GPU-backed model (test/src/model.cpp:59-75, :271-288)
    for rid in range(g.root_count):
        a, b, c = g.compute_lh(rid), g.compute_lh(rid), g.compute_lh_root(rid)
        assert np.isfinite(a) and a < 0 and a == b and a == c


def test_empirical_frequencies_and_random_rates_identical(libs):
    g, o = pair(libs, "101.phy", K=4, uniform=False)
    for a, b in zip(g.get_params(), o.get_params()):
        assert np.array_equal(bits(a), bits(b))


def test_sweep_and_root_ranking_identical(libs):
    g, o = pair(libs, "101.phy", K=4, uniform=False)
    g.compute_lh(0)
    o.compute_lh(0)
    a, b = g.sweep_root_lh(), o.sweep_root_lh()
    assert np.array_equal(bits(a), bits(b))
    for mode in (g.SWEEP_SEQUENTIAL, g.SWEEP_PATH, g.SWEEP_DIRECTED):
        # the reference's own loop (move_root + compute_lh_root per root), the same operations in one
        # engine call, the directed-CLV pass: same bits, from a different current root too
        g.compute_lh(7, 0.2)
        g.set_sweep_mode(mode)
        c = g.sweep_root_lh()
        assert np.array_equal(bits(a), bits(c)), mode
    assert np.array_equal(np.argsort(-a, kind="stable"), np.argsort(-b, kind="stable"))


def test_optimize_alpha_identical(libs):
    g, o = pair(libs, K=4)
    for rid in range(g.root_count):
        g.compute_lh(rid)
        o.compute_lh(rid)
        for atol in (1e-7, 1e-14):
            assert g.optimize_alpha(rid, 0.5, atol).hex() == o.optimize_alpha(rid, 0.5, atol).hex()
    assert g.optimize_root_location(2, 0.1) == o.optimize_root_location(2, 0.1)


def test_search_chooses_identical_root_alpha_and_likelihood(libs):
    for (g, o) in (pair(libs, K=1), synthetic_pair(libs)):
        g.compute_lh(0)
        o.compute_lh(0)
        rg = g.search(2, 0.0, 1e-3, 1e-3, 1e-3, 1e12, strategy="modified_mad")
        ro = o.search(2, 0.0, 1e-3, 1e-3, 1e-3, 1e12, strategy="modified_mad")
        assert rg[0] == ro[0]                       # chosen root branch
        assert rg[1].hex() == ro[1].hex()           # optimised alpha
        assert rg[2].hex() == ro[2].hex()           # final log-likelihood
        for a, b in zip(g.get_params(), o.get_params()):
            assert np.array_equal(bits(a), bits(b))  # optimised rates / frequencies / category rates


def test_exhaustive_mode_lwr_identical(libs):
    g, o = synthetic_pair(libs, n=8, S=1500, K=4, seed=21)
    g.compute_lh(0)
    o.compute_lh(0)
    ig, lg, ag = g.exhaustive_search(1e-3, 1e-3, 1e-3, 1e12)
    io, lo, ao = o.exhaustive_search(1e-3, 1e-3, 1e-3, 1e12)
    assert np.array_equal(ig, io) and np.array_equal(bits(lg), bits(lo)) and np.array_equal(bits(ag), bits(ao))
    wg, wo = g.lwr(lg), o.lwr(lo)
    assert np.array_equal(bits(wg), bits(wo))
    assert np.array_equal(np.argsort(-wg, kind="stable"), np.argsort(-wo, kind="stable"))   # LWR ranking
    assert g.newick() == o.newick()                                                        # annotated output tree


def test_multi_partition_model(libs):
    """config 4 shape in miniature: independent parameters per partition, summed log-likelihood"""
    top = synth.random_tree(16, 5)
    rates, freqs = synth.random_params(6)
    aln = synth.simulate_alignment(top, 4000, 7, rates, freqs, capi.gamma_cats(1.0, 4))
    parts = [(0, 1000), (1000, 2500), (2500, 4000)]
    ms = []
    for lib in libs:
        tree = capi.RootedTree(synth.to_newick(top), lib=lib)
        m = capi.Model(tree, aln, rate_cats=4, compress=True, seed=3, partitions=parts)
        m.initialize_partitions(uniform_freqs=False)
        ms.append(m)
    g, o = ms
    for rid in (0, 5, 11):
        assert g.compute_lh(rid).hex() == o.compute_lh(rid).hex()
        assert g.compute_lh_root(rid, 0.25).hex() == o.compute_lh_root(rid, 0.25).hex()


def test_batched_root_only_evaluations_on_the_engine(libs):
    """DESIGN 5.5 on the CUDA engine: compute_dlh / optimize_alpha with their root-only evaluations
    handed over as fused batches (rdk_root_loglikelihood_multi: 2 per slope, 5 before the first
    decision of optimize_alpha, a whole dyadic level) and issued one by one (the reference's call
    sequence, src/model.cpp:481-519,679-794) return the same bits, and the batched model did batch"""
    g, _ = synthetic_pair(libs, n=20, S=2500, K=4, seed=21)
    g.compute_lh(0)
    assert g.batched_probes
    for rid in range(0, g.root_count, 3):
        got = {}
        for batched in (True, False):
            g.set_batched_probes(batched)
            g.compute_lh(rid)
            got[batched] = [v for x in (0.0, 0.37, 1.0) for v in g.compute_dlh(rid, x)]
            got[batched] += [g.optimize_alpha(rid, 0.5, atol) for atol in (1e-7, 1e-14)]
            got[batched].append(g.compute_lh_root(rid, 0.3))
        assert np.array_equal(bits(got[True]), bits(got[False])), rid
    c = g.probe_counters()
    assert c["fused_batches"] > 0 and c["fused_evaluations"] >= 2 * c["fused_batches"]
    g.close()


# bench.py's exhaustive-mode sample (cfg2: 500 taxa x 100 000 sites, UNREST+G4, root branch 0 optimised to
# convergence) as recorded on a B200 with RootDigger's own vendored L-BFGS-B (lib/lbfgsb) linked into the host:
# profiles/r02_bench_final2_n1.json, e2e.exhaustive.  Thousands of L-BFGS-B steps lead to this value, so
# its bits and the number of root evaluations pin the optimiser's trajectory.
RECORDED_EXHAUSTIVE_BEST_LLH = -9474150.440101244
RECORDED_EXHAUSTIVE_ROOT_EVALUATIONS = 57553


def test_exhaustive_branch_reproduces_the_run_recorded_with_the_reference_lbfgsb():
    import ctypes as C
    from cases import Case
    case = Case(500, 100000, 4, seed=0x5EED0002, data="evolved", alpha=1.0, gamma_cats=capi.gamma_cats)
    m = capi.Model(capi.RootedTree(case.newick), case.aln, 4)
    m.initialize_partitions()
    m.set_params(rates=case.rates, freqs=case.freqs)
    m.set_sweep_mode(m.SWEEP_DIRECTED)
    m.compute_lh(0, 0.5)
    m.sweep_root_lh()
    part = C.cast(m.L.rdh_model_partition(m.h, 0), C.POINTER(capi.PartitionStruct))
    L = capi.load_engine()

    def root_evals():
        s = capi.Stats()
        L.rdk_partition_stats(part, C.byref(s))
        return s.asdict()["root_evals"]

    before = root_evals()
    ids, llh, _ = m.exhaustive_search(1e-7, 1e-7, 1e-12, 1e4, rank=0, num_tasks=m.root_count)
    evaluations = root_evals() - before
    m.close()
    assert list(ids) == [0]
    assert float(llh[0]).hex() == RECORDED_EXHAUSTIVE_BEST_LLH.hex()
    assert evaluations == RECORDED_EXHAUSTIVE_ROOT_EVALUATIONS
