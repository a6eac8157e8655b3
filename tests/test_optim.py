"""The optimiser components of root_digger_b200/host/optim.hpp on their own, on analytic functions
(CPU; the host library compiled against the oracle carries the same code).  What they do inside
model_t -- the reference's trajectories, bit for bit -- is held by tests/test_reference_sources.py
against the reference's own src/model.cpp (brents :606-676, bfgs_params :1430-1522)."""
import math

import numpy as np
import pytest

import oracle_build
from root_digger_b200 import capi


@pytest.fixture(scope="module")
def lib():
    return capi.load_tree_lib(oracle_build.build_host_on_oracle())


def concave(peak, curvature=3.0):
    """a log-likelihood-like function with its maximum at `peak`: slope changes sign there"""
    return lambda x: (-curvature * (x - peak) ** 2 - 100.0, -2.0 * curvature * (x - peak))


@pytest.mark.parametrize("peak", [0.5, 0.123456789, 0.9, 1e-3])
def test_slope_root_finds_the_peak(lib, peak):
    x, value, slope, probes = capi.slope_root(concave(peak), 0.0, 1.0, 1e-12, lib=lib)
    assert abs(x - peak) < 1e-9
    assert value == pytest.approx(-100.0, abs=1e-12)
    assert abs(slope) < 1e-8
    assert 0 < probes <= 64


def test_slope_root_on_a_transcendental_slope(lib):
    # slope = cos(3x) on [0, 1]: root at pi/6; value = sin(3x)/3
    x, value, slope, probes = capi.slope_root(lambda t: (math.sin(3 * t) / 3, math.cos(3 * t)), 0.0, 1.0, 1e-14,
                                              lib=lib)
    assert abs(x - math.pi / 6) < 1e-10 and abs(value - 1 / 3) < 1e-12 and probes <= 64


def test_slope_root_returns_a_sample_it_evaluated(lib):
    seen = []

    def fn(x):
        seen.append(x)
        return concave(0.3)(x)

    x, value, slope, probes = capi.slope_root(fn, 0.0, 1.0, 1e-10, lib=lib)
    assert x in seen and len(seen) == probes + 2
    assert all(0.0 <= s <= 1.0 for s in seen), "the iterates stay inside the bracket"


def test_slope_root_refuses_a_non_bracket(lib):
    with pytest.raises(RuntimeError, match="don't bracket"):
        capi.slope_root(concave(2.0), 0.0, 1.0, lib=lib)  # slope positive at both ends
    with pytest.raises(RuntimeError, match="don't bracket"):
        capi.slope_root(lambda x: (0.0, float("nan")), 0.0, 1.0, lib=lib)


def test_slope_root_gives_up_after_64_iterations(lib):
    # the sign change sits immediately right of 0 and the tolerance is relative to the estimate
    # (2 |x| eps): every step halves the bracket towards 0 and 64 halvings do not get there
    with pytest.raises(RuntimeError, match="failed to converge"):
        capi.slope_root(lambda x: (0.0, 1.0 if x == 0.0 else -1.0), 0.0, 1.0, 0.0, lib=lib)


def test_slope_root_keeps_the_larger_residual_as_its_estimate(lib):
    """Q1 of optim.hpp (the reference's rank test, src/model.cpp:624-631): the current estimate is
    the bracket end with the LARGER |slope|, so an end that is already flat (1e-13 <= the 1e-12
    floor) does not end the search at once as it would in textbook Brent -- the bracket is walked
    down to it"""
    x, _, slope, probes = capi.slope_root(lambda t: (0.0, 1e-13 if t == 0.0 else -1.0), 0.0, 1.0, 1e-9, lib=lib)
    assert probes > 10 and 0.0 < x < 1e-8 and slope == -1.0


def test_minimize_in_box_quadratic(lib):
    target = np.array([0.3, 0.7, 0.55])
    x, f_end, calls = capi.minimize_in_box(lambda v: float(np.sum((v - target) ** 2)), [0.5, 0.5, 0.5], 1e-4, 1.0,
                                           lib=lib)
    # forward differences of step 1e-4 bias the gradient by h: the minimum is found to about h/2
    assert np.allclose(x, target, atol=1e-4) and f_end < 1e-7 and calls > 5


def test_minimize_in_box_respects_the_box(lib):
    seen = []

    def fn(v):
        seen.append(v.copy())
        return float(np.sum((v - 2.0) ** 2))  # unconstrained minimum outside the box

    x, f_end, _ = capi.minimize_in_box(fn, [0.5, 0.25], 0.2, 1.0, lib=lib)
    assert np.allclose(x, [1.0, 1.0], atol=1e-9)
    pts = np.array(seen)
    assert pts.min() >= 0.2 - 1e-12 and pts.max() <= 1.0 + 1e-4 + 1e-12  # + the difference step


def test_minimize_in_box_evaluation_protocol(lib):
    """Q3 / Q4 of optim.hpp: the start is evaluated first, the final point last (and is what stays
    installed), every gradient costs n shifted evaluations after one at the point itself"""
    seen = []

    def fn(v):
        seen.append(v.copy())
        return float((v[0] - 0.4) ** 2 + 2 * (v[1] - 0.6) ** 2)

    x0 = np.array([0.9, 0.1])
    x, f_end, calls = capi.minimize_in_box(fn, x0, 1e-4, 1.0, lib=lib)
    assert calls == len(seen) and np.array_equal(seen[0], x0)
    assert np.array_equal(seen[-1], x) and f_end == fn(x)
    # the first round: the point, then one coordinate shifted by max(1e-4 |x_i|, 1e-4) at a time
    assert np.array_equal(seen[1], x0)
    assert seen[2][0] == x0[0] + 1e-4 and seen[2][1] == x0[1]
    assert seen[3][0] == x0[0] and seen[3][1] == x0[1] + 1e-4


def test_minimize_in_box_keeps_the_start_when_the_end_is_worse(lib):
    """Q4: an objective that gets WORSE wherever the optimiser goes leaves x at the start"""
    x0 = np.array([0.5])
    calls = {"n": 0}

    def fn(v):
        calls["n"] += 1
        return -1.0 if calls["n"] == 1 else float(calls["n"])  # the start is the best point ever seen

    x, f_end, _ = capi.minimize_in_box(fn, x0, 1e-4, 1.0, lib=lib)
    assert np.array_equal(x, x0) and f_end > -1.0


def test_minimize_in_box_refuses_non_finite_objectives(lib):
    def fn(v):
        return float("inf") if v[0] > 0.5 else float(v[0])

    with pytest.raises(RuntimeError, match="not finite"):
        capi.minimize_in_box(fn, [0.5], 1e-4, 1.0, lib=lib)


# ---------------------------------------------------------------------------------------------
# rd::unit_segment_search_t against the restated reference (oracle/alpha_oracle.py)
# ---------------------------------------------------------------------------------------------
import alpha_oracle  # noqa: E402  (oracle/ is on the path through conftest)

TAU = 2.0 * math.pi
SURFACES = {
    # name: (f, which branch of optimize_alpha it is there to reach)
    "peak_0.3": (lambda x: -3.0 * (x - 0.3) ** 2 - 100.0, "bracket -> Brent"),
    "peak_0.9": (lambda x: -40.0 * (x - 0.9) ** 2 - 5.0, "bracket -> Brent"),
    "peak_tiny": (lambda x: -1e-3 * (x - 0.123456789) ** 2 - 7000.0, "bracket, small slopes"),
    "log_like": (lambda x: 300.0 * math.log(0.2 + x) + 200.0 * math.log(1.3 - x) - 9000.0, "bracket -> Brent"),
    "rising": (lambda x: 3.0 * x - 50.0, "same sign, no turn: upper end"),
    "falling": (lambda x: -2.0 * x - 50.0, "same sign, no turn: lower end"),
    "rising_turn_1/4": (lambda x: x + 0.3 * math.sin(2 * TAU * x) - 80.0, "same sign, turn at 1/4 (level 2)"),
    "falling_turn_1/4": (lambda x: -(x + 0.3 * math.sin(2 * TAU * x)) - 80.0, "same sign, turn at 1/4 (level 2)"),
    "rising_turn_inner_wins": (lambda x: 0.2 * x + 0.3 * math.sin(2 * TAU * x) - 80.0,
                               "same sign, turn at 1/4, a refinement beats both ends"),
    "rising_turn_1/16": (lambda x: x + 1.05 * math.sin(8 * TAU * x) / (8 * TAU) - 80.0,
                         "same sign, turn only at 1/16 (level 16)"),
    "flat": (lambda x: -123.0, "flat end"),
    "cubic": (lambda x: (x - 0.5) ** 3 - 10.0, "same sign, flat grid point at 1/2, no turn"),
    "impossible_below_0.3": (lambda x: -math.inf if x < 0.3 else -5.0 * (x - 0.6) ** 2 - 3.0,
                             "-inf at both evaluations of the lower end: slope 0 there"),
    "impossible_everywhere": (lambda x: -math.inf, "-inf everywhere"),
    "valley": (lambda x: 4.0 * (x - 0.45) ** 2 - 20.0, "bracket around a MINIMUM: an end wins"),
}


def bits(x):
    return np.float64(x).view(np.uint64)


@pytest.mark.parametrize("name", sorted(SURFACES))
@pytest.mark.parametrize("atol", [1e-7, 1e-14])
def test_segment_search_is_the_reference_algorithm(lib, name, atol):
    """one evaluation at a time (look_ahead off) the component IS the reference's call sequence: the
    same abscissae in the same order and the same answer, bit for bit; with batches ahead of need the
    answer is unchanged and the number of engine calls drops"""
    f = SURFACES[name][0]
    for x_now in (0.5, 0.0, 1.0):
        want, xs = alpha_oracle.optimize_alpha(f, x_now, atol)
        got, batches = capi.argmax_on_segment(f, x_now, atol, look_ahead=False, lib=lib)
        flat = [x for b in batches for x in b]
        assert bits(got) == bits(want), (name, got, want)
        assert [bits(x) for x in flat] == [bits(x) for x in xs], name
        assert all(len(b) <= 2 for b in batches)
        ahead, batches_ahead = capi.argmax_on_segment(f, x_now, atol, look_ahead=True, lib=lib)
        assert bits(ahead) == bits(want), (name, ahead, want)
        assert len(batches_ahead) <= len(batches) - 2 and len(batches_ahead[0]) == 5
        consumed = {bits(x) for x in xs}
        assert consumed <= {bits(x) for b in batches_ahead for x in b}, "nothing the decision needs is skipped"


def test_segment_search_reaches_every_branch(lib):
    """the surfaces above do take the branches they are named for (read off the evaluation log)"""
    def log_of(name, atol=1e-7):
        return alpha_oracle.optimize_alpha(SURFACES[name][0], 0.5, atol)

    assert len(log_of("flat")[1]) == 5 and log_of("flat")[0] == 0.0
    assert log_of("impossible_everywhere") == (0.0, [0.5, 0.0, 1e-8, 1.0, 1.0 - 1e-8])
    x, xs = log_of("rising")
    assert x == 1.0 and len(xs) == 5 + 2 * 31          # the whole grid, then the upper end
    x, xs = log_of("falling")
    assert x == 0.0 and len(xs) == 5 + 2 * 31
    x, xs = log_of("cubic")
    assert x == 0.5 and len(xs) == 5 + 2 * 31          # the flat grid point wins
    x, xs = log_of("rising_turn_1/4")
    assert xs[5:9] == [0.5, 0.5 + 1e-8, 0.25, 0.25 + 1e-8] and x == 1.0 and len(xs) > 9   # the upper end wins
    x, xs = log_of("rising_turn_inner_wins")
    assert xs[7] == 0.25 and 0.0 < x < 1.0 and abs(0.2 + 0.6 * TAU * math.cos(2 * TAU * x)) < 1e-5
    x, xs = log_of("rising_turn_1/16")
    assert xs[5 + 2 * 7] == 1.0 / 16.0 and len(xs) > 5 + 2 * 8   # 1 + 2 + 4 grid points before level 16
    x, xs = log_of("valley")
    assert x in (0.0, 1.0) and len(xs) > 5
    x, xs = log_of("peak_0.3", 1e-14)
    assert abs(x - 0.3) < 1e-7 and 5 < len(xs) < 5 + 2 * 64


@pytest.mark.parametrize("x", [0.0, 0.25, 1.0 - 1e-8, 1.0 - 0.5e-8, 1.0])
def test_slope_is_the_reference_forward_difference(lib, x):
    for name in ("log_like", "peak_0.9", "impossible_below_0.3", "impossible_everywhere"):
        f = SURFACES[name][0]
        want = alpha_oracle.compute_dlh(alpha_oracle.Trace(f), x)
        got = capi.slope_on_segment(f, x, lib=lib)
        assert [bits(v) for v in got] == [bits(v) for v in want], (name, x, got, want)


def test_segment_search_reports_nan_only_where_the_reference_would(lib):
    bad_at_end = lambda x: math.nan if x > 0.9 else -x  # noqa: E731
    with pytest.raises(alpha_oracle.NotANumber):
        alpha_oracle.optimize_alpha(bad_at_end, 0.5, 1e-7)
    for ahead in (False, True):
        with pytest.raises(RuntimeError, match="not a number"):
            capi.argmax_on_segment(bad_at_end, 0.5, 1e-7, look_ahead=ahead, lib=lib)
    # NaN at 3/4 only: the scan of level 2 turns at 1/4 and never gets there -- the batch that
    # evaluated 3/4 ahead of need must not fail either
    base = SURFACES["rising_turn_1/4"][0]
    poisoned = lambda x: math.nan if abs(x - 0.75) < 3e-8 else base(x)  # noqa: E731
    want, xs = alpha_oracle.optimize_alpha(poisoned, 0.5, 1e-7)
    assert all(abs(x - 0.75) > 3e-8 for x in xs)
    got, batches = capi.argmax_on_segment(poisoned, 0.5, 1e-7, look_ahead=True, lib=lib)
    assert bits(got) == bits(want) and any(abs(x - 0.75) < 3e-8 for b in batches for x in b)


# ---------------------------------------------------------------------------------------------
# rd::minimize_in_box against the restated reference driver (oracle/bfgs_oracle.py)
# ---------------------------------------------------------------------------------------------
import bfgs_oracle  # noqa: E402

OBJECTIVES = {
    "quadratic": (lambda v: sum((a - t) ** 2 for a, t in zip(v, (0.3, 0.7, 0.55))), [0.5, 0.5, 0.5], 1e-4, 1.0),
    "rosenbrock": (lambda v: (1 - v[0]) ** 2 + 100.0 * (v[1] - v[0] ** 2) ** 2, [0.2, 0.9], 1e-4, 1e4),
    "at_the_bound": (lambda v: sum((a - 2.0) ** 2 for a in v), [0.5, 0.25], 0.2, 1.0),
    "neg_log_like": (lambda v: -(300 * math.log(v[0] / sum(v)) + 500 * math.log(v[1] / sum(v))
                                 + 200 * math.log(v[2] / sum(v))), [1 / 3, 1 / 3, 1 / 3], 1e-4, 1.0 - 3e-4),
    "twelve_rates": (lambda v: sum((math.log(a) - math.log(0.05 * (i + 1))) ** 2 for i, a in enumerate(v)) - 9000.0,
                     [1.0 / 12] * 12, 1e-4, 1e4),
    "gets_worse": (lambda v: -abs(v[0] - 0.5) * 0.0 + (0.0 if v[0] == 0.5 else 1.0 + v[0]), [0.5], 1e-4, 1.0),
}


@pytest.mark.parametrize("name", sorted(OBJECTIVES))
@pytest.mark.parametrize("pgtol,factr", [(1e-7, 1e4), (1e-3, 1e12)])
def test_minimize_in_box_is_the_reference_driver(lib, name, pgtol, factr):
    """the same points evaluated in the same order, the same vector handed back and the same final
    objective as the reference's bfgs_params (src/model.cpp:1430-1522) around the same setulb"""
    from root_digger_b200 import _build
    fn, x0, lo, hi = OBJECTIVES[name]
    want_f, want_x, want_trace = bfgs_oracle.bfgs_params(_build.build_lbfgsb(), x0, lo, hi, 1e-4, pgtol, factr, fn)
    seen = []

    def logged(v):
        seen.append(v.tolist())
        return fn(v.tolist())

    x, f_end, calls = capi.minimize_in_box(logged, x0, lo, hi, pgtol=pgtol, factr=factr, lib=lib)
    as_bits = lambda rows: [[bits(a) for a in r] for r in rows]  # noqa: E731
    assert calls == len(want_trace) and as_bits(seen) == as_bits(want_trace), name
    assert bits(f_end) == bits(want_f) and [bits(a) for a in x] == [bits(a) for a in want_x], name


# ---------------------------------------------------------------------------------------------
# setulb itself (root_digger_b200/lbfgsb) against an independent L-BFGS-B 3.0: scipy's
# ---------------------------------------------------------------------------------------------
def _rosenbrock(x):
    f = np.sum(100.0 * (x[1:] - x[:-1] ** 2) ** 2 + (1.0 - x[:-1]) ** 2)
    g = np.zeros_like(x)
    g[:-1] = -400.0 * x[:-1] * (x[1:] - x[:-1] ** 2) - 2.0 * (1.0 - x[:-1])
    g[1:] += 200.0 * (x[1:] - x[:-1] ** 2)
    return f, g


def _run_setulb(path, fg, x0, lo, hi, m, factr, pgtol):
    """setulb driven to its end with the analytic gradient -> every point it asked f and g at"""
    import ctypes as C
    L = C.CDLL(str(path))
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    L.setulb.argtypes = [ip, ip, dp, dp, dp, ip, dp, dp, dp, dp, dp, ip, ip, ip, ip, ip, ip, dp]
    n = len(x0)
    x, lower, upper = (C.c_double * n)(*x0), (C.c_double * n)(*([lo] * n)), (C.c_double * n)(*([hi] * n))
    nbd, f, g = (C.c_int * n)(*([2] * n)), C.c_double(0.0), (C.c_double * n)()
    wa, iwa = (C.c_double * (2 * m * n + 5 * n + 11 * m * m + 8 * m))(), (C.c_int * (3 * n))()
    task, csave, iprint = C.c_int(bfgs_oracle.START), C.c_int(0), C.c_int(-1)
    lsave, isave, dsave = (C.c_int * 4)(), (C.c_int * 44)(), (C.c_double * 29)()
    n_c, m_c, factr_c, pgtol_c = C.c_int(n), C.c_int(m), C.c_double(factr), C.c_double(pgtol)
    points = []
    while True:
        L.setulb(C.byref(n_c), C.byref(m_c), x, lower, upper, nbd, C.byref(f), g, C.byref(factr_c), C.byref(pgtol_c),
                 wa, iwa, C.byref(task), C.byref(iprint), C.byref(csave), lsave, isave, dsave)
        if bfgs_oracle.FG <= task.value <= bfgs_oracle.FG_END:
            points.append(np.array(x[:]))
            fv, gv = fg(points[-1])
            f.value, g[:] = fv, gv.tolist()
        elif task.value != bfgs_oracle.NEW_X:
            return points


@pytest.mark.parametrize("n,lo,hi,m,seed", [(2, -2.0, 2.0, 10, 1), (8, 0.2, 5.0, 20, 2), (12, 0.0, 0.9, 20, 3),
                                            (25, -0.5, 2.0, 3, 4)])
def test_setulb_follows_an_independent_lbfgsb(n, lo, hi, m, seed):
    """bounded Rosenbrock from a seeded start: the same number of evaluations as scipy's L-BFGS-B and
    the same points up to rounding (scipy sums through LAPACK / BLAS in another order)"""
    optimize = pytest.importorskip("scipy.optimize")
    from root_digger_b200 import _build
    x0 = np.random.default_rng(seed).uniform(lo, hi, n)
    ours = _run_setulb(_build.build_lbfgsb(), _rosenbrock, x0, lo, hi, m, 1e7, 1e-5)
    theirs = []

    def logged(x):
        theirs.append(x.copy())
        return _rosenbrock(x)

    optimize.fmin_l_bfgs_b(logged, x0.copy(), bounds=[(lo, hi)] * n, m=m, factr=1e7, pgtol=1e-5, maxiter=10 ** 5,
                           maxfun=10 ** 5)
    assert len(ours) == len(theirs) > 5
    assert max(np.max(np.abs(a - b)) for a, b in zip(ours, theirs)) < 1e-8
