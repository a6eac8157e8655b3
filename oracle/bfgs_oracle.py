"""TEST INFRASTRUCTURE -- CPU restatement of the reference's L-BFGS-B driver with the likelihood
replaced by any objective.

Restates `bfgs_params` (src/model.cpp:1430-1522) statement by statement around the L-BFGS-B 3.0 the
host drives (`setulb` in lib/liblbfgsb.so, built from root_digger_b200/lbfgsb): the objective is
evaluated after every return of setulb whatever the task (:1486-1487), the gradient is a forward difference with h = max(epsilon |x_i|, epsilon) (:1488-1501), the loop
ends on any task but FG / NEW_X or after 500 rounds, the caller's vector receives the final point
only if it is not worse than the start (:1510-1511) while the LAST point stays installed.

tests/test_optim.py compares rd::minimize_in_box (root_digger_b200/host/optim.hpp) with this, bit
for bit: the returned vector, the final objective and the whole sequence of evaluated points.
Only tests/ may import this module.
"""
import ctypes as C
import math

START, NEW_X, FG, FG_END = 1, 2, 10, 15  # lib/lbfgsb/lbfgsb.h:70-77


def bfgs_params(setulb_lib_path, initial_params, p_min, p_max, epsilon, pgtol, factor, objective):
    """-> (score, parameters the caller is left with, [points evaluated, in order])"""
    lib = C.CDLL(str(setulb_lib_path))
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    lib.setulb.argtypes = [ip, ip, dp, dp, dp, ip, dp, dp, dp, dp, dp, ip, ip, ip, ip, ip, ip, dp]
    trace = []

    def compute_lh(params):  # set_func + compute_lh of the reference, always called as a pair
        trace.append(list(params))
        return float(objective(list(params)))

    n = len(initial_params)
    task = C.c_int(START)
    n_params = C.c_int(n)
    initial_params = list(initial_params)
    score = C.c_double(compute_lh(initial_params))
    initial_score = score.value
    csave = C.c_int(0)
    gradient = (C.c_double * n)()
    max_corrections = C.c_int(20)
    m = 20
    wa = (C.c_double * ((2 * m + 5) * n + 12 * m * (m + 1)))()
    iwa = (C.c_int * (3 * n))()
    parameters = (C.c_double * n)(*initial_params)
    param_min = (C.c_double * n)(*([p_min] * n))
    param_max = (C.c_double * n)(*([p_max] * n))
    lsave, isave, dsave = (C.c_int * 4)(), (C.c_int * 44)(), (C.c_double * 29)()
    bound_type = (C.c_int * n)(*([2] * n))
    iprint = C.c_int(-1)
    factor_c, pgtol_c = C.c_double(factor), C.c_double(pgtol)
    iters = 0
    while iters < 500:
        lib.setulb(C.byref(n_params), C.byref(max_corrections), parameters, param_min, param_max, bound_type,
                   C.byref(score), gradient, C.byref(factor_c), C.byref(pgtol_c), wa, iwa, C.byref(task),
                   C.byref(iprint), C.byref(csave), lsave, isave, dsave)
        score.value = compute_lh(parameters)
        if FG <= task.value <= FG_END:
            for i in range(n):
                h = epsilon * abs(parameters[i])
                if h < epsilon:
                    h = epsilon
                temp = parameters[i]
                parameters[i] += h
                dlh = compute_lh(parameters)
                if not math.isfinite(dlh):
                    raise RuntimeError("dlh is not finite")
                gradient[i] = (dlh - score.value) / h
                if not math.isfinite(gradient[i]):
                    raise RuntimeError("gradient is not finite")
                parameters[i] = temp
        elif task.value != NEW_X:
            break
        iters += 1
    score.value = compute_lh(parameters)
    if initial_score >= score.value:
        initial_params = list(parameters)
    return score.value, initial_params, trace
