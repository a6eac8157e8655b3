"""GPU tests of the engine's failure paths: a call that fails leaves the partition in a state from
which the next calls compute what they would have computed without it."""
import pytest

from cases import Case, compute_lh, same_bits

pytestmark = pytest.mark.gpu


def test_refused_sweep_leaves_no_evaluation_recorded():
    """a sweep refused at placement 2 (a child CLV index out of range) has recorded the evaluations of
    placements 0 and 1 by then: the call drops them, so neither the next flush nor the next evaluation
    runs one of them"""
    from root_digger_b200.capi import EngineError, Partition
    case = Case(10, 991, 4, seed=1000 + 10 + 991, data="evolved", weights="random")
    g = Partition(case.n, case.S, case.K)
    case.setup(g)
    sched = case.full_schedule(0, 0.5)
    want = compute_lh(g, sched, case.root_clv, case.root_scaler)
    before = g.stats()
    pm_off, mi, bl, op_off, ops = case.sweep_schedule(list(range(case.tree.root_count)), 0.5)
    ops[op_off[3] - 1].child1_clv_index = g.tips + g.clv_buffers  # the root operation of placement 2
    with pytest.raises(EngineError):
        g.sweep_root_placements(pm_off, mi, bl, op_off, ops, case.root_clv, case.root_scaler)
    g.flush()
    got = compute_lh(g, sched, case.root_clv, case.root_scaler)
    assert same_bits([got], [want])
    assert g.stats()["root_evals"] == before["root_evals"] + 1
