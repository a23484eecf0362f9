"""GPU tests (-m gpu) of what an evaluation reports for each flag set: the status of a Jacobian-only evaluation, and the
number of kernel launches per evaluation (DESIGN.md section 4)."""
import numpy as np
import pytest

import towr_b200 as tb
from towr_b200 import capi
from towr_b200.configs import synthetic_iterates

pytestmark = pytest.mark.gpu

GJ = capi.EVAL_G | capi.EVAL_JAC


def _problem(name):
    return tb.Problem(tb.make_formulation(name).to_spec())


@pytest.fixture(scope="module", params=["anymal_trot_block", "hyq_gallop_gap"])
def problem(request):
    """Config 2 (fixed durations) and config 4 (optimised durations: DynTailOut and PhaseJac run as well)."""
    return _problem(request.param)


def _nan_node(p, X, b):
    """X with one base-lin node value of instance b set to NaN (enters every dynamic sample of the node's polynomials)."""
    (start, count), = [(s, c) for nm, s, c in p.variable_sets() if nm == "base-lin"]
    X = X.copy()
    X[b, start + count // 2] = np.nan
    return X


def test_jacobian_only_status_matches_full_evaluation(problem):
    p = problem
    B = 40   # two tiles, the second one ragged
    bt = p.batch(B)
    X = synthetic_iterates(p, B)
    for Xi, expect in ((X, np.zeros(B, np.int32)), (_nan_node(p, X, 33), None)):
        full = bt.eval_host(Xi, flags=GJ)
        only_j = bt.eval_host(Xi, flags=capi.EVAL_JAC)
        assert np.array_equal(only_j["status"], full["status"])
        assert np.array_equal(only_j["jac"], full["jac"], equal_nan=True)
        if expect is not None:
            assert np.array_equal(full["status"], expect)
    flagged = np.flatnonzero(full["status"])
    assert list(flagged) == [33] and full["status"][33] == 1


def test_jacobian_only_status_after_non_finite_evaluation(problem):
    """The dynamic units' value rows are written by every evaluation, so a Jacobian-only evaluation of finite iterates
    reports status 0 even right after an evaluation that left NaN values in the same shared memory."""
    p = problem
    B = 256
    bt = p.batch(B)
    X = synthetic_iterates(p, B)
    bad = bt.eval_host(np.full_like(X, np.nan), flags=GJ)
    assert (bad["status"] & 1).all()
    for _ in range(3):
        assert not bt.eval_host(X, flags=capi.EVAL_JAC)["status"].any()


def test_launches_per_eval():
    """TransposeInP + RomNodeOut + DynOut; + CostKernel with cost terms; with optimised durations + DynTailOut (Jacobian)
    + PhaseJac."""
    bt = _problem("anymal_trot_block").batch(64)
    for flags in (capi.EVAL_G, capi.EVAL_JAC, GJ, capi.EVAL_ALL):
        assert bt.launches_per_eval(flags) == 3
    f = tb.make_formulation("anymal_trot_block")
    f.params_.costs_ = [(capi.COST_FORCES, 1.0)]
    bc = tb.Problem(f.to_spec()).batch(64)
    assert bc.launches_per_eval(GJ) == 3 and bc.launches_per_eval(capi.EVAL_ALL) == 4
    bd = _problem("hyq_gallop_gap").batch(64)
    assert bd.launches_per_eval(GJ) == 5 and bd.launches_per_eval(capi.EVAL_JAC) == 5 and bd.launches_per_eval(capi.EVAL_G) == 4
