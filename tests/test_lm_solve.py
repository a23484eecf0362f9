"""Solving batches to a tolerance on the device: twb_batch_lm_trial_device (the step with damping per instance, written to
x_trial, with merit, predicted decrease and the solve status), twb_batch_lm_accept_device (the gain-ratio decision) and
BatchedLevenbergMarquardt.solve on top of them.

The trial step is pinned bit for bit to the existing step and, with mu per instance, to the extended-precision step of
tests/lm_reference.py.  Accept / reject decisions are compared with the numpy rule of tests/lm_solve_reference.py on the
SAME inputs (never on two independently walked trajectories, where a decision near the threshold can go either way)."""
import ctypes as C

import numpy as np
import pytest

import towr_b200 as tb
from towr_b200 import capi
import lm_reference as ref
import lm_solve_reference as sref
from test_lm_step import CAP, CG, EPS, F64_RUNS, MU, PATH_CASES, _bits, _cuda, _edge_inputs, _problem, _violation64

# End-to-end runs: iteration budget and tolerance on max |s r|.  Measured on a B200 (1000 W limit, profiles/lm_solve_n1.json):
# with tol 1e-6 no instance of either 4096-instance workload converges within 60 iterations (median max |s r| 4.6 on the
# config-5 shard, 0.29 on the base-ROM workload), so the tolerance here is one that part of each batch reaches, to give the
# checks on converged instances something to check (at tol 1: 1254 and 3114 of 4096 converged).  No floor on the converged
# fraction beyond "some" is pinned.
TOL = 1.0
BUDGET = 60


# ---- CPU: the reference rule ----------------------------------------------------------------------------------------------

def test_reference_accept_rule():
    acc, rho, mu, nu, stalled = sref.accept(1.0, 0.5, 0.5, True, 1e-2, 8.0, 1e-4, 1e-12, 1e10)
    assert acc and rho == 1.0 and nu == 2.0 and not stalled and mu == 1e-2 * (1.0 / 3.0)
    acc, rho, mu, nu, stalled = sref.accept(1.0, 0.5, 0.9, True, 1e-2, 8.0, 0.5, 1e-12, 1e10)     # rho = 0.2 <= eta
    assert not acc and mu == 8e-2 and nu == 16.0 and not stalled
    assert not sref.accept(1.0, 0.0, 0.5, True, 1e-2, 2.0, 1e-4, 1e-12, 1e10)[0]                  # predicted = 0
    assert not sref.accept(1.0, -1.0, 2.0, True, 1e-2, 2.0, 1e-4, 1e-12, 1e10)[0]                 # predicted < 0, rho > 0
    assert not sref.accept(1.0, 0.5, 0.1, False, 1e-2, 2.0, 1e-4, 1e-12, 1e10)[0]                 # non-finite g_trial
    assert sref.accept(1.0, 0.5, 0.9, True, 6e9, 2.0, 0.9, 1e-12, 1e10)[4]                        # 1.2e10 > mu_max
    assert sref.accept(1.0, 1.0, 0.0, True, 1e-12, 2.0, 1e-4, 1e-12, 1e10)[2] == 1e-12            # mu_min floor


def test_reference_merit_and_predicted_against_dense_algebra():
    rng = np.random.default_rng(4)
    m, n = 30, 20
    mask = rng.random((m, n)) < 0.3
    J = np.where(mask, rng.standard_normal((m, n)) * 3.0, 0.0)
    row_ptr = np.concatenate([[0], np.cumsum(mask.sum(axis=1))])
    pat = ref.Pattern(row_ptr, np.nonzero(mask)[1], n)
    g, x, xt = rng.standard_normal(m), rng.standard_normal(n), rng.standard_normal(n)
    gl, gu = np.full(m, -0.3), np.full(m, 0.3)
    s = 1 / np.maximum(np.abs(J).max(axis=1), 1.0)
    phi0 = 0.5 * np.sum((s * ref.violation(g, gl, gu)) ** 2)
    lin = 0.5 * np.sum((s * ref.violation(g + J @ (xt - x), gl, gu)) ** 2)
    merit, pred = sref.merit_and_predicted(pat, x, xt, g, J[mask], gl, gu)
    assert np.isclose(merit, phi0, rtol=1e-14) and np.isclose(pred, phi0 - lin, rtol=1e-12, atol=1e-14)


# ---- GPU helpers ----------------------------------------------------------------------------------------------------------

def _trial(bt, X, g, jac, xl, xu, mu, gl=None, gu=None, status=None, tol=0.0, cg_iters=CG, cap=CAP):
    """One trial call from numpy inputs; returns numpy outputs (the inputs are not changed)."""
    import torch
    B, p = bt.B, bt.problem
    st = _cuda(np.zeros(B)).to(torch.int32) if status is None else torch.from_numpy(np.asarray(status, np.int32)).cuda()
    out = dict(x_trial=torch.full((B, p.n), 7.0, dtype=torch.float64, device="cuda"),
               row_scale=torch.full((B, p.m), 7.0, dtype=torch.float64, device="cuda"),
               merit=torch.full((B,), 7.0, dtype=torch.float64, device="cuda"),
               predicted=torch.full((B,), 7.0, dtype=torch.float64, device="cuda"),
               violation=torch.full((B,), 7.0, dtype=torch.float64, device="cuda"))
    x = _cuda(X)
    bt.lm_trial_device(x, _cuda(g), _cuda(jac), _cuda(np.broadcast_to(mu, (B,))), st, out["x_trial"], out["row_scale"], out["merit"],
                       out["predicted"], _cuda(xl), _cuda(xu), None if gl is None else _cuda(gl), None if gu is None else _cuda(gu),
                       cap, cg_iters, tol, out["violation"])
    torch.cuda.synchronize()
    assert np.array_equal(_bits(x.cpu().numpy()), _bits(X))          # x is only read
    res = {k: v.cpu().numpy() for k, v in out.items()}
    res["status"] = st.cpu().numpy()
    return res


def _step(bt, X, g, jac, xl, xu, gl=None, gu=None):
    import torch
    x = _cuda(X)
    viol = torch.full((bt.B,), 7.0, dtype=torch.float64, device="cuda")
    bt.lm_step_device(x, _cuda(g), _cuda(jac), _cuda(xl), _cuda(xu), MU, CAP, CG, viol,
                      g_lower=None if gl is None else _cuda(gl), g_upper=None if gu is None else _cuda(gu))
    torch.cuda.synchronize()
    return x.cpu().numpy(), viol.cpu().numpy()


def _instance_bounds(p, g, B, seed):
    from test_lm_instance_bounds import _instance_bounds as make
    return make(p, g, B, seed)


def _evaluated(case, B, seed):
    """g and J from twb_batch_eval_device at perturbed goal-instance starts (as test_lm_step does): (bt, X, g, jac, xl, xu)
    as numpy arrays, and the batch."""
    import torch
    p = _problem(case)
    rng = np.random.default_rng(seed)
    goals = np.column_stack([rng.uniform(0.3, 2.5, B), rng.uniform(-0.4, 0.4, B), np.full(B, 0.5), np.zeros(B), np.zeros(B),
                             rng.uniform(-0.5, 0.5, B)])
    bt = p.batch(B)
    x0, xl, xu = bt.goal_instances_device(_cuda(goals))
    X = torch.minimum(torch.maximum(x0 + 0.01 * _cuda(rng.standard_normal((B, p.n))), xl), xu)
    g = torch.empty((B, p.m), dtype=torch.float64, device="cuda")
    jac = torch.empty((B, p.nnz), dtype=torch.float64, device="cuda")
    status = torch.empty(B, dtype=torch.int32, device="cuda")
    bt.eval_device(X, g=g, jac=jac, status=status)
    torch.cuda.synchronize()
    assert not status.any().item()
    return bt, X.cpu().numpy(), g.cpu().numpy(), jac.cpu().numpy(), xl.cpu().numpy(), xu.cpu().numpy()


# ---- GPU: the trial step --------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_trial_with_one_mu_is_the_existing_step(case):
    """mu[b] = MU everywhere: x_trial and violation are the bits twb_batch_lm_step_device writes into x and violation (and
    twb_batch_lm_step_bounds_device with per-instance bounds), for every instance left RUNNING.  Instance 0 has no violated
    row: with tol = 0 it is CONVERGED and x_trial = x (the step would only project it)."""
    p = _problem(case)
    B = 10
    X, g, jac, xl, xu = _edge_inputs(p, B, seed=301)
    bt = p.batch(B)
    for gl, gu in ((None, None), _instance_bounds(p, g, B, seed=302)):
        x_step, v_step = _step(bt, X, g, jac, xl, xu, gl, gu)
        t = _trial(bt, X, g, jac, xl, xu, MU, gl, gu)
        assert t["status"][0] == capi.LM_CONVERGED and np.all(t["status"][1:] == capi.LM_RUNNING)
        assert np.array_equal(_bits(t["x_trial"][1:]), _bits(x_step[1:]))
        assert np.array_equal(_bits(t["x_trial"][0]), _bits(X[0])) and t["predicted"][0] == 0.0
        assert np.array_equal(_bits(t["violation"]), _bits(v_step))


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_trial_with_damping_per_instance_matches_the_extended_precision_step(case, record_property):
    """mu[b] spread over 1e-6 ... 1e2.  x_trial against the longdouble step under test_lm_step's yardstick (8 x the worst of
    F64_RUNS relabelled float64 steps, or 64 eps ||dx||); row_scale bit for bit 1 / max(1, max |J_row|); merit and predicted
    against longdouble values at the kernel's own x_trial (which separates them from the conjugate gradients' rounding)
    within 8 x the error of the plain float64 statement, or 64 eps of the larger of the two norms."""
    if not ref.LONGDOUBLE_IS_WIDER:
        pytest.skip("np.longdouble is not wider than float64 here")
    p = _problem(case)
    B = 9
    X, g, jac, xl, xu = _edge_inputs(p, B, seed=311)
    mu = np.logspace(-6, 2, B)
    _, _, gl, gu = p.bounds()
    t = _trial(p.batch(B), X, g, jac, xl, xu, mu)
    assert np.all(t["status"][1:] == capi.LM_RUNNING)
    row_ptr, col_idx = p.row_ptr(), p.structure()[1]
    pat = ref.Pattern(row_ptr, col_idx, p.n)
    worst = dict(x=0.0, merit=0.0, predicted=0.0)
    for b in range(1, B):
        dld, _ = ref.lm_capped_step(pat, g[b], jac[b], gl, gu, mu[b], CAP, CG, np.longdouble)
        xld = np.minimum(np.maximum(X[b].astype(np.longdouble) + dld, xl[b].astype(np.longdouble)), xu[b].astype(np.longdouble))
        runs = ref.relabelled_float64_steps(X[b], g[b], jac[b], xl[b], xu[b], gl, gu, row_ptr, col_idx, mu[b], CAP, CG, F64_RUNS, b)
        err_f64 = max(float(np.max(np.abs(x.astype(np.longdouble) - xld))) for x in runs)
        err_gpu = float(np.max(np.abs(t["x_trial"][b].astype(np.longdouble) - xld)))
        bound = max(err_f64, 64 * EPS * float(np.max(np.abs(dld))))
        assert err_gpu <= 8 * bound, (b, err_gpu, err_f64)
        worst["x"] = max(worst["x"], err_gpu / bound)
        assert np.array_equal(_bits(t["row_scale"][b]), _bits(1.0 / np.maximum(pat.row_max_abs(jac[b]), 1.0))), b
        assert t["violation"][b] == _violation64(pat, gl, gu, g[b], jac[b])
        m_ld, p_ld = sref.merit_and_predicted(pat, X[b], t["x_trial"][b], g[b], jac[b], gl, gu, np.longdouble)
        m_64, p_64 = sref.merit_and_predicted(pat, X[b], t["x_trial"][b], g[b], jac[b], gl, gu, np.float64)
        scale = float(max(m_ld, m_ld - p_ld))
        for name, gpu, ld, f64 in (("merit", t["merit"][b], m_ld, m_64), ("predicted", t["predicted"][b], p_ld, p_64)):
            bnd = max(float(abs(np.longdouble(f64) - ld)), 64 * EPS * scale)
            err = float(abs(np.longdouble(gpu) - ld))
            assert err <= 8 * bnd, (name, b, gpu, float(ld), f64)
            worst[name] = max(worst[name], err / bnd)
    record_property(f"lm_trial_mu_per_instance_{case}", worst)


# ---- GPU: the acceptance --------------------------------------------------------------------------------------------------

def _accept(bt, X, x_trial, g_trial, row_scale, merit, predicted, mu, nu, status, iterations, eta=1e-4, mu_min=1e-12, mu_max=1e10,
            gl=None, gu=None):
    import torch
    c = lambda a: _cuda(a)
    ci = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.int32)).cuda()
    t = dict(x=c(X), mu=c(mu), nu=c(nu), status=ci(status), iterations=ci(iterations))
    bt.lm_accept_device(t["x"], c(x_trial), c(g_trial), c(row_scale), c(merit), c(predicted), t["mu"], t["nu"], t["status"],
                        t["iterations"], None if gl is None else c(gl), None if gu is None else c(gu), eta, mu_min, mu_max)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in t.items()}


def _check_against_rule(X, x_trial, g_trial, row_scale, merit, predicted, mu, nu, status, iterations, out, gl, gu, eta, mu_min, mu_max,
                        exact_phi=False):
    """Every RUNNING instance against sref.accept on the same inputs (phi_t in numpy's summation order): decision, x, status
    and iterations equal wherever |rho - eta| > 1e-9 max(1, |rho|).  On the same decision nu and a rejection's mu are the
    rule's bits; an acceptance's mu depends on rho, so it is the rule's bits where phi_t is exact in both orders
    (`exact_phi`: one non-zero term) and within 1e-12 relative otherwise.  Instances that are not RUNNING are untouched.
    Returns the device's decisions."""
    decisions = {}
    for b in range(X.shape[0]):
        if status[b] != capi.LM_RUNNING:
            for k, ref_v in (("x", X), ("mu", mu), ("nu", nu)):
                assert np.array_equal(_bits(out[k][b]), _bits(ref_v[b])), (k, b)
            assert out["status"][b] == status[b] and out["iterations"][b] == iterations[b], b
            continue
        glb, gub = (gl[b], gu[b]) if gl.ndim == 2 else (gl, gu)
        phi_t = sref.half_norm2(row_scale[b], g_trial[b], glb, gub)
        acc, rho, mu_r, nu_r, stalled = sref.accept(merit[b], predicted[b], phi_t, bool(np.all(np.isfinite(g_trial[b]))), mu[b], nu[b],
                                                    eta, mu_min, mu_max)
        dev_acc = bool(out["nu"][b] == 2.0)          # a rejection doubles nu >= 2
        if not abs(rho - eta) <= 1e-9 * max(1.0, abs(rho)):
            assert dev_acc == acc, (b, rho, eta)
        assert out["iterations"][b] == iterations[b] + 1, b
        decisions[b] = dev_acc
        if dev_acc != acc:
            continue
        assert out["nu"][b] == nu_r, b
        if acc:
            assert np.array_equal(_bits(out["x"][b]), _bits(x_trial[b])), b
            if exact_phi:
                assert np.array_equal(_bits(out["mu"][b]), _bits(mu_r)), (b, out["mu"][b], mu_r)
            else:
                assert abs(out["mu"][b] - mu_r) <= 1e-12 * mu_r, (b, out["mu"][b], mu_r)
            assert out["status"][b] == capi.LM_RUNNING, b
        else:
            assert np.array_equal(_bits(out["x"][b]), _bits(X[b])), b
            assert np.array_equal(_bits(out["mu"][b]), _bits(mu_r)), b
            assert out["status"][b] == (capi.LM_STALLED if stalled else capi.LM_RUNNING), b
    return decisions


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_accept_on_device_produced_inputs_follows_the_numpy_rule(case):
    """Trial on evaluated inputs with mu spread over 1e-6 ... 1e2, g at x_trial from twb_batch_eval_device, then the accept
    call against the numpy rule on exactly these inputs, for two values of eta."""
    import torch
    from towr_b200.solver import BatchedLevenbergMarquardt  # noqa: F401
    B = 16
    bt, X, g, jac, xl, xu = _evaluated(case, B, seed=321)
    mu = np.logspace(-6, 2, B)
    _, _, gl, gu = bt.problem.bounds()
    nu = np.full(B, 2.0)
    its = np.arange(B, dtype=np.int32)
    seen = set()
    for cap in (CAP, 5.0):                        # the large cap lets Gauss-Newton steps overshoot: rejections
        t = _trial(bt, X, g, jac, xl, xu, mu, tol=1e-300, cap=cap)
        gt = torch.empty((B, bt.problem.m), dtype=torch.float64, device="cuda")
        bt.eval_device(_cuda(t["x_trial"]), g=gt, flags=capi.EVAL_G)
        torch.cuda.synchronize()
        g_trial = gt.cpu().numpy()
        for eta in (1e-4, 0.75, 0.999):
            out = _accept(bt, X, t["x_trial"], g_trial, t["row_scale"], t["merit"], t["predicted"], mu, nu, t["status"], its, eta=eta)
            seen |= set(_check_against_rule(X, t["x_trial"], g_trial, t["row_scale"], t["merit"], t["predicted"], mu, nu, t["status"],
                                             its, out, gl, gu, eta, 1e-12, 1e10).values())
    assert seen == {True, False}, "expected both accepted and rejected trials"


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_accept_on_crafted_inputs(case):
    """Crafted merit / predicted / g_trial with unit row scales: one violated row of size v gives phi_t = v^2 / 2 exactly.
    predicted = 0 and < 0, NaN and +Inf in g_trial, rho far
    above and below eta, mu overflowing mu_max (STALLED), the mu_min floor, and instances that are not RUNNING."""
    p = _problem(case)
    _, _, gl, gu = p.bounds()
    fin = np.flatnonzero((np.abs(gl) < 1e10) & (np.abs(gu) < 1e10))
    row = int(fin[0])
    inside = np.where(np.abs(gl) < 1e10, gl, np.where(np.abs(gu) < 1e10, gu, 0.0))
    # (merit, predicted, violation v of `row`, mu, nu, status, special)
    rows = [
        (1.0, 0.0, 0.5, 1e-2, 2.0, 0, None),          # predicted = 0: reject
        (1.0, -0.5, 0.5, 1e-2, 2.0, 0, None),         # predicted < 0: reject
        (1.0, 0.5, 0.0, 1e-2, 2.0, 0, "nan"),         # NaN in g_trial: reject
        (1.0, 0.5, 0.0, 1e-2, 2.0, 0, "inf"),         # +Inf in g_trial: reject
        (2.0, 1.0, 0.0, 1e-2, 8.0, 0, None),          # rho = 2: accept, mu / 3, nu = 2
        (2.0, 1.5, 1.0, 1e-2, 2.0, 0, None),          # phi_t = 0.5, rho = 1: accept
        (1.0, 0.5, 2.0, 1e-2, 4.0, 0, None),          # phi_t = 2 > merit: reject, mu * 4, nu = 8
        (1.0, 0.5, 2.0, 6e9, 2.0, 0, None),           # reject: 1.2e10 > mu_max: STALLED
        (1.0, 1.0, 0.0, 2e-12, 2.0, 0, None),         # rho = 1: mu / 3 < mu_min = 1e-12: floored
        (1.0, 1.0, 0.0, 1e-2, 2.0, capi.LM_CONVERGED, None),
        (1.0, 1.0, 0.0, 1e-2, 2.0, capi.LM_STALLED, None),
        (1.0, 1.0, 0.0, 1e-2, 2.0, capi.LM_NONFINITE, None),
    ]
    B = len(rows)
    rng = np.random.default_rng(331)
    X = rng.standard_normal((B, p.n)); x_trial = X + 0.01 * rng.standard_normal((B, p.n))
    g_trial = np.tile(inside, (B, 1))
    merit, pred, mu, nu = (np.array([r[k] for r in rows], np.float64) for k in (0, 1, 3, 4))
    status = np.array([r[5] for r in rows], np.int32)
    its = np.full(B, 5, np.int32)
    for b, r in enumerate(rows):
        g_trial[b, row] = gu[row] + r[2]
        if r[6] == "nan":
            g_trial[b, rng.integers(p.m)] = np.nan
        elif r[6] == "inf":
            g_trial[b, rng.integers(p.m)] = np.inf
    scale = np.ones((B, p.m))
    bt = p.batch(B)
    out = _accept(bt, X, x_trial, g_trial, scale, merit, pred, mu, nu, status, its, eta=0.5)
    dec = _check_against_rule(X, x_trial, g_trial, scale, merit, pred, mu, nu, status, its, out, gl, gu, 0.5, 1e-12, 1e10, exact_phi=True)
    assert [dec[b] for b in range(9)] == [False, False, False, False, True, True, False, False, True]
    assert out["mu"][4] == 1e-2 * (1.0 / 3.0) and out["nu"][4] == 2.0
    assert out["mu"][6] == 4e-2 and out["nu"][6] == 8.0
    assert out["status"][7] == capi.LM_STALLED and out["mu"][7] == 1.2e10
    assert out["mu"][8] == 1e-12
    assert list(out["status"][9:]) == [capi.LM_CONVERGED, capi.LM_STALLED, capi.LM_NONFINITE]


# ---- GPU: solve iterations ------------------------------------------------------------------------------------------------

def _solver(case, B, seed, goals_perm=None):
    import torch
    from towr_b200.solver import BatchedLevenbergMarquardt
    p = _problem(case)
    rng = np.random.default_rng(seed)
    goals = np.column_stack([rng.uniform(0.3, 2.5, B), rng.uniform(-0.4, 0.4, B), np.full(B, 0.5), np.zeros(B), np.zeros(B),
                             rng.uniform(-0.5, 0.5, B)])
    noise = rng.standard_normal((B, p.n))
    if goals_perm is not None:
        goals, noise = goals[goals_perm], noise[goals_perm]
    bt = p.batch(B)
    x0, xl, xu = bt.goal_instances_device(_cuda(goals))
    X = torch.minimum(torch.maximum(x0 + 0.01 * _cuda(noise), xl), xu)
    return BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu), X


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_finished_instances_stay_put(case):
    """Instances preset to CONVERGED, STALLED and NONFINITE keep x, mu, nu and iterations bit for bit over further
    iterations (x_trial = x for them); an instance with a NaN in x becomes NONFINITE with x untouched and violation NaN; the
    RUNNING neighbours walk exactly as in a batch without the special instances."""
    import torch
    B = 8
    lm, X0 = _solver(case, B, seed=341)
    st_ref = lm.solve_state()
    X_ref = X0.clone()
    st = lm.solve_state()
    X = X0.clone()
    X[4, 3] = float("nan")
    st.status[1], st.status[2], st.status[3] = capi.LM_CONVERGED, capi.LM_STALLED, capi.LM_NONFINITE
    st.mu[1:4] = torch.tensor([3e-3, 5e9, 7e-2], dtype=torch.float64, device="cuda")
    st.nu[1:4] = 16.0
    st.iterations[1:4] = torch.tensor([3, 9, 1], dtype=torch.int32, device="cuda")
    keep = {k: getattr(st, k)[1:4].clone() for k in ("mu", "nu", "iterations")}
    X_keep = X.clone()
    for _ in range(4):
        lm.iterate(X_ref, st_ref, 1e-300)
        lm.iterate(X, st, 1e-300)
    torch.cuda.synchronize()
    special = [1, 2, 3, 4]
    for k in ("mu", "nu"):
        assert np.array_equal(_bits(getattr(st, k)[1:4].cpu().numpy()), _bits(keep[k].cpu().numpy())), k
    assert torch.equal(st.iterations[1:4], keep["iterations"])
    assert np.array_equal(_bits(X[special].cpu().numpy()), _bits(X_keep[special].cpu().numpy()))
    assert np.array_equal(_bits(st.x_trial[special].cpu().numpy()), _bits(X_keep[special].cpu().numpy()))
    assert st.status[4].item() == capi.LM_NONFINITE and np.isnan(st.violation[4].item()) and st.iterations[4].item() == 0
    assert [st.status[b].item() for b in (1, 2, 3)] == [capi.LM_CONVERGED, capi.LM_STALLED, capi.LM_NONFINITE]
    rest = [0, 5, 6, 7]
    assert np.array_equal(_bits(X[rest].cpu().numpy()), _bits(X_ref[rest].cpu().numpy()))
    for k in ("mu", "nu", "violation", "merit", "predicted"):
        assert np.array_equal(_bits(getattr(st, k)[rest].cpu().numpy()), _bits(getattr(st_ref, k)[rest].cpu().numpy())), k
    assert torch.equal(st.iterations[rest], st_ref.iterations[rest]) and torch.equal(st.status[rest], st_ref.status[rest])
    assert st_ref.iterations.min().item() == 4 and not torch.equal(X_ref, X0)


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_solve_is_deterministic_and_permutation_equivariant(case):
    B = 10
    perm = np.random.default_rng(351).permutation(B)
    lm, X0 = _solver(case, B, seed=352)
    outs = []
    for _ in range(2):
        X = X0.clone()
        outs.append((X,) + tuple(lm.solve(X, 12, 1e-8)))
    lmp, Xp = _solver(case, B, seed=352, goals_perm=perm)
    outp = (Xp,) + tuple(lmp.solve(Xp, 12, 1e-8))
    for a, b, c in zip(outs[0], outs[1], outp):
        a, b, c = a.cpu().numpy(), b.cpu().numpy(), c.cpu().numpy()
        bits = (lambda t: _bits(t)) if a.dtype == np.float64 else (lambda t: t)
        assert np.array_equal(bits(a), bits(b))
        assert np.array_equal(bits(c), bits(a[perm]))
    assert outs[0][2].min().item() >= 1


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_graph_replay_of_a_solve_iteration_equals_the_eager_iteration(case, monkeypatch):
    """The four calls of one iteration captured in a torch.cuda.CUDAGraph (after a first eager iteration, which uploads the
    pattern) and replayed twice equal two eager iterations bit for bit.  The batch's own evaluation graphs are off
    (TWB_GRAPH=0), so that its kernels are captured directly into the outer graph."""
    import torch
    monkeypatch.setenv("TWB_GRAPH", "0")
    B = 6
    lm, X0 = _solver(case, B, seed=361)
    tol = 1e-300

    def reset(st, X):
        X.copy_(X0); st.mu.fill_(lm.mu); st.nu.fill_(2.0); st.status.zero_(); st.iterations.zero_()

    st, X = lm.solve_state(), X0.clone()
    lm.iterate(X, st, tol)
    torch.cuda.synchronize()
    reset(st, X)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        lm.iterate(X, st, tol)
    st_e, X_e = lm.solve_state(), X0.clone()
    for _ in range(2):
        lm.iterate(X_e, st_e, tol)
    torch.cuda.synchronize()
    reset(st, X)
    graph.replay(); graph.replay()
    torch.cuda.synchronize()
    assert not torch.equal(X_e, X0)
    assert np.array_equal(_bits(X.cpu().numpy()), _bits(X_e.cpu().numpy()))
    for k in ("mu", "nu", "violation", "merit", "predicted", "x_trial", "row_scale"):
        assert np.array_equal(_bits(getattr(st, k).cpu().numpy()), _bits(getattr(st_e, k).cpu().numpy())), k
    assert torch.equal(st.status, st_e.status) and torch.equal(st.iterations, st_e.iterations)


@pytest.mark.gpu
def test_bad_arguments_are_rejected_and_enqueue_nothing():
    import torch
    p = _problem("hopper")
    B = 3
    bt = p.batch(B)
    X, g, jac, xl, xu = (_cuda(a) for a in _edge_inputs(p, B, seed=371))
    gl = _cuda(np.tile(p.bounds()[2], (B, 1))); gu = _cuda(np.tile(p.bounds()[3], (B, 1)))
    f = lambda *shape: torch.full(shape, 7.0, dtype=torch.float64, device="cuda")
    x = X.clone(); mu = f(B); nu = f(B); xt = f(B, p.n); rsc = f(B, p.m); mer = f(B); pred = f(B); viol = f(B)
    gt = g.clone()
    status = torch.full((B,), 0, dtype=torch.int32, device="cuda"); its = torch.full((B,), 5, dtype=torch.int32, device="cuda")
    v = lambda t: C.c_void_p(t.data_ptr())
    lib, h = capi.lib, bt._h
    nan = float("nan")

    def trial(**kw):
        a = dict(b=h, x=v(x), g=v(g), jac=v(jac), xl=v(xl), xu=v(xu), gl=v(gl), gu=v(gu), mu=v(mu), cap=CAP, cg=CG, tol=1e-6,
                 st=v(status), xt=v(xt), rs=v(rsc), merit=v(mer), pred=v(pred), viol=v(viol), stream=None)
        a.update(kw)
        return lib.twb_batch_lm_trial_device(*a.values())

    def accept(**kw):
        a = dict(b=h, x=v(x), xt=v(xt), gt=v(gt), gl=v(gl), gu=v(gu), rs=v(rsc), merit=v(mer), pred=v(pred), mu=v(mu), nu=v(nu),
                 st=v(status), its=v(its), eta=1e-4, mu_min=1e-12, mu_max=1e10, stream=None)
        a.update(kw)
        return lib.twb_batch_lm_accept_device(*a.values())

    bad_trial = [dict(b=None), dict(x=None), dict(g=None), dict(jac=None), dict(mu=None), dict(st=None), dict(xt=None), dict(rs=None),
                 dict(merit=None), dict(pred=None), dict(xl=None), dict(xu=None), dict(gl=None), dict(gu=None), dict(cap=0.0),
                 dict(cap=nan), dict(cg=-1), dict(cg=10001), dict(tol=-1e-9), dict(tol=nan)]
    bad_accept = [dict(b=None), dict(x=None), dict(xt=None), dict(gt=None), dict(rs=None), dict(merit=None), dict(pred=None),
                  dict(mu=None), dict(nu=None), dict(st=None), dict(its=None), dict(gl=None), dict(gu=None), dict(eta=-1e-9),
                  dict(eta=1.0), dict(eta=nan), dict(mu_min=0.0), dict(mu_min=2e10), dict(mu_min=nan), dict(mu_max=nan)]
    assert [trial(**k) for k in bad_trial] == [capi.ERR_INVALID] * len(bad_trial)
    assert [accept(**k) for k in bad_accept] == [capi.ERR_INVALID] * len(bad_accept)
    with pytest.raises(capi.TowrB200Error):
        bt.lm_trial_device(x, g, jac, mu, status, xt, rsc, mer, pred, xl, xu, cap=-1.0)
    from test_lm_step import TOO_LARGE, _problem_of
    big = _problem_of(*TOO_LARGE)
    bb = big.batch(2)
    z = lambda *s: torch.zeros(s, dtype=torch.float64, device="cuda")
    assert lib.twb_batch_lm_trial_device(bb._h, v(z(2, big.n)), v(z(2, big.m)), v(z(2, big.nnz)), None, None, None, None, v(z(2)), CAP, CG,
                                         1e-6, v(torch.zeros(2, dtype=torch.int32, device="cuda")), v(z(2, big.n)), v(z(2, big.m)),
                                         v(z(2)), v(z(2)), None, None) == capi.ERR_UNSUPPORTED
    torch.cuda.synchronize()
    assert torch.equal(x, X) and torch.equal(gt, g)
    for t in (mu, nu, xt, rsc, mer, pred, viol):
        assert bool((t == 7.0).all())
    assert bool((status == 0).all()) and bool((its == 5).all())
    assert trial() == capi.OK and accept() == capi.OK          # the batch still serves valid calls
    torch.cuda.synchronize()
    assert bool((its == 6).all()) or bool((status != 0).any())


# ---- GPU: end to end ------------------------------------------------------------------------------------------------------

def _walk(lm, X, tol, budget):
    """The solve's iterations one at a time, checking after each that every accepted trial decreased the merit
    (phi_t < phi0, phi_t recomputed in torch from g_trial and the row scales).  Returns the solve state."""
    import torch
    st = lm.solve_state()
    accepted = 0
    for _ in range(budget):
        before = st.iterations.clone()
        lm.iterate(X, st, tol)
        acc = (st.iterations > before) & (st.nu == 2.0)
        v = lm._violation(st.g_trial)
        phi_t = 0.5 * ((st.row_scale * v) ** 2).sum(dim=1)
        assert bool((phi_t[acc] < st.merit[acc]).all())
        accepted += int(acc.sum())
        if not bool((st.status == capi.LM_RUNNING).any()):
            break
    lm.iterate(X, st, tol, cg_iters=0)
    torch.cuda.synchronize()
    assert accepted > 0
    return st


def _check_converged(lm, X, st, tol, gl, gu):
    """Re-evaluate the converged instances at their returned x: scaled violation <= tol (float64 on the host)."""
    import torch
    bt, p = lm.batch, lm.p
    g = torch.empty((lm.B, p.m), dtype=torch.float64, device="cuda")
    jac = torch.empty((lm.B, p.nnz), dtype=torch.float64, device="cuda")
    bt.eval_device(X, g=g, jac=jac, flags=capi.EVAL_G | capi.EVAL_JAC)
    torch.cuda.synchronize()
    conv = np.flatnonzero(st.status.cpu().numpy() == capi.LM_CONVERGED)
    pat = ref.Pattern(p.row_ptr(), p.structure()[1], p.n)
    viol = st.violation.cpu().numpy()
    for chunk in np.array_split(conv, max(1, len(conv) // 256)):
        if not len(chunk):
            continue
        gh, jh = g[chunk].cpu().numpy(), jac[chunk].cpu().numpy()
        for k, b in enumerate(chunk):
            glb, gub = (gl[b], gu[b]) if gl.ndim == 2 else (gl, gu)
            v = _violation64(pat, glb, gub, gh[k], jh[k])
            assert v <= tol and v == viol[b], (b, v, viol[b])
    return conv


def _record(record_property, name, st, budget):
    counts = np.bincount(st.status.cpu().numpy(), minlength=4)
    rec = {"instances": int(counts.sum()), "budget": budget, "tol": TOL, "running": int(counts[0]), "converged": int(counts[1]),
           "stalled": int(counts[2]), "nonfinite": int(counts[3]), "iterations_max": int(st.iterations.max())}
    record_property(name, rec)
    return counts


@pytest.mark.gpu
def test_solve_config5_shard(record_property):
    """4096 goal-randomised Anymal instances on mixed Slope / Chimney / Gap terrains (the set-up of
    test_device_resident_multistart_loop_config5_matches_oracle_driven_loop), solved to TOL within BUDGET iterations."""
    import torch
    import oracle_lib
    from towr_b200.solver import BatchedLevenbergMarquardt
    spec = tb.make_formulation("anymal_trot_mixed").to_spec()
    p = tb.Problem(spec)
    B = 4096
    rng = np.random.default_rng(77)
    terr = rng.choice([tb.SLOPE, tb.CHIMNEY, tb.GAP], B).astype(np.int32)
    goals = np.column_stack([rng.uniform(1.0, 2.0, B), rng.uniform(-0.2, 0.2, B), np.full(B, 0.5), np.zeros(B), np.zeros(B), rng.uniform(-0.2, 0.2, B)])
    bt = p.batch(B); bt.set_terrains(terr)
    x0, xl, xu = bt.goal_instances_device(torch.from_numpy(goals).cuda())
    X0 = torch.minimum(torch.maximum(x0 + 0.01 * torch.from_numpy(rng.standard_normal((B, p.n))).cuda(), xl), xu)
    lm = BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu)
    X = X0.clone()
    st = _walk(lm, X, TOL, BUDGET)
    Xs = X0.clone()
    status, its, viol, mu = lm.solve(Xs, BUDGET, TOL)                # the solve itself walks the same iterations
    assert torch.equal(Xs, X) and torch.equal(status, st.status) and torch.equal(its, st.iterations)
    assert np.array_equal(_bits(viol.cpu().numpy()), _bits(st.violation.cpu().numpy()))
    counts = _record(record_property, "lm_solve_config5_shard", st, BUDGET)
    assert counts[capi.LM_NONFINITE] == 0 and counts[capi.LM_CONVERGED] > 0
    _, _, gl, gu = p.bounds()
    conv = _check_converged(lm, X, st, TOL, gl, gu)
    # the oracle at the returned x of converged instances of every terrain
    o = oracle_lib.Oracle(spec)
    pat = ref.Pattern(p.row_ptr(), p.structure()[1], p.n)
    Xh = X.cpu().numpy()
    for t in (tb.SLOPE, tb.CHIMNEY, tb.GAP):
        for b in conv[terr[conv] == t][:4]:
            o.set_terrain(int(t))
            r = o.eval(Xh[b])
            assert r["rc"] == 0
            assert _violation64(pat, gl, gu, r["g"], r["jac"]) <= TOL, (b, t)


@pytest.mark.gpu
def test_solve_base_rom_with_instance_bounds(record_property):
    """4096 Anymal instances with BaseMotionConstraint, each from its own measured state and solved against its own
    constraint bounds (scripts/lm_bounds_bench.py's workload)."""
    import torch
    from towr_b200.solver import BatchedLevenbergMarquardt
    from test_state_instances import _random_states
    f = tb.make_formulation("anymal_trot_block_base_rom")
    p = tb.Problem(f.to_spec())
    B = 4096
    rng = np.random.default_rng(707)
    bt = p.batch(B)
    x0, xl, xu, gl, gu = bt.state_instances_device(torch.from_numpy(_random_states(f, rng, B)).cuda(), want_g_bounds=True)
    X = torch.minimum(torch.maximum(x0 + 0.01 * torch.from_numpy(rng.standard_normal((B, p.n))).cuda(), xl), xu)
    lm = BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu, g_lower=gl, g_upper=gu)
    st = _walk(lm, X, TOL, BUDGET)
    counts = _record(record_property, "lm_solve_base_rom", st, BUDGET)
    assert counts[capi.LM_NONFINITE] == 0 and counts[capi.LM_CONVERGED] > 0
    _check_converged(lm, X, st, TOL, gl.cpu().numpy(), gu.cpu().numpy())
