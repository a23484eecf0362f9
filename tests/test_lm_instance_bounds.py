"""twb_batch_lm_step_bounds_device: the Levenberg-Marquardt step of twb_batch_lm_step_device with one row of constraint bounds
per instance, on every launch path, against the float64 and extended-precision statement of the step in
tests/lm_reference.py; and BatchedLevenbergMarquardt driven by the per-instance bounds of twb_batch_state_instances_device
(BaseMotionConstraint rows around each instance's own initial base height) against the oracle-driven numpy twin."""
import ctypes as C

import numpy as np
import pytest

import towr_b200 as tb
from towr_b200 import capi
import lm_reference as ref
from test_lm_step import CASES, CG, CAP, EPS, F64_RUNS, MU, PATH_CASES, _bits, _cuda, _edge_inputs, _problem, _violation64, lm_path

pytestmark = pytest.mark.gpu


def _step(bt, X, g, jac, xl, xu, gl=None, gu=None, cg_iters=CG):
    """One device step from numpy inputs (gl / gu (B, m) or None: the problem's bounds): (x_new, violation) as numpy."""
    import torch
    x = _cuda(X)
    viol = torch.full((bt.B,), 7.0, dtype=torch.float64, device="cuda")
    bt.lm_step_device(x, _cuda(g), _cuda(jac), _cuda(xl), _cuda(xu), MU, CAP, cg_iters, viol,
                      g_lower=None if gl is None else _cuda(gl), g_upper=None if gu is None else _cuda(gu))
    torch.cuda.synchronize()
    return x.cpu().numpy(), viol.cpu().numpy()


def _instance_bounds(p, g, B, seed):
    """Per-instance constraint bounds: the problem's shifted by a random offset per row (inequality rows also widened),
    about a tenth of the rows of each instance unbounded below (-Inf) and another tenth above (+Inf); instance 0's bounds
    contain its g, so r = 0 there."""
    rng = np.random.default_rng(seed)
    _, _, gl0, gu0 = p.bounds()
    fin_l, fin_u = np.abs(gl0) < 1e10, np.abs(gu0) < 1e10
    d = rng.uniform(-0.2, 0.2, (B, p.m))
    w = np.where(gl0 < gu0, rng.uniform(0.0, 0.05, (B, p.m)), 0.0)
    gl = np.where(fin_l, gl0 + d - w, gl0)
    gu = np.where(fin_u, gu0 + d + w, gu0)
    gl[rng.random((B, p.m)) < 0.1] = -np.inf
    gu[rng.random((B, p.m)) < 0.1] = np.inf
    gl[0] = np.minimum(gl[0], g[0]); gu[0] = np.maximum(gu[0], g[0])
    return gl, gu


def _compare_with_reference(p, X, g, jac, xl, xu, gl, gu, x_gpu, v_gpu):
    """test_lm_step's criterion with instance b's own constraint bounds gl[b], gu[b]: ||x_gpu - x_ld|| <= 8 max(worst of
    F64_RUNS relabelled float64 steps' error, 64 eps ||dx_ld||), and the violation equals the float64 one exactly."""
    row_ptr, col_idx = p.row_ptr(), p.structure()[1]
    pat = ref.Pattern(row_ptr, col_idx, p.n)
    worst = 0.0
    for b in range(X.shape[0]):
        dld, _ = ref.lm_capped_step(pat, g[b], jac[b], gl[b], gu[b], MU, CAP, CG, np.longdouble)
        xld = np.minimum(np.maximum(X[b].astype(np.longdouble) + dld, xl[b].astype(np.longdouble)), xu[b].astype(np.longdouble))
        runs = ref.relabelled_float64_steps(X[b], g[b], jac[b], xl[b], xu[b], gl[b], gu[b], row_ptr, col_idx, MU, CAP, CG, F64_RUNS, b)
        err_f64 = max(float(np.max(np.abs(x.astype(np.longdouble) - xld))) for x in runs)
        err_gpu = float(np.max(np.abs(x_gpu[b].astype(np.longdouble) - xld)))
        bound = max(err_f64, 64 * EPS * float(np.max(np.abs(dld))))
        ratio = err_gpu / bound if bound > 0 else (0.0 if err_gpu == 0 else np.inf)
        assert ratio <= 8.0, (b, err_gpu, err_f64, float(np.max(np.abs(dld))))
        assert v_gpu[b] == _violation64(pat, gl[b], gu[b], g[b], jac[b]), b
        worst = max(worst, ratio)
    return worst


@pytest.mark.parametrize("case", PATH_CASES)
def test_problem_bounds_per_instance_give_the_old_bits(case):
    """Per-instance bounds equal to the problem's (broadcast to (B, m)) and both NULL: bit for bit twb_batch_lm_step_device."""
    import torch
    p = _problem(case)
    B = 10
    X, g, jac, xl, xu = _edge_inputs(p, B, seed=201)
    bt = p.batch(B)
    _, _, gl0, gu0 = p.bounds()
    x_old, v_old = _step(bt, X, g, jac, xl, xu)
    x_new, v_new = _step(bt, X, g, jac, xl, xu, np.tile(gl0, (B, 1)), np.tile(gu0, (B, 1)))
    assert np.array_equal(_bits(x_new), _bits(x_old)) and np.array_equal(_bits(v_new), _bits(v_old))
    x = _cuda(X)
    viol = torch.full((B,), 7.0, dtype=torch.float64, device="cuda")
    v = lambda t: C.c_void_p(t.data_ptr())
    assert capi.lib.twb_batch_lm_step_bounds_device(bt._h, v(x), v(_cuda(g)), v(_cuda(jac)), v(_cuda(xl)), v(_cuda(xu)), None, None,
                                                    MU, CAP, CG, v(viol), None) == capi.OK
    torch.cuda.synchronize()
    assert np.array_equal(_bits(x.cpu().numpy()), _bits(x_old)) and np.array_equal(_bits(viol.cpu().numpy()), _bits(v_old))


@pytest.mark.parametrize("case", PATH_CASES)
def test_instance_bounds_match_the_extended_precision_reference(case, record_property):
    if not ref.LONGDOUBLE_IS_WIDER:
        pytest.skip("np.longdouble is not wider than float64 here")
    p = _problem(case)
    B = 8
    X, g, jac, xl, xu = _edge_inputs(p, B, seed=211)
    X[0] = np.clip(X[0], xl[0], xu[0])                    # instance 0: inside its bounds, so no projection either
    gl, gu = _instance_bounds(p, g, B, seed=212)
    bt = p.batch(B)
    x_gpu, v_gpu = _step(bt, X, g, jac, xl, xu, gl, gu)
    assert np.array_equal(_bits(x_gpu[0]), _bits(X[0])) and v_gpu[0] == 0.0          # r = 0: no step at all
    assert np.all(np.isfinite(v_gpu)) and np.all(v_gpu[1:] > 0.0)                       # +-Inf bounds are no error
    worst = _compare_with_reference(p, X, g, jac, xl, xu, gl, gu, x_gpu, v_gpu)
    x_shared, v_shared = _step(bt, X, g, jac, xl, xu)
    assert not np.array_equal(x_gpu[1:], x_shared[1:]) and not np.array_equal(v_gpu, v_shared)   # the bounds were used
    record_property(f"lm_instance_bounds_{case}", {"path": lm_path(p.n, p.m, p.nnz), "instances": B, "worst_ratio_over_f64_bound": worst})


@pytest.mark.parametrize("case", PATH_CASES)
def test_instances_are_independent_under_permutation(case):
    p = _problem(case)
    B = 9
    X, g, jac, xl, xu = _edge_inputs(p, B, seed=221)
    gl, gu = _instance_bounds(p, g, B, seed=222)
    bt = p.batch(B)
    x1, v1 = _step(bt, X, g, jac, xl, xu, gl, gu)
    perm = np.random.default_rng(223).permutation(B)
    x2, v2 = _step(bt, X[perm], g[perm], jac[perm], xl[perm], xu[perm], gl[perm], gu[perm])
    assert np.array_equal(_bits(x2), _bits(x1[perm])) and np.array_equal(_bits(v2), _bits(v1[perm]))


@pytest.mark.parametrize("case", PATH_CASES)
def test_nan_bound_leaves_the_instance_unchanged(case):
    """A NaN in one instance's g_lower or g_upper counts like a non-finite g: that instance keeps its x bit for bit and reports
    violation NaN; the other instances equal a run without the NaN bit for bit."""
    p = _problem(case)
    B = 6
    X, g, jac, xl, xu = _edge_inputs(p, B, seed=231)
    gl, gu = _instance_bounds(p, g, B, seed=232)
    rng = np.random.default_rng(233)
    glb, gub = gl.copy(), gu.copy()
    glb[1, rng.integers(p.m)] = np.nan
    gub[4, rng.integers(p.m)] = np.nan
    bt = p.batch(B)
    x_ref, v_ref = _step(bt, X, g, jac, xl, xu, gl, gu)
    x_bad, v_bad = _step(bt, X, g, jac, xl, xu, glb, gub)
    clean = np.array([0, 2, 3, 5])
    assert np.array_equal(_bits(x_bad[clean]), _bits(x_ref[clean])) and np.array_equal(_bits(v_bad[clean]), _bits(v_ref[clean]))
    for b in (1, 4):
        assert np.array_equal(_bits(x_bad[b]), _bits(X[b])), b
        assert np.isnan(v_bad[b]), (b, v_bad[b])


def test_bad_bound_arguments_are_rejected_and_leave_x_untouched():
    import torch
    p = _problem("hopper")
    B = 3
    bt = p.batch(B)
    X, g, jac, xl, xu = (_cuda(a) for a in _edge_inputs(p, B, seed=241))
    gl, gu = (_cuda(a) for a in _instance_bounds(p, g.cpu().numpy(), B, seed=242))
    x = X.clone()
    viol = torch.full((B,), 7.0, dtype=torch.float64, device="cuda")
    v = lambda t: C.c_void_p(t.data_ptr())
    step = lambda *a: capi.lib.twb_batch_lm_step_bounds_device(*a)
    h = bt._h
    calls = [
        step(h, v(x), v(g), v(jac), v(xl), v(xu), v(gl), None, MU, CAP, CG, v(viol), None),
        step(h, v(x), v(g), v(jac), v(xl), v(xu), None, v(gu), MU, CAP, CG, v(viol), None),
        step(h, v(x), v(g), v(jac), None, None, v(gl), None, MU, CAP, CG, v(viol), None),
        step(None, v(x), v(g), v(jac), v(xl), v(xu), v(gl), v(gu), MU, CAP, CG, v(viol), None),
        step(h, v(x), v(g), v(jac), v(xl), None, v(gl), v(gu), MU, CAP, CG, v(viol), None),
        step(h, v(x), v(g), v(jac), v(xl), v(xu), v(gl), v(gu), -1.0, CAP, CG, v(viol), None),
        step(h, v(x), v(g), v(jac), v(xl), v(xu), v(gl), v(gu), MU, CAP, -1, v(viol), None),
    ]
    assert calls == [capi.ERR_INVALID] * len(calls)
    wrong = [gl[:, :-1].contiguous(), gl.to(torch.float32), gl.cpu(), gl.t().contiguous().t(), gl.reshape(-1), gl[:-1].contiguous()]
    for bad in wrong:
        with pytest.raises(AssertionError):
            bt.lm_step_device(x, g, jac, xl, xu, MU, CAP, CG, viol, g_lower=bad, g_upper=gu)
        with pytest.raises(AssertionError):
            bt.lm_step_device(x, g, jac, xl, xu, MU, CAP, CG, viol, g_lower=gl, g_upper=bad)
    with pytest.raises(AssertionError):
        bt.lm_step_device(x, g, jac, xl, xu, MU, CAP, CG, viol, g_lower=gl)
    torch.cuda.synchronize()
    assert torch.equal(x, X) and bool((viol == 7.0).all())
    assert step(h, v(x), v(g), v(jac), v(xl), v(xu), v(gl), v(gu), MU, CAP, CG, v(viol), None) == capi.OK   # still serves
    torch.cuda.synchronize()
    assert bool(torch.isfinite(viol).all())


@pytest.mark.parametrize("case", PATH_CASES)
def test_graph_replay_with_instance_bounds_equals_the_eager_step(case):
    import torch
    p = _problem(case)
    B = 6
    bt = p.batch(B)
    Xh, gh, jh, xlh, xuh = _edge_inputs(p, B, seed=251)
    X1, g, jac, xl, xu = (_cuda(a) for a in (Xh, gh, jh, xlh, xuh))
    X2 = _cuda(_edge_inputs(p, B, seed=252)[0])
    gl, gu = (_cuda(a) for a in _instance_bounds(p, gh, B, seed=253))
    viol = torch.empty(B, dtype=torch.float64, device="cuda")
    bt.lm_step_device(X1.clone(), g, jac, xl, xu, MU, CAP, CG, viol, g_lower=gl, g_upper=gu)     # first call: pattern upload
    torch.cuda.synchronize()
    x = X1.clone()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        bt.lm_step_device(x, g, jac, xl, xu, MU, CAP, CG, viol, g_lower=gl, g_upper=gu)
    for X in (X1, X2):
        eager_x = X.clone()
        eager_v = torch.empty(B, dtype=torch.float64, device="cuda")
        bt.lm_step_device(eager_x, g, jac, xl, xu, MU, CAP, CG, eager_v, g_lower=gl, g_upper=gu)
        x.copy_(X)
        viol.fill_(7.0)
        graph.replay()
        torch.cuda.synchronize()
        assert not torch.equal(eager_x, X)
        assert np.array_equal(_bits(x.cpu().numpy()), _bits(eager_x.cpu().numpy()))
        assert np.array_equal(_bits(viol.cpu().numpy()), _bits(eager_v.cpu().numpy()))


def _scaled_violation(g, jac, gl, gu, pat):
    """max_i |s_i r_i| per instance, in float64 on the host."""
    return np.array([_violation64(pat, gl[b], gu[b], g[b], jac[b]) for b in range(g.shape[0])])


def test_device_pipeline_from_measured_states_with_base_rom():
    """4096 Anymal instances with BaseMotionConstraint, each with its own start (initial base z spread by +-0.05) and goal:
    setup on the device with the per-instance constraint bounds, then 12 Levenberg-Marquardt iterations against them.  The
    first violation is measured against each instance's own LZ band, and the oracle-driven numpy twin with the instance's
    bounds walks a subsample of 8 instances to the same iterates."""
    import torch
    from towr_b200.solver import BatchedLevenbergMarquardt
    from test_solver_loop import LevenbergMarquardtReference
    from test_state_instances import _base_z_rows, _random_states
    import oracle_lib
    f = tb.make_formulation("anymal_trot_block_base_rom")
    spec = f.to_spec()
    p = tb.Problem(spec)
    B, iters = 4096, 12
    rng = np.random.default_rng(707)
    S = _random_states(f, rng, B)
    bt = p.batch(B)
    x0, xl, xu, gl, gu = bt.state_instances_device(torch.from_numpy(S).cuda(), want_g_bounds=True)
    X = torch.minimum(torch.maximum(x0 + 0.01 * torch.from_numpy(rng.standard_normal((B, p.n))).cuda(), xl), xu)
    starts = X.cpu().numpy().copy()
    lm = BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu, g_lower=gl, g_upper=gu)
    hist = torch.empty((iters, B), dtype=torch.float64, device="cuda")
    hist[0] = lm.step(X)
    g1, j1 = lm.g.cpu().numpy(), lm.jac_vals.cpu().numpy()          # the first evaluation, at the starts
    for it in range(1, iters):
        hist[it] = lm.step(X)
    hist = hist.cpu().numpy(); X_gpu = X.cpu().numpy()
    assert np.isfinite(hist).all() and not lm.status.any().item()
    assert not np.array_equal(X_gpu, starts)
    gl_h, gu_h = gl.cpu().numpy(), gu.cpu().numpy()
    _, _, pgl, pgu = p.bounds()
    pat = ref.Pattern(p.row_ptr(), p.structure()[1], p.n)
    own = _scaled_violation(g1, j1, gl_h, gu_h, pat)
    assert np.array_equal(hist[0], own)
    rows = _base_z_rows(p)
    band_differs = np.flatnonzero(np.any(gl_h[:, rows] != pgl[rows], axis=1))
    assert band_differs.size > 0
    shared = _scaled_violation(g1[band_differs], j1[band_differs], np.tile(pgl, (band_differs.size, 1)), np.tile(pgu, (band_differs.size, 1)), pat)
    assert np.any(shared != hist[0, band_differs])
    o = oracle_lib.Oracle(spec)
    xl_h, xu_h = xl.cpu().numpy(), xu.cpu().numpy()
    for b in rng.choice(B, 8, replace=False):
        twin = LevenbergMarquardtReference(o, p, spec.terrain, xl_h[b], xu_h[b])
        twin.gl, twin.gu = gl_h[b], gu_h[b]
        x = starts[b].copy()
        for it in range(iters):
            x, v = twin.step(x)
            assert abs(v - hist[it, b]) <= 1e-6 * max(1e-9, abs(v)), (b, it)
        assert np.allclose(x, X_gpu[b], rtol=0, atol=1e-8), (b, float(np.abs(x - X_gpu[b]).max()))


def test_native_step_matches_the_tensor_algebra_step_with_instance_bounds():
    import torch
    from towr_b200.solver import BatchedLevenbergMarquardt
    from test_state_instances import _random_states
    f = tb.make_formulation("anymal_trot_block_base_rom")
    p = tb.Problem(f.to_spec())
    B = 70
    rng = np.random.default_rng(808)
    bt = p.batch(B)
    x0, xl, xu, gl, gu = bt.state_instances_device(torch.from_numpy(_random_states(f, rng, B)).cuda(), want_g_bounds=True)
    X0 = torch.minimum(torch.maximum(x0 + 0.01 * torch.from_numpy(rng.standard_normal((B, p.n))).cuda(), xl), xu)
    Xa, Xb = X0.clone(), X0.clone()
    a = BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu, g_lower=gl, g_upper=gu, native=True)
    b = BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu, g_lower=gl, g_upper=gu, native=False)
    shared = BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu, native=True)
    v_shared = shared.step(X0.clone())
    for it in range(4):
        va, vb = a.step(Xa), b.step(Xb)
        torch.cuda.synchronize()
        if it == 0:
            assert not torch.equal(va, v_shared)                 # the instances' own bounds are in use
        assert torch.allclose(va, vb, rtol=1e-12, atol=1e-14)
        assert torch.allclose(Xa, Xb, rtol=1e-8, atol=1e-10), (it, float((Xa - Xb).abs().max()))
    assert not torch.equal(Xa, X0)
