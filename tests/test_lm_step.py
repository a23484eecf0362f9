"""twb_batch_lm_step_device (towr_b200/csrc/lm_kernel.cu) on every launch path, one step at a time, against the plain float64
and extended-precision statement of the same step in tests/lm_reference.py.

LaunchLmStep picks one of three kernels from the problem's size: the row-scaled Jacobian values Js in shared memory or
re-read from global memory, with 16-bit or 32-bit pattern indices.  The cases below are chosen so that every kernel runs
(test_cases_cover_every_launch_path states which case takes which).  The CPU tests at the top check the reference itself."""
import ctypes as C
import functools

import numpy as np
import pytest

import towr_b200 as tb
from towr_b200 import capi
from towr_b200.configs import synthetic_iterates, synthetic_iterates_fast
import lm_reference as ref

MU, CAP, CG = 1e-2, 0.1, 25          # BatchedLevenbergMarquardt's defaults
EPS = np.finfo(np.float64).eps
SMEM_J_BYTES = 220 * 1024            # LaunchLmStep: vectors + Js up to this size keep Js in shared memory
VECTOR_BYTES = 200 * 1024            # twb_batch_lm_step_device: larger solver vectors are TWB_ERR_UNSUPPORTED

# name: (recipe, make_formulation keywords, optimise the phase durations on top of the recipe)
CASES = {
    "hopper": ("hopper", {}, False),
    "anymal_trot_block": ("anymal_trot_block", {}, False),
    "biped_walk_stairs_durations": ("biped_walk_stairs", {}, True),
    "hyq_gallop_gap": ("hyq_gallop_gap", {}, False),                 # BASELINE config 4 (the recipe optimises durations)
    "hyq_gallop_gap_3s": ("hyq_gallop_gap", {"t_total": 3.0}, False),
}
TOO_LARGE = ("anymal_trot_block", {"t_total": 24.0}, False)
# one case per kernel, each with a Jacobian pattern of full column rank (mu = 0 leaves Js^T Js regular on random values)
PATH_CASES = ["hopper", "biped_walk_stairs_durations", "hyq_gallop_gap_3s"]

needs_longdouble = pytest.mark.skipif(not ref.LONGDOUBLE_IS_WIDER, reason="np.longdouble is not wider than float64 here")


def _problem_of(recipe, kw, optimise):
    f = tb.make_formulation(recipe, **kw)
    if optimise:
        f.params_.OptimizePhaseDurations()
    return tb.Problem(f.to_spec())


@functools.lru_cache(maxsize=None)
def _problem(case):
    return _problem_of(*CASES[case])


def lm_path(n, m, nnz):
    """The kernel LaunchLmStep runs for these dimensions (capi.cc rejects the vectors first when they are too large)."""
    vec = 8 * (2 * m + 4 * n + 32)
    if vec > VECTOR_BYTES:
        return "unsupported"
    js = "smem" if vec + 8 * nnz <= SMEM_J_BYTES else "global"
    return js + ("/idx16" if max(n, m, nnz) < 65536 else "/idx32")


def _path(p):
    return lm_path(p.n, p.m, p.nnz)


def _bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def _random_system(rng, m, n, density=0.3):
    """A random CSR pattern with one empty row and one empty column, and values on it."""
    mask = rng.random((m, n)) < density
    mask[m // 2] = False
    mask[:, n // 3] = False
    J = np.where(mask, rng.standard_normal((m, n)) * rng.choice([0.5, 3.0, 2e3], m)[:, None], 0.0)
    row_ptr = np.concatenate([[0], np.cumsum(mask.sum(axis=1))])
    return J, row_ptr, np.nonzero(mask)[1], J[mask]


# ---- CPU: the cases and the reference ------------------------------------------------------------------------------------

def test_cases_cover_every_launch_path():
    paths = {case: _path(_problem(case)) for case in CASES}
    assert set(paths.values()) == {"smem/idx16", "global/idx16", "global/idx32"}, paths
    assert {paths[c] for c in PATH_CASES} == {"smem/idx16", "global/idx16", "global/idx32"}
    assert paths["hyq_gallop_gap"] == "global/idx16"
    assert _path(_problem_of(*TOO_LARGE)) == "unsupported"
    # Js in shared memory needs 8 nnz bytes <= 220 KiB, so nnz < 28 160 < 65 536: 32-bit indices never meet that kernel
    assert SMEM_J_BYTES // 8 < 65536


def test_reference_products_against_dense_algebra():
    rng = np.random.default_rng(3)
    J, row_ptr, col_idx, vals = _random_system(rng, 23, 17)
    pat = ref.Pattern(row_ptr, col_idx, 17)
    v, u = rng.standard_normal(17), rng.standard_normal(23)
    assert np.allclose(pat.matvec(vals, v), J @ v, rtol=1e-14, atol=1e-12)
    assert np.allclose(pat.rmatvec(vals[pat.by_col], u), J.T @ u, rtol=1e-14, atol=1e-12)
    assert np.array_equal(pat.row_max_abs(vals), np.abs(J).max(axis=1))
    assert pat.matvec(vals, v)[23 // 2] == 0.0 and pat.rmatvec(vals[pat.by_col], u)[17 // 3] == 0.0


@needs_longdouble
def test_reference_float64_agrees_with_longdouble_on_a_well_conditioned_system():
    """mu = 5 keeps Js^T Js + mu I within a condition number of 4, so 25 iterations converge in both precisions and the
    float64 step is the longdouble one to a few roundings of x.  (Where CG stops short of convergence, or just reaches
    it, float64 and longdouble iterates can differ by far more: the device tests compare against float64's own error.)"""
    rng = np.random.default_rng(5)
    m, n = 40, 25
    _, row_ptr, col_idx, vals = _random_system(rng, m, n)
    g = rng.standard_normal(m)
    gl, gu = np.full(m, -0.2), np.full(m, 0.3)
    gl[::5] = gu[::5] = 0.1                                   # equality rows
    x = rng.standard_normal(n)
    xl, xu = np.full(n, -1.0), np.full(n, 1.0)
    args = (x, g, vals, xl, xu, gl, gu, row_ptr, col_idx, 5.0, 10.0, 25)
    x64, v64 = ref.lm_step(*args, dtype=np.float64)
    xld, vld = ref.lm_step(*args, dtype=np.longdouble)
    assert x64.dtype == np.float64 and xld.dtype == np.longdouble
    assert np.max(np.abs(x64 - xld)) <= 4 * EPS
    assert abs(v64 - vld) <= 4 * EPS * vld
    assert not np.array_equal(x64, np.clip(x, xl, xu))          # the step moved x


@needs_longdouble
def test_reference_cg_with_n_iterations_solves_the_damped_normal_equations():
    """cg_iters = n, a large mu and no cap: the step is the solution of (Js^T Js + mu I) dx = -Js^T rs, here from
    np.linalg.solve refined with residuals in longdouble (LAPACK has no longdouble)."""
    rng = np.random.default_rng(8)
    m, n, mu = 30, 20, 4.0
    J, row_ptr, col_idx, vals = _random_system(rng, m, n)
    g = 2.0 * rng.standard_normal(m)
    gl, gu = np.full(m, -0.5), np.full(m, 0.5)
    pat = ref.Pattern(row_ptr, col_idx, n)
    dx, viol = ref.lm_capped_step(pat, g, vals, gl, gu, mu, 1e9, n, dtype=np.longdouble)
    L = np.longdouble
    Jl = J.astype(L)
    s = 1 / np.maximum(np.abs(Jl).max(axis=1), L(1))
    Js = Jl * s[:, None]
    rs = s * ref.violation(g.astype(L), gl.astype(L), gu.astype(L))
    A = Js.T @ Js + L(mu) * np.eye(n, dtype=L)
    b = -(Js.T @ rs)
    A64 = A.astype(np.float64)
    sol = np.linalg.solve(A64, b.astype(np.float64)).astype(L)
    for _ in range(3):
        sol = sol + np.linalg.solve(A64, (b - A @ sol).astype(np.float64))
    assert viol == np.max(np.abs(rs))
    assert np.max(np.abs(dx - sol)) <= 1e-17 * np.max(np.abs(sol))
    assert np.max(np.abs(dx - sol)) < 1e-14 * np.max(np.abs(sol.astype(np.float64)))   # far inside float64's reach


# ---- GPU ------------------------------------------------------------------------------------------------------------------

def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda()


def _step(bt, X, g, jac, xl=None, xu=None, mu=MU, cap=CAP, cg_iters=CG):
    """One device step from numpy inputs: (x_new, violation) as numpy arrays; the inputs are not changed."""
    import torch
    x = _cuda(X)
    viol = torch.full((bt.B,), 7.0, dtype=torch.float64, device="cuda")
    bt.lm_step_device(x, _cuda(g), _cuda(jac), None if xl is None else _cuda(xl), None if xu is None else _cuda(xu),
                      mu, cap, cg_iters, viol)
    torch.cuda.synchronize()
    return x.cpu().numpy(), viol.cpu().numpy()


def _violation64(pat, gl, gu, g, jac):
    """max_i |s_i r_i| in float64: every operation is one IEEE rounding, so the kernel must give this value exactly."""
    s = 1.0 / np.maximum(pat.row_max_abs(jac), 1.0)
    return np.max(np.abs(s * ref.violation(g, gl, gu)))


F64_RUNS = 8                         # float64 runs in different summation orders that make the accuracy yardstick


def _compare_with_reference(p, X, g, jac, xl, xu, x_gpu, v_gpu, mu=MU):
    """Per instance: ||x_gpu - x_ld|| <= 8 max(||x_f64 - x_ld||, 64 eps ||dx_ld||) (max norms; x_ld, dx_ld: the longdouble
    step), where ||x_f64 - x_ld|| is the worst of F64_RUNS float64 steps that differ only in summation order
    (lm_reference.relabelled_float64_steps): the kernel is no less accurate than a straightforward float64 step.  One
    float64 run is no yardstick: on these inputs its error moves by up to 140 x with the summation order alone, while no
    order's error exceeded 3 x the worst of seven others.  The violation must equal the float64 one exactly.  Returns the
    worst ratio of the left side to the right side / 8 and the worst absolute errors of the kernel and of float64."""
    _, _, gl, gu = p.bounds()
    row_ptr, col_idx = p.row_ptr(), p.structure()[1]
    pat = ref.Pattern(row_ptr, col_idx, p.n)
    worst = dict(ratio=0.0, err_gpu=0.0, err_f64=0.0)
    for b in range(X.shape[0]):
        dld, _ = ref.lm_capped_step(pat, g[b], jac[b], gl, gu, mu, CAP, CG, np.longdouble)
        xld = np.minimum(np.maximum(X[b].astype(np.longdouble) + dld, xl[b].astype(np.longdouble)), xu[b].astype(np.longdouble))
        runs = ref.relabelled_float64_steps(X[b], g[b], jac[b], xl[b], xu[b], gl, gu, row_ptr, col_idx, mu, CAP, CG, F64_RUNS, b)
        err_f64 = max(float(np.max(np.abs(x.astype(np.longdouble) - xld))) for x in runs)
        err_gpu = float(np.max(np.abs(x_gpu[b].astype(np.longdouble) - xld)))
        bound = max(err_f64, 64 * EPS * float(np.max(np.abs(dld))))
        ratio = err_gpu / bound if bound > 0 else (0.0 if err_gpu == 0 else np.inf)
        assert ratio <= 8.0, (b, err_gpu, err_f64, float(np.max(np.abs(dld))))
        assert v_gpu[b] == _violation64(pat, gl, gu, g[b], jac[b]), b
        worst = dict(ratio=max(worst["ratio"], ratio), err_gpu=max(worst["err_gpu"], err_gpu), err_f64=max(worst["err_f64"], err_f64))
    return worst


def _edge_inputs(p, B, seed):
    """Random Jacobian values on the problem's pattern and g / x that reach the edges of the step:
    rows whose largest |entry| is below 1 (s = 1), around 30, or near 1e4; g below g_lower, above g_upper and inside (equality
    rows: on the bound); x on its bounds, outside them and inside; per-instance variable bounds.  Instance 0 has no
    violated row.  Returns numpy (X, g, jac, x_lower, x_upper)."""
    rng = np.random.default_rng(seed)
    xl0, xu0, gl, gu = p.bounds()
    row_of = np.repeat(np.arange(p.m), np.diff(p.row_ptr()))
    mag = np.array([0.9, 30.0, 1e4])[rng.integers(0, 3, (B, p.m))]
    jac = rng.uniform(-1.0, 1.0, (B, p.nnz)) * mag[:, row_of]
    lo_f, up_f = np.abs(gl) < 1e10, np.abs(gu) < 1e10          # +-1e20 stands for "no bound"
    step = rng.uniform(0.01, 0.5, (B, p.m))
    inside = np.where(lo_f & up_f, gl + (gu - gl) * rng.uniform(0.0, 1.0, (B, p.m)),
                      np.where(lo_f, gl + step, np.where(up_f, gu - step, step - 0.25)))
    kind = rng.integers(0, 3, (B, p.m))
    g = np.where((kind == 0) & lo_f, gl - step, np.where((kind == 1) & up_f, gu + step, inside))
    g[0] = np.clip(g[0], gl, gu)
    widen = lambda bnd, sign: np.where(np.abs(bnd) < 1e10, bnd + sign * rng.uniform(0.0, 0.05, (B, p.n)), bnd)
    xl, xu = widen(xl0, -1.0), widen(xu0, 1.0)
    X = synthetic_iterates(p, B, seed=seed)
    kind = rng.integers(0, 6, (B, p.n))
    off = rng.uniform(0.01, 0.3, (B, p.n))
    X = np.where(kind == 0, xl, np.where(kind == 1, xu, X))
    X = np.where((kind == 2) & (np.abs(xl) < 1e10), xl - off, np.where((kind == 3) & (np.abs(xu) < 1e10), xu + off, X))
    return X, g, jac, xl, xu


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_step_on_evaluated_inputs_matches_the_extended_precision_reference(case, record_property):
    """g and the Jacobian from twb_batch_eval_device on synthetic iterates around goal-randomised initial guesses, with the
    goal instances' own variable bounds; one device step against the float64 and longdouble references."""
    if not ref.LONGDOUBLE_IS_WIDER:
        pytest.skip("np.longdouble is not wider than float64 here")
    import torch
    p = _problem(case)
    B = 12
    rng = np.random.default_rng(61)
    goals = np.column_stack([rng.uniform(0.3, 2.5, B), rng.uniform(-0.4, 0.4, B), np.full(B, 0.5), np.zeros(B), np.zeros(B),
                             rng.uniform(-0.5, 0.5, B)])
    bt = p.batch(B)
    x0, xl, xu = bt.goal_instances_device(_cuda(goals))
    X = _cuda(synthetic_iterates_fast(p, B, seed=62, x0=x0.cpu().numpy()))
    g = torch.empty((B, p.m), dtype=torch.float64, device="cuda")
    jac = torch.empty((B, p.nnz), dtype=torch.float64, device="cuda")
    status = torch.empty(B, dtype=torch.int32, device="cuda")
    bt.eval_device(X, g=g, jac=jac, status=status)
    torch.cuda.synchronize()
    assert not status.any().item()
    Xh, gh, jh, xlh, xuh = (t.cpu().numpy() for t in (X, g, jac, xl, xu))
    x_gpu, v_gpu = _step(bt, Xh, gh, jh, xlh, xuh)
    worst = _compare_with_reference(p, Xh, gh, jh, xlh, xuh, x_gpu, v_gpu)
    record_property(f"lm_step_{case}", {"path": _path(p), "n": p.n, "m": p.m, "nnz": p.nnz, "instances": B, "inputs": "evaluated",
                                        "worst_ratio_over_f64_bound": worst["ratio"], "worst_abs_err_gpu": worst["err_gpu"],
                                        "worst_abs_err_f64": worst["err_f64"]})
    assert not np.array_equal(x_gpu, np.clip(Xh, xlh, xuh))


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_step_on_edge_inputs_matches_the_extended_precision_reference(case, record_property):
    if not ref.LONGDOUBLE_IS_WIDER:
        pytest.skip("np.longdouble is not wider than float64 here")
    p = _problem(case)
    B = 12
    X, g, jac, xl, xu = _edge_inputs(p, B, seed=71)
    x_gpu, v_gpu = _step(p.batch(B), X, g, jac, xl, xu)
    worst = _compare_with_reference(p, X, g, jac, xl, xu, x_gpu, v_gpu)
    record_property(f"lm_step_edges_{case}", {"path": _path(p), "instances": B, "inputs": "edges",
                                              "worst_ratio_over_f64_bound": worst["ratio"], "worst_abs_err_gpu": worst["err_gpu"],
                                              "worst_abs_err_f64": worst["err_f64"]})


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_exact_invariants_of_the_step(case):
    """What must hold bit for bit (the library builds with -fmad=false, divisions are IEEE): the violation, the bounds,
    the projection alone when there is no step, the cap, determinism, independence of the instances' order, and NULL
    bounds meaning the problem's own."""
    p = _problem(case)
    B = 10
    X, g, jac, xl, xu = _edge_inputs(p, B, seed=81)
    bt = p.batch(B)
    x1, v1 = _step(bt, X, g, jac, xl, xu)
    _, _, gl, gu = p.bounds()
    pat = ref.Pattern(p.row_ptr(), p.structure()[1], p.n)
    for b in range(B):
        assert v1[b] == _violation64(pat, gl, gu, g[b], jac[b]), b
    assert v1[0] == 0.0 and np.all(v1[1:] > 0.0)
    assert np.all(xl <= x1) and np.all(x1 <= xu)
    assert np.array_equal(x1[0], np.clip(X[0], xl[0], xu[0]))            # r = 0: the projection alone
    assert not np.array_equal(x1[1:], np.clip(X[1:], xl[1:], xu[1:]))
    inside = (xl <= X) & (X <= xu)
    moved = np.abs(x1 - X)
    assert np.all(moved[inside] <= (CAP * (1 + 4 * EPS) + np.spacing(np.abs(X)))[inside])
    x2, v2 = _step(bt, X, g, jac, xl, xu)
    assert np.array_equal(_bits(x2), _bits(x1)) and np.array_equal(_bits(v2), _bits(v1))
    perm = np.random.default_rng(82).permutation(B)
    x3, v3 = _step(bt, X[perm], g[perm], jac[perm], xl[perm], xu[perm])
    assert np.array_equal(_bits(x3), _bits(x1[perm])) and np.array_equal(_bits(v3), _bits(v1[perm]))
    x4, v4 = _step(bt, X, g, jac, xl, xu, cg_iters=0)
    assert np.array_equal(x4, np.clip(X, xl, xu)) and np.array_equal(_bits(v4), _bits(v1))
    pxl, pxu, _, _ = p.bounds()
    xa, va = _step(bt, X, g, jac)
    xb, vb = _step(bt, X, g, jac, np.tile(pxl, (B, 1)), np.tile(pxu, (B, 1)))
    assert np.array_equal(_bits(xa), _bits(xb)) and np.array_equal(_bits(va), _bits(vb))
    assert np.all(pxl <= xa) and np.all(xa <= pxu)


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_mu_zero_is_accepted_where_the_normal_matrix_is_regular(case, record_property):
    if not ref.LONGDOUBLE_IS_WIDER:
        pytest.skip("np.longdouble is not wider than float64 here")
    p = _problem(case)
    B = 4
    X, g, jac, xl, xu = _edge_inputs(p, B, seed=91)
    row_of = np.repeat(np.arange(p.m), np.diff(p.row_ptr()))
    col_idx = p.structure()[1]
    for b in range(B):                                       # Js^T Js is regular: Js has full column rank
        J = np.zeros((p.m, p.n))
        J[row_of, col_idx] = jac[b]
        assert np.linalg.matrix_rank(J / np.maximum(np.abs(J).max(axis=1), 1.0)[:, None]) == p.n
    x_gpu, v_gpu = _step(p.batch(B), X, g, jac, xl, xu, mu=0.0)
    assert np.all(np.isfinite(x_gpu)) and np.all(np.isfinite(v_gpu))
    assert np.all(xl <= x_gpu) and np.all(x_gpu <= xu)
    worst = _compare_with_reference(p, X, g, jac, xl, xu, x_gpu, v_gpu, mu=0.0)
    record_property(f"lm_step_mu0_{case}", {"path": _path(p), "instances": B, "worst_ratio_over_f64_bound": worst["ratio"]})


@pytest.mark.gpu
def test_bad_arguments_are_rejected_and_leave_x_untouched():
    """mu < 0, cap <= 0, cg_iters outside [0, 10000], one bound NULL, NULL pointers: TWB_ERR_INVALID; solver vectors over
    200 KiB: TWB_ERR_UNSUPPORTED.  Nothing is enqueued: x and the violation keep their values."""
    import torch
    p = _problem("hopper")
    B = 3
    bt = p.batch(B)
    X, g, jac, xl, xu = (_cuda(a) for a in _edge_inputs(p, B, seed=101))
    x = X.clone()
    viol = torch.full((B,), 7.0, dtype=torch.float64, device="cuda")
    v = lambda t: C.c_void_p(t.data_ptr())
    lib, h = capi.lib, bt._h
    step = lambda *a: lib.twb_batch_lm_step_device(*a)
    calls = [
        step(None, v(x), v(g), v(jac), v(xl), v(xu), MU, CAP, CG, v(viol), None),
        step(h, None, v(g), v(jac), v(xl), v(xu), MU, CAP, CG, v(viol), None),
        step(h, v(x), None, v(jac), v(xl), v(xu), MU, CAP, CG, v(viol), None),
        step(h, v(x), v(g), None, v(xl), v(xu), MU, CAP, CG, v(viol), None),
        step(h, v(x), v(g), v(jac), v(xl), None, MU, CAP, CG, v(viol), None),
        step(h, v(x), v(g), v(jac), None, v(xu), MU, CAP, CG, v(viol), None),
        step(h, v(x), v(g), v(jac), v(xl), v(xu), -1e-300, CAP, CG, v(viol), None),
        step(h, v(x), v(g), v(jac), v(xl), v(xu), float("nan"), CAP, CG, v(viol), None),
        step(h, v(x), v(g), v(jac), v(xl), v(xu), MU, 0.0, CG, v(viol), None),
        step(h, v(x), v(g), v(jac), v(xl), v(xu), MU, -0.1, CG, v(viol), None),
        step(h, v(x), v(g), v(jac), v(xl), v(xu), MU, float("nan"), CG, v(viol), None),
        step(h, v(x), v(g), v(jac), v(xl), v(xu), MU, CAP, -1, v(viol), None),
        step(h, v(x), v(g), v(jac), v(xl), v(xu), MU, CAP, 10001, v(viol), None),
    ]
    assert calls == [capi.ERR_INVALID] * len(calls)
    with pytest.raises(capi.TowrB200Error) as err:
        bt.lm_step_device(x, g, jac, xl, xu, MU, 0.0, CG, viol)
    assert err.value.code == capi.ERR_INVALID
    big = _problem_of(*TOO_LARGE)
    bb = big.batch(2)
    xb = _cuda(synthetic_iterates(big, 2))
    xb0 = xb.clone()
    gb = torch.zeros((2, big.m), dtype=torch.float64, device="cuda")
    jb = torch.zeros((2, big.nnz), dtype=torch.float64, device="cuda")
    vb = torch.full((2,), 7.0, dtype=torch.float64, device="cuda")
    assert lib.twb_batch_lm_step_device(bb._h, v(xb), v(gb), v(jb), None, None, MU, CAP, CG, v(vb), None) == capi.ERR_UNSUPPORTED
    with pytest.raises(capi.TowrB200Error) as err:
        bb.lm_step_device(xb, gb, jb, violation=vb)
    assert err.value.code == capi.ERR_UNSUPPORTED
    torch.cuda.synchronize()
    assert torch.equal(x, X) and torch.equal(xb, xb0)
    assert bool((viol == 7.0).all()) and bool((vb == 7.0).all())
    # the range's ends are accepted, and the batch still serves valid calls
    assert step(h, v(x), v(g), v(jac), v(xl), v(xu), 0.0, CAP, 0, v(viol), None) == capi.OK
    assert step(h, v(x), v(g), v(jac), v(xl), v(xu), MU, CAP, 10000, v(viol), None) == capi.OK
    torch.cuda.synchronize()
    assert bool(torch.isfinite(x).all()) and bool(torch.isfinite(viol).all())


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_graph_replay_equals_the_eager_step(case):
    """After the first call (which uploads the pattern with cudaMalloc / cudaMemcpy) the step only enqueues: captured in a
    CUDA graph, its replay equals the eager step bit for bit, for two different inputs."""
    import torch
    p = _problem(case)
    B = 6
    bt = p.batch(B)
    X1, g, jac, xl, xu = (_cuda(a) for a in _edge_inputs(p, B, seed=111))
    X2 = _cuda(_edge_inputs(p, B, seed=112)[0])
    viol = torch.empty(B, dtype=torch.float64, device="cuda")
    bt.lm_step_device(X1.clone(), g, jac, xl, xu, MU, CAP, CG, viol)      # warm-up
    torch.cuda.synchronize()
    x = X1.clone()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        bt.lm_step_device(x, g, jac, xl, xu, MU, CAP, CG, viol)
    for X in (X1, X2):
        eager_x = X.clone()
        eager_v = torch.empty(B, dtype=torch.float64, device="cuda")
        bt.lm_step_device(eager_x, g, jac, xl, xu, MU, CAP, CG, eager_v)
        x.copy_(X)
        viol.fill_(7.0)
        graph.replay()
        torch.cuda.synchronize()
        assert not torch.equal(eager_x, X)
        assert np.array_equal(_bits(x.cpu().numpy()), _bits(eager_x.cpu().numpy()))
        assert np.array_equal(_bits(viol.cpu().numpy()), _bits(eager_v.cpu().numpy()))


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_non_finite_inputs_leave_the_instance_unchanged(case):
    """A NaN or an Inf in one g entry, one Jacobian entry or one x entry of an instance: that instance keeps its x bit for
    bit and reports violation NaN (a clipped step would move it to its bounds); every other instance of the batch equals
    a run without the non-finite entries bit for bit."""
    p = _problem(case)
    B = 9
    X, g, jac, xl, xu = _edge_inputs(p, B, seed=121)
    rng = np.random.default_rng(122)
    Xb, gb, jb = X.copy(), g.copy(), jac.copy()
    gb[1, rng.integers(p.m)] = np.nan
    gb[2, rng.integers(p.m)] = np.inf
    gb[3, rng.integers(p.m)] = -np.inf
    jb[4, rng.integers(p.nnz)] = np.nan
    jb[5, rng.integers(p.nnz)] = -np.inf
    Xb[6, rng.integers(p.n)] = np.nan
    Xb[7, rng.integers(p.n)] = np.inf
    marked = np.arange(1, 8)
    clean = np.array([0, 8])
    bt = p.batch(B)
    x_ref, v_ref = _step(bt, X, g, jac, xl, xu)
    x_bad, v_bad = _step(bt, Xb, gb, jb, xl, xu)
    assert np.array_equal(_bits(x_bad[clean]), _bits(x_ref[clean])) and np.array_equal(_bits(v_bad[clean]), _bits(v_ref[clean]))
    for b in marked:
        assert np.array_equal(_bits(x_bad[b]), _bits(Xb[b])), b
        assert np.isnan(v_bad[b]), (b, v_bad[b])
    # the same with the problem's own bounds (bound_stride 0) and without a violation output
    import torch
    x = _cuda(Xb)
    bt.lm_step_device(x, _cuda(gb), _cuda(jb), None, None, MU, CAP, CG, None)
    torch.cuda.synchronize()
    assert np.array_equal(_bits(x.cpu().numpy()[marked]), _bits(Xb[marked]))
