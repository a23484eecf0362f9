"""The trust-region step rule of the one-call solve (twb_lm_solve_options.step_rule = TWB_LM_STEP_TRUST): conjugate
gradients on the variables not held at a bound, a radius per instance that adapts to the gain ratio, and STALLED when the
radius collapses.  The cap rule stays the default and keeps its bits.

One iteration is compared with the numpy restatement of tests/lm_trust_reference.py, and the radius update with the numpy
rule on the device's own trial (the same x_trial, g and g_trial), so that a decision near a threshold cannot go two ways."""
import ctypes as C
import functools
import os
import subprocess
import types

import numpy as np
import pytest

import towr_b200 as tb
from towr_b200 import capi
import lm_reference as ref
import lm_solve_reference as sref
import lm_trust_reference as tref
from test_lm_step import EPS, F64_RUNS, PATH_CASES, _bits, _cuda, _violation64
from test_lm_solve import _check_converged, _solver
from test_lm_solve_device import FIELDS, _base_rom, _config5_shard, _one_call

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRUST_FIELDS = FIELDS + ("step_rule", "radius_max")
BUDGET = 60


# ---- CPU ------------------------------------------------------------------------------------------------------------------

def test_options_struct_matches_the_header(tmp_path):
    """sizeof and offsetof of twb_lm_solve_options, new fields included, from a C compiler against the ctypes structure;
    the step-rule constants against capi."""
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "towr_b200.h"\nint main(void) {\n'
                   '  printf("size %zu\\n", sizeof(twb_lm_solve_options));\n'
                   '  printf("cap_rule %d\\n", TWB_LM_STEP_CAP);\n  printf("trust_rule %d\\n", TWB_LM_STEP_TRUST);\n'
                   + "".join(f'  printf("{f} %zu\\n", offsetof(twb_lm_solve_options, {f}));\n' for f in TRUST_FIELDS) + "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(capi.LmSolveOptions)
    for f in TRUST_FIELDS:
        assert int(got[f]) == getattr(capi.LmSolveOptions, f).offset, f
    assert (int(got["cap_rule"]), int(got["trust_rule"])) == (capi.LM_STEP_CAP, capi.LM_STEP_TRUST) == (0, 1)


def test_default_options_keep_the_cap_rule():
    o = capi.LmSolveOptions()
    capi.lib.twb_lm_solve_options_default(C.byref(o))
    assert o.step_rule == capi.LM_STEP_CAP and o.radius_max == 1e3
    assert (o.mu0, o.cap, o.tol, o.eta, o.mu_min, o.mu_max, o.cg_iters, o.max_iters) == (1e-2, 0.1, 1e-6, 1e-4, 1e-12, 1e10, 25, 60)


def _random_box_problem(rng, m=40, n=24):
    mask = rng.random((m, n)) < 0.3
    J = np.where(mask, rng.standard_normal((m, n)) * 3.0, 0.0)
    pat = ref.Pattern(np.concatenate([[0], np.cumsum(mask.sum(axis=1))]), np.nonzero(mask)[1], n)
    x = rng.standard_normal(n)
    lo, up = x - rng.uniform(0.1, 1.0, n), x + rng.uniform(0.1, 1.0, n)
    lo[:4], up[4:8], lo[8:10], up[8:10] = x[:4], x[4:8], x[8:10], x[8:10]      # on the lower, the upper, both bounds
    return pat, J, mask, x, lo, up, rng.standard_normal(m), np.full(m, -0.2), np.full(m, 0.2)


def test_reference_step_is_the_free_set_newton_step():
    """With as many CG iterations as free variables and a radius it does not reach, the reference step solves
    (Js^T Js + mu I) dx = -gamma on the free set (dense algebra), leaves every frozen variable's bits and moves no variable
    outside its bounds."""
    rng = np.random.default_rng(5)
    pat, J, mask, x, lo, up, g, gl, gu = _random_box_problem(rng)
    s = 1 / np.maximum(np.abs(J).max(axis=1), 1.0)
    Js = J * s[:, None]
    gamma = Js.T @ (s * ref.violation(g, gl, gu))
    assert np.allclose(tref.gradient(pat, g, J[mask], gl, gu), gamma, rtol=1e-13, atol=1e-14)
    fz = tref.frozen(x, lo, up, gamma)
    assert fz[8:10].all() and fz[:4].tolist() == (gamma[:4] > 0).tolist() and fz[4:8].tolist() == (gamma[4:8] < 0).tolist()
    free = ~fz
    mu = 1e-1
    A = Js.T @ Js + mu * np.eye(pat.n)
    dx = np.zeros(pat.n)
    dx[free] = np.linalg.solve(A[np.ix_(free, free)], -gamma[free])
    xt, fz_ref, step_norm = tref.trust_step(pat, x, g, J[mask], lo, up, gl, gu, mu, 1e6, int(free.sum()) + 5)
    assert np.array_equal(fz_ref, fz)
    assert np.array_equal(_bits(xt[fz]), _bits(x[fz]))
    assert np.allclose(xt, np.clip(x + dx, lo, up), rtol=1e-9, atol=1e-12)
    assert np.all(xt >= lo) and np.all(xt <= up) and step_norm == np.max(np.abs(xt - x))
    xt, _, step_norm = tref.trust_step(pat, x, g, J[mask], lo, up, gl, gu, mu, 1e-3, 25)     # the radius binds
    assert step_norm <= 1e-3 * (1 + 4 * EPS)


def test_reference_radius_rule():
    assert tref.radius_update(0.1, 0.1, False, 0.9, 1e3, 1.0) == (0.025, False)              # rejected: shrink
    assert tref.radius_update(0.1, 0.1, True, 0.2, 1e3, 1.0) == (0.025, False)               # rho < 0.25: shrink
    assert tref.radius_update(0.1, 0.1, True, 0.8, 1e3, 1.0) == (0.2, False)                 # rho > 0.75 at the edge: grow
    assert tref.radius_update(0.1, 0.1, True, 0.8, 0.15, 1.0) == (0.15, False)               # ... up to radius_max
    assert tref.radius_update(0.1, 0.05, True, 0.8, 1e3, 1.0) == (0.1, False)                # inside the region: hold
    assert tref.radius_update(0.1, 0.1, True, 0.5, 1e3, 1.0) == (0.1, False)                 # 0.25 <= rho <= 0.75: hold
    assert tref.radius_update(0.1, 0.0, False, np.nan, 1e3, 1.0) == (0.0, True)              # no step: collapsed
    assert tref.radius_update(0.1, 4e-12, False, 0.0, 1e3, 10.0) == (1e-12, True)            # below 1e-12 max |x|
    assert tref.radius_update(0.1, 4e-12, False, 0.0, 1e3, 0.5) == (1e-12, False)


# ---- GPU helpers ----------------------------------------------------------------------------------------------------------

def _trust(lm, X, max_iters, tol, **kw):
    """_one_call with the trust-region rule; keywords override the solver's own mu0, cap and cg_iters."""
    import torch
    args = dict(max_iters=max_iters, tol=tol, mu0=lm.mu, cap=lm.cap, cg_iters=lm.cg_iters, step_rule="trust")
    args.update(kw)
    out = lm.batch.lm_solve_device(X, lm.xl_full, lm.xu_full, lm.gl_full, lm.gu_full, **args)
    torch.cuda.synchronize()
    return (X.cpu().numpy(),) + tuple(t.cpu().numpy() for t in out)


def _eval(bt, X):
    """g and J at X (torch), as numpy arrays."""
    import torch
    g = torch.empty((bt.B, bt.problem.m), dtype=torch.float64, device="cuda")
    jac = torch.empty((bt.B, bt.problem.nnz), dtype=torch.float64, device="cuda")
    st = torch.empty(bt.B, dtype=torch.int32, device="cuda")
    bt.eval_device(X, g=g, jac=jac, status=st)
    torch.cuda.synchronize()
    return g.cpu().numpy(), jac.cpu().numpy()


def _bounds(lm):
    xl, xu = lm.xl_full.cpu().numpy(), lm.xu_full.cpu().numpy()
    gl, gu = (np.broadcast_to(a.cpu().numpy(), (lm.B, lm.p.m)) for a in (lm.gl, lm.gu))
    return xl, xu, gl, gu


def _craft_bounds(lm, X0):
    """Bounds through X0 (the solver's per-instance x_lower / x_upper, changed in place; X0, g and J stay as they are): for
    every fourth of the variables with the largest |gamma| per instance, a box of width 1 with x on the bound the descent
    direction -gamma leaves through (outward: frozen), for the next such variable on the other one (inward: free)."""
    g, jac = _eval(lm.batch, X0)
    x = X0.cpu().numpy()
    xl, xu, gl, gu = _bounds(lm)
    xl, xu = xl.copy(), xu.copy()
    pat = ref.Pattern(lm.p.row_ptr(), lm.p.structure()[1], lm.p.n)
    for b in range(lm.B):
        gamma = tref.gradient(pat, g[b], jac[b], gl[b], gu[b])
        cand = np.flatnonzero((xl[b] < xu[b]) & (np.abs(gamma) > 0))
        pick = cand[np.argsort(-np.abs(gamma[cand]))][:max(2, len(cand) // 10)]
        for k, j in enumerate(pick[::2]):
            at_lower = (gamma[j] > 0) == (k % 2 == 0)
            xl[b, j], xu[b, j] = (x[b, j], x[b, j] + 1.0) if at_lower else (x[b, j] - 1.0, x[b, j])
    lm.xl_full.copy_(_cuda(xl))
    lm.xu_full.copy_(_cuda(xu))


# ---- GPU: the cap rule is unchanged -------------------------------------------------------------------------------------

def _assert_same_bits(a, b):
    for u, v in zip(a[:5], b[:5]):
        assert np.array_equal(_bits(u), _bits(v)) if u.dtype == np.float64 else np.array_equal(u, v)
    assert np.array_equal(a[5], b[5]) and a[6][0] == b[6][0]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_the_cap_rule_with_any_radius_max_is_the_default(case):
    lm, X0 = _solver(case, 10, seed=501)
    default = _one_call(lm, X0.clone(), 30, 1e-2)
    for radius_max in (0.0, 0.05, 1e3, float("nan")):
        _assert_same_bits(_one_call(lm, X0.clone(), 30, 1e-2, step_rule="cap", radius_max=radius_max), default)


@functools.lru_cache(maxsize=None)
def _workload(name):
    return (_config5_shard if name == "config5_shard" else _base_rom)()


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["config5_shard", "base_rom"])
def test_the_cap_rule_is_unchanged_on_4096_instances(workload):
    lm, X0 = _workload(workload)
    _assert_same_bits(_one_call(lm, X0.clone(), BUDGET, 1e-6, step_rule="cap", radius_max=0.0), _one_call(lm, X0.clone(), BUDGET, 1e-6))


# ---- GPU: one iteration against numpy -------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("inputs", ["evaluated", "crafted"])
@pytest.mark.parametrize("case", PATH_CASES)
def test_one_iteration_against_the_numpy_rule(case, inputs, record_property):
    """max_iters = 1 from X0.  The reference trial from the device's g and J at X0: frozen variables keep their bits, clearly
    moved free ones move, max |x_new - x| <= cap, an accepted x matches the extended-precision reference step under the
    yardstick of tests/test_lm_solve.py (8 x the worst of F64_RUNS relabelled float64 steps, or 64 eps max |dx|), and status,
    iterations and the accept decision follow the numpy rule evaluated at the float64 reference trial point."""
    import torch
    lm, X0 = _solver(case, 8, seed=511)
    if inputs == "crafted":
        _craft_bounds(lm, X0)
    x0 = X0.cpu().numpy()
    g, jac = _eval(lm.batch, X0)
    xl, xu, gl, gu = _bounds(lm)
    row_ptr, col_idx = lm.p.row_ptr(), lm.p.structure()[1]
    pat = ref.Pattern(row_ptr, col_idx, lm.p.n)
    x, status, its, viol, mu, counts, loops = _trust(lm, X0.clone(), 1, 1e-6)
    xt = np.stack([tref.trust_step(pat, x0[b], g[b], jac[b], xl[b], xu[b], gl[b], gu[b], lm.mu, lm.cap, lm.cg_iters)[0] for b in range(lm.B)])
    fz = np.stack([tref.trust_step(pat, x0[b], g[b], jac[b], xl[b], xu[b], gl[b], gu[b], lm.mu, lm.cap, lm.cg_iters)[1] for b in range(lm.B)])
    gt, _ = _eval(lm.batch, torch.from_numpy(xt).cuda())
    worst, n_frozen_by_gradient = 0.0, 0
    for b in range(lm.B):
        assert np.array_equal(_bits(x[b][fz[b]]), _bits(x0[b][fz[b]])), b
        n_frozen_by_gradient += int(np.sum(fz[b] & (xl[b] < xu[b])))
        assert np.max(np.abs(x[b] - x0[b])) <= lm.cap * (1 + 4 * EPS) + 4 * EPS * np.max(np.abs(x0[b]))
        runs = tref.relabelled_trust_steps(x0[b], g[b], jac[b], xl[b], xu[b], gl[b], gu[b], row_ptr, col_idx, lm.mu, lm.cap, lm.cg_iters,
                                           F64_RUNS, b)
        xt_ld = tref.trust_step(pat, x0[b], g[b], jac[b], xl[b], xu[b], gl[b], gu[b], lm.mu, lm.cap, lm.cg_iters, np.longdouble)[0]
        spread = max(float(np.max(np.abs(r - xt_ld))) for r in runs)
        tol = max(8 * spread, 64 * EPS * np.max(np.abs(xt[b] - x0[b])))
        merit, pred = sref.merit_and_predicted(pat, x0[b], xt[b], g[b], jac[b], gl[b], gu[b])
        s = sref.row_scales(pat, jac[b])
        acc, rho, mu1, _, stalled = sref.accept(merit, pred, sref.half_norm2(s, gt[b], gl[b], gu[b]), bool(np.isfinite(gt[b]).all()),
                                               lm.mu, 2.0, 1e-4, 1e-12, 1e10)
        _, collapsed = tref.radius_update(lm.cap, np.max(np.abs(xt[b] - x0[b])), acc, rho, 1e3, np.max(np.abs(xt[b] if acc else x0[b])))
        moved = ~np.equal(_bits(x[b]), _bits(x0[b]))
        if abs(rho - 1e-4) > 1e-6:                   # the decision is not at the threshold
            assert moved.any() == acc, (b, rho)
        if moved.any():
            err = float(np.max(np.abs(x[b] - xt_ld)))
            assert err <= tol, (b, err, tol)
            worst = max(worst, err / tol)
            assert moved[~fz[b] & (np.abs(xt[b] - x0[b]) > tol)].all(), b
        assert its[b] == 1
        assert status[b] == (capi.LM_STALLED if stalled or collapsed else capi.LM_CONVERGED if viol[b] <= 1e-6 else capi.LM_RUNNING), b
    assert loops[0] == 1 and np.array_equal(counts, np.bincount(status, minlength=4))
    if inputs == "crafted":
        assert n_frozen_by_gradient > 0
    record_property(f"trust_one_iteration_{case}_{inputs}", {"worst_err_over_tol": worst, "frozen_by_gradient": n_frozen_by_gradient})


# ---- GPU: the radius update -----------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_the_radius_update_follows_the_rule(case, record_property):
    """max_iters = 1 with first radii that make the trials overshoot or stop inside the region, that reach its edge (with and
    without the radius_max clamp), and with eta = 0.999999, which rejects nearly every trial.  The rule is evaluated on the device's own trial: the step_norm it reports, its x_trial
    (the returned x when accepted) and g there, so the radius must match bit for bit; rho is recomputed in float64 and
    instances within 1e-9 of a threshold are not judged."""
    import torch
    lm, X0 = _solver(case, 10, seed=521)
    x0 = X0.cpu().numpy()
    g, jac = _eval(lm.batch, X0)
    xl, xu, gl, gu = _bounds(lm)
    pat = ref.Pattern(lm.p.row_ptr(), lm.p.structure()[1], lm.p.n)
    seen = set()
    for cap, radius_max, eta in ((10.0, 1e3, 1e-4), (1e-4, 1e3, 1e-4), (1e-4, 1.5e-4, 1e-4), (1e-4, 1e-4, 1e-4), (0.1, 1e3, 1e-4),
                                 (0.1, 1e3, 0.999999)):
        x, status, its, viol, mu, counts, loops = _trust(lm, X0.clone(), 1, 1e-6, cap=cap, radius_max=radius_max, eta=eta)
        radius, step_norm = lm.batch.lm_solve_radius()
        gx, _ = _eval(lm.batch, torch.from_numpy(x).cuda())
        for b in range(lm.B):
            acc = not np.array_equal(_bits(x[b]), _bits(x0[b]))
            assert step_norm[b] <= cap * (1 + 4 * EPS) + 4 * EPS * np.max(np.abs(x0[b]))
            if not acc:
                assert radius[b] == 0.25 * step_norm[b], b
                seen.add("shrink (rejected)")
                continue
            assert step_norm[b] == np.max(np.abs(x[b] - x0[b])), b
            merit, pred = sref.merit_and_predicted(pat, x0[b], x[b], g[b], jac[b], gl[b], gu[b])
            rho = (merit - sref.half_norm2(sref.row_scales(pat, jac[b]), gx[b], gl[b], gu[b])) / pred
            if min(abs(rho - tref.LOW), abs(rho - tref.HIGH)) < 1e-9:
                continue
            want, collapsed = tref.radius_update(cap, step_norm[b], True, rho, radius_max, np.max(np.abs(x[b])))
            assert radius[b] == want, (b, cap, radius_max, rho, radius[b], want)
            assert (status[b] == capi.LM_STALLED) == (collapsed or mu[b] > 1e10), b
            edge = rho > tref.HIGH and step_norm[b] >= tref.EDGE * cap
            seen.add("shrink" if rho < tref.LOW else ("clamp" if 2 * cap > radius_max else "grow") if edge else "hold")
    record_property(f"trust_radius_branches_{case}", sorted(seen))
    assert {"grow", "clamp", "hold"} <= seen and ("shrink" in seen or "shrink (rejected)" in seen), seen


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_a_collapsed_radius_stalls_the_instance(case):
    """Instance 2 with every variable fixed (x_lower = x_upper = x): its free set is empty, the trial does not move, the
    radius becomes 0.25 x 0 and the instance is STALLED after one iteration with x bit for bit; the other instances run
    exactly as in a batch without it."""
    import torch
    lm, X0 = _solver(case, 6, seed=531)
    clean = _trust(lm, X0.clone(), 5, 1e-6)
    lm.xl_full[2] = X0[2]
    lm.xu_full[2] = X0[2]
    x, status, its, viol, mu, counts, loops = _trust(lm, X0.clone(), 5, 1e-6)
    radius, step_norm = lm.batch.lm_solve_radius()
    assert status[2] == capi.LM_STALLED and its[2] == 1 and radius[2] == 0.0 and step_norm[2] == 0.0
    assert np.array_equal(_bits(x[2]), _bits(X0[2].cpu().numpy()))
    rest = [0, 1, 3, 4, 5]
    for a, c in zip((x, status, its, viol, mu), clean[:5]):
        assert np.array_equal(_bits(a[rest]) if a.dtype == np.float64 else a[rest], _bits(c[rest]) if c.dtype == np.float64 else c[rest])
    torch.cuda.synchronize()


# ---- GPU: invariants ------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_deterministic_and_permutation_equivariant(case):
    B = 10
    perm = np.random.default_rng(541).permutation(B)
    lm, X0 = _solver(case, B, seed=542)
    a = _trust(lm, X0.clone(), 20, 1e-8)
    b = _trust(lm, X0.clone(), 20, 1e-8)
    lmp, Xp = _solver(case, B, seed=542, goals_perm=perm)
    c = _trust(lmp, Xp, 20, 1e-8)
    _assert_same_bits(a, b)
    for u, w in zip(a[:5], c[:5]):
        assert np.array_equal(_bits(w), _bits(u[perm])) if u.dtype == np.float64 else np.array_equal(w, u[perm])
    assert np.array_equal(a[5], c[5]) and a[6][0] == c[6][0]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_a_nan_instance_is_isolated(case):
    lm, X0 = _solver(case, 8, seed=551)
    clean = _trust(lm, X0.clone(), 20, 1e-6)
    X = X0.clone()
    X[3, 5] = float("nan")
    Xn = X.cpu().numpy()
    x, status, its, viol, mu, counts, loops = _trust(lm, X, 20, 1e-6)
    assert status[3] == capi.LM_NONFINITE and np.isnan(viol[3]) and its[3] == 0
    assert np.array_equal(_bits(x[3]), _bits(Xn[3]))
    rest = [0, 1, 2, 4, 5, 6, 7]
    for a, c in zip((x, status, its, viol, mu), clean[:5]):
        assert np.array_equal(_bits(a[rest]) if a.dtype == np.float64 else a[rest], _bits(c[rest]) if c.dtype == np.float64 else c[rest])


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_a_zero_budget_runs_only_the_tail(case):
    """max_iters = 0: x keeps its bits, every radius is the first one (cap), and status and violation are the cap rule's."""
    lm, X0 = _solver(case, 10, seed=561)
    cap_run = _one_call(lm, X0.clone(), 0, 1e-2)
    dev = _trust(lm, X0.clone(), 0, 1e-2)
    radius, _ = lm.batch.lm_solve_radius()
    assert dev[6][0] == 0 and np.all(dev[2] == 0) and np.all(radius == lm.cap)
    assert np.array_equal(_bits(dev[0]), _bits(X0.cpu().numpy()))
    _assert_same_bits(dev, cap_run)


@pytest.mark.gpu
def test_the_graph_is_reused_per_rule():
    lm, X0 = _solver("hopper", 6, seed=571)
    bt = lm.batch
    n0 = bt.lm_solve_graphs_instantiated()
    first = _trust(lm, X0.clone(), 15, 1e-6)
    assert bt.lm_solve_graphs_instantiated() == n0 + 1
    _assert_same_bits(_trust(lm, X0.clone(), 15, 1e-6), first)              # the same options: the cached graph
    assert bt.lm_solve_graphs_instantiated() == n0 + 1
    cap = _one_call(lm, X0.clone(), 15, 1e-6)                              # the other rule: one more graph
    assert bt.lm_solve_graphs_instantiated() == n0 + 2
    _assert_same_bits(_trust(lm, X0.clone(), 15, 1e-6), first)
    _assert_same_bits(_one_call(lm, X0.clone(), 15, 1e-6), cap)
    assert bt.lm_solve_graphs_instantiated() == n0 + 2
    _trust(lm, X0.clone(), 15, 1e-6, radius_max=2.0)                        # another radius_max: another graph
    assert bt.lm_solve_graphs_instantiated() == n0 + 3


@pytest.mark.gpu
def test_bad_arguments_are_rejected_and_touch_nothing():
    """An unknown step_rule, and with the trust-region rule radius_max < cap or NaN: TWB_ERR_INVALID, nothing enqueued, no
    output touched, no graph built.  The radius read-back is TWB_ERR_INVALID before the batch's first trust-region solve."""
    import torch
    lm, X0 = _solver("hopper", 3, seed=581)
    bt = lm.batch
    B = bt.B
    with pytest.raises(capi.TowrB200Error):
        bt.lm_solve_radius()
    x = X0.clone()
    st = torch.full((B,), 5, dtype=torch.int32, device="cuda"); its = st.clone()
    viol = torch.full((B,), 7.0, dtype=torch.float64, device="cuda"); mu = viol.clone()
    counts = torch.full((4,), 5, dtype=torch.int32, device="cuda"); loops = torch.full((1,), 5, dtype=torch.int32, device="cuda")
    v = lambda t: C.c_void_p(t.data_ptr())

    def call(**kw):
        o = capi.LmSolveOptions()
        capi.lib.twb_lm_solve_options_default(C.byref(o))
        for k, val in kw.items():
            setattr(o, k, val)
        return capi.lib.twb_batch_lm_solve_device(bt._h, v(x), v(lm.xl_full), v(lm.xu_full), None, None, C.byref(o), v(st), v(its), v(viol),
                                                  v(mu), v(counts), v(loops), None)

    bad = [dict(step_rule=2), dict(step_rule=-1), dict(step_rule=1, radius_max=0.05), dict(step_rule=1, radius_max=float("nan")),
           dict(step_rule=1, cap=2e3)]
    assert [call(**k) for k in bad] == [capi.ERR_INVALID] * len(bad)
    torch.cuda.synchronize()
    assert torch.equal(x, X0) and bool((st == 5).all()) and bool((its == 5).all()) and bool((counts == 5).all()) and loops.item() == 5
    assert bool((viol == 7.0).all()) and bool((mu == 7.0).all())
    assert bt.lm_solve_graphs_instantiated() == 0
    assert call(step_rule=1, radius_max=0.1) == capi.OK                     # radius_max == cap is valid
    torch.cuda.synchronize()
    assert int(counts.sum()) == B
    with pytest.raises(AssertionError):
        bt.lm_solve_device(x, step_rule="dogleg")


# ---- GPU: end to end ------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["config5_shard", "base_rom"])
def test_the_trust_region_rule_lowers_the_violation_on_4096_instances(workload, record_property):
    """60 iterations of both rules at tol 1e-6: the trust-region rule's median max |s r| is below the cap rule's and no
    instance is NONFINITE.  At tol 1e-2 the converged instances pass a re-evaluation and, on the config-5 shard, a subsample
    passes the oracle.  The converged counts are recorded, not pinned."""
    import torch
    import oracle_lib
    lm, X0 = _workload(workload)
    cap = _one_call(lm, X0.clone(), BUDGET, 1e-6)
    trust = _trust(lm, X0.clone(), BUDGET, 1e-6)
    assert trust[5][capi.LM_NONFINITE] == 0
    med_cap, med_trust = float(np.median(cap[3])), float(np.median(trust[3]))
    assert med_trust < med_cap, (med_trust, med_cap)
    X = X0.clone()
    x, status, its, viol, mu, counts, loops = _trust(lm, X, BUDGET, 1e-2)
    assert counts[capi.LM_NONFINITE] == 0
    gl, gu = lm.gl.cpu().numpy(), lm.gu.cpu().numpy()
    st = types.SimpleNamespace(status=torch.from_numpy(status), violation=torch.from_numpy(viol))
    conv = _check_converged(lm, torch.from_numpy(x).cuda(), st, 1e-2, gl, gu)
    if workload == "config5_shard":
        spec = tb.make_formulation("anymal_trot_mixed").to_spec()
        terr = np.random.default_rng(77).choice([tb.SLOPE, tb.CHIMNEY, tb.GAP], lm.B).astype(np.int32)   # _config5_shard's draw
        o = oracle_lib.Oracle(spec)
        pat = ref.Pattern(lm.p.row_ptr(), lm.p.structure()[1], lm.p.n)
        for t in (tb.SLOPE, tb.CHIMNEY, tb.GAP):
            for b in conv[terr[conv] == t][:4]:
                o.set_terrain(int(t))
                r = o.eval(x[b])
                assert r["rc"] == 0
                assert _violation64(pat, gl, gu, r["g"], r["jac"]) <= 1e-2, (b, t)
    record_property(f"trust_region_{workload}", {
        "median_violation_cap": med_cap, "median_violation_trust": med_trust,
        "counts_tol_1e-6": {"cap": cap[5].tolist(), "trust": trust[5].tolist()}, "counts_tol_1e-2_trust": counts.tolist(),
        "loop_count_tol_1e-2": int(loops[0])})


# ---- GPU: C++ -------------------------------------------------------------------------------------------------------------

EXE = os.path.join(ROOT, "tests", "cpp", "_build", "ifopt_trust_solve_test")


@pytest.mark.gpu
def test_batched_problem_solve_with_the_trust_region_rule_equals_the_c_call():
    """BatchedProblem::Solve(opt) with step_rule TWB_LM_STEP_TRUST (tests/cpp/ifopt_trust_solve_test.cc) against
    twb_batch_lm_solve_device on the same instances, bit for bit."""
    import torch
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    libdir = os.path.dirname(capi.LIB_PATH)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", os.path.join(ROOT, "tests", "cpp", "ifopt_trust_solve_test.cc"),
                           "-o", EXE, "-L" + libdir, "-ltowr_b200", "-Wl,-rpath," + libdir, "-Wl,-rpath,/usr/local/cuda/lib64"])
    out = subprocess.run([EXE], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stdout[-2000:] + out.stderr
    vals, results = {}, {}
    for line in out.stdout.splitlines():
        parts = line.split()
        if parts and parts[0] in ("state", "x"):
            vals[(parts[0], int(parts[1]))] = np.array([float.fromhex(v) for v in parts[2:]])
        elif parts and parts[0] == "result":
            results[int(parts[1])] = (int(parts[2]), int(parts[3]), float.fromhex(parts[4]), float.fromhex(parts[5]))
    B = len(results)
    p = tb.Problem(tb.make_formulation("anymal_trot_block_base_rom").to_spec())
    S = np.stack([vals[("state", k)] for k in range(B)])
    x0, xl, xu, gl, gu = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in p.state_instances(S))
    bt = p.batch(B)
    X = x0.clone()
    status, its, viol, mu, _, _ = bt.lm_solve_device(X, xl, xu, gl, gu, max_iters=30, tol=1e-2, step_rule="trust", radius_max=50.0)
    torch.cuda.synchronize()
    Xh = X.cpu().numpy()
    assert not np.array_equal(Xh, x0.cpu().numpy())
    for b in range(B):
        assert np.array_equal(_bits(vals[("x", b)]), _bits(Xh[b])), b
        st, it, v, m = results[b]
        assert (st, it) == (status[b].item(), its[b].item()), b
        assert np.array_equal(_bits(np.float64(v)), _bits(viol[b].cpu().numpy())), b
        assert np.array_equal(_bits(np.float64(m)), _bits(mu[b].cpu().numpy())), b
