"""A whole solve in one call: twb_batch_lm_solve_device runs the loop of BatchedLevenbergMarquardt.solve (evaluation, trial,
g-only evaluation at the trial point, acceptance) as a CUDA graph whose WHILE node stops at the iteration after which no
instance is RUNNING.  BatchedLevenbergMarquardt.solve is the reference: finished instances do not move, so stopping at the
exact iteration instead of the next multiple of check_every changes no bit of the result."""
import ctypes as C
import inspect
import os
import subprocess

import numpy as np
import pytest

import towr_b200 as tb
from towr_b200 import capi
from towr_b200.solver import BatchedLevenbergMarquardt
from test_lm_step import PATH_CASES, TOO_LARGE, _bits, _cuda, _problem_of
from test_lm_solve import BUDGET, TOL, _solver

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOLVE_CALLS = ("twb_lm_solve_options_default", "twb_batch_lm_solve_device", "twb_batch_lm_solve_host", "twb_batch_lm_solve_graph_stats")
FIELDS = ("mu0", "cap", "tol", "eta", "mu_min", "mu_max", "cg_iters", "max_iters")


# ---- CPU ------------------------------------------------------------------------------------------------------------------

def test_solve_calls_are_exported_and_declared():
    for name in SOLVE_CALLS:
        assert name in capi.EXPORTS, name
        assert hasattr(capi.lib, name), name
    with open(os.path.join(ROOT, "include", "towr_b200.h")) as fh:
        header = fh.read()
    for name in SOLVE_CALLS:
        assert f" {name}(" in header, name


def test_options_struct_matches_the_header(tmp_path):
    """sizeof and offsetof of twb_lm_solve_options from a C compiler against the ctypes structure."""
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "towr_b200.h"\nint main(void) {\n'
                   '  printf("size %zu\\n", sizeof(twb_lm_solve_options));\n'
                   + "".join(f'  printf("{f} %zu\\n", offsetof(twb_lm_solve_options, {f}));\n' for f in FIELDS) + "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(capi.LmSolveOptions)
    for f in FIELDS:
        assert int(got[f]) == getattr(capi.LmSolveOptions, f).offset, f


def test_default_options_are_the_defaults_of_solve():
    o = capi.LmSolveOptions()
    capi.lib.twb_lm_solve_options_default(C.byref(o))
    init = inspect.signature(BatchedLevenbergMarquardt.__init__).parameters
    solve = inspect.signature(BatchedLevenbergMarquardt.solve).parameters
    assert (o.mu0, o.cap, o.cg_iters) == (init["mu"].default, init["cap"].default, init["cg_iters"].default)
    assert (o.eta, o.mu_min, o.mu_max) == (solve["eta"].default, solve["mu_min"].default, solve["mu_max"].default)
    assert (o.tol, o.max_iters) == (1e-6, 60)


# ---- GPU helpers ----------------------------------------------------------------------------------------------------------

def _one_call(lm, X, max_iters, tol, **kw):
    """The one-call solve with the solver's own bounds and parameters; numpy results (X, status, iterations, violation, mu,
    counts, loop count) after a synchronise."""
    import torch
    out = lm.batch.lm_solve_device(X, lm.xl_full, lm.xu_full, lm.gl_full, lm.gu_full, max_iters=max_iters, tol=tol, mu0=lm.mu,
                                   cap=lm.cap, cg_iters=lm.cg_iters, **kw)
    torch.cuda.synchronize()
    return (X.cpu().numpy(),) + tuple(t.cpu().numpy() for t in out)


def _reference(lm, X, max_iters, tol, **kw):
    import torch
    res = lm.solve(X, max_iters, tol, **kw)
    torch.cuda.synchronize()
    return (X.cpu().numpy(),) + tuple(t.cpu().numpy() for t in res)


def _assert_same(dev, ref):
    """X, status, iterations, violation and mu bit for bit; the counts are the histogram of the status."""
    for k, (a, b) in enumerate(zip(dev[:5], ref[:5])):
        if a.dtype == np.float64:
            assert np.array_equal(_bits(a), _bits(b)), ("x", "status", "iterations", "violation", "mu")[k]
        else:
            assert np.array_equal(a, b), ("x", "status", "iterations", "violation", "mu")[k]
    assert np.array_equal(dev[5], np.bincount(dev[1], minlength=4))


def _first_finished_iteration(lm, X, budget, tol, **kw):
    """The eager loop one iteration at a time: the first k after which no instance is RUNNING (None within the budget)."""
    st = lm.solve_state()
    for k in range(1, budget + 1):
        lm.iterate(X, st, tol, **kw)
        if not bool((st.status == capi.LM_RUNNING).any()):
            return k
    return None


# ---- GPU: against the reference -------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_one_call_equals_the_python_solve(case):
    lm, X0 = _solver(case, 10, seed=401)
    ref = _reference(lm, X0.clone(), BUDGET, TOL)
    dev = _one_call(lm, X0.clone(), BUDGET, TOL)
    _assert_same(dev, ref)
    assert 1 <= dev[6][0] <= BUDGET


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
@pytest.mark.parametrize("tol, mu_max", [(TOL, 1e10), (TOL, 1e-1), (1e-2, 1e-1)])
def test_the_loop_stops_at_the_first_iteration_with_nothing_running(case, tol, mu_max, record_property):
    """loop_count == min(k, budget) for k the first iteration after which the eager loop has no RUNNING instance; a low
    mu_max makes instances stall early, so that k falls inside the budget.  The results equal the reference's too."""
    lm, X0 = _solver(case, 10, seed=411)
    k = _first_finished_iteration(lm, X0.clone(), BUDGET, tol, mu_max=mu_max)
    dev = _one_call(lm, X0.clone(), BUDGET, tol, mu_max=mu_max)
    assert dev[6][0] == (BUDGET if k is None else k)
    _assert_same(dev, _reference(lm, X0.clone(), BUDGET, tol, mu_max=mu_max, check_every=1))
    record_property(f"first_finished_{case}_{tol}_{mu_max}", k)


def _config5_shard():
    import torch
    spec = tb.make_formulation("anymal_trot_mixed").to_spec()
    p = tb.Problem(spec)
    B = 4096
    rng = np.random.default_rng(77)
    terr = rng.choice([tb.SLOPE, tb.CHIMNEY, tb.GAP], B).astype(np.int32)
    goals = np.column_stack([rng.uniform(1.0, 2.0, B), rng.uniform(-0.2, 0.2, B), np.full(B, 0.5), np.zeros(B), np.zeros(B), rng.uniform(-0.2, 0.2, B)])
    bt = p.batch(B); bt.set_terrains(terr)
    x0, xl, xu = bt.goal_instances_device(torch.from_numpy(goals).cuda())
    X0 = torch.minimum(torch.maximum(x0 + 0.01 * torch.from_numpy(rng.standard_normal((B, p.n))).cuda(), xl), xu)
    return BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu), X0


def _base_rom():
    import torch
    from test_state_instances import _random_states
    f = tb.make_formulation("anymal_trot_block_base_rom")
    p = tb.Problem(f.to_spec())
    B = 4096
    rng = np.random.default_rng(707)
    bt = p.batch(B)
    x0, xl, xu, gl, gu = bt.state_instances_device(torch.from_numpy(_random_states(f, rng, B)).cuda(), want_g_bounds=True)
    X0 = torch.minimum(torch.maximum(x0 + 0.01 * torch.from_numpy(rng.standard_normal((B, p.n))).cuda(), xl), xu)
    return BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu, g_lower=gl, g_upper=gu), X0


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["config5_shard", "base_rom"])
def test_one_call_equals_the_python_solve_on_4096_instances(workload, record_property):
    """The two 4096-instance workloads of test_lm_solve.py: the config-5 shard against the problem's constraint bounds, the
    base-ROM batch from measured states against per-instance constraint bounds."""
    lm, X0 = (_config5_shard if workload == "config5_shard" else _base_rom)()
    ref = _reference(lm, X0.clone(), BUDGET, TOL)
    dev = _one_call(lm, X0.clone(), BUDGET, TOL)
    _assert_same(dev, ref)
    assert dev[5][capi.LM_CONVERGED] > 0
    record_property(f"lm_solve_device_{workload}", {"counts": dev[5].tolist(), "loop_count": int(dev[6][0])})


# ---- GPU: edge cases ------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_a_tolerance_met_at_the_start_runs_one_iteration(case):
    """Every instance meets the tolerance at x0: the first body's trial marks all CONVERGED, the accept touches none, the loop
    stops after one iteration and x keeps its bits."""
    lm, X0 = _solver(case, 10, seed=421)
    x, status, its, viol, mu, counts, loops = _one_call(lm, X0.clone(), BUDGET, 1e300)
    assert loops[0] == 1 and np.all(status == capi.LM_CONVERGED) and np.all(its == 0)
    assert np.array_equal(_bits(x), _bits(X0.cpu().numpy())) and np.all(mu == lm.mu)
    assert counts.tolist() == [0, 10, 0, 0]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_a_zero_budget_runs_only_the_tail(case):
    lm, X0 = _solver(case, 10, seed=431)
    _, _, _, v0, _, _, _ = _one_call(lm, X0.clone(), 0, 1e300)
    tol = float(np.median(v0))            # part of the batch meets it at x0
    dev = _one_call(lm, X0.clone(), 0, tol)
    x, status, its, viol, mu, counts, loops = dev
    assert loops[0] == 0 and np.all(its == 0)
    assert np.array_equal(_bits(x), _bits(X0.cpu().numpy()))
    assert np.array_equal(status, np.where(viol <= tol, capi.LM_CONVERGED, capi.LM_RUNNING))
    assert 0 < counts[capi.LM_CONVERGED] < 10
    _assert_same(dev, _reference(lm, X0.clone(), 0, tol))


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_a_nan_in_x_leaves_that_instance_and_no_other(case):
    lm, X0 = _solver(case, 8, seed=441)
    clean = _one_call(lm, X0.clone(), 20, TOL)
    X = X0.clone()
    X[3, 5] = float("nan")
    Xn = X.cpu().numpy()
    x, status, its, viol, mu, counts, loops = _one_call(lm, X, 20, TOL)
    assert status[3] == capi.LM_NONFINITE and np.isnan(viol[3]) and its[3] == 0
    assert np.array_equal(_bits(x[3]), _bits(Xn[3]))
    rest = [0, 1, 2, 4, 5, 6, 7]
    for a, b in zip((x, status, its, viol, mu), clean[:5]):
        assert np.array_equal(a[rest].view(np.int64) if a.dtype == np.float64 else a[rest],
                              b[rest].view(np.int64) if b.dtype == np.float64 else b[rest])


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATH_CASES)
def test_deterministic_and_permutation_equivariant(case):
    B = 10
    perm = np.random.default_rng(451).permutation(B)
    lm, X0 = _solver(case, B, seed=452)
    a = _one_call(lm, X0.clone(), 20, 1e-8)
    b = _one_call(lm, X0.clone(), 20, 1e-8)
    lmp, Xp = _solver(case, B, seed=452, goals_perm=perm)
    c = _one_call(lmp, Xp, 20, 1e-8)
    for u, v, w in zip(a[:5], b[:5], c[:5]):
        bits = _bits if u.dtype == np.float64 else (lambda t: t)
        assert np.array_equal(bits(u), bits(v)) and np.array_equal(bits(w), bits(u[perm]))
    assert np.array_equal(a[5], c[5]) and a[6][0] == c[6][0]


@pytest.mark.gpu
def test_repeated_calls_reuse_the_graph_until_the_terrains_change():
    import torch
    lm, X0 = _solver("hopper", 6, seed=461)
    bt = lm.batch
    n0 = bt.lm_solve_graphs_instantiated()
    X = X0.clone()
    kw = dict(max_iters=15, tol=TOL, mu0=lm.mu)
    out = bt.lm_solve_device(X, lm.xl_full, lm.xu_full, **kw)
    torch.cuda.synchronize()
    first = [t.clone() for t in (X,) + tuple(out)]
    n1 = bt.lm_solve_graphs_instantiated()
    assert n1 == n0 + 1
    X.copy_(X0)
    bt.lm_solve_device(X, lm.xl_full, lm.xu_full, out=out, **kw)
    torch.cuda.synchronize()
    assert bt.lm_solve_graphs_instantiated() == n1                     # the cached graph
    for a, b in zip(first, (X,) + tuple(out)):
        assert torch.equal(a.view(torch.int64) if a.dtype == torch.float64 else a, b.view(torch.int64) if b.dtype == torch.float64 else b)
    X.copy_(X0)
    bt.lm_solve_device(X, lm.xl_full, lm.xu_full, out=out, max_iters=14, tol=TOL, mu0=lm.mu)   # other options: another graph
    torch.cuda.synchronize()
    assert bt.lm_solve_graphs_instantiated() == n1 + 1
    bt.set_terrains(None)                                         # every instance on the problem's own terrain, as before
    X.copy_(X0)
    bt.lm_solve_device(X, lm.xl_full, lm.xu_full, out=out, **kw)
    torch.cuda.synchronize()
    assert bt.lm_solve_graphs_instantiated() == n1 + 2                 # rebuilt after set_terrains
    for a, b in zip(first, (X,) + tuple(out)):                    # the same terrain: the same result
        assert torch.equal(a.view(torch.int64) if a.dtype == torch.float64 else a, b.view(torch.int64) if b.dtype == torch.float64 else b)


@pytest.mark.gpu
def test_bad_arguments_are_rejected_and_touch_nothing():
    import torch
    lm, X0 = _solver("hopper", 3, seed=471)
    bt, p = lm.batch, lm.p
    B = bt.B
    x = X0.clone()
    xl, xu = lm.xl_full, lm.xu_full
    gl, gu = (_cuda(np.tile(a, (B, 1))) for a in p.bounds()[2:])
    st = torch.full((B,), 5, dtype=torch.int32, device="cuda"); its = st.clone()
    viol = torch.full((B,), 7.0, dtype=torch.float64, device="cuda"); mu = viol.clone()
    counts = torch.full((4,), 5, dtype=torch.int32, device="cuda"); loops = torch.full((1,), 5, dtype=torch.int32, device="cuda")
    v = lambda t: C.c_void_p(t.data_ptr())
    nan = float("nan")

    def call(stream=None, **kw):
        o = capi.LmSolveOptions()
        capi.lib.twb_lm_solve_options_default(C.byref(o))
        for k in FIELDS:
            if k in kw:
                setattr(o, k, kw.pop(k))
        a = dict(b=bt._h, x=v(x), xl=v(xl), xu=v(xu), gl=v(gl), gu=v(gu), opt=C.byref(o), st=v(st), its=v(its), viol=v(viol), mu=v(mu),
                 counts=v(counts), loops=v(loops), stream=stream)
        a.update(kw)
        return capi.lib.twb_batch_lm_solve_device(*a.values())

    bad = [dict(b=None), dict(x=None), dict(opt=None), dict(st=None), dict(its=None), dict(viol=None), dict(mu=None), dict(xl=None),
           dict(xu=None), dict(gl=None), dict(gu=None), dict(max_iters=-1), dict(tol=-1e-9), dict(tol=nan), dict(eta=-1e-9), dict(eta=1.0),
           dict(eta=nan), dict(mu_min=0.0), dict(mu_min=2e10), dict(mu_min=nan), dict(mu_max=nan), dict(mu0=0.0), dict(mu0=-1.0),
           dict(mu0=nan), dict(cg_iters=-1), dict(cg_iters=10001), dict(cap=0.0), dict(cap=nan)]
    assert [call(**k) for k in bad] == [capi.ERR_INVALID] * len(bad)
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        rc = call(stream=C.c_void_p(side.cuda_stream))
    assert rc == capi.ERR_UNSUPPORTED
    big = _problem_of(*TOO_LARGE)
    bb = big.batch(2)
    z = lambda *s: torch.zeros(s, dtype=torch.float64, device="cuda")
    zi = lambda *s: torch.zeros(s, dtype=torch.int32, device="cuda")
    o = capi.LmSolveOptions()
    capi.lib.twb_lm_solve_options_default(C.byref(o))
    assert capi.lib.twb_batch_lm_solve_device(bb._h, v(z(2, big.n)), None, None, None, None, C.byref(o), v(zi(2)), v(zi(2)), v(z(2)), v(z(2)),
                                              None, None, None) == capi.ERR_UNSUPPORTED
    torch.cuda.synchronize()
    assert torch.equal(x, X0) and bool((st == 5).all()) and bool((its == 5).all()) and bool((counts == 5).all()) and loops.item() == 5
    assert bool((viol == 7.0).all()) and bool((mu == 7.0).all())
    assert bt.lm_solve_graphs_instantiated() == 0
    assert call() == capi.OK                                     # the batch still serves a valid call
    torch.cuda.synchronize()
    assert loops.item() >= 1 and int(counts.sum()) == B
