"""Per-instance start states (twb_problem_state_instances / twb_batch_state_instances_device): instances of one structure
class that differ in NlpFormulation::initial_base_, final_base_ and initial_ee_W_.  The host builder is checked bit for bit
against the oracle built on each instance's own formulation; the device kernel against the host builder, on height grids,
inside guard zones, under CUDA graph capture, and as the setup of a device-resident solver loop."""
import ctypes as C

import numpy as np
import pytest

import towr_b200 as tb
from towr_b200 import capi
import oracle_lib

RECIPES = ("hopper", "anymal_trot_block", "biped_walk_stairs", "hyq_gallop_gap", "anymal_trot_block_base_rom")


def _random_states(f, rng, count):
    """`count` state records around the formulation's own: base position / yaw offsets, base velocities, Euler angles within
    +-0.3 rad, feet shifted in x / y / z, non-zero final velocities (the default Parameters bound all of them)."""
    S = np.tile(f.state_record(), (count, 1))
    n_ee = len(f.initial_ee_W_)
    S[:, 0:2] += rng.uniform(-0.3, 0.3, (count, 2)); S[:, 2] += rng.uniform(-0.05, 0.05, count)     # initial base position
    S[:, 3:6] = rng.uniform(-0.5, 0.5, (count, 3))                                                   # initial base velocity
    S[:, 6:9] = rng.uniform(-0.3, 0.3, (count, 3))                                                   # initial Euler angles
    S[:, 9:12] = rng.uniform(-0.5, 0.5, (count, 3))                                                  # initial angular velocity
    S[:, 12:14] += rng.uniform(-0.5, 0.5, (count, 2)); S[:, 14] += rng.uniform(-0.05, 0.05, count)  # goal position
    S[:, 15:18] = rng.uniform(-0.3, 0.3, (count, 3))                                                 # final velocity
    S[:, 18:21] = rng.uniform(-0.3, 0.3, (count, 3))                                                 # goal Euler angles
    S[:, 21:24] = rng.uniform(-0.3, 0.3, (count, 3))                                                 # final angular velocity
    S[:, 24:24 + 3 * n_ee] += rng.uniform(-0.05, 0.05, (count, 3 * n_ee))                            # initial feet
    return S


def _formulation_with_state(name, rec):
    """The recipe's NlpFormulation with its three state fields set from one state record."""
    f = tb.make_formulation(name)
    for node, off in ((f.initial_base_.lin, 0), (f.initial_base_.ang, 6), (f.final_base_.lin, 12), (f.final_base_.ang, 18)):
        node.p = np.array(rec[off:off + 3]); node.v = np.array(rec[off + 3:off + 6])
    f.initial_ee_W_ = [np.array(rec[24 + 3 * e:27 + 3 * e]) for e in range(len(f.initial_ee_W_))]
    return f


def _base_z_rows(p):
    sets = [c for c in p.constraint_sets() if c[0] == "baseMotion"]
    return np.concatenate([np.arange(r0 + 5, r0 + nr, 6) for _, r0, nr in sets]).astype(int) if sets else np.zeros(0, int)


# ---- host builder (no GPU) ---------------------------------------------------------------------------------------------

def test_state_record_layout():
    f = tb.make_formulation("anymal_trot_block")
    f.initial_base_.lin.v[:] = (0.1, 0.2, 0.3); f.final_base_.ang.v[:] = (-0.1, -0.2, -0.3)
    rec, s = f.state_record(), f.to_spec()
    assert rec.shape == (capi.STATE_DOUBLES,)
    fields = ("initial_base_lin_pos", "initial_base_lin_vel", "initial_base_ang_pos", "initial_base_ang_vel",
              "final_base_lin_pos", "final_base_lin_vel", "final_base_ang_pos", "final_base_ang_vel")
    for k, name in enumerate(fields):
        assert list(rec[3 * k:3 * k + 3]) == list(getattr(s, name)), name
    for e in range(4):
        assert list(rec[24 + 3 * e:27 + 3 * e]) == list(s.initial_ee_W[e])
    hop = tb.make_formulation("hopper").state_record()            # one foot: the other three slots stay 0
    assert np.all(hop[27:] == 0.0)
    with pytest.raises(ValueError):
        tb.pack_states([f.initial_base_], [], [f.initial_ee_W_])


def test_state_instances_match_oracle_bit_for_bit():
    """For every recipe, 5 random start / goal states: x0, variable bounds and constraint bounds of the unchanged problem's
    twb_problem_state_instances equal those of the oracle built on each instance's own formulation, bit for bit."""
    rng = np.random.default_rng(101)
    for name in RECIPES:
        base = tb.make_formulation(name)
        p = tb.Problem(base.to_spec())
        S = _random_states(base, rng, 5)
        x0, xl, xu, gl, gu = p.state_instances(S)
        for i in range(len(S)):
            f = _formulation_with_state(name, S[i])
            assert np.array_equal(f.state_record(), S[i])
            o = oracle_lib.Oracle(f.to_spec())
            oxl, oxu, ogl, ogu = o.bounds()
            assert np.array_equal(x0[i], o.x0()), (name, i)
            assert np.array_equal(xl[i], oxl) and np.array_equal(xu[i], oxu), (name, i)
            assert np.array_equal(gl[i], ogl) and np.array_equal(gu[i], ogu), (name, i)
        _, _, pgl, pgu = p.bounds()
        rows = _base_z_rows(p)
        other = np.setdiff1d(np.arange(p.m), rows)
        assert np.all(gl[:, other] == pgl[other]) and np.all(gu[:, other] == pgu[other]), name
        if name.endswith("_base_rom"):
            assert rows.size > 0
            assert np.unique(gl[:, rows[0]]).size == len(S) and np.unique(gu[:, rows[-1]]).size == len(S)   # differ per instance
            assert np.allclose(gl[:, rows], (S[:, 2] - 0.02)[:, None], rtol=0, atol=1e-15)
        else:
            assert rows.size == 0


def test_spec_state_reproduces_the_problem():
    for name in RECIPES:
        f = tb.make_formulation(name)
        p = tb.Problem(f.to_spec())
        x0, xl, xu, gl, gu = p.state_instances(f.state_record()[None])
        pxl, pxu, pgl, pgu = p.bounds()
        assert np.array_equal(x0[0], p.GetVariableValues()), name
        assert np.array_equal(xl[0], pxl) and np.array_equal(xu[0], pxu), name
        assert np.array_equal(gl[0], pgl) and np.array_equal(gu[0], pgu), name


def test_goal_only_states_reproduce_goal_instances():
    rng = np.random.default_rng(5)
    for name in RECIPES:
        f = tb.make_formulation(name)
        p = tb.Problem(f.to_spec())
        G = 6
        goals = np.column_stack([rng.uniform(0.3, 2.5, G), rng.uniform(-0.4, 0.4, G), np.full(G, 0.5), rng.uniform(-0.3, 0.3, (G, 2)),
                                 rng.uniform(-0.5, 0.5, G)])
        S = np.tile(f.state_record(), (G, 1))
        S[:, 12:15] = goals[:, :3]; S[:, 18:21] = goals[:, 3:]
        x0, xl, xu, gl, gu = p.state_instances(S)
        gx0, gxl, gxu = p.goal_instances(goals)
        assert np.array_equal(x0, gx0) and np.array_equal(xl, gxl) and np.array_equal(xu, gxu), name
        _, _, pgl, pgu = p.bounds()
        assert np.all(gl == pgl) and np.all(gu == pgu), name


def test_state_instances_argument_errors():
    f = tb.make_formulation("hopper")
    p = tb.Problem(f.to_spec())
    S = np.ascontiguousarray(f.state_record()[None])
    x0 = np.empty(p.n)
    dp = C.POINTER(C.c_double)
    assert capi.lib.twb_problem_state_instances(p._h, 1, None, x0.ctypes.data_as(dp), None, None, None, None) == capi.ERR_INVALID
    for n_states in (0, -1):
        assert capi.lib.twb_problem_state_instances(p._h, n_states, S.ctypes.data_as(dp), x0.ctypes.data_as(dp), None, None, None,
                                                    None) == capi.ERR_INVALID
    assert capi.lib.twb_problem_state_instances(None, 1, S.ctypes.data_as(dp), x0.ctypes.data_as(dp), None, None, None, None) == capi.ERR_INVALID
    # every output NULL is allowed on the host (nothing to write); one output alone equals the full call's
    assert capi.lib.twb_problem_state_instances(p._h, 1, S.ctypes.data_as(dp), None, None, None, None, None) == capi.OK
    assert capi.lib.twb_problem_state_instances(p._h, 1, S.ctypes.data_as(dp), x0.ctypes.data_as(dp), None, None, None, None) == capi.OK
    assert np.array_equal(x0, p.GetVariableValues())


# ---- device kernel -----------------------------------------------------------------------------------------------------

def _device_call(bt, states, x0=None, lo=None, up=None, gl=None, gu=None, stream=None):
    import torch
    ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    s = torch.cuda.current_stream() if stream is None else stream
    return capi.lib.twb_batch_state_instances_device(bt._h, ptr(states), ptr(x0), ptr(lo), ptr(up), ptr(gl), ptr(gu), C.c_void_p(s.cuda_stream))


@pytest.mark.gpu
def test_state_instances_on_the_device_match_the_host():
    """Device kernel against the host builder for every recipe at B = 70 and at ragged B = 1 and 37 (rtol 1e-14 on x0 and
    the x bounds: sincos(yaw) may differ from the host's libm in the last place); constraint bounds equal."""
    import torch
    rng = np.random.default_rng(202)
    for name in RECIPES:
        f = tb.make_formulation(name)
        p = tb.Problem(f.to_spec())
        for B in (70, 1, 37):
            S = _random_states(f, rng, B)
            x0h, xlh, xuh, glh, guh = p.state_instances(S)
            bt = p.batch(B)
            x0, lo, up, gl, gu = bt.state_instances_device(torch.from_numpy(S).cuda(), want_g_bounds=True)
            torch.cuda.synchronize()
            assert np.allclose(x0.cpu().numpy(), x0h, rtol=1e-14, atol=1e-15), (name, B)
            assert np.allclose(lo.cpu().numpy(), xlh, rtol=1e-14, atol=0) and np.allclose(up.cpu().numpy(), xuh, rtol=1e-14, atol=0), (name, B)
            assert np.array_equal(gl.cpu().numpy(), glh) and np.array_equal(gu.cpu().numpy(), guh), (name, B)
            x1, l1, u1, g1, h1 = bt.state_instances_device(torch.from_numpy(S).cuda())      # defaults: no constraint bounds
            assert g1 is None and h1 is None and torch.equal(x1, x0) and torch.equal(l1, lo) and torch.equal(u1, up)


@pytest.mark.gpu
def test_state_instances_on_height_grids():
    """TWB_GRID_CSV and TWB_GRID_MAP as the instances' terrain: the last base-lin node z and the final footholds follow the
    grid under each instance's own goal."""
    import torch
    rng = np.random.default_rng(303)
    f = tb.make_formulation("anymal_trot_block")
    p = tb.Problem(f.to_spec())
    nominal = np.array(tb.robot_info(tb.ANYMAL)["nominal_stance"])
    sets = {name: (s, k) for name, s, k in p.variable_sets()}
    s_lin, n_lin = sets["base-lin"]
    B = 33
    sx, sy, res, pos = 60, 40, 0.1, (1.0, 0.0)
    xs = pos[0] + sx * res / 2 - res / 2 - res * np.arange(sx)
    ys = pos[1] + sy * res / 2 - res / 2 - res * np.arange(sy)
    H = (0.15 * np.sin(2.0 * xs)[:, None] * np.cos(1.5 * ys)[None, :] + 0.02 * rng.standard_normal((sx, sy))).astype(np.float32)
    grid = rng.integers(0, 4, (12, 20)) * 0.04
    for terrain, y_range, tol in ((tb.GRID_CSV, (0.3, 1.0), 1e-12), (tb.GRID_MAP, (-0.5, 0.5), 1e-6)):
        bt = p.batch(B); bt.set_terrains(np.full(B, terrain, np.int32))
        if terrain == tb.GRID_CSV:
            bt.set_grid_terrain(grid); oracle_lib.set_grid(grid)
        else:
            bt.set_grid_map(H, res, pos); oracle_lib.set_grid_map(H, res, pos)
        S = _random_states(f, rng, B)
        S[:, 12] = rng.uniform(0.5, 2.5, B); S[:, 13] = rng.uniform(*y_range, B)
        x0, _, _, _, _ = bt.state_instances_device(torch.from_numpy(S).cuda(), want_bounds=False)
        x0 = x0.cpu().numpy()
        for b in range(B):
            h = oracle_lib.terrain_point(terrain, S[b, 12], S[b, 13])[0]
            assert abs(x0[b, s_lin + n_lin - 6 + 2] - (h - nominal[0][2])) < tol, (terrain, b)    # last base-lin node, z
            yaw = S[b, 20]
            for e in range(len(nominal)):
                s_e, k_e = sets[f"ee-motion_{e}"]
                w = S[b, 12:14] + np.array([[np.cos(yaw), -np.sin(yaw)], [np.sin(yaw), np.cos(yaw)]]) @ nominal[e][:2]
                foot = x0[b, s_e + k_e - 3:s_e + k_e]            # the last node is a stance node: its shared x, y, z
                assert np.allclose(foot[:2], w, rtol=0, atol=1e-12), (terrain, b, e)
                assert abs(foot[2] - oracle_lib.terrain_point(terrain, w[0], w[1])[0]) < tol, (terrain, b, e)
        assert np.ptp(x0[:, s_lin + n_lin - 6 + 2]) > 0.01                                        # the grid shows


@pytest.mark.gpu
def test_state_instances_write_exactly_their_outputs():
    """Every output between two guard zones: the guards stay intact and every element is written; NULL outputs are skipped;
    argument errors enqueue nothing."""
    import torch
    f = tb.make_formulation("anymal_trot_block_base_rom")
    p = tb.Problem(f.to_spec())
    B = 37
    S = torch.from_numpy(_random_states(f, np.random.default_rng(404), B)).cuda()
    bt = p.batch(B)
    guard, sentinel = 4096, -7.25e300

    def guarded(count):
        buf = torch.full((count + 2 * guard,), sentinel, dtype=torch.float64, device="cuda")
        return buf, buf[guard:guard + count]
    bufs = [guarded(B * k) for k in (p.n, p.n, p.n, p.m, p.m)]
    views = [v for _, v in bufs]
    assert _device_call(bt, S, *views) == capi.OK
    torch.cuda.synchronize()
    for (buf, v), count in zip(bufs, (B * p.n,) * 3 + (B * p.m,) * 2):
        assert bool((buf[:guard] == sentinel).all()) and bool((buf[guard + count:] == sentinel).all()), "write outside the array"
        assert not bool((v == sentinel).any()), "element left unwritten"
    full = [v.clone() for v in views]
    for k in range(5):                                   # one output at a time: the others stay untouched
        for buf, _ in bufs:
            buf.fill_(sentinel)
        only = [views[j] if j == k else None for j in range(5)]
        assert _device_call(bt, S, *only) == capi.OK
        torch.cuda.synchronize()
        assert torch.equal(views[k], full[k])
        for j in range(5):
            if j != k:
                assert bool((bufs[j][0] == sentinel).all()), (k, j)
    for buf, _ in bufs:
        buf.fill_(sentinel)
    assert _device_call(bt, None, *views) == capi.ERR_INVALID
    assert _device_call(bt, S) == capi.ERR_INVALID
    with pytest.raises(AssertionError):
        bt.state_instances_device(S[:, :6].contiguous())
    torch.cuda.synchronize()
    assert all(bool((buf == sentinel).all()) for buf, _ in bufs)


@pytest.mark.gpu
def test_state_instances_graph_capture():
    """One CUDA graph capture of the call on a non-default stream, replayed for two state sets, gives the direct call's
    results."""
    import torch
    f = tb.make_formulation("hyq_gallop_gap")
    p = tb.Problem(f.to_spec())
    B = 45
    rng = np.random.default_rng(505)
    sets = [torch.from_numpy(_random_states(f, rng, B)).cuda() for _ in range(2)]
    bt = p.batch(B)
    direct = [bt.state_instances_device(s, want_g_bounds=True) for s in sets]
    torch.cuda.synchronize()
    st = torch.empty_like(sets[0])
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        out = bt.state_instances_device(st, want_g_bounds=True)
    for s, ref in zip(sets, direct):
        st.copy_(s)
        graph.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(out, ref))
    assert not torch.equal(direct[0][0], direct[1][0])


@pytest.mark.gpu
def test_device_pipeline_from_measured_states():
    """4096 Anymal instances with their own starts and goals: setup on the device, then 12 Levenberg-Marquardt iterations on
    the per-instance x bounds.  The start-bound variables keep each instance's record after every step, every violation is
    finite, and the oracle-driven numpy twin walks a subsample of 8 instances to the same iterates."""
    import torch
    from towr_b200.solver import BatchedLevenbergMarquardt
    from test_solver_loop import LevenbergMarquardtReference
    f = tb.make_formulation("anymal_trot_block")
    spec = f.to_spec()
    p = tb.Problem(spec)
    B, iters = 4096, 12
    rng = np.random.default_rng(606)
    S = _random_states(f, rng, B)
    bt = p.batch(B)
    x0, xl, xu, _, _ = bt.state_instances_device(torch.from_numpy(S).cuda())
    X = torch.minimum(torch.maximum(x0 + 0.01 * torch.from_numpy(rng.standard_normal((B, p.n))).cuda(), xl), xu)
    starts = X.cpu().numpy().copy()
    sets = {name: s for name, s, _ in p.variable_sets()}
    fixed = [(sets["base-lin"] + np.arange(6), np.r_[0:6]), (sets["base-ang"] + np.arange(6), np.r_[6:12])]
    for e in range(spec.n_ee):                            # node 0 position of each foot: a stance pair (x, y, z) or a swing node
        local = np.array([0, 1, 2]) if spec.in_contact_at_start[e] else np.array([0, 2, 4])
        fixed.append((sets[f"ee-motion_{e}"] + local, 24 + 3 * e + np.arange(3)))
    cols = np.concatenate([c for c, _ in fixed]); recs = torch.from_numpy(S[:, np.concatenate([r for _, r in fixed])]).cuda()
    lm = BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu)
    hist = torch.empty((iters, B), dtype=torch.float64, device="cuda")
    for it in range(iters):
        hist[it] = lm.step(X)
        assert torch.equal(X[:, cols], recs), it
    hist = hist.cpu().numpy(); X_gpu = X.cpu().numpy()
    assert np.isfinite(hist).all() and not lm.status.any().item()
    assert not np.array_equal(X_gpu, starts)
    o = oracle_lib.Oracle(spec)
    xl_h, xu_h = xl.cpu().numpy(), xu.cpu().numpy()
    for b in rng.choice(B, 8, replace=False):
        ref = LevenbergMarquardtReference(o, p, spec.terrain, xl_h[b], xu_h[b])
        x = starts[b].copy()
        for it in range(iters):
            x, v = ref.step(x)
            assert abs(v - hist[it, b]) <= 1e-6 * max(1e-9, abs(v)), (b, it)
        assert np.allclose(x, X_gpu[b], rtol=0, atol=1e-8), (b, float(np.abs(x - X_gpu[b]).max()))
