"""Device-pointer post-processing (twb_batch_*_device): trajectory, initial guesses, footstep plans and contact sets from
iterates that stay on the GPU — equal to the host-pointer calls bit for bit, the fused footstep-plan kernel equal to a
scan of the sampled trajectory bit for bit, stream-ordered and capturable in a CUDA graph."""
import ctypes as C

import numpy as np
import pytest

import towr_b200 as tb
from towr_b200 import capi
from towr_b200.configs import _renormalise, synthetic_iterates, synthetic_iterates_fast
import oracle_lib

pytestmark = pytest.mark.gpu

TIMES = np.array([0.0, 0.013, 0.4, 0.99, 1.0, 1.37, 2.0])
HORIZON = 2.0


def _polys():
    from test_oracle import _polys_for_lookup
    return _polys_for_lookup()


def _problem(name, optimise=False):
    f = tb.make_formulation(name)
    if optimise and not f.params_.IsOptimizeTimings():
        f.params_.OptimizePhaseDurations()
    return tb.Problem(f.to_spec())


def _spread_durations(p, X, seed, lo=0.35, hi=1.65):
    """durations x U[lo, hi], renormalised so that their sum stays below T (as test_durations_spread_widely_over_a_tile)"""
    rng = np.random.default_rng(seed)
    x0 = p.GetVariableValues()
    for sname, start, count in p.variable_sets():
        if sname.startswith("ee-schedule"):
            X[:, start:start + count] = _renormalise(p, sname, x0[start:start + count] * rng.uniform(lo, hi, (X.shape[0], count)))
    return X


def _host_plans(bt, X, T):
    """twb_batch_footstep_plan_host with the full (B, max_states, V) output (NaN-filled first: every row must be written)"""
    ms, nv = bt.footstep_plan_dims()
    out = np.full((bt.B, ms, nv), np.nan)
    count = np.full(bt.B, -7, np.int32)
    X = np.ascontiguousarray(X, np.float64)
    capi.check(capi.lib.twb_batch_footstep_plan_host(bt._h, X.ctypes.data_as(C.c_void_p), float(T), count.ctypes.data_as(C.c_void_p),
                                                     out.ctypes.data_as(C.c_void_p)))
    return out, count


def _host_contact_sets(bt, plans, count, polygons):
    ms, nv = bt.footstep_plan_dims()
    offs, verts = tb.pack_polygons(polygons)
    cs = np.full((bt.B, ms, (nv - 2) // 4), -7, np.int32)
    capi.check(capi.lib.twb_batch_nearest_planes_host(bt._h, plans.ctypes.data_as(C.c_void_p), count.ctypes.data_as(C.c_void_p),
                                                      offs.ctypes.data_as(C.c_void_p), len(polygons), verts.ctypes.data_as(C.c_void_p),
                                                      cs.ctypes.data_as(C.c_void_p)))
    return cs


def _device_polys(polygons):
    import torch
    offs, verts = tb.pack_polygons(polygons)
    return torch.from_numpy(offs).cuda(), torch.from_numpy(verts).cuda()


def _scan_reference(traj, T, dt=0.01):
    """fpowr::ExtractFootstepPlan's rule (footstep_plan_extractor.h:68-133) on a sampled trajectory (n_samples, 19 + 13 n_ee):
    the first state and every change of the contact set, t += dt, durations as differences, the last one up to T."""
    n_ee = (traj.shape[1] - 19) // 13
    flags = traj[:, [19 + 13 * e for e in range(n_ee)]]
    states, t = [], 0.0
    for k in range(traj.shape[0]):
        if k == 0 or not np.array_equal(flags[k], flags[k - 1]):
            if states:
                states[-1][1] = t - states[-1][0]
            row = [t, 0.0]
            for e in range(n_ee):
                row += [traj[k, 19 + 13 * e]] + list(traj[k, 20 + 13 * e:23 + 13 * e])
            states.append(row)
        t += dt
    states[-1][1] = T - states[-1][0]
    return np.array(states)


CASES = [("hopper", False, 5, 0.05), ("anymal_trot_block", False, 33, 0.01), ("biped_walk_stairs", False, 101, 0.02),
         ("hyq_gallop_gap", True, 37, 0.02)]


@pytest.mark.parametrize("name,optimise,B,dt", CASES)
def test_device_variants_equal_host_variants(name, optimise, B, dt):
    """Trajectory, initial guesses, footstep plans with their counts and contact sets: device == host, bit for bit (Biped:
    interleaved tiles; HyQ: optimised durations)."""
    import torch
    p = _problem(name, optimise)
    X = synthetic_iterates(p, B)
    if optimise:
        X = _spread_durations(p, X, 5)
    bt = p.batch(B)
    polys = _polys()
    traj_h = bt.sample_trajectory(X, dt)
    ig_h = bt.initial_guesses(X, TIMES)
    plans_h, count_h = _host_plans(bt, X, HORIZON)
    cs_h = _host_contact_sets(bt, plans_h, count_h, polys)
    assert np.all(count_h >= 2) and not np.isnan(plans_h).any()

    xd = torch.from_numpy(X).cuda()
    traj_d = bt.sample_trajectory_device(xd, dt)
    ig_d = bt.initial_guesses_device(xd, TIMES)
    plans_d, count_d = bt.footstep_plans_device(xd, HORIZON)
    cs_d = bt.nearest_planes_device(plans_d, count_d, *_device_polys(polys))
    torch.cuda.synchronize()
    assert np.array_equal(traj_d.cpu().numpy(), traj_h)
    assert np.array_equal(ig_d.cpu().numpy(), ig_h)
    assert np.array_equal(count_d.cpu().numpy(), count_h)
    assert np.array_equal(plans_d.cpu().numpy(), plans_h)
    assert np.array_equal(cs_d.cpu().numpy(), cs_h)
    for b in range(B):   # unused rows: 0 in the plan, -1 in the contact sets
        assert not plans_h[b, count_h[b]:].any() and np.all(cs_h[b, count_h[b]:] == -1)


def _check_scan(p, X, bt=None):
    import torch
    B = X.shape[0]
    bt = bt or p.batch(B)
    traj = bt.sample_trajectory(X, 0.01)
    plans_h, count_h = _host_plans(bt, X, HORIZON)
    plans_d, count_d = bt.footstep_plans_device(torch.from_numpy(X).cuda(), HORIZON)
    plans_d, count_d = plans_d.cpu().numpy(), count_d.cpu().numpy()
    for b in range(B):
        ref = _scan_reference(traj[b], HORIZON)
        assert count_h[b] == len(ref) and count_d[b] == len(ref), (b, count_h[b], count_d[b], len(ref))
        assert np.array_equal(plans_h[b, :len(ref)], ref, equal_nan=True), (b, np.nanmax(np.abs(plans_h[b, :len(ref)] - ref)))
        assert np.array_equal(plans_d[b, :len(ref)], ref, equal_nan=True), b
        assert not plans_h[b, len(ref):].any() and not plans_d[b, len(ref):].any()
    return count_h


@pytest.mark.parametrize("name", ["anymal_trot_block", "biped_walk_stairs"])
def test_footstep_plan_is_the_scan_of_the_trajectory_fixed_durations(name):
    p = _problem(name)
    _check_scan(p, synthetic_iterates(p, 45))


@pytest.mark.parametrize("name,B", [("hyq_gallop_gap", 64), ("biped_walk_stairs", 37)])
def test_footstep_plan_is_the_scan_of_the_trajectory_spread_durations(name, B):
    """Optimised durations x U[0.35, 1.65]: the instances of a tile change contact at very different steps."""
    p = _problem(name, optimise=True)
    _check_scan(p, _spread_durations(p, synthetic_iterates(p, B), 99))


def test_footstep_plan_is_the_scan_of_the_trajectory_durations_past_the_horizon():
    """Iterates whose phase durations sum to T or more (status bit 1 of an evaluation): the last phase is empty or
    negative; the walk still follows the trajectory's phase search exactly."""
    p = _problem("hyq_gallop_gap", optimise=True)
    B = 40
    X = synthetic_iterates(p, B)
    spec = p.spec
    for sname, start, count in p.variable_sets():
        if sname.startswith("ee-schedule"):
            ee = int(sname[len("ee-schedule"):])
            t_total = sum(spec.phase_durations[ee][i] for i in range(spec.n_phases[ee]))
            d = X[:, start:start + count]
            for b, factor in ((0, 1.0), (1, 1.05), (2, 1.5), (7, 3.0), (31, 1.2), (39, 1.0)):   # sum = factor x T
                d[b] *= factor * t_total / d[b].sum()
    out = p.batch(B).eval_host(X)
    assert (out["status"][[1, 2, 7, 31]] & 2).all()
    _check_scan(p, X)


def test_device_calls_are_stream_ordered_and_capturable():
    """On a non-default stream: one warm-up call per entry point, then footstep plans -> nearest planes -> trajectory ->
    initial guesses captured in one CUDA graph (global capture mode: any allocation or synchronisation would fail it),
    replayed for two iterate sets copied into the captured input."""
    import torch
    p = _problem("anymal_trot_block")
    B, dt = 70, 0.02
    bt = p.batch(B)
    polys = _polys()
    offs_d, verts_d = _device_polys(polys)
    s = torch.cuda.Stream()
    X1 = synthetic_iterates(p, B)
    X2 = synthetic_iterates(p, B, seed=777)
    with torch.cuda.stream(s):
        xin = torch.from_numpy(X1).cuda()
        plans, count = bt.footstep_plans_device(xin, HORIZON, stream=s)
        cs = bt.nearest_planes_device(plans, count, offs_d, verts_d, stream=s)
        traj = bt.sample_trajectory_device(xin, dt, stream=s)
        ig = bt.initial_guesses_device(xin, TIMES, stream=s)
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        bt.footstep_plans_device(xin, HORIZON, out=(plans, count))
        bt.nearest_planes_device(plans, count, offs_d, verts_d, out=cs)
        bt.sample_trajectory_device(xin, dt, out=traj)
        bt.initial_guesses_device(xin, TIMES, out=ig)
    for X in (X2, X1):
        with torch.cuda.stream(s):
            xin.copy_(torch.from_numpy(X).cuda())
            g.replay()
        s.synchronize()
        plans_h, count_h = _host_plans(bt, X, HORIZON)
        assert np.array_equal(count.cpu().numpy(), count_h)
        assert np.array_equal(plans.cpu().numpy(), plans_h)
        assert np.array_equal(cs.cpu().numpy(), _host_contact_sets(bt, plans_h, count_h, polys))
        assert np.array_equal(traj.cpu().numpy(), bt.sample_trajectory(X, dt))
        assert np.array_equal(ig.cpu().numpy(), bt.initial_guesses(X, TIMES))


def test_footstep_plans_at_the_config5_size():
    """Config 5 (Anymal trot, mixed Slope / Chimney / Gap terrains, B = 65 536) on one GPU: fixed durations give every
    instance the same number of footstep states; sampled instances against the oracle's fpowr::ExtractFootstepPlan."""
    import torch
    spec = tb.make_formulation("anymal_trot_mixed").to_spec()
    p = tb.Problem(spec)
    B = 65536
    bt = p.batch(B)
    bt.set_terrains(np.array([tb.SLOPE, tb.CHIMNEY, tb.GAP] * (B // 3 + 1), np.int32)[:B])
    X = synthetic_iterates_fast(p, B)
    plans, count = bt.footstep_plans_device(torch.from_numpy(X).cuda(), HORIZON)
    plans, count = plans.cpu().numpy(), count.cpu().numpy()
    assert np.all(count == count[0]) and count[0] >= 2
    o = oracle_lib.Oracle(spec)
    for b in np.random.default_rng(5).choice(B, 24, replace=False):
        ref = o.footstep_plan(X[b], HORIZON)
        got = plans[b, :count[b]]
        assert got.shape == ref.shape, (b, got.shape, ref.shape)
        flags = [2 + 4 * e for e in range(4)]
        assert np.array_equal(got[:, 0], ref[:, 0]) and np.array_equal(got[:, flags], ref[:, flags])
        assert np.all(np.abs(got - ref) <= 1e-12 * np.abs(ref) + 1e-13), (b, np.abs(got - ref).max())
        assert abs(got[:, 1].sum() - HORIZON) < 1e-9


def test_device_calls_reject_bad_arguments():
    """Null pointers, dt <= 0, n_times <= 0, n_polys < 0: TWB_ERR_INVALID and nothing enqueued (the outputs keep their
    sentinel values)."""
    import torch
    p = _problem("anymal_trot_block")
    B = 33
    bt = p.batch(B)
    x = torch.from_numpy(synthetic_iterates(p, B)).cuda()
    ms, nv = bt.footstep_plan_dims()
    traj = torch.full((B, 201, 19 + 13 * 4), 7.0, dtype=torch.float64, device="cuda")
    ig = torch.full((B, TIMES.size, 49), 7.0, dtype=torch.float64, device="cuda")
    plans = torch.full((B, ms, nv), 7.0, dtype=torch.float64, device="cuda")
    count = torch.full((B,), 7, dtype=torch.int32, device="cuda")
    cs = torch.full((B, ms, 4), 7, dtype=torch.int32, device="cuda")
    offs, verts = _device_polys(_polys())
    v = lambda t: C.c_void_p(t.data_ptr())
    times = TIMES.ctypes.data_as(C.c_void_p)
    lib, h = capi.lib, bt._h
    calls = [
        lib.twb_batch_sample_trajectory_device(None, v(x), 0.01, v(traj), None),
        lib.twb_batch_sample_trajectory_device(h, None, 0.01, v(traj), None),
        lib.twb_batch_sample_trajectory_device(h, v(x), 0.01, None, None),
        lib.twb_batch_sample_trajectory_device(h, v(x), 0.0, v(traj), None),
        lib.twb_batch_sample_trajectory_device(h, v(x), -0.01, v(traj), None),
        lib.twb_batch_sample_trajectory_device(h, v(x), float("nan"), v(traj), None),
        lib.twb_batch_initial_guess_device(h, None, times, TIMES.size, v(ig), None),
        lib.twb_batch_initial_guess_device(h, v(x), None, TIMES.size, v(ig), None),
        lib.twb_batch_initial_guess_device(h, v(x), times, 0, v(ig), None),
        lib.twb_batch_initial_guess_device(h, v(x), times, TIMES.size, None, None),
        lib.twb_batch_footstep_plan_device(h, None, HORIZON, v(count), v(plans), None),
        lib.twb_batch_footstep_plan_device(h, v(x), HORIZON, None, v(plans), None),
        lib.twb_batch_footstep_plan_device(h, v(x), HORIZON, v(count), None, None),
        lib.twb_batch_nearest_planes_device(h, None, v(count), v(offs), offs.numel() - 1, v(verts), v(cs), None),
        lib.twb_batch_nearest_planes_device(h, v(plans), None, v(offs), offs.numel() - 1, v(verts), v(cs), None),
        lib.twb_batch_nearest_planes_device(h, v(plans), v(count), None, offs.numel() - 1, v(verts), v(cs), None),
        lib.twb_batch_nearest_planes_device(h, v(plans), v(count), v(offs), offs.numel() - 1, None, v(cs), None),
        lib.twb_batch_nearest_planes_device(h, v(plans), v(count), v(offs), -1, v(verts), v(cs), None),
        lib.twb_batch_nearest_planes_device(h, v(plans), v(count), v(offs), offs.numel() - 1, v(verts), None, None),
    ]
    assert calls == [capi.ERR_INVALID] * len(calls)
    with pytest.raises(capi.TowrB200Error) as err:
        bt.sample_trajectory_device(x, 0.0)
    assert err.value.code == capi.ERR_INVALID
    torch.cuda.synchronize()
    for t in (traj, ig, plans, count, cs):
        assert bool((t == 7).all())
    # the same batch still serves valid calls afterwards
    plans2, count2 = bt.footstep_plans_device(x, HORIZON)
    assert np.array_equal(plans2.cpu().numpy(), _host_plans(bt, x.cpu().numpy(), HORIZON)[0])
