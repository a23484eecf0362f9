"""Per-instance terrains for batched plan requests: several grid_map elevation layers per batch with a map index per instance
(twb_batch_set_grid_maps), and one planar-region set per instance for the nearest-plane lookup
(twb_batch_nearest_planes_ranges_*).  The GPU results are checked against the oracle on each instance's own map, and bit for
bit against batches that hold only that instance's map or polygon list."""
import ctypes as C

import numpy as np
import pytest

import towr_b200 as tb
from towr_b200 import capi
from towr_b200.configs import synthetic_iterates, synthetic_iterates_fast
import oracle_lib
from tolerance import check_rows, check_sets

def _grid_map(rng, sx, sy, res, pos):
    """a smooth elevation layer with noise, heights[ix, iy] at the cell centres of grid_map's convention"""
    xs = pos[0] + sx * res / 2 - res / 2 - res * np.arange(sx)
    ys = pos[1] + sy * res / 2 - res / 2 - res * np.arange(sy)
    a, wx, wy = rng.uniform(0.05, 0.2), rng.uniform(1.0, 3.0), rng.uniform(1.0, 2.0)
    H = a * np.sin(wx * xs + rng.uniform(0, 3))[:, None] * np.cos(wy * ys)[None, :] + 0.02 * rng.standard_normal((sx, sy))
    return H.astype(np.float32), res, pos


def _five_maps(rng):
    """five maps that differ in size, resolution (0.03 - 0.1 m) and position, each covering the feet of the iterates"""
    geo = ((60, 40, 0.1, (1.0, 0.0)), (110, 70, 0.05, (1.1, 0.05)), (160, 110, 0.03, (0.9, -0.05)), (70, 50, 0.07, (1.05, 0.1)),
           (56, 44, 0.085, (0.95, -0.1)))
    return [_grid_map(rng, *g) for g in geo]


def _many_maps(rng, count):
    maps = []
    for _ in range(count):
        res = rng.uniform(0.05, 0.1)
        sx, sy = int(np.ceil(5.0 / res)) + int(rng.integers(0, 8)), int(np.ceil(3.5 / res)) + int(rng.integers(0, 8))
        maps.append(_grid_map(rng, sx, sy, res, (1.0 + rng.uniform(-0.1, 0.1), rng.uniform(-0.1, 0.1))))
    return maps


def _set_maps_raw(bt, n_maps, maps, idx):
    """twb_batch_set_grid_maps on raw arrays (no Python checks): returns the status code"""
    heights = np.concatenate([np.ascontiguousarray(h, np.float32).ravel() for h, _, _ in maps]) if maps else np.zeros(1, np.float32)
    sizes = np.array([h.shape for h, _, _ in maps] or [(1, 1)], np.int32)
    geometry = np.array([(r, p[0], p[1]) for _, r, p in maps] or [(1.0, 0.0, 0.0)], np.float64)
    idx = None if idx is None else np.ascontiguousarray(idx, np.int32)
    return capi.lib.twb_batch_set_grid_maps(bt._h, n_maps, heights.ctypes.data_as(C.POINTER(C.c_float)), sizes.ctypes.data_as(C.POINTER(C.c_int)),
                                            geometry.ctypes.data_as(C.POINTER(C.c_double)),
                                            None if idx is None else idx.ctypes.data_as(C.POINTER(C.c_int)))


# ---- no GPU ------------------------------------------------------------------------------------------------------------

def test_pack_polygon_sets():
    sq = lambda x0: np.array([[x0, 0.0], [x0, 1.0], [x0 + 1.0, 1.0], [x0, 0.0]])
    sets = [[sq(0.0), sq(2.0)], [], [sq(5.0)], [sq(7.0), sq(8.0), sq(9.0)]]
    offs, verts, ranges = tb.pack_polygon_sets(sets)
    assert ranges.dtype == np.int32 and ranges.shape == (4, 2)
    assert ranges.tolist() == [[0, 2], [2, 0], [2, 1], [3, 3]]
    flat = [q for s in sets for q in s]
    offs_ref, verts_ref = tb.pack_polygons(flat)
    assert np.array_equal(offs, offs_ref) and np.array_equal(verts, verts_ref)
    for b, s in enumerate(sets):
        first, count = ranges[b]
        for j, q in enumerate(s):
            k = first + j
            assert np.array_equal(verts[offs[k]:offs[k + 1]], q)
    offs0, verts0, ranges0 = tb.pack_polygon_sets([[], []])
    assert offs0.tolist() == [0] and verts0.shape == (0, 2) and ranges0.tolist() == [[0, 0], [0, 0]]


def test_python_argument_checks():
    """set_grid_maps checks its arguments before the library is called (a Batch without a device handle suffices)"""
    bt = tb.Batch.__new__(tb.Batch)
    bt.B, bt._h = 4, None
    H = np.zeros((3, 2), np.float32)
    with pytest.raises(AssertionError):
        bt.set_grid_maps([(H, 0.1, (0.0, 0.0))], map_of_instance=np.zeros(3, np.int32))   # one index per instance
    with pytest.raises(AssertionError):
        bt.set_grid_maps([(np.zeros(6, np.float32), 0.1, (0.0, 0.0))])                    # a layer is 2-D
    with pytest.raises(AssertionError):
        bt.footstep_contact_sets_per_instance(np.zeros((4, 1)), 2.0, [[]] * 3)             # one polygon list per instance


def test_null_batch_is_rejected():
    assert capi.lib.twb_batch_set_grid_maps(None, 0, None, None, None, None) == capi.ERR_INVALID


# ---- GPU ---------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", ["anymal_trot_block", "biped_walk_stairs"])
def test_per_instance_maps_against_the_oracle(name, record_property):
    """Five maps, random indices at a ragged B; every fourth instance is on TWB_SLOPE with a nonzero (ignored) map index.
    The oracle holds one map: map k is set and the instances on map k are compared (Biped: odd row length, interleaved tiles)."""
    rng = np.random.default_rng(41)
    maps = _five_maps(rng)
    B = 45
    terr = np.where(np.arange(B) % 4 == 3, tb.SLOPE, tb.GRID_MAP).astype(np.int32)
    idx = rng.permutation(np.arange(B) % 5).astype(np.int32)
    idx[terr == tb.SLOPE] = rng.integers(1, 5, int((terr == tb.SLOPE).sum()))
    spec = tb.make_formulation(name).to_spec(); p = tb.Problem(spec)
    X = synthetic_iterates(p, B)
    bt = p.batch(B); bt.set_terrains(terr); bt.set_grid_maps(maps, idx)
    out = bt.eval_host(X)
    assert not out["status"].any()
    rp = p.row_ptr()
    for k in range(5):
        sel = np.flatnonzero((idx == k) | (terr == tb.SLOPE)) if k == 0 else np.flatnonzero((idx == k) & (terr == tb.GRID_MAP))
        assert sel.size > 0
        oracle_lib.set_grid_map(*maps[k])
        ref = oracle_lib.batch_eval(spec, X[sel], terrain_ids=terr[sel])
        assert ref["rc"] == 0
        bad_j, strict_j, worst_j = check_rows(out["jac"][sel], ref["jac"], rp)
        bad_g, strict_g, worst_g = check_sets(out["g"][sel], ref["g"], p.constraint_sets())
        # worst error / tolerance and the fraction of entries that miss the bare 1e-12 / 1e-14 criterion, per map
        record_property(f"parity_map_{k}", {"B": int(sel.size), "res": maps[k][1], "size": list(maps[k][0].shape),
                                            "jac": {"violations": bad_j, "worst_err_over_tol": worst_j, "strict_miss_fraction": strict_j},
                                            "g": {"violations": bad_g, "worst_err_over_tol": worst_g, "strict_miss_fraction": strict_g}})
        assert bad_j == 0 and bad_g == 0, (k, bad_j, bad_g, worst_j, worst_g)
    # the instances really stand on different maps: one iterate evaluated on every map gives different terrain rows
    (_, r0, nr), = [c for c in p.constraint_sets() if c[0] == "terrain-ee-motion_0"]
    X5 = np.repeat(X[:1], 5, axis=0)
    b5 = p.batch(5); b5.set_terrains(np.full(5, tb.GRID_MAP, np.int32)); b5.set_grid_maps(maps, np.arange(5))
    g5 = b5.eval_host(X5)["g"][:, r0:r0 + nr]
    assert len({g5[k].tobytes() for k in range(5)}) == 5


def _eval_device(bt, X, p):
    import torch
    g = torch.empty((bt.B, p.m), dtype=torch.float64, device="cuda")
    jac = torch.empty((bt.B, p.nnz), dtype=torch.float64, device="cuda")
    status = torch.empty(bt.B, dtype=torch.int32, device="cuda")
    bt.eval_device(X, g=g, jac=jac, status=status)
    torch.cuda.synchronize()
    return g, jac, status


@pytest.mark.gpu
@pytest.mark.parametrize("B,path", [(4096, "device"), (10000, "device"), (4096, "host")])
def test_many_maps_equal_single_map_batches(B, path):
    """64 maps, every instance on TWB_GRID_MAP: each instance's rows equal, bit for bit, those of a batch that holds only its
    map (set_grid_map).  B = 10 000 walks 4096-instance chunks inside the graph; "host" is eval_host's 512-instance pipeline."""
    import torch
    rng = np.random.default_rng(B + len(path))
    maps = _many_maps(rng, 64)
    p = tb.Problem(tb.make_formulation("anymal_trot_block").to_spec())
    X = synthetic_iterates_fast(p, B, seed=B)
    idx = rng.integers(0, 64, B).astype(np.int32)
    allgrid = np.full(B, tb.GRID_MAP, np.int32)
    bt = p.batch(B); bt.set_terrains(allgrid); bt.set_grid_maps(maps, idx)
    single = p.batch(B); single.set_terrains(allgrid)
    if path == "device":
        Xd = torch.from_numpy(X).cuda()
        run = lambda b: _eval_device(b, Xd, p)
    else:
        run = lambda b: tuple(torch.from_numpy(b.eval_host(X)[k]) for k in ("g", "jac", "status"))
    g, jac, status = run(bt)
    assert not bool(status.any())
    for k in range(64):
        members = np.flatnonzero(idx == k)
        sample = torch.from_numpy(rng.choice(members, min(16, members.size), replace=False)).to(g.device)
        single.set_grid_map(*maps[k])
        g1, jac1, status1 = run(single)
        assert torch.equal(g[sample], g1[sample]) and torch.equal(jac[sample], jac1[sample]) and torch.equal(status[sample], status1[sample]), k


@pytest.mark.gpu
def test_single_map_call_is_the_one_map_set():
    """set_grid_map(H) and set_grid_maps([H]) give identical g, Jacobian and status (eval_host and eval_device)."""
    import torch
    rng = np.random.default_rng(43)
    H = _grid_map(rng, 60, 40, 0.1, (1.0, 0.0))
    B = 70
    terr = np.where(np.arange(B) % 3 == 2, tb.BLOCK, tb.GRID_MAP).astype(np.int32)
    p = tb.Problem(tb.make_formulation("anymal_trot_block").to_spec())
    X = synthetic_iterates(p, B)
    a = p.batch(B); a.set_terrains(terr); a.set_grid_map(*H)
    b = p.batch(B); b.set_terrains(terr); b.set_grid_maps([H])
    oa, ob = a.eval_host(X), b.eval_host(X)
    for key in ("g", "jac", "status"):
        assert np.array_equal(oa[key], ob[key]), key
    Xd = torch.from_numpy(X).cuda()
    assert all(torch.equal(u, v) for u, v in zip(_eval_device(a, Xd, p), _eval_device(b, Xd, p)))
    assert np.array_equal(_eval_device(a, Xd, p)[1].cpu().numpy(), oa["jac"])


@pytest.mark.gpu
def test_setter_semantics():
    """Either call order of set_terrains / set_grid_maps, replacing maps behind a cached graph, rejected calls that keep the
    previous maps, and removing the maps."""
    import torch
    rng = np.random.default_rng(44)
    maps = _five_maps(rng)
    B = 64
    terr = np.where(np.arange(B) % 4 == 3, tb.GAP, tb.GRID_MAP).astype(np.int32)
    idx = (np.arange(B) % 5).astype(np.int32)
    p = tb.Problem(tb.make_formulation("anymal_trot_block").to_spec())
    Xd = torch.from_numpy(synthetic_iterates(p, B)).cuda()
    a = p.batch(B); a.set_terrains(terr); a.set_grid_maps(maps, idx)
    b = p.batch(B); b.set_grid_maps(maps, idx); b.set_terrains(terr)
    ref = _eval_device(a, Xd, p)
    assert all(torch.equal(u, v) for u, v in zip(ref, _eval_device(b, Xd, p)))
    b.set_terrains(None); b.set_terrains(terr)          # the map indices survive a reset of the terrain ids
    assert all(torch.equal(u, v) for u, v in zip(ref, _eval_device(b, Xd, p)))

    # replacing the maps after a graph was captured: the results of a fresh batch
    other = [maps[k] for k in (4, 3, 2, 1, 0)]
    idx2 = ((np.arange(B) * 3) % 5).astype(np.int32)
    a.set_grid_maps(other, idx2)
    fresh = p.batch(B); fresh.set_terrains(terr); fresh.set_grid_maps(other, idx2)
    new = _eval_device(a, Xd, p)
    assert all(torch.equal(u, v) for u, v in zip(new, _eval_device(fresh, Xd, p)))
    assert not torch.equal(new[0], ref[0])

    # rejected calls keep the previous maps and indices
    bad_idx = idx2.copy(); bad_idx[7] = 5
    nan_pos = [(h, r, (np.nan, 0.0)) if k == 2 else (h, r, pos) for k, (h, r, pos) in enumerate(other)]
    zero_res = [(h, 0.0 if k == 1 else r, pos) for k, (h, r, pos) in enumerate(other)]
    for n_maps, mp, ix in ((5, other, bad_idx), (5, other, -idx2 - 1), (5, nan_pos, idx2), (5, zero_res, idx2), (-1, other, idx2),
                           ((1 << 27) + 1, other, idx2)):
        assert _set_maps_raw(a, n_maps, mp, ix) == capi.ERR_INVALID, n_maps
        assert all(torch.equal(u, v) for u, v in zip(new, _eval_device(a, Xd, p)))
    with pytest.raises(tb.TowrB200Error):
        a.set_grid_map(np.zeros((0, 3), np.float32), 0.1)
    assert all(torch.equal(u, v) for u, v in zip(new, _eval_device(a, Xd, p)))

    # removing the maps: TWB_GRID_MAP instances are outside the map everywhere (FLT_MAX heights), like a batch without maps
    a.set_grid_maps([])
    none = p.batch(B); none.set_terrains(terr)
    g0, _, _ = _eval_device(a, Xd, p)
    assert torch.equal(g0, _eval_device(none, Xd, p)[0])
    (_, r0, nr), = [c for c in p.constraint_sets() if c[0] == "terrain-ee-motion_0"]
    grid_rows = g0[torch.from_numpy(terr == tb.GRID_MAP).cuda(), r0:r0 + nr]
    assert bool((grid_rows < -1e30).all())
    a.set_grid_maps(other, idx2); a.set_grid_map(None, 1.0)  # a NULL single-map call removes every map too
    assert torch.equal(g0, _eval_device(a, Xd, p)[0])


@pytest.mark.gpu
def test_setup_kernels_read_each_instance_map():
    """goal_instances_device and state_instances_device: the goal z and the final footholds follow each instance's own map."""
    import torch
    from test_state_instances import _random_states
    rng = np.random.default_rng(45)
    maps = _five_maps(rng)
    f = tb.make_formulation("anymal_trot_block")
    p = tb.Problem(f.to_spec())
    nominal = np.array(tb.robot_info(tb.ANYMAL)["nominal_stance"])
    sets = {name: (s, k) for name, s, k in p.variable_sets()}
    s_lin, n_lin = sets["base-lin"]
    B = 35
    idx = (np.arange(B) % 5).astype(np.int32)
    bt = p.batch(B); bt.set_terrains(np.full(B, tb.GRID_MAP, np.int32)); bt.set_grid_maps(maps, idx)
    S = _random_states(f, rng, B)
    S[:, 12] = rng.uniform(0.5, 2.0, B); S[:, 13] = rng.uniform(-0.5, 0.5, B)
    goals = np.concatenate([S[:, 12:15], S[:, 18:21]], axis=1)
    x_state = bt.state_instances_device(torch.from_numpy(S).cuda(), want_bounds=False)[0].cpu().numpy()
    x_goal = bt.goal_instances_device(torch.from_numpy(goals).cuda(), want_bounds=False)[0].cpu().numpy()
    for k in range(5):
        oracle_lib.set_grid_map(*maps[k])
        for b in np.flatnonzero(idx == k):
            h = oracle_lib.terrain_point(tb.GRID_MAP, S[b, 12], S[b, 13])[0]
            yaw = S[b, 20]
            for x0 in (x_state, x_goal):
                assert abs(x0[b, s_lin + n_lin - 6 + 2] - (h - nominal[0][2])) < 1e-6, (k, b)
                for e in range(len(nominal)):
                    s_e, k_e = sets[f"ee-motion_{e}"]
                    w = S[b, 12:14] + np.array([[np.cos(yaw), -np.sin(yaw)], [np.sin(yaw), np.cos(yaw)]]) @ nominal[e][:2]
                    assert abs(x0[b, s_e + k_e - 1] - oracle_lib.terrain_point(tb.GRID_MAP, w[0], w[1])[0]) < 1e-6, (k, b, e)
    assert len({round(float(x_state[b, s_lin + n_lin - 4]), 9) for b in range(5)}) > 1     # the maps show


def _polygon_sets(rng, count):
    """`count` planar-region sets: squares and a triangle scattered over the plans' footholds, one set empty"""
    sets = []
    for i in range(count):
        if i == 1:
            sets.append([]); continue
        polys = []
        for _ in range(int(rng.integers(1, 6))):
            x0, y0, w, h = rng.uniform(-0.5, 2.5), rng.uniform(-0.8, 0.3), rng.uniform(0.2, 1.2), rng.uniform(0.2, 0.8)
            polys.append(np.array([[x0, y0], [x0, y0 + h], [x0 + w, y0 + h], [x0 + w, y0], [x0, y0]]))
        if i % 3 == 0:
            polys.append(np.array([[2.5, 0.0], [3.0, 0.8], [3.5, 0.0], [2.5, 0.0]]))
        sets.append(polys)
    return sets


def _plans(bt, p, seed):
    import torch
    Xd = torch.from_numpy(synthetic_iterates(p, bt.B, seed=seed)).cuda()
    plans, count = bt.footstep_plans_device(Xd, 2.0)
    torch.cuda.synchronize()
    return plans, count


@pytest.mark.gpu
def test_nearest_planes_by_range():
    """_ranges_device and _ranges_host equal the shared-list call run on each instance's own polygon list; empty ranges give
    -1; device ranges outside the list are clamped; a graph captured on a side stream replays; argument errors."""
    import torch
    rng = np.random.default_rng(46)
    p = tb.Problem(tb.make_formulation("anymal_trot_block").to_spec())
    B = 40
    bt = p.batch(B)
    plans, count = _plans(bt, p, 46)
    sets = _polygon_sets(rng, 6)
    per_instance = [sets[b % 6] for b in range(B)]
    offs, verts, ranges = tb.pack_polygon_sets(per_instance)
    od, vd, rd = (torch.from_numpy(a).cuda() for a in (offs, verts, ranges))
    cs_dev = bt.nearest_planes_ranges_device(plans, count, rd, od, vd)
    torch.cuda.synchronize()
    cs_dev = cs_dev.cpu().numpy()
    ph, ch = plans.cpu().numpy(), count.cpu().numpy()
    ms, nv = bt.footstep_plan_dims()
    cs_host = np.full((B, ms, (nv - 2) // 4), -7, np.int32)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    capi.check(capi.lib.twb_batch_nearest_planes_ranges_host(bt._h, ptr(ph), ptr(ch), ptr(ranges), ptr(offs), len(offs) - 1, ptr(verts), ptr(cs_host)))
    assert np.array_equal(cs_dev, cs_host)
    for s in range(6):
        o1, v1 = tb.pack_polygons(sets[s])
        ref = np.full_like(cs_host, -7)
        capi.check(capi.lib.twb_batch_nearest_planes_host(bt._h, ptr(ph), ptr(ch), ptr(o1), len(o1) - 1, ptr(v1), ptr(ref)))
        members = np.arange(s, B, 6)
        assert np.array_equal(cs_host[members], ref[members]), s
    assert (cs_host[np.arange(1, B, 6)] == -1).all()                 # the empty set
    assert cs_host.max() > 0 and (cs_host >= 0).any()

    # the Python wrapper of the host path
    plans_l, sets_l = bt.footstep_contact_sets_per_instance(synthetic_iterates(p, B, seed=46), 2.0, per_instance)
    assert all(np.array_equal(sets_l[b], cs_host[b, :ch[b]]) for b in range(B))

    # device ranges outside the list are clamped to it; the index counts from the clamped first polygon
    n_polys = len(offs) - 1
    wild = ranges.copy()
    wild[0] = (-3, 5); wild[2] = (n_polys - 2, 10); wild[3] = (n_polys + 5, 2); wild[4] = (-10, 3); wild[5] = (4, -2)
    clamped = wild.astype(np.int64)
    lo = np.clip(clamped[:, 0], 0, n_polys); hi = np.clip(clamped[:, 0] + clamped[:, 1], lo, n_polys)
    clamped = np.stack([lo, hi - lo], axis=1).astype(np.int32)
    cs_wild = bt.nearest_planes_ranges_device(plans, count, torch.from_numpy(wild).cuda(), od, vd).cpu().numpy()
    ref = np.full_like(cs_host, -7)
    capi.check(capi.lib.twb_batch_nearest_planes_ranges_host(bt._h, ptr(ph), ptr(ch), ptr(clamped), ptr(offs), n_polys, ptr(verts), ptr(ref)))
    assert np.array_equal(cs_wild, ref)
    assert (cs_wild[[3, 4, 5]] == -1).all()

    # one graph capture on a non-default stream, replayed for two plan sets
    plans2, count2 = _plans(bt, p, 47)
    direct = [bt.nearest_planes_ranges_device(pl, c, rd, od, vd).clone() for pl, c in ((plans, count), (plans2, count2))]
    pin, cin = torch.empty_like(plans), torch.empty_like(count)
    out = torch.empty_like(direct[0])
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        bt.nearest_planes_ranges_device(pin, cin, rd, od, vd, out=out, stream=side)
    for (pl, c), d in zip(((plans, count), (plans2, count2)), direct):
        pin.copy_(pl); cin.copy_(c)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, d)
    assert not torch.equal(direct[0], direct[1])

    # argument errors
    lib, v = capi.lib, lambda t: C.c_void_p(t.data_ptr())
    h = bt._h
    for rc in (lib.twb_batch_nearest_planes_ranges_device(h, v(plans), v(count), None, v(od), n_polys, v(vd), v(out), None),
               lib.twb_batch_nearest_planes_ranges_device(h, v(plans), v(count), v(rd), v(od), -1, v(vd), v(out), None),
               lib.twb_batch_nearest_planes_ranges_device(h, None, v(count), v(rd), v(od), n_polys, v(vd), v(out), None),
               lib.twb_batch_nearest_planes_ranges_host(h, ptr(ph), ptr(ch), None, ptr(offs), n_polys, ptr(verts), ptr(cs_host))):
        assert rc == capi.ERR_INVALID
    for bad in ((-1, 1), (0, -1), (n_polys - 1, 2)):
        r = ranges.copy(); r[9] = bad
        assert lib.twb_batch_nearest_planes_ranges_host(h, ptr(ph), ptr(ch), ptr(r), ptr(offs), n_polys, ptr(verts), ptr(cs_host)) == capi.ERR_INVALID


@pytest.mark.gpu
def test_pipeline_with_per_instance_states_and_maps():
    """4096 Anymal instances, each with its own start state and map: state setup, 8 Levenberg-Marquardt iterations, footstep
    plans, contact sets by range.  Every instance's iterates, plans and contact sets equal, bit for bit, those of the same
    pipeline on a batch that holds only that instance's map."""
    import torch
    from towr_b200.solver import BatchedLevenbergMarquardt
    from test_state_instances import _random_states
    f = tb.make_formulation("anymal_trot_block")
    p = tb.Problem(f.to_spec())
    B, iters, n_maps = 4096, 8, 16
    rng = np.random.default_rng(47)
    maps = _many_maps(rng, n_maps)
    idx = rng.integers(0, n_maps, B).astype(np.int32)
    S = _random_states(f, rng, B)
    S[:, 12] = rng.uniform(0.5, 2.0, B); S[:, 13] = rng.uniform(-0.5, 0.5, B)
    Sd = torch.from_numpy(S).cuda()
    noise = torch.from_numpy(0.01 * rng.standard_normal((B, p.n))).cuda()
    sets = _polygon_sets(rng, 7)
    offs, verts, ranges = tb.pack_polygon_sets([sets[b % 7] for b in range(B)])
    od, vd, rd = (torch.from_numpy(a).cuda() for a in (offs, verts, ranges))
    allgrid = np.full(B, tb.GRID_MAP, np.int32)

    def pipeline(bt):
        x0, xl, xu, _, _ = bt.state_instances_device(Sd)
        X = torch.minimum(torch.maximum(x0 + noise, xl), xu)
        lm = BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu)
        for _ in range(iters):
            lm.step(X)
        plans, count = bt.footstep_plans_device(X, 2.0)
        cs = bt.nearest_planes_ranges_device(plans, count, rd, od, vd)
        torch.cuda.synchronize()
        return X, plans, count, cs, lm.status.clone()

    bt = p.batch(B); bt.set_terrains(allgrid); bt.set_grid_maps(maps, idx)
    X, plans, count, cs, status = pipeline(bt)
    assert torch.isfinite(X).all() and not bool(status.any())
    single = p.batch(B); single.set_terrains(allgrid)
    for k in range(n_maps):
        single.set_grid_map(*maps[k])
        X1, plans1, count1, cs1, _ = pipeline(single)
        m = torch.from_numpy(np.flatnonzero(idx == k)).cuda()
        assert torch.equal(X[m], X1[m]), k
        assert torch.equal(plans[m], plans1[m]) and torch.equal(count[m], count1[m]) and torch.equal(cs[m], cs1[m]), k
    assert (cs >= 0).any()
