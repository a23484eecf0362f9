"""Times the evaluation step (g + Jacobian, twb_batch_eval_device) of Anymal trot on per-instance grid_map terrains, one GPU,
CUDA events around every step, median, the iterates rotating over 8 sets as in bench.py (so that inputs and outputs exceed
the 126 MB L2), at B = 4096 and B = 65 536:
  (a) every instance on the analytic Block terrain (the bench.py workload);
  (b) every instance on one shared 160 x 160 map at 0.03 m (twb_batch_set_grid_map);
  (c) every instance on its own 160 x 160 map at 0.03 m (twb_batch_set_grid_maps: 4096 / 65 536 maps, 420 MB / 6.7 GB);
and (d) the nearest-plane lookup by ranges (twb_batch_nearest_planes_ranges_device) against the shared-list call, at the
sizes of postproc_device_bench.py: every range pointing at the one shared list of 32 stepping stones, and every instance
with its own copy of them.  --profile adds a torch.profiler pass over (b) and (c) (kernel times; a separate pass).

    python scripts/grid_maps_bench.py --out-dir DIR [--profile]
    python scripts/grid_maps_bench.py --out-dir DIR --package-root OTHER_TREE --sections ab --tag parent

--package-root imports towr_b200 from another checkout (e.g. the parent commit, built) to time (a) and (b) with the same
script.  Writes <out-dir>/grid_maps_n1<tag>.json (the committed copy: profiles/grid_maps_n1.json).  Needs a CUDA device."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

RECIPE = "anymal_trot_block"
SIZES = (4096, 65536)
N_SETS = 8
MAP = (160, 160, 0.03, (1.0, 0.0))   # size_x, size_y, resolution, position: 4.8 m x 4.8 m around the iterates' feet


def time_steps(fn, warmup, iters, stream):
    """median of CUDA events around each call of fn(i) on `stream`, in microseconds"""
    import numpy as np
    import torch
    for i in range(warmup):
        fn(i)
    stream.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for i, (a, b) in enumerate(ev):
        a.record(stream)
        fn(i)
        b.record(stream)
    stream.synchronize()
    us = np.array([1e3 * a.elapsed_time(b) for a, b in ev])
    return {"median_us": float(np.median(us)), "min_us": float(us.min()), "max_us": float(us.max()), "calls": int(us.size)}


def base_map(seed):
    import numpy as np
    sx, sy, res, pos = MAP
    rng = np.random.default_rng(seed)
    xs = pos[0] + sx * res / 2 - res / 2 - res * np.arange(sx)
    ys = pos[1] + sy * res / 2 - res / 2 - res * np.arange(sy)
    return (0.15 * np.sin(2.0 * xs)[:, None] * np.cos(1.5 * ys)[None, :] + 0.02 * rng.standard_normal((sx, sy))).astype(np.float32)


def set_own_maps(tb, bt, B):
    """B maps of MAP's geometry, map b = the base layer + 0.001 b m, instance b on map b (one contiguous host array)"""
    import numpy as np
    sx, sy, res, pos = MAP
    heights = np.empty((B, sx, sy), np.float32)
    heights[:] = base_map(1)
    heights += (0.001 * np.arange(B, dtype=np.float32))[:, None, None]
    sizes = np.tile(np.array([sx, sy], np.int32), (B, 1))
    geometry = np.tile(np.array([res, pos[0], pos[1]], np.float64), (B, 1))
    idx = np.arange(B, dtype=np.int32)
    tb.capi.check(tb.capi.lib.twb_batch_set_grid_maps(bt._h, B, heights.ctypes.data_as(C.POINTER(C.c_float)), sizes.ctypes.data_as(C.POINTER(C.c_int)),
                                                      geometry.ctypes.data_as(C.POINTER(C.c_double)), idx.ctypes.data_as(C.POINTER(C.c_int))))
    return heights.nbytes


def eval_cases(tb, p, B, sections, args):
    import numpy as np
    import torch
    from towr_b200.configs import synthetic_iterates_fast
    dev = torch.device("cuda", 0)
    s = torch.cuda.Stream()
    Xs = [torch.from_numpy(synthetic_iterates_fast(p, B, seed=100 + k)).to(dev) for k in range(N_SETS)]
    g = torch.empty((B, p.m), dtype=torch.float64, device=dev)
    jac = torch.empty((B, p.nnz), dtype=torch.float64, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    res, profiled = {}, {}
    iters = args.iters if B <= 4096 else max(20, args.iters // 4)
    for case in sections:
        if case not in "abc":
            continue
        bt = p.batch(B)
        map_bytes = 0
        if case in "bc":
            bt.set_terrains(np.full(B, tb.GRID_MAP, np.int32))
        if case == "b":
            sx, sy, res_m, pos = MAP
            bt.set_grid_map(base_map(1), res_m, pos); map_bytes = 4 * sx * sy
        if case == "c":
            map_bytes = set_own_maps(tb, bt, B)
        step = lambda i: bt.eval_device(Xs[i % N_SETS], g=g, jac=jac, status=status, stream=s)
        t = time_steps(step, max(args.warmup, N_SETS), iters, s)
        t.update({"evals_per_s": B / (t["median_us"] * 1e-6), "map_bytes": map_bytes, "status_clear": not bool(status.any())})
        res[case] = t
        if args.profile and case in "bc":
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for i in range(3 * N_SETS):
                    step(i)
                s.synchronize()
            kern = {}
            for e in prof.key_averages():
                total = getattr(e, "device_time_total", None)
                if total is None:
                    total = e.cuda_time_total
                if total > 0 and e.count > 0:
                    kern[e.key[:120]] = {"avg_us": total / e.count, "launches": e.count}
            profiled[case] = kern
        del bt
        torch.cuda.empty_cache()
    if "a" in res and "b" in res:
        res["b_over_a"] = res["b"]["median_us"] / res["a"]["median_us"]
    if "b" in res and "c" in res:
        res["c_over_b"] = res["c"]["median_us"] / res["b"]["median_us"]
    if profiled:
        res["profile"] = profiled
    return res


def stepping_stones():
    """the 32 closed 0.5 m squares of postproc_device_bench.py"""
    import numpy as np
    polys = []
    for i in range(8):
        for j in range(4):
            x0, y0 = -1.0 + 0.5 * i, -1.0 + 0.5 * j
            polys.append(np.array([[x0, y0], [x0 + 0.5, y0], [x0 + 0.5, y0 + 0.5], [x0, y0 + 0.5], [x0, y0]]))
    return polys


def nearest_planes_case(tb, label, recipe, B, mixed, args):
    import numpy as np
    import torch
    from towr_b200.configs import synthetic_iterates_fast
    p = tb.Problem(tb.make_formulation(recipe).to_spec())
    bt = p.batch(B)
    if mixed:
        bt.set_terrains(np.array([tb.SLOPE, tb.CHIMNEY, tb.GAP] * (B // 3 + 1), np.int32)[:B])
    s = torch.cuda.Stream()
    polys = stepping_stones()
    with torch.cuda.stream(s):
        xd = torch.from_numpy(synthetic_iterates_fast(p, B, seed=3)).cuda()
        plans, count = bt.footstep_plans_device(xd, 2.0, stream=s)
        offs, verts = (torch.from_numpy(a).cuda() for a in tb.pack_polygons(polys))
        shared_ranges = torch.tensor([[0, len(polys)]] * B, dtype=torch.int32).cuda()
        o2, v2, r2 = (torch.from_numpy(a).cuda() for a in tb.pack_polygon_sets([polys] * B))
        cs = bt.nearest_planes_device(plans, count, offs, verts, stream=s)
        cs_r = torch.empty_like(cs); cs_own = torch.empty_like(cs)
    s.synchronize()
    calls = {
        "shared_list": lambda i: bt.nearest_planes_device(plans, count, offs, verts, out=cs, stream=s),
        "ranges_into_shared_list": lambda i: bt.nearest_planes_ranges_device(plans, count, shared_ranges, offs, verts, out=cs_r, stream=s),
        "ranges_own_copy_per_instance": lambda i: bt.nearest_planes_ranges_device(plans, count, r2, o2, v2, out=cs_own, stream=s),
    }
    res = {"label": label, "recipe": recipe, "B": B, "polygons_per_instance": len(polys),
           "own_copy_vertex_bytes": int(v2.numel() * 8)}
    for k, fn in calls.items():
        res[k] = time_steps(fn, args.warmup, args.iters, s)
    res["identical_contact_sets"] = bool(torch.equal(cs, cs_r) and torch.equal(cs, cs_own))
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out-dir", required=True, help="directory that receives grid_maps_n1<tag>.json")
    ap.add_argument("--sections", default="abcd", help="which of (a) .. (d) to run")
    ap.add_argument("--package-root", default=ROOT, help="checkout whose towr_b200 is imported (default: this one)")
    ap.add_argument("--tag", default="", help="suffix of the output file name")
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--profile", action="store_true", help="add a torch.profiler pass over (b) and (c)")
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.package_root))
    import torch
    import towr_b200 as tb
    if not torch.cuda.is_available():
        sys.exit("grid_maps_bench: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    p = tb.Problem(tb.make_formulation(RECIPE).to_spec())
    result = {"gpu": smi.stdout.strip(), "package": tb.__file__, "recipe": RECIPE, "n": p.n, "m": p.m, "nnz": p.nnz,
              "map": {"size": list(MAP[:2]), "resolution": MAP[2], "position": list(MAP[3])}, "iterate_sets": N_SETS,
              "timing": "CUDA events around every eval_device step on one stream (graph replay), median", "eval": {}}
    for B in SIZES:
        result["eval"][str(B)] = eval_cases(tb, p, B, args.sections, args)
    if "d" in args.sections:
        result["nearest_planes"] = [nearest_planes_case(tb, "anymal_trot_block_4096", "anymal_trot_block", 4096, False, args),
                                    nearest_planes_case(tb, "config5_anymal_trot_mixed_65536", "anymal_trot_mixed", 65536, True, args)]
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, f"grid_maps_n1{args.tag}.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
