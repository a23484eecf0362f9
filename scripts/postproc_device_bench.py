"""Times the fpowr post-processing calls on one GPU: the four device-pointer calls (CUDA events, one pair per call), the
host-pointer calls end to end (host clock; each call ends in its own synchronise), and the footstep plan of an older build
of the library (--parent-lib: the trajectory kernel + one-thread-per-instance scan pair) against the fused kernel,
alternating old and new in the same process.  Workloads: Anymal trot / Block at B = 4096 and the config-5 recipe (Anymal
trot, mixed Slope / Chimney / Gap terrains) at B = 65 536.  Kernel times come from a separate torch.profiler pass.

    python scripts/postproc_device_bench.py --out-dir DIR [--parent-lib path/to/old/libtowr_b200.so]

Writes <out-dir>/postproc_device_n1.json (the committed copy: profiles/postproc_device_n1.json).  Needs a CUDA device."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import towr_b200 as tb  # noqa: E402
from towr_b200.configs import synthetic_iterates_fast  # noqa: E402
from bench import read_peak  # noqa: E402

HORIZON = 2.0
IG_TIMES = np.linspace(0.0, 2.0, 41)
WORKLOADS = [   # (label, recipe, B, trajectory dt, per-instance terrains)
    ("anymal_trot_block_4096", "anymal_trot_block", 4096, 0.01, False),
    ("config5_anymal_trot_mixed_65536", "anymal_trot_mixed", 65536, 0.05, True),
]


def stepping_stones():
    """32 closed 0.5 m squares over x in [-1, 3], y in [-1, 1]"""
    polys = []
    for i in range(8):
        for j in range(4):
            x0, y0 = -1.0 + 0.5 * i, -1.0 + 0.5 * j
            polys.append(np.array([[x0, y0], [x0 + 0.5, y0], [x0 + 0.5, y0 + 0.5], [x0, y0 + 0.5], [x0, y0]]))
    return polys


def stats(us):
    us = np.asarray(us)
    return {"median_us": float(np.median(us)), "mean_us": float(us.mean()), "min_us": float(us.min()), "max_us": float(us.max()), "calls": int(us.size)}


def time_device(fn, warmup, iters, stream):
    """CUDA events around each call on `stream`"""
    for _ in range(warmup):
        fn()
    stream.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        a.record(stream)
        fn()
        b.record(stream)
    stream.synchronize()
    return stats([1e3 * a.elapsed_time(b) for a, b in ev])


def time_host(fn, warmup, iters):
    """host clock around each call (the host-pointer calls synchronise before they return)"""
    for _ in range(warmup):
        fn()
    us = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        us.append(1e6 * (time.perf_counter() - t0))
    return stats(us)


class OldLibrary:
    """An older build of libtowr_b200.so loaded next to the current one: its own problem and batch of the same spec"""

    def __init__(self, path, spec, B):
        self.lib = L = C.CDLL(os.path.abspath(path))
        P = C.c_void_p
        L.twb_problem_create.argtypes = [C.POINTER(tb.capi.Spec), C.POINTER(P)]
        L.twb_batch_create.argtypes = [P, C.c_int, C.c_int, C.POINTER(P)]
        L.twb_batch_footstep_plan_host.argtypes = [P, P, C.c_double, P, P]
        L.twb_batch_destroy.argtypes = [P]
        L.twb_problem_destroy.argtypes = [P]
        self.p, self.b = P(), P()
        assert L.twb_problem_create(C.byref(spec), C.byref(self.p)) == 0
        assert L.twb_batch_create(self.p, B, 0, C.byref(self.b)) == 0

    def footstep_plan_host(self, X, count, out):
        assert self.lib.twb_batch_footstep_plan_host(self.b, X.ctypes.data_as(C.c_void_p), HORIZON, count.ctypes.data_as(C.c_void_p),
                                                     out.ctypes.data_as(C.c_void_p)) == 0

    def close(self):
        self.lib.twb_batch_destroy(self.b)
        self.lib.twb_problem_destroy(self.p)


def host_plans(bt, X, count, out):
    tb.capi.check(tb.capi.lib.twb_batch_footstep_plan_host(bt._h, X.ctypes.data_as(C.c_void_p), HORIZON, count.ctypes.data_as(C.c_void_p),
                                                           out.ctypes.data_as(C.c_void_p)))


def profile_kernels(calls, stream, reps):
    """device time per kernel name (torch.profiler, CUDA activities), averaged over its launches"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            for fn in calls:
                fn()
        stream.synchronize()
    out = {}
    for e in prof.key_averages():
        total = getattr(e, "device_time_total", None)
        if total is None:
            total = e.cuda_time_total
        if total > 0 and e.count > 0 and "Memcpy" not in e.key and "Memset" not in e.key:
            out[e.key] = {"avg_us": total / e.count, "launches": e.count}
    return out


def run_workload(label, recipe, B, dt, mixed, args, hbm_gbs):
    spec = tb.make_formulation(recipe).to_spec()
    p = tb.Problem(spec)
    bt = p.batch(B)
    if mixed:
        bt.set_terrains(np.array([tb.SLOPE, tb.CHIMNEY, tb.GAP] * (B // 3 + 1), np.int32)[:B])
    X = np.ascontiguousarray(synthetic_iterates_fast(p, B, seed=3))
    ms, V = bt.footstep_plan_dims()
    n_ee = (V - 2) // 4
    polys = stepping_stones()
    offs, verts = tb.pack_polygons(polys)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        xd = torch.from_numpy(X).cuda()
        offs_d, verts_d = torch.from_numpy(offs).cuda(), torch.from_numpy(verts).cuda()
        traj = bt.sample_trajectory_device(xd, dt, stream=s)
        ig = bt.initial_guesses_device(xd, IG_TIMES, stream=s)
        plans, count = bt.footstep_plans_device(xd, HORIZON, stream=s)
        cs = bt.nearest_planes_device(plans, count, offs_d, verts_d, stream=s)
    s.synchronize()
    calls = {
        "sample_trajectory": lambda: bt.sample_trajectory_device(xd, dt, out=traj, stream=s),
        "initial_guesses": lambda: bt.initial_guesses_device(xd, IG_TIMES, out=ig, stream=s),
        "footstep_plans": lambda: bt.footstep_plans_device(xd, HORIZON, out=(plans, count), stream=s),
        "nearest_planes": lambda: bt.nearest_planes_device(plans, count, offs_d, verts_d, out=cs, stream=s),
    }
    res = {"recipe": recipe, "B": B, "n": p.n, "trajectory_dt": dt, "trajectory_samples": int(traj.shape[1]),
           "initial_guess_times": int(IG_TIMES.size), "max_states": ms, "n_values": V, "polygons": len(polys),
           "n_states": sorted(set(count.cpu().numpy().tolist()))}
    res["device_calls"] = {k: time_device(fn, args.warmup, args.iters, s) for k, fn in calls.items()}

    # host-pointer variants end to end: H2D of x (pageable), kernels, D2H, synchronise
    h_traj = np.empty(tuple(traj.shape)); h_ig = np.empty(tuple(ig.shape))
    h_plans = np.empty((B, ms, V)); h_count = np.empty(B, np.int32); h_cs = np.empty((B, ms, n_ee), np.int32)
    L, ptr = tb.capi.lib, lambda a: a.ctypes.data_as(C.c_void_p)
    host = {
        "sample_trajectory": lambda: tb.capi.check(L.twb_batch_sample_trajectory_host(bt._h, ptr(X), dt, ptr(h_traj))),
        "initial_guesses": lambda: tb.capi.check(L.twb_batch_initial_guess_host(bt._h, ptr(X), ptr(IG_TIMES), IG_TIMES.size, ptr(h_ig))),
        "footstep_plans": lambda: host_plans(bt, X, h_count, h_plans),
        "nearest_planes": lambda: tb.capi.check(L.twb_batch_nearest_planes_host(bt._h, ptr(h_plans), ptr(h_count), ptr(offs), len(polys),
                                                                                ptr(verts), ptr(h_cs))),
    }
    res["host_calls"] = {k: time_host(fn, 2, args.iters) for k, fn in host.items()}
    res["device_equals_host"] = bool(np.array_equal(plans.cpu().numpy(), h_plans) and np.array_equal(count.cpu().numpy(), h_count)
                                     and np.array_equal(cs.cpu().numpy(), h_cs) and np.array_equal(traj.cpu().numpy(), h_traj)
                                     and np.array_equal(ig.cpu().numpy(), h_ig))

    if args.parent_lib:   # footstep plan, host path: the older build's kernel pair against the fused kernel, alternating
        old = OldLibrary(args.parent_lib, spec, B)
        o_plans = np.zeros((B, ms, V)); o_count = np.empty(B, np.int32)
        n_plans = np.zeros((B, ms, V)); n_count = np.empty(B, np.int32)
        old.footstep_plan_host(X, o_count, o_plans); host_plans(bt, X, n_count, n_plans)
        t_old, t_new = [], []
        for _ in range(args.iters):
            for fn, acc in ((lambda: old.footstep_plan_host(X, o_count, o_plans), t_old), (lambda: host_plans(bt, X, n_count, n_plans), t_new)):
                t0 = time.perf_counter(); fn(); acc.append(1e6 * (time.perf_counter() - t0))
        res["footstep_host_old_vs_new"] = {"old_pair": stats(t_old), "fused": stats(t_new),
                                           "identical_outputs": bool(np.array_equal(o_plans, n_plans) and np.array_equal(o_count, n_count))}
        old.close()

    # kernel times, profiler on (a separate pass)
    kern = profile_kernels(list(calls.values()), s, 20)
    res["kernels"] = kern
    fused = [v for k, v in kern.items() if "FootstepPlanKernel" in k]
    if fused:
        t_us = fused[0]["avg_us"]
        nbytes = B * (8 * p.n + 8 * ms * V + 4)
        res["fused_footstep_kernel"] = {"avg_us": t_us, "algorithmic_bytes": nbytes, "bytes_per_instance": {"read": 8 * p.n, "written": 8 * ms * V + 4},
                                        "achieved_gbs": nbytes / (t_us * 1e-6) / 1e9, "fraction_of_hbm": nbytes / (t_us * 1e-6) / (hbm_gbs * 1e9)}
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--parent-lib", default=None, help="an older build of libtowr_b200.so to time the footstep plan against")
    ap.add_argument("--parent-label", default="older build", help="what --parent-lib was built from (recorded in the JSON)")
    ap.add_argument("--out-dir", required=True, help="directory that receives postproc_device_n1.json")
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--only", default=None, help="run one workload label")
    args = ap.parse_args()
    assert args.iters >= 20
    if not torch.cuda.is_available():
        sys.exit("postproc_device_bench: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    hbm_gbs, hbm_src = read_peak()
    result = {"gpu": smi.stdout.strip(), "hbm_gbs": hbm_gbs, "hbm_source": hbm_src, "iters": args.iters, "warmup": args.warmup,
              "parent_lib": args.parent_label if args.parent_lib else None, "workloads": {}}
    for label, recipe, B, dt, mixed in WORKLOADS:
        if args.only and label != args.only:
            continue
        result["workloads"][label] = run_workload(label, recipe, B, dt, mixed, args, hbm_gbs)
        torch.cuda.empty_cache()
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "postproc_device_n1.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
