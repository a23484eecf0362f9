"""Times twb_batch_state_instances_device (per-instance start states: x0, variable bounds and, optionally, constraint bounds
for every instance of a batch) on one GPU with CUDA events, for Anymal trot / Block at B = 4096 and B = 65 536, with and
without the constraint bounds; twb_batch_goal_instances_device (x0 and variable bounds from goals only) is timed next to
it.  The achieved bandwidth counts the bytes the call must write: 3 * 8 * n per instance for x0 and the variable bounds,
plus 2 * 8 * m for the constraint bounds (the reads, 288 bytes of state record per instance and the per-problem tables,
are left out).  At B = 4096 the outputs (about 60 / 120 MB) fit the 126 MB L2, at B = 65 536 they do not.

    python scripts/state_instances_bench.py --out-dir DIR

Writes <out-dir>/state_instances_n1.json (the committed copy: profiles/state_instances_n1.json).  Needs a CUDA device."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import towr_b200 as tb  # noqa: E402
from bench import read_peak  # noqa: E402

RECIPE = "anymal_trot_block"
SIZES = (4096, 65536)


def random_states(f, B, seed):
    """B state records around the recipe's own (the distribution of tests/test_state_instances.py)"""
    rng = np.random.default_rng(seed)
    S = np.tile(f.state_record(), (B, 1))
    n_ee = len(f.initial_ee_W_)
    S[:, 0:2] += rng.uniform(-0.3, 0.3, (B, 2)); S[:, 2] += rng.uniform(-0.05, 0.05, B)
    S[:, 3:12] = rng.uniform(-0.3, 0.3, (B, 9))
    S[:, 12:14] += rng.uniform(-0.5, 0.5, (B, 2)); S[:, 14] += rng.uniform(-0.05, 0.05, B)
    S[:, 15:24] = rng.uniform(-0.3, 0.3, (B, 9))
    S[:, 24:24 + 3 * n_ee] += rng.uniform(-0.05, 0.05, (B, 3 * n_ee))
    return S


def time_events(fn, warmup, iters, stream):
    """median of CUDA events around each call on `stream`, in microseconds"""
    for _ in range(warmup):
        fn()
    stream.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        a.record(stream)
        fn()
        b.record(stream)
    stream.synchronize()
    us = np.array([1e3 * a.elapsed_time(b) for a, b in ev])
    return {"median_us": float(np.median(us)), "min_us": float(us.min()), "max_us": float(us.max()), "calls": int(us.size)}


def run_size(p, f, B, args, hbm_gbs):
    L = tb.capi.lib
    bt = p.batch(B)
    dev = torch.device("cuda", 0)
    states = torch.from_numpy(random_states(f, B, seed=B)).to(dev)
    goals = states[:, [12, 13, 14, 18, 19, 20]].contiguous()
    x0, lo, up = (torch.empty((B, p.n), dtype=torch.float64, device=dev) for _ in range(3))
    gl, gu = (torch.empty((B, p.m), dtype=torch.float64, device=dev) for _ in range(2))
    s = torch.cuda.Stream()
    ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    sp = C.c_void_p(s.cuda_stream)
    calls = {
        "state_instances": (lambda: tb.capi.check(L.twb_batch_state_instances_device(bt._h, ptr(states), ptr(x0), ptr(lo), ptr(up), None, None, sp)),
                            3 * 8 * p.n),
        "state_instances_with_g_bounds": (lambda: tb.capi.check(L.twb_batch_state_instances_device(bt._h, ptr(states), ptr(x0), ptr(lo), ptr(up), ptr(gl),
                                                                                                   ptr(gu), sp)),
                                          3 * 8 * p.n + 2 * 8 * p.m),
        "goal_instances": (lambda: tb.capi.check(L.twb_batch_goal_instances_device(bt._h, ptr(goals), ptr(x0), ptr(lo), ptr(up), sp)), 3 * 8 * p.n),
    }
    res = {"B": B}
    for name, (fn, per_instance) in calls.items():
        t = time_events(fn, args.warmup, args.iters, s)
        nbytes = B * per_instance
        t.update({"bytes_written": nbytes, "bytes_written_per_instance": per_instance, "achieved_gbs": nbytes / (t["median_us"] * 1e-6) / 1e9,
                  "fraction_of_hbm": nbytes / (t["median_us"] * 1e-6) / (hbm_gbs * 1e9)})
        res[name] = t
    # the timed outputs are the host builder's (spot check of 16 instances)
    L.twb_batch_state_instances_device(bt._h, ptr(states), ptr(x0), ptr(lo), ptr(up), ptr(gl), ptr(gu), sp)
    s.synchronize()
    pick = np.linspace(0, B - 1, 16).astype(int)
    hx0, hxl, hxu, hgl, hgu = p.state_instances(states[pick].cpu().numpy())
    res["spot_check_16_vs_host"] = bool(np.allclose(x0[pick].cpu().numpy(), hx0, rtol=1e-14, atol=1e-15)
                                        and np.allclose(lo[pick].cpu().numpy(), hxl, rtol=1e-14, atol=0)
                                        and np.array_equal(gl[pick].cpu().numpy(), hgl) and np.array_equal(gu[pick].cpu().numpy(), hgu))
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out-dir", required=True, help="directory that receives state_instances_n1.json")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("state_instances_bench: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    hbm_gbs, hbm_src = read_peak()
    f = tb.make_formulation(RECIPE)
    p = tb.Problem(f.to_spec())
    result = {"gpu": smi.stdout.strip(), "hbm_gbs": hbm_gbs, "hbm_source": hbm_src, "recipe": RECIPE, "n": p.n, "m": p.m,
              "iters": args.iters, "warmup": args.warmup, "sizes": {}}
    for B in SIZES:
        result["sizes"][str(B)] = run_size(p, f, B, args, hbm_gbs)
        torch.cuda.empty_cache()
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "state_instances_n1.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
