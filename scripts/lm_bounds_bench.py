"""Times the device-resident solver loop with the problem's shared constraint bounds against the same loop with one row of
constraint bounds per instance (twb_batch_lm_step_device vs twb_batch_lm_step_bounds_device), on one GPU with CUDA events:
Anymal trot / Block at B = 4096 (BASELINE configs[1]) and the same recipe with BaseMotionConstraint, whose LZ rows follow
each instance's initial base height.  Every instance starts from its own measured state (twb_batch_state_instances_device,
which also yields the per-instance bounds).  Per recipe and bound mode: `--iters` solver iterations (eval_device + step)
and, separately, `--iters` steps alone on fixed g / Jacobian values; the two modes alternate over `--reps` repetitions
after one warm-up run each, and the median, min and max are reported.  The per-instance bounds add 2 * 8 * m bytes of reads
per instance to a step that reads 8 * nnz bytes of Jacobian values; the g / Jacobian arrays at B = 4096 (about 0.5 GB)
do not fit the 126 MB L2.

    python scripts/lm_bounds_bench.py --out-dir DIR

Writes <out-dir>/lm_bounds_n1.json (the committed copy: profiles/lm_bounds_n1.json).  Needs a CUDA device."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import towr_b200 as tb  # noqa: E402
from towr_b200.solver import BatchedLevenbergMarquardt  # noqa: E402

RECIPES = ("anymal_trot_block", "anymal_trot_block_base_rom")
B = 4096


def random_states(f, count, seed):
    """state records around the recipe's own (the distribution of tests/test_state_instances.py): initial base z +-0.05"""
    rng = np.random.default_rng(seed)
    S = np.tile(f.state_record(), (count, 1))
    n_ee = len(f.initial_ee_W_)
    S[:, 0:2] += rng.uniform(-0.3, 0.3, (count, 2)); S[:, 2] += rng.uniform(-0.05, 0.05, count)
    S[:, 3:12] = rng.uniform(-0.3, 0.3, (count, 9))
    S[:, 12:14] += rng.uniform(-0.5, 0.5, (count, 2)); S[:, 14] += rng.uniform(-0.05, 0.05, count)
    S[:, 15:24] = rng.uniform(-0.3, 0.3, (count, 9))
    S[:, 24:24 + 3 * n_ee] += rng.uniform(-0.05, 0.05, (count, 3 * n_ee))
    return S


def stats(ms):
    ms = np.asarray(ms)
    return {"median_ms": float(np.median(ms)), "min_ms": float(ms.min()), "max_ms": float(ms.max()), "runs": int(ms.size)}


def run_recipe(name, args):
    f = tb.make_formulation(name)
    p = tb.Problem(f.to_spec())
    dev = torch.device("cuda", 0)
    bt = p.batch(B)
    x0, xl, xu, gl, gu = bt.state_instances_device(torch.from_numpy(random_states(f, B, seed=11)).to(dev), want_g_bounds=True)
    X0 = torch.minimum(torch.maximum(x0 + 0.01 * torch.from_numpy(np.random.default_rng(12).standard_normal((B, p.n))).to(dev), xl), xu)
    solvers = {"shared_bounds": BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu),
               "instance_bounds": BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu, g_lower=gl, g_upper=gu)}
    finals, hists = {}, {}
    for mode, lm in solvers.items():           # warm-up (graph capture, pattern upload, module load) and the outputs
        X = X0.clone()
        hists[mode] = lm.run(X, args.iters)
        finals[mode] = X
    torch.cuda.synchronize()
    loop = {mode: [] for mode in solvers}
    step = {mode: [] for mode in solvers}
    for rep in range(args.reps):
        for mode in (list(solvers) if rep % 2 == 0 else list(solvers)[::-1]):
            lm = solvers[mode]
            X = X0.clone()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record(); lm.run(X, args.iters); b.record()
            torch.cuda.synchronize()
            loop[mode].append(a.elapsed_time(b))
            # the step alone, on the g / Jacobian values of the last evaluation
            a.record()
            for _ in range(args.iters):
                bt.lm_step_device(X, lm.g, lm.jac_vals, lm.xl_full, lm.xu_full, lm.mu, lm.cap, lm.cg_iters, lm.viol,
                                  g_lower=lm.gl_full, g_upper=lm.gu_full)
            b.record()
            torch.cuda.synchronize()
            step[mode].append(a.elapsed_time(b))
    same = bool(torch.equal(finals["shared_bounds"], finals["instance_bounds"]) and torch.equal(hists["shared_bounds"], hists["instance_bounds"]))
    res = {"n": p.n, "m": p.m, "nnz": p.nnz, "instances": B, "iterations": args.iters, "cg_iters": solvers["shared_bounds"].cg_iters,
           "extra_bytes_per_instance_step": 2 * 8 * p.m, "jacobian_bytes_per_instance_step": 8 * p.nnz,
           "results_identical_between_modes": same,
           "violation_median_first_last": {mode: [float(h[0].median()), float(h[-1].median())] for mode, h in hists.items()}}
    for mode in solvers:
        res[mode] = {"loop": stats(loop[mode]), "step_only": stats(step[mode])}
    res["loop_median_ratio_instance_over_shared"] = res["instance_bounds"]["loop"]["median_ms"] / res["shared_bounds"]["loop"]["median_ms"]
    res["step_median_ratio_instance_over_shared"] = res["instance_bounds"]["step_only"]["median_ms"] / res["shared_bounds"]["step_only"]["median_ms"]
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out-dir", required=True, help="directory that receives lm_bounds_n1.json")
    ap.add_argument("--iters", type=int, default=12)
    ap.add_argument("--reps", type=int, default=6)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("lm_bounds_bench: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    result = {"gpu": smi.stdout.strip(), "timing": "CUDA events around each run, modes alternating, after one warm-up run per mode",
              "recipes": {}}
    for name in RECIPES:
        result["recipes"][name] = run_recipe(name, args)
        torch.cuda.empty_cache()
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "lm_bounds_n1.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
