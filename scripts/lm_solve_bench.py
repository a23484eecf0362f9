"""Measures BatchedLevenbergMarquardt.solve (trial step, g-only evaluation at the trial point, gain-ratio acceptance) on one
GPU with CUDA events, on two workloads of 4096 instances:

  config5_shard  Anymal trot on mixed Slope / Chimney / Gap terrains, goal-randomised initial guesses and bounds from
                 twb_batch_goal_instances_device, 1 % perturbations (tests/test_solver_loop.py's config-5 shard)
  base_rom       Anymal trot / Block with BaseMotionConstraint, every instance from its own measured state with its own
                 constraint bounds (twb_batch_state_instances_device; scripts/lm_bounds_bench.py's workload)

Per workload: the time of one `run` iteration (evaluation + step) against one solve iteration (evaluation + trial + g-only
evaluation + acceptance), both over the first `--iters` iterations from the same start; the g-only evaluation alone; the
whole solve to `--tol` with a budget of `--budget` iterations; and the histogram of the solve statuses after every
iteration.  Timed runs alternate after one warm-up run each; the median, min and max are reported.

    python scripts/lm_solve_bench.py --out-dir DIR

Writes <out-dir>/lm_solve_n1.json (the committed copy: profiles/lm_solve_n1.json).  Needs a CUDA device."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import towr_b200 as tb  # noqa: E402
from towr_b200 import capi  # noqa: E402
from towr_b200.solver import BatchedLevenbergMarquardt  # noqa: E402
from lm_bounds_bench import random_states  # noqa: E402

B = 4096
STATUS_NAMES = ("running", "converged", "stalled", "nonfinite")


def config5_shard():
    p = tb.Problem(tb.make_formulation("anymal_trot_mixed").to_spec())
    rng = np.random.default_rng(77)
    terr = rng.choice([tb.SLOPE, tb.CHIMNEY, tb.GAP], B).astype(np.int32)
    goals = np.column_stack([rng.uniform(1.0, 2.0, B), rng.uniform(-0.2, 0.2, B), np.full(B, 0.5), np.zeros(B), np.zeros(B),
                             rng.uniform(-0.2, 0.2, B)])
    bt = p.batch(B); bt.set_terrains(terr)
    x0, xl, xu = bt.goal_instances_device(torch.from_numpy(goals).cuda())
    X0 = torch.minimum(torch.maximum(x0 + 0.01 * torch.from_numpy(rng.standard_normal((B, p.n))).cuda(), xl), xu)
    return p, bt, X0, BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu)


def base_rom():
    f = tb.make_formulation("anymal_trot_block_base_rom")
    p = tb.Problem(f.to_spec())
    bt = p.batch(B)
    x0, xl, xu, gl, gu = bt.state_instances_device(torch.from_numpy(random_states(f, B, seed=11)).cuda(), want_g_bounds=True)
    X0 = torch.minimum(torch.maximum(x0 + 0.01 * torch.from_numpy(np.random.default_rng(12).standard_normal((B, p.n))).cuda(), xl), xu)
    return p, bt, X0, BatchedLevenbergMarquardt(bt, x_lower=xl, x_upper=xu, g_lower=gl, g_upper=gu)


def stats(ms):
    ms = np.asarray(ms)
    return {"median_ms": float(np.median(ms)), "min_ms": float(ms.min()), "max_ms": float(ms.max()), "runs": int(ms.size)}


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def measure(name, make, args):
    p, bt, X0, lm = make()
    K = args.iters
    # warm-up of every argument set (evaluation graphs, pattern upload, module load)
    lm.run(X0.clone(), 1)
    lm.solve(X0.clone(), 1, args.tol)
    torch.cuda.synchronize()
    runs = {"run": [], "solve_iterations": [], "g_only_eval": []}
    st_last = None
    for rep in range(args.reps):
        order = ("run", "solve_iterations") if rep % 2 == 0 else ("solve_iterations", "run")
        for mode in order:
            X = X0.clone()
            if mode == "run":
                runs[mode].append(timed(lambda: lm.run(X, K)) / K)
            else:
                st = lm.solve_state()
                runs[mode].append(timed(lambda: [lm.iterate(X, st, args.tol) for _ in range(K)]) / K)
                st_last = st
        runs["g_only_eval"].append(timed(lambda: [bt.eval_device(st_last.x_trial, g=st_last.g_trial, flags=capi.EVAL_G) for _ in range(K)]) / K)
    # the whole solve, and the status histogram after every iteration (a separate, untimed walk of the same iterations)
    solve_ms, result = [], None
    for rep in range(args.reps):
        X = X0.clone()
        out = []
        solve_ms.append(timed(lambda: out.append(lm.solve(X, args.budget, args.tol))))
        result = out[0]
    status, iterations, violation, mu = (t.cpu().numpy() for t in result)
    X = X0.clone()
    st = lm.solve_state()
    hist = []
    for it in range(args.budget):
        lm.iterate(X, st, args.tol)
        hist.append(np.bincount(st.status.cpu().numpy(), minlength=4).tolist())
    lm.iterate(X, st, args.tol, cg_iters=0)
    same = bool(np.array_equal(st.status.cpu().numpy(), status) and np.array_equal(st.iterations.cpu().numpy(), iterations))
    res = {"n": p.n, "m": p.m, "nnz": p.nnz, "instances": B, "cg_iters": lm.cg_iters, "tol": args.tol, "eta": 1e-4,
           "timed_iterations": K,
           "per_iteration": {"run_ms": stats(runs["run"]), "solve_iteration_ms": stats(runs["solve_iterations"]),
                             "g_only_eval_ms": stats(runs["g_only_eval"])},
           "solve_iteration_over_run_iteration": float(np.median(runs["solve_iterations"]) / np.median(runs["run"])),
           "solve": {"budget": args.budget, "check_every": 4, "ms": stats(solve_ms),
                     "status_counts": dict(zip(STATUS_NAMES, np.bincount(status, minlength=4).tolist())),
                     "iterations_median_max": [float(np.median(iterations)), int(iterations.max())],
                     "violation_median_of_converged": float(np.median(violation[status == 1])) if (status == 1).any() else None,
                     "violation_median_of_running": float(np.median(violation[status == 0])) if (status == 0).any() else None,
                     "mu_median": float(np.median(mu)),
                     "violation_quantiles_10_25_50_75_90": [float(q) for q in np.quantile(violation, [0.1, 0.25, 0.5, 0.75, 0.9])]},
           "status_histogram_after_iteration": {"columns": list(STATUS_NAMES), "rows": hist},
           "histogram_walk_matches_solve": same}
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out-dir", required=True, help="directory that receives lm_solve_n1.json")
    ap.add_argument("--iters", type=int, default=12, help="iterations per timed run")
    ap.add_argument("--budget", type=int, default=60, help="iteration budget of the solve")
    ap.add_argument("--tol", type=float, default=1e-6, help="tolerance on the largest scaled violation")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("lm_solve_bench: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    result = {"gpu": smi.stdout.strip(),
              "timing": "CUDA events around each run, run / solve iterations alternating, after one warm-up run each",
              "workloads": {}}
    for name, make in (("config5_shard", config5_shard), ("base_rom", base_rom)):
        result["workloads"][name] = measure(name, make, args)
        torch.cuda.empty_cache()
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "lm_solve_n1.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({k: {kk: v[kk] for kk in ("per_iteration", "solve")} for k, v in result["workloads"].items()}, indent=1))


if __name__ == "__main__":
    main()
