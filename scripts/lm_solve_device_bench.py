"""Measures the one-call solve (twb_batch_lm_solve_device: the loop of BatchedLevenbergMarquardt.solve as a CUDA graph with a
device-side WHILE node) against the Python loop (BatchedLevenbergMarquardt.solve, which reads one flag every `check_every`
iterations), on one GPU, on the two 4096-instance workloads of scripts/lm_solve_bench.py (config5_shard, base_rom).

Per workload and tolerance (--tols), at a budget of --budget iterations:
  * wall time (host clock around the call and a device synchronise) of the one-call solve and of the Python solve at
    check_every 1 and 4; the modes alternate, after one warm-up run of each (the first one-call run builds its graph);
  * the host time spent inside the one-call solve (it only enqueues; after the first call it launches the cached graph);
  * loop iterations run (one call) and the largest iteration count (Python), and whether the results are bit-identical.
Per workload: the time per loop iteration of the one-call solve, (T(budget) - T(0)) / loop iterations at tol 0 — T(0)
is the start and the tail — against the Python iteration (four calls, CUDA events over --iters eager iterations).

    python scripts/lm_solve_device_bench.py --out-dir DIR

Writes <out-dir>/lm_solve_device_n1.json (the committed copy: profiles/lm_solve_device_n1.json).  Needs a CUDA device."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from lm_solve_bench import base_rom, config5_shard, stats, timed  # noqa: E402


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0)


def measure(make, args):
    p, bt, X0, lm = make()
    X = X0.clone()
    out = None

    def one_call(max_iters, tol):
        nonlocal out
        X.copy_(X0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = bt.lm_solve_device(X, lm.xl_full, lm.xu_full, lm.gl_full, lm.gu_full, max_iters=max_iters, tol=tol, mu0=lm.mu, cap=lm.cap,
                                 cg_iters=lm.cg_iters, out=out)
        host_ms = 1e3 * (time.perf_counter() - t0)
        torch.cuda.synchronize()
        return host_ms

    def python(tol, check_every):
        X.copy_(X0)
        return lm.solve(X, args.budget, tol, check_every=check_every)

    res = {"n": p.n, "m": p.m, "nnz": p.nnz, "instances": bt.B, "budget": args.budget, "cg_iters": lm.cg_iters, "tolerances": {}}
    for tol in args.tols:
        first_host_ms = one_call(args.budget, tol)          # builds and instantiates the graph
        python(tol, 1); python(tol, 4)
        modes = ("one_call", "python_check_every_1", "python_check_every_4")
        ms = {m: [] for m in modes}
        host = []
        for rep in range(args.reps):
            for m in (modes if rep % 2 == 0 else modes[::-1]):
                if m == "one_call":
                    h = []
                    ms[m].append(wall(lambda: h.append(one_call(args.budget, tol))))
                    host.append(h[0])
                else:
                    ms[m].append(wall(lambda: python(tol, int(m[-1]))))
        one_call(args.budget, tol)
        dev = [X.cpu().numpy()] + [t.cpu().numpy() for t in out]
        ref = [t.cpu().numpy() for t in python(tol, 4)]
        ref = [X.cpu().numpy()] + ref
        same = all(np.array_equal(a.view(np.int64) if a.dtype == np.float64 else a, b.view(np.int64) if b.dtype == np.float64 else b)
                   for a, b in zip(dev[:5], ref[:5]))
        res["tolerances"][str(tol)] = {
            "wall_ms": {m: stats(v) for m, v in ms.items()},
            "host_ms_inside_one_call": {"first_call": first_host_ms, "later_calls": stats(host)},
            "loop_iterations_one_call": int(dev[6][0]), "iterations_max_python": int(ref[2].max()),
            "status_counts": dev[5].tolist(), "bit_identical_to_python_solve": bool(same)}
    # time per loop iteration: tol 0 keeps every finite instance RUNNING until it stalls
    one_call(args.budget, 0.0); one_call(0, 0.0)
    t_full, t_tail, loops = [], [], []
    for rep in range(args.reps):
        t_full.append(wall(lambda: one_call(args.budget, 0.0)))
        loops.append(int(out[5][0]))
        t_tail.append(wall(lambda: one_call(0, 0.0)))
    st = lm.solve_state()
    X.copy_(X0)
    lm.iterate(X, st, 0.0)
    eager = []
    for rep in range(args.reps):
        X.copy_(X0)
        st = lm.solve_state()
        eager.append(timed(lambda: [lm.iterate(X, st, 0.0) for _ in range(args.iters)]) / args.iters)
    per_it = [(f - t) / max(n, 1) for f, t, n in zip(t_full, t_tail, loops)]
    res["per_iteration"] = {"one_call_loop_iteration_ms": stats(per_it), "python_iteration_ms": stats(eager),
                            "one_call_budget_ms": stats(t_full), "one_call_start_and_tail_ms": stats(t_tail), "loop_iterations": loops,
                            "ratio_one_call_over_python": float(np.median(per_it) / np.median(eager))}
    res["graphs_instantiated"] = bt.lm_solve_graphs_instantiated()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out-dir", required=True, help="directory that receives lm_solve_device_n1.json")
    ap.add_argument("--budget", type=int, default=60, help="iteration budget of the solve")
    ap.add_argument("--tols", type=float, nargs="+", default=[1.0, 1e-6], help="tolerances on the largest scaled violation")
    ap.add_argument("--iters", type=int, default=12, help="eager Python iterations per timed run")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("lm_solve_device_bench: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    result = {"gpu": smi.stdout.strip(),
              "timing": "host clock around each solve and a device synchronise, modes alternating after one warm-up run each; "
                        "Python iterations with CUDA events",
              "workloads": {}}
    for name, make in (("config5_shard", config5_shard), ("base_rom", base_rom)):
        result["workloads"][name] = measure(make, args)
        torch.cuda.empty_cache()
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "lm_solve_device_n1.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
