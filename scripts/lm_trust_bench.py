"""Measures the two step rules of the one-call solve (twb_batch_lm_solve_device: TWB_LM_STEP_CAP, the default, and
TWB_LM_STEP_TRUST) on one GPU, on the two 4096-instance workloads of scripts/lm_solve_bench.py (its set-up functions):

  config5_shard  Anymal trot on mixed Slope / Chimney / Gap terrains, goal-randomised starts, 1 % perturbations
  base_rom       Anymal trot / Block with BaseMotionConstraint, per-instance states and constraint bounds

Per workload and rule:
  - the time of one loop iteration: CUDA events around a solve with tol 0 and a budget of --budget iterations minus a solve
    with budget 0 (the start and the tail), over the loop iterations it ran; runs of the two rules alternate after one
    warm-up each.  Finished instances only copy x, so the same over the first --early iterations, where nearly every
    instance still runs, is recorded too;
  - the status counts after --budget iterations at tol 1e-6 and at tol 1e-2;
  - the quantiles of max |s r| at the returned x, and max |s r| and the status of the first six instances (the instances a
    per-instance CPU restatement of the loop is cheap enough to run on);
  - for the trust-region rule, the radius and step_norm of those six instances after each loop iteration (a solve with
    budget k for k = 1 .. --budget, twb_batch_lm_solve_radius), and the status counts after --early iterations.

    python scripts/lm_trust_bench.py --out-dir DIR

Writes <out-dir>/lm_trust_n1.json (the committed copy: profiles/lm_trust_n1.json).  Needs a CUDA device."""
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

from lm_solve_bench import STATUS_NAMES, base_rom, config5_shard, stats, timed  # noqa: E402

RULES = ("cap", "trust")


def solve(lm, X0, rule, max_iters, tol):
    """One solve from a copy of X0: (elapsed ms, status, violation, loop count, mu)."""
    X = X0.clone()
    out = []
    ms = timed(lambda: out.append(lm.batch.lm_solve_device(X, lm.xl_full, lm.xu_full, lm.gl_full, lm.gu_full, max_iters=max_iters, tol=tol,
                                                           mu0=lm.mu, cap=lm.cap, cg_iters=lm.cg_iters, step_rule=rule)))
    status, _, violation, mu, _, loop_count = out[0]
    return ms, status.cpu().numpy(), violation.cpu().numpy(), int(loop_count.item()), mu.cpu().numpy()


def measure(make, args):
    p, bt, X0, lm = make()
    for rule in RULES:                            # warm-up: the first call of an argument set builds its graph
        for k in (0, args.budget):
            solve(lm, X0, rule, k, 0.0)
    for rule in RULES:
        solve(lm, X0, rule, args.early, 0.0)
    res = {"n": p.n, "m": p.m, "nnz": p.nnz, "instances": int(X0.shape[0]), "cg_iters": lm.cg_iters, "cap": lm.cap, "budget": args.budget,
           "rules": {}}
    for key, budget in (("", args.budget), ("early_", args.early)):
        loop_ms = {r: [] for r in RULES}
        loops = {}
        for rep in range(args.reps):
            for rule in (RULES if rep % 2 == 0 else RULES[::-1]):
                full, status, _, n_loop, _ = solve(lm, X0, rule, budget, 0.0)
                tail = solve(lm, X0, rule, 0, 0.0)[0]
                loops[rule] = {"loop_iterations": n_loop, "status_counts_after": np.bincount(status, minlength=4).tolist()}
                loop_ms[rule].append((full - tail) / max(n_loop, 1))
        res[key + "loop_iteration_ms"] = {r: stats(loop_ms[r]) for r in RULES}
        res[key + "loops_timed"] = loops
        res[key + "trust_over_cap_iteration"] = float(np.median(loop_ms["trust"]) / np.median(loop_ms["cap"]))
    trace = {"radius": [], "step_norm": [], "status": []}
    for k in range(1, args.budget + 1):
        _, status, _, _, _ = solve(lm, X0, "trust", k, 1e-6)
        radius, step_norm = lm.batch.lm_solve_radius()
        for name, v in (("radius", radius), ("step_norm", step_norm), ("status", status)):
            trace[name].append(v[:6].tolist())
    res["trust_first_six_by_iteration"] = trace
    for rule in RULES:
        rec = {}
        for tol in (1e-6, 1e-2):
            _, status, violation, n_loop, mu = solve(lm, X0, rule, args.budget, tol)
            stalled = status == 2
            rec[f"tol_{tol:g}"] = {"status_counts": dict(zip(STATUS_NAMES, np.bincount(status, minlength=4).tolist())), "loop_count": n_loop,
                                   # STALLED through mu > mu_max (both rules) or through a collapsed radius (trust only)
                                   "stalled_by_mu": int(np.sum(stalled & (mu > 1e10))), "stalled_by_radius": int(np.sum(stalled & (mu <= 1e10))),
                                   "violation_median_of_stalled": float(np.median(violation[stalled])) if stalled.any() else None,
                                   "violation_quantiles_10_25_50_75_90": [float(q) for q in np.quantile(violation, [0.1, 0.25, 0.5, 0.75, 0.9])],
                                   "first_six": {"violation": violation[:6].tolist(), "status": status[:6].tolist()}}
        res["rules"][rule] = rec
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out-dir", required=True, help="directory that receives lm_trust_n1.json")
    ap.add_argument("--budget", type=int, default=60, help="iteration budget of every solve")
    ap.add_argument("--early", type=int, default=5, help="iterations of the second timing")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("lm_trust_bench: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    result = {"gpu": smi.stdout.strip(),
              "timing": "CUDA events around one-call solves (tol 0, budget minus budget 0, over the loop iterations run), the two "
                        "rules alternating after one warm-up each",
              "workloads": {}}
    for name, make in (("config5_shard", config5_shard), ("base_rom", base_rom)):
        result["workloads"][name] = measure(make, args)
        torch.cuda.empty_cache()
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "lm_trust_n1.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
