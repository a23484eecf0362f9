#!/usr/bin/env python
"""bench.py — NLP evals/sec (constraints + sparse Jacobian, fp64), Anymal batch.

A "step" is one batched evaluation (g and all CSR Jacobian values) of B
independent Anymal fly-trot / Block-terrain problem instances
(BASELINE.json configs[1], B = 4096 per GPU, weak scaling: every rank owns its
own 4096 instances, no data-path collective).

  python bench.py [--gpus N] [--steps K] [--warmup W]          # CUDA arm
  python bench.py --dump-outputs DIR [...]                      # + the outputs of the last timed step as DIR/*.npy
  python bench.py --impl reference [...]                        # CPU restatement arm (oracle, all host cores)
  torchrun --nproc-per-node N bench.py --gpus N ...             # N > 1

Prints ONE JSON line (rank 0).  See DESIGN.md §6 for how every field is measured.
Writes nothing into the tree: the build lock lives in the temporary directory.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOAD = "anymal_trot_block"   # --workload overrides (other BASELINE configs; not the driver's line)
BATCH_PER_GPU = 4096
DESCR = {
    "anymal_trot_block": "BASELINE configs[1]: Anymal fly-trot C1, Block terrain, T=2.0 s",
    "biped_walk_stairs": "BASELINE configs[2]: Biped walk C0, Stairs, fpowr recipe, T=2.0 s",
    "hyq_gallop_gap": "BASELINE configs[3]: HyQ gallop C4, Gap terrain, phase durations optimised, T=2.0 s",
    "anymal_trot_mixed": "BASELINE configs[4], one GPU's shard: Anymal fly-trot C1, terrains drawn from Slope/Chimney/Gap per instance",
    "hopper": "BASELINE configs[0]: Monoped hopper, FlatGround, T=2.0 s",
}
METRIC = "nlp_evals_per_sec"
UNIT = "evals/s"
DUMP_BYTES = 48 << 20      # --dump-outputs: at most this many bytes of instances (g + jac + status, as float64)


def read_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.samples.append([s.strip() for s in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx = float(s[1])
                for nm, v in zip(names, s[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def load_spec_fixture(workload):
    """twb_spec of a bench workload from tests/golden/bench_specs.json, as a ctypes struct defined by towr_b200/_spec.py loaded
    BY FILE PATH: neither the towr_b200 package nor libtowr_b200.so is touched (reference arm)."""
    import importlib.util
    sp = importlib.util.spec_from_file_location("twb_spec_struct", os.path.join(ROOT, "towr_b200", "_spec.py"))
    mod = importlib.util.module_from_spec(sp); sp.loader.exec_module(mod)
    fx = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_specs.json")))
    return mod.Spec.from_buffer_copy(bytes.fromhex(fx[workload]))


def oracle_iterates(spec, batch, seed=1234):
    """The iterate distribution of towr_b200.configs.synthetic_iterates_fast (x0 + sigma N(0,1); sigma 0.05 / 0.2 / 10 / 50),
    built from the ORACLE's x0 and variable-set layout only."""
    import importlib.util
    import numpy as np
    import oracle_lib
    sp_ = importlib.util.spec_from_file_location("twb_spec_struct", os.path.join(ROOT, "towr_b200", "_spec.py"))
    mod = importlib.util.module_from_spec(sp_); sp_.loader.exec_module(mod)
    o = oracle_lib.Oracle(spec)
    x0 = o.x0()
    sig = np.zeros(o.n)
    sets = o.variable_sets()
    for name, start, count in sets:
        idx = np.arange(count)
        if name.startswith("base-"):
            sig[start:start + count] = np.where((idx % 6) < 3, 0.05, 0.2)
        elif name.startswith("ee-motion"):
            sig[start:start + count] = np.where(np.array(mod.motion_velocity_mask(spec, int(name[len("ee-motion_"):]))), 0.2, 0.05)
        elif name.startswith("ee-force"):
            sig[start:start + count] = np.where((idx % 2) == 0, 10.0, 50.0)
    rng = np.random.default_rng(seed)
    X = x0 + sig * rng.standard_normal((batch, o.n))
    for name, start, count in sets:
        if name.startswith("ee-schedule"):
            ee = int(name[len("ee-schedule"):])
            t_total = sum(spec.phase_durations[ee][i] for i in range(spec.n_phases[ee]))
            d = x0[start:start + count] * rng.uniform(0.9, 1.1, (batch, count))
            X[:, start:start + count] = d * np.minimum(1.0, 0.98 * t_total / d.sum(axis=-1, keepdims=True))
        if name == "base-ang":
            blk = X[:, start:start + count].reshape(batch, -1, 6)
            blk[:, :, :3] = np.clip(blk[:, :, :3], -1.0, 1.0)
    return X, o


def make_problem():
    import towr_b200 as tb
    spec = tb.make_formulation(WORKLOAD).to_spec()
    return tb, spec, tb.Problem(spec)


def kernel_breakdown(p, B):
    """Per-kernel durations from a second, serialised pass (TWB_PROFILE=1: every kernel on one stream, CUDA events
    around each launch) in a child process, with each kernel's own algorithmic bytes.  The timed region of the main
    pass runs the three output kernels concurrently on three streams, so their durations are not separable there."""
    env = dict(os.environ, TWB_PROFILE="1")
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--quick", "--steps", "30", "--warmup", "5",
                              "--workload", WORKLOAD, "--batch", str(B)],
                             capture_output=True, text=True, timeout=300, env=env).stderr
    except Exception:
        return None
    rows = {}
    for nm, r0, nr in p.constraint_sets():
        rows[nm] = (r0, nr)
    rp = p.row_ptr()
    def share(pred):
        nz = sum(int(rp[r0 + nr] - rp[r0]) for nm, (r0, nr) in rows.items() if pred(nm))
        mm = sum(nr for nm, (r0, nr) in rows.items() if pred(nm))
        return 8 * B * (nz + mm)
    alg = {"DynOut": share(lambda n: n == "dynamic"), "RomOut": share(lambda n: n.startswith("rangeofmotion")),
           "NodeOut": share(lambda n: n != "dynamic" and not n.startswith(("rangeofmotion", "totalduration"))),
           "RomNodeOut": share(lambda n: n != "dynamic" and not n.startswith("totalduration")),
           "TransposeIn": 2 * 8 * B * p.n, "TransposeOut": 2 * 8 * B * p.m}
    res = {}
    for line in out.splitlines():
        parts = line.split()
        if line.startswith("[twb profile]") and "avg" in parts:
            name, us = parts[2], float(parts[parts.index("avg") + 1])
            res[name] = {"avg_us": us}
            if name == "TransposeIn":
                res[name]["note"] = "first kernel of a step: includes the host launch gap of the serialised pass (ncu: 8 us)"
                continue
            if name in alg and us > 0:
                res[name]["algorithmic_bytes"] = alg[name]
                res[name]["gbs"] = alg[name] / (us * 1e-6) / 1e9
    return res or None


def host_threads():
    """Host threads the CPU legs use: every core this process may run on (torchrun exports OMP_NUM_THREADS=1,
    which must not throttle the CPU arm — the thread count is passed to the oracle explicitly)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_arm(spec, problem, X, threads, target_seconds=12.0):
    """Times the CPU restatement (oracle) on a bounded sample of the same iterates: whole passes over the batch
    (at most 4096 instances each) until ~target_seconds of CPU work have been done."""
    import oracle_lib
    sample = min(len(X), 4096)
    oracle_lib.batch_eval(spec, X[:min(sample, 4 * threads)], threads=threads)      # warm-up (thread pool, page faults)
    done, t0 = 0, time.perf_counter()
    while True:
        r = oracle_lib.batch_eval(spec, X[:sample], threads=threads)
        assert r["rc"] == 0
        done += sample
        dt = time.perf_counter() - t0
        if dt >= target_seconds or done >= 64 * sample:
            return done / dt, done, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle_lib
    spec = load_spec_fixture(WORKLOAD)            # no towr_b200 import, no libtowr_b200.so in this process
    threads = host_threads()
    X, p = oracle_iterates(spec, 2048)
    assert "towr_b200" not in sys.modules
    # each step: a bounded sample of the workload sized for ~1.5 s of CPU time
    t0 = time.perf_counter(); oracle_lib.batch_eval(spec, X[:max(threads, 8)], threads=threads)
    per_eval = (time.perf_counter() - t0) / max(threads, 8)
    sample = int(max(threads, min(len(X), 1.5 / per_eval)))
    for _ in range(args.warmup):
        oracle_lib.batch_eval(spec, X[:sample], threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle_lib.batch_eval(spec, X[:sample], threads=threads)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{WORKLOAD} ({DESCR.get(WORKLOAD, WORKLOAD)}), n={p.n} m={p.m} nnz={p.nnz}",
                   "note": "reference arm = CPU restatement of towr's evaluation (oracle port, g++ -O3, OpenMP over instances; towr itself "
                           "needs Eigen+ifopt, absent here); spec from tests/golden/bench_specs.json, the product library is not loaded"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{sample} instances per step, OpenMP over instances"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa_node(local):
    """Multi-GPU runs: pin this rank's host threads to the CPUs next to its GPU (NVML's CPU affinity mask), so that the
    pinned host buffers of the end-to-end leg are first-touched on the GPU's NUMA node and the D2H copies of the ranks do
    not all cross one socket link.  Returns the number of CPUs bound to (0: left alone)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def run_config5(args, tb, dev, world, rank, local):
    """BASELINE configs[4], the north-star size: 65 536 Anymal multi-start instances on mixed Slope / Chimney / Gap terrains,
    split over the ranks with shard_range (STRONG scaling: 65 536 / N instances per GPU).  Device-timed like the headline;
    after every step the per-instance cost / status are all-gathered over NCCL (outside the timed region)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from towr_b200.configs import synthetic_iterates_fast
    from towr_b200.sharding import gather_cost_status, shard_range
    total = 65536
    lo, hi = shard_range(total, rank, world)
    nb = hi - lo
    spec = tb.make_formulation("anymal_trot_mixed").to_spec()
    p = tb.Problem(spec)
    batch = p.batch(nb, device=local)
    batch.set_terrains(np.random.default_rng(7).choice([tb.SLOPE, tb.CHIMNEY, tb.GAP], total).astype(np.int32)[lo:hi])
    rng_sets = [torch.from_numpy(synthetic_iterates_fast(p, nb, seed=99 + 13 * rank + 1000 * r)).to(dev) for r in range(2)]
    g = torch.empty((nb, p.m), dtype=torch.float64, device=dev)
    jac = torch.empty((nb, p.nnz), dtype=torch.float64, device=dev)
    status = torch.zeros(nb, dtype=torch.int32, device=dev)
    cost = torch.zeros(nb, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream(dev)
    flags = tb.EVAL_G | tb.EVAL_JAC
    steps = max(3, min(args.steps, 10))
    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier(); torch.cuda.synchronize(dev)
    for i in range(3):
        batch.eval_device(rng_sets[i % 2], g=g, jac=jac, status=status, flags=flags, stream=stream)
    barrier()
    total_ms, gathered, flagged = 0.0, 0, 0
    for i in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record(stream)
        batch.eval_device(rng_sets[i % 2], g=g, jac=jac, status=status, flags=flags, stream=stream)
        b.record(stream)
        barrier()
        total_ms += a.elapsed_time(b)
        cost_all, status_all = gather_cost_status(cost.cpu().numpy(), status.cpu().numpy(), total, device=dev)   # NCCL all_gather (N > 1)
        gathered, flagged = len(status_all), int((status_all != 0).sum())
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    del batch, g, jac
    torch.cuda.empty_cache()
    bytes_per_eval = 8 * (p.n + p.m + p.nnz)
    achieved_per_gpu = bytes_per_eval * nb / (ms * 1e-3) / 1e9
    return {"workload": "BASELINE configs[4]: Anymal fly-trot C1 multi-start, terrains drawn from Slope / Chimney / Gap per instance",
            "instances_total": total, "instances_per_gpu": nb, "scaling": "strong", "steps": steps, "ms_per_step": ms,
            "value": total / (ms * 1e-3), "unit": UNIT, "roofline_frac_per_gpu": achieved_per_gpu / read_peak()[0],
            "collective": {"op": "all_gather of per-instance cost (f64) + status (i32) after every step, outside the timed region",
                           "backend": "nccl" if world > 1 else "none (one rank: local copy)", "gathered_instances": gathered, "flagged": flagged}}


def dump_outputs(out_dir, g, jac, status):
    """Writes what the caller of twb_batch_eval_device received: g[k][m], jac[k][nnz] (CSR values) and status[k] (as float64)
    of k instances.  k is the whole batch when it fits DUMP_BYTES, else a fixed, seeded sample of instances in ascending
    order, so that two builds run with the same arguments can be compared output for output."""
    import numpy as np
    import torch
    B = g.shape[0]
    k = min(B, DUMP_BYTES // (8 * (g.shape[1] + jac.shape[1] + 1)))
    idx = torch.from_numpy(np.sort(np.random.default_rng(0).choice(B, k, replace=False))).to(g.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("g", g), ("jac", jac), ("status", status)):
        np.save(os.path.join(out_dir, f"{name}.npy"), t[idx].to(torch.float64).cpu().numpy())


def run_cuda(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from towr_b200.configs import synthetic_iterates_fast

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (towr_b200 has no CPU evaluation path; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = bind_to_gpu_numa_node(local) if world > 1 and not os.environ.get("TWB_NO_NUMA_BIND") else 0
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    tb, spec, p = make_problem()
    B = args.batch or BATCH_PER_GPU
    batch = p.batch(B, device=local)
    if WORKLOAD == "anymal_trot_mixed":
        batch.set_terrains(np.random.default_rng(7 + rank).choice([tb.SLOPE, tb.CHIMNEY, tb.GAP], B).astype(np.int32))

    # ---- inputs: a ring of distinct iterate sets, together larger than L2 (126 MB)
    n_ring = 8
    Xh = synthetic_iterates_fast(p, B, seed=1234 + rank)
    ring = []
    for r in range(n_ring):
        Xr = Xh if r == 0 else synthetic_iterates_fast(p, B, seed=1234 + rank + 1000 * r)
        ring.append(torch.from_numpy(Xr).to(dev))
    g = torch.empty((B, p.m), dtype=torch.float64, device=dev)
    jac = torch.empty((B, p.nnz), dtype=torch.float64, device=dev)
    status = torch.zeros(B, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev)
    flags = tb.EVAL_G | tb.EVAL_JAC

    def step(i):
        batch.eval_device(ring[i % n_ring], g=g, jac=jac, status=status, flags=flags, stream=stream)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    sampler = ClockSampler(local) if rank == 0 and not args.quick else None
    if sampler:
        sampler.start()
    for i in range(n_ring):      # setup: one evaluation per argument set, so that every set's CUDA graph is captured and instantiated
        step(i)                  # before the warm-up (a one-time cost per argument set, like loading the module)
    sync_all()
    for i in range(max(args.warmup, 3)):
        step(i)
    sync_all()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    sync_all()
    ev[0].record(stream)
    for i in range(args.steps):
        step(i)
        ev[i + 1].record(stream)
    sync_all()
    total_ms = ev[0].elapsed_time(ev[-1])
    per_step = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps))
    if args.dump_outputs and rank == 0:    # before the clock-sampling steps below overwrite g / jac
        dump_outputs(args.dump_outputs, g, jac, status)
    if sampler:
        # the timed region lasts a few milliseconds; keep the same loop running ~1 s more so that nvidia-smi (one
        # sample per ~60 ms) sees the clocks under this load; these steps are not part of any reported number
        t_end = time.perf_counter() + 1.0
        i = 0
        while time.perf_counter() < t_end:
            step(i); i += 1
            if i % 64 == 0:
                torch.cuda.synchronize(dev)
        torch.cuda.synchronize(dev)
        sampler.stop_flag = True
    assert int(status.sum().item()) == 0, "non-finite values flagged"
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    value = world * B * args.steps / (total_ms * 1e-3)

    if args.quick:
        if rank == 0:
            print(json.dumps({"value": value, "ms_per_step": total_ms / args.steps, "ms_best": per_step[0],
                              "frac": 8 * (p.n + p.m + p.nnz) * B / (total_ms / args.steps * 1e-3) / 1e9 / read_peak()[0]}), flush=True)
        return
    # ---- end to end through the host-pointer C ABI call: pinned host buffers, H2D + D2H inside the timed region
    xs_pinned = torch.from_numpy(Xh).pin_memory()
    out = {"g": torch.empty((B, p.m), dtype=torch.float64).pin_memory().numpy(),
           "jac": torch.empty((B, p.nnz), dtype=torch.float64).pin_memory().numpy(),
           "status": torch.empty(B, dtype=torch.int32).pin_memory().numpy()}
    x_np = xs_pinned.numpy()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        batch.eval_host(x_np, flags=flags, out=out)
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        batch.eval_host(x_np, flags=flags, out=out)      # synchronises internally; result is on the host
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * B * e2e_steps / float(te.item())
    h2d = B * p.n * 8
    d2h = B * (p.m + p.nnz) * 8 + B * 4
    # the PCIe ceiling of this box for that step, measured in the same run on the same buffers: a bare pinned D2H copy of
    # the step's output bytes (all ranks at once, max over ranks) — what the step would cost if the GPU computed in zero time
    jac_pinned = torch.from_numpy(out["jac"]); g_pinned = torch.from_numpy(out["g"])
    cs = torch.cuda.Stream(dev)
    with torch.cuda.stream(cs):
        jac_pinned.copy_(jac, non_blocking=True); g_pinned.copy_(g, non_blocking=True)
    cs.synchronize(); sync_all()
    best = float("inf")
    for _ in range(5):   # the best of five: a ceiling must not be lowered by a disturbed repetition
        sync_all()
        t0 = time.perf_counter()
        with torch.cuda.stream(cs):
            jac_pinned.copy_(jac, non_blocking=True); g_pinned.copy_(g, non_blocking=True)
        cs.synchronize()
        best = min(best, time.perf_counter() - t0)
    tc = torch.tensor([best], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tc, op=dist.ReduceOp.MAX)
    d2h_ceiling_s = float(tc.item())
    config5 = run_config5(args, tb, dev, world, rank, local) if not os.environ.get("TWB_NO_CONFIG5") else None

    if rank == 0:
        import oracle_lib
        peak, peak_src = read_peak()
        bytes_per_eval = 8 * (p.n + p.m + p.nnz)
        avg_kernel_ms = total_ms / args.steps       # one evaluation (all its kernels) per step
        achieved = bytes_per_eval * B / (avg_kernel_ms * 1e-3) / 1e9
        threads = host_threads()
        cpu_value, cpu_sample, cpu_dt = cpu_arm(spec, p, Xh, threads)
        kernels = kernel_breakdown(p, B)
        dominant = None
        if kernels:
            cand = [(k, v) for k, v in kernels.items() if "gbs" in v and k.endswith("Out") and k != "TransposeOut"]
            if cand:
                k, v = max(cand, key=lambda kv: kv[1]["avg_us"])
                dominant = {"name": k, "avg_launch_ms": v["avg_us"] * 1e-3, "algorithmic_bytes_per_launch": v["algorithmic_bytes"],
                            "achieved": v["gbs"], "frac": v["gbs"] / peak, "how": "serialised pass, CUDA events around each launch"}
        traffic, traffic_kernels = None, {}
        tpath = os.path.join(ROOT, "profiles", "traffic_bytes_per_launch.json")
        if os.path.exists(tpath) and WORKLOAD == "anymal_trot_block" and B == BATCH_PER_GPU:
            try:
                tj = json.load(open(tpath))
                traffic, traffic_kernels = tj.get("dram_bytes_per_launch"), tj.get("kernels", {})
            except Exception:
                traffic = None
        if dominant and dominant["name"] in traffic_kernels:
            dominant["traffic"] = traffic_kernels[dominant["name"]]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{WORKLOAD} ({DESCR.get(WORKLOAD, WORKLOAD)}), "
                                   f"{B} instances per GPU, n={p.n} m={p.m} nnz={p.nnz}",
                       "batch_per_gpu": B, "outputs": "g[B][m] + jac[B][nnz] (CSR values), fp64",
                       "l2": f"inputs rotate over {n_ring} distinct iterate sets ({n_ring * B * p.n * 8 / 1e6:.0f} MB) and each step "
                             f"writes {B * (p.m + p.nnz) * 8 / 1e6:.0f} MB of outputs (> 126 MB L2)",
                       "iterates": "x0 + sigma*N(0,1), sigma 0.05 pos / 0.2 vel / 10 N force (SURVEY §8d)"},
            "ms_per_step_median": per_step[len(per_step) // 2], "ms_per_step_best": per_step[0],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": "static: ncu --set full capture committed under profiles/ (traffic_bytes_per_launch.json, taken with the same command in a separate profiler run), not measured in this run",
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": bytes_per_eval * B, "avg_launch_ms": avg_kernel_ms,
                         "kernel": "whole evaluation, replayed as one CUDA graph: TransposeIn -> RomNodeOut | DynOut (two branches; the "
                                   "constraint values are written by the output CTAs themselves, no TransposeOut with fixed durations); "
                                   "CUDA events on the launching stream around every step of the timed region",
                         "dominant_kernel": dominant},
            "kernels": kernels,
            "cpu_baseline": {"value": cpu_value, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": f"{cpu_sample} evaluations of instances of the same batch, OpenMP over instances, {cpu_dt:.1f} s"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "api": "twb_batch_eval_host (pinned host buffers; H2D, kernels and D2H pipelined in chunks of 512 instances)",
                    "host_cpus_bound_per_rank": numa_cpus,
                    "ceiling": {"value": world * B / d2h_ceiling_s, "unit": UNIT, "d2h_gbs_per_rank": (d2h - 4 * B) / d2h_ceiling_s / 1e9,
                                "how": "bare pinned D2H copy of the step's g + jac bytes on every rank at once, max over ranks, same run"},
                    "frac_of_ceiling": e2e_value / (world * B / d2h_ceiling_s)},
            "config5": config5,
            "gpu_launches": args.steps * batch.launches_per_eval(flags),
            "clocks": sampler.summary() if sampler else None,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    os.environ.setdefault("NCCL_DEBUG", "WARN")   # keeps NCCL's version banner off stdout: rank 0 prints ONE JSON line
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--quick", action="store_true", help="kernel timing only (tuning sweeps): skip e2e and the CPU arm")
    ap.add_argument("--workload", default=None, help="recipe name of towr_b200.configs (default: BASELINE configs[1])")
    ap.add_argument("--batch", type=int, default=0, help="instances per GPU (default 4096)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write g, jac and status of the last timed step as DIR/<name>.npy (float64; rank 0's "
                         f"instances, a fixed seeded sample of them when the batch exceeds {DUMP_BYTES >> 20} MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl cuda (the reference arm sizes its sample by time)")
    global WORKLOAD
    if args.workload:
        WORKLOAD = args.workload
    import fcntl
    import __graft_entry__ as ge
    # every rank builds under one file lock: the first one runs make, the others find everything up to date — nobody
    # imports a half-written library (torchrun starts all ranks at once).  The lock is per user and per tree, outside it.
    lock_path = os.path.join(tempfile.gettempdir(),
                             f"towr_b200-build-{os.getuid()}-{hashlib.sha1(ROOT.encode()).hexdigest()[:16]}.lock")
    with open(lock_path, "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        ge.build(quiet=True, import_package=(args.impl != "reference"))
        fcntl.flock(lock, fcntl.LOCK_UN)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
