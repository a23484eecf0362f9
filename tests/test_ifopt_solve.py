"""BatchedProblem::Solve in the C++ ifopt layer (include/towr_b200_ifopt.hpp), driven by tests/cpp/ifopt_solve_test.cc: without
a device batch it returns TWB_ERR_NO_DEVICE; on the GPU, after SetStates, it equals twb_batch_lm_solve_device on the same
inputs bit for bit, and GpuProblem(batch, b).GetVariableValues() serves the solved row."""
import os
import subprocess

import numpy as np
import pytest

import towr_b200 as tb
from towr_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "_build", "ifopt_solve_test")


def _run(*args):
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    libdir = os.path.dirname(capi.LIB_PATH)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", os.path.join(ROOT, "tests", "cpp", "ifopt_solve_test.cc"),
                           "-o", EXE, "-L" + libdir, "-ltowr_b200", "-Wl,-rpath," + libdir, "-Wl,-rpath,/usr/local/cuda/lib64"])
    out = subprocess.run([EXE, *args], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stdout[-2000:] + out.stderr
    return out.stdout


def test_solve_without_a_device_batch_returns_no_device():
    _run()


@pytest.mark.gpu
def test_batched_problem_solve_equals_the_c_call():
    import torch
    vals, results = {}, {}
    for line in _run("--gpu").splitlines():
        parts = line.split()
        if parts and parts[0] in ("state", "x"):
            vals[(parts[0], int(parts[1]))] = np.array([float.fromhex(v) for v in parts[2:]])
        elif parts and parts[0] == "result":
            results[int(parts[1])] = (int(parts[2]), int(parts[3]), float.fromhex(parts[4]), float.fromhex(parts[5]))
    B = len(results)
    p = tb.Problem(tb.make_formulation("anymal_trot_block_base_rom").to_spec())
    S = np.stack([vals[("state", k)] for k in range(B)])
    x0, xl, xu, gl, gu = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in p.state_instances(S))
    bt = p.batch(B)
    X = x0.clone()
    status, its, viol, mu, counts, loops = bt.lm_solve_device(X, xl, xu, gl, gu, max_iters=30, tol=1.0)
    torch.cuda.synchronize()
    Xh = X.cpu().numpy()
    assert not np.array_equal(Xh, x0.cpu().numpy())
    for b in range(B):
        assert np.array_equal(vals[("x", b)].view(np.int64), Xh[b].view(np.int64)), b
        st, it, v, m = results[b]
        assert (st, it) == (status[b].item(), its[b].item()), b
        assert np.array_equal(np.float64(v).view(np.int64), viol[b].cpu().numpy().view(np.int64)), b
        assert np.array_equal(np.float64(m).view(np.int64), mu[b].cpu().numpy().view(np.int64)), b
