"""Per-instance start states in the C++ ifopt layer (include/towr_b200_ifopt.hpp: BatchedProblem::SetStates and the bounds the
GpuProblem views serve), driven by tests/cpp/ifopt_states_test.cc without a GPU and checked bit for bit against
twb_problem_state_instances through the Python binding."""
import os
import subprocess

import numpy as np

import towr_b200 as tb
from towr_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "_build", "ifopt_states_test")


def _run():
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    libdir = os.path.dirname(capi.LIB_PATH)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", os.path.join(ROOT, "tests", "cpp", "ifopt_states_test.cc"),
                           "-o", EXE, "-L" + libdir, "-ltowr_b200", "-Wl,-rpath," + libdir, "-Wl,-rpath,/usr/local/cuda/lib64"])
    out = subprocess.run([EXE], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stdout[-2000:] + out.stderr
    vals = {}
    for line in out.stdout.splitlines():
        parts = line.split()
        if len(parts) >= 2 and parts[0] not in ("dims", "ok"):
            vals[(parts[0], int(parts[1]))] = np.array([float.fromhex(v) for v in parts[2:]])
    return vals


def test_set_states_serves_each_instances_own_bounds():
    vals = _run()
    p = tb.Problem(tb.make_formulation("anymal_trot_block_base_rom").to_spec())
    # the C++ recipe is the Python one: same dimensions, initial guess and bounds
    xl, xu, gl, gu = p.bounds()
    assert np.array_equal(vals[("problem_x0", 0)], p.GetVariableValues())
    assert np.array_equal(vals[("problem_gl", 0)], gl)
    # without SetStates the views serve the problem's bounds and initial guess
    for key, want in (("x0", p.GetVariableValues()), ("xl", xl), ("xu", xu), ("gl", gl), ("gu", gu)):
        assert np.array_equal(vals[("spec_" + key, 1)], want), key
    S = np.stack([vals[("state", k)] for k in range(3)])
    assert S.shape == (3, capi.STATE_DOUBLES)
    x0, sxl, sxu, sgl, sgu = p.state_instances(S)
    for b in range(3):
        for key, want in (("x0", x0[b]), ("xl", sxl[b]), ("xu", sxu[b]), ("gl", sgl[b]), ("gu", sgu[b])):
            got = vals[("inst_" + key, b)]
            assert np.array_equal(got.view(np.int64), want.view(np.int64)), (b, key)
    # the base-ROM rows make the instances' constraint bounds differ from each other and from the problem's
    assert not np.array_equal(sgl[0], gl) and not np.array_equal(sgl[0], sgl[2]) and not np.array_equal(sgu[1], sgu[2])
    # instance 3 got no state record: the problem's
    for key, want in (("x0", p.GetVariableValues()), ("xl", xl), ("xu", xu), ("gl", gl), ("gu", gu)):
        assert np.array_equal(vals[("inst_" + key, 3)], want), key
