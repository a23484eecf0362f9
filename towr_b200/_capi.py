"""ctypes binding of include/towr_b200.h (the C ABI of libtowr_b200.so).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C
towr_b200/csrc``.  There is no Python or CPU fallback for the evaluation path:
if the shared library is missing, importing this module raises.
"""
import ctypes as C
import os

from ._spec import *   # noqa: F401,F403  (Spec, the enums and size limits)
from ._spec import Spec


# TWB_LIB: developer knob for tuning sweeps (scripts/build_variants.sh) — another build of the same library
LIB_PATH = os.environ.get("TWB_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libtowr_b200.so")


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(towr_b200 has no fallback path)")
    lib = C.CDLL(LIB_PATH)
    P, D, I = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)
    sig = {
        "twb_spec_default": (C.c_int, [C.POINTER(Spec), C.c_int]),
        "twb_spec_optimize_phase_durations": (C.c_int, [C.POINTER(Spec)]),
        "twb_spec_set_gait": (C.c_int, [C.POINTER(Spec), C.c_int, C.c_int, C.c_double]),
        "twb_robot_info": (C.c_int, [C.c_int, I, D, D, D, D]),
        "twb_terrain_height": (C.c_double, [C.c_int, C.c_double, C.c_double]),
        "twb_problem_create": (C.c_int, [C.POINTER(Spec), C.POINTER(P)]),
        "twb_problem_destroy": (None, [P]),
        "twb_problem_dims": (C.c_int, [P, I, I, I]),
        "twb_problem_structure": (C.c_int, [P, I, I]),
        "twb_problem_row_ptr": (C.c_int, [P, I]),
        "twb_problem_bounds": (C.c_int, [P, D, D, D, D]),
        "twb_problem_x0": (C.c_int, [P, D]),
        "twb_problem_has_cost": (C.c_int, [P]),
        "twb_problem_goal_instances": (C.c_int, [P, C.c_int, D, D, D, D]),
        "twb_layout_num_variable_sets": (C.c_int, [P]),
        "twb_layout_variable_set": (C.c_int, [P, C.c_int, C.c_char_p, C.c_int, I, I]),
        "twb_layout_num_constraint_sets": (C.c_int, [P]),
        "twb_layout_constraint_set": (C.c_int, [P, C.c_int, C.c_char_p, C.c_int, I, I]),
        "twb_batch_create": (C.c_int, [P, C.c_int, C.c_int, C.POINTER(P)]),
        "twb_batch_destroy": (None, [P]),
        "twb_batch_set_terrains": (C.c_int, [P, I]),
        "twb_batch_set_grid_terrain": (C.c_int, [P, D, C.c_int, C.c_int]),
        "twb_batch_set_grid_map": (C.c_int, [P, C.POINTER(C.c_float), C.c_int, C.c_int, C.c_double, C.c_double, C.c_double]),
        "twb_batch_goal_instances_device": (C.c_int, [P, P, P, P, P, P]),
        "twb_batch_eval_device": (C.c_int, [P, P, P, P, P, P, P, C.c_uint, P]),
        "twb_batch_eval_host": (C.c_int, [P, P, P, P, P, P, P, C.c_uint]),
        "twb_batch_lm_step_device": (C.c_int, [P, P, P, P, P, P, C.c_double, C.c_double, C.c_int, P, P]),
        "twb_problem_trajectory_dims": (C.c_int, [P, C.c_double, I, I]),
        "twb_batch_sample_trajectory_host": (C.c_int, [P, P, C.c_double, P]),
        "twb_batch_initial_guess_host": (C.c_int, [P, P, P, C.c_int, P]),
        "twb_problem_footstep_plan_dims": (C.c_int, [P, I, I]),
        "twb_batch_footstep_plan_host": (C.c_int, [P, P, C.c_double, P, P]),
        "twb_batch_nearest_planes_host": (C.c_int, [P, P, P, P, C.c_int, P, P]),
        "twb_batch_sample_trajectory_device": (C.c_int, [P, P, C.c_double, P, P]),
        "twb_batch_initial_guess_device": (C.c_int, [P, P, P, C.c_int, P, P]),
        "twb_batch_footstep_plan_device": (C.c_int, [P, P, C.c_double, P, P, P]),
        "twb_batch_nearest_planes_device": (C.c_int, [P, P, P, P, C.c_int, P, P, P]),
        "twb_batch_linear_equality_host": (C.c_int, [P, P, C.c_int, P, C.c_int, P]),
        "twb_batch_soft_constraint_host": (C.c_int, [P, C.c_int, P, P, P]),
        "twb_batch_launches_per_eval": (C.c_int, [P, C.c_uint]),
        "twb_last_error": (C.c_char_p, []),
        "twb_version": (C.c_char_p, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib, list(sig)


lib, EXPORTS = _load()


class TowrB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"towr_b200 error {code}: {msg}")
        self.code = code


def check(rc):
    if rc != OK:
        raise TowrB200Error(rc, lib.twb_last_error().decode())
