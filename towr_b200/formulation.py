"""Host-side mirror of the reference interface for the NLP-evaluation path.

``NlpFormulation`` / ``Parameters`` / ``BaseState`` / ``GaitGenerator`` keep the
field and method names of the reference (towr/include/towr/nlp_formulation.h:
100-105, parameters.h:139-214, variables/state.h, initialization/
gait_generator.h) so a towr user fills them the same way; ``Problem`` stands
where ``ifopt::Problem`` stands (structure, bounds, initial guess, evaluation),
for a whole batch of instances.  All work happens in libtowr_b200.so.
"""
import ctypes as C

import numpy as np

from . import _capi as capi
from ._capi import lib, check


class Node:
    """towr::Node (variables/state.h): value and first derivative."""

    def __init__(self):
        self.p = np.zeros(3)
        self.v = np.zeros(3)


class BaseState:
    """towr::BaseState: lin (x,y,z) and ang (roll,pitch,yaw) nodes."""

    def __init__(self):
        self.lin = Node()
        self.ang = Node()


class Parameters:
    """towr::Parameters (parameters.cc:40-73 defaults come from the C ABI)."""

    def __init__(self, robot=capi.MONOPED):
        s = capi.Spec()
        check(lib.twb_spec_default(C.byref(s), robot))
        self.ee_phase_durations_ = []
        self.ee_in_contact_at_start_ = []
        self.constraints_ = [s.constraints[i] for i in range(s.n_constraints)]
        self.costs_ = []
        self.dt_constraint_dynamic_ = s.dt_constraint_dynamic
        self.dt_constraint_range_of_motion_ = s.dt_constraint_range_of_motion
        self.dt_constraint_base_motion_ = s.dt_constraint_base_motion
        self.duration_base_polynomial_ = s.duration_base_polynomial
        self.ee_polynomials_per_swing_phase_ = s.ee_polynomials_per_swing_phase
        self.force_polynomials_per_stance_phase_ = s.force_polynomials_per_stance_phase
        self.force_limit_in_normal_direction_ = s.force_limit_in_normal_direction
        self.bounds_final_lin_pos_ = [d for d in range(3) if s.bounds_final_lin_pos[d]]
        self.bounds_final_lin_vel_ = [d for d in range(3) if s.bounds_final_lin_vel[d]]
        self.bounds_final_ang_pos_ = [d for d in range(3) if s.bounds_final_ang_pos[d]]
        self.bounds_final_ang_vel_ = [d for d in range(3) if s.bounds_final_ang_vel[d]]
        self.bound_phase_duration_ = (s.bound_phase_duration_min, s.bound_phase_duration_max)

    def OptimizePhaseDurations(self):
        self.constraints_.append(capi.C_TOTAL_TIME)

    def IsOptimizeTimings(self):
        return capi.C_TOTAL_TIME in self.constraints_

    def GetEECount(self):
        return len(self.ee_in_contact_at_start_)

    def GetPhaseCount(self, ee):
        return len(self.ee_phase_durations_[ee])

    def GetTotalTime(self):
        return float(sum(self.ee_phase_durations_[0])) if self.ee_phase_durations_ else 0.0


class GaitGenerator:
    """towr::GaitGenerator::MakeGaitGenerator(n_ee) + SetCombo + GetPhaseDurations."""

    def __init__(self, n_ee):
        self.n_ee = n_ee
        self.combo = 0

    @staticmethod
    def MakeGaitGenerator(leg_count):
        return GaitGenerator(leg_count)

    def SetCombo(self, combo):
        self.combo = int(combo)

    def _spec(self, t_total):
        s = capi.Spec()
        check(lib.twb_spec_set_gait(C.byref(s), self.n_ee, self.combo, float(t_total)))
        return s

    def GetPhaseDurations(self, t_total, ee):
        s = self._spec(t_total)
        return [s.phase_durations[ee][i] for i in range(s.n_phases[ee])]

    def IsInContactAtStart(self, ee):
        return bool(self._spec(1.0).in_contact_at_start[ee])


def robot_info(robot):
    n_ee, mass = C.c_int(), C.c_double()
    inertia = (C.c_double * 6)()
    nominal = ((C.c_double * 3) * capi.MAX_EE)()
    dev = (C.c_double * 3)()
    check(lib.twb_robot_info(robot, C.byref(n_ee), C.byref(mass), inertia,
                             C.cast(nominal, C.POINTER(C.c_double)), dev))
    return dict(n_ee=n_ee.value, mass=mass.value, inertia=list(inertia),
                nominal_stance=[list(nominal[e]) for e in range(n_ee.value)], max_dev=list(dev))


def terrain_height(terrain, x, y):
    return lib.twb_terrain_height(int(terrain), float(x), float(y))


class NlpFormulation:
    """towr::NlpFormulation: public fields + to_spec() instead of Get*Sets()."""

    def __init__(self, robot=capi.MONOPED, terrain=capi.FLAT):
        self.initial_base_ = BaseState()
        self.final_base_ = BaseState()
        self.initial_ee_W_ = []
        self.model_ = robot
        self.terrain_ = terrain
        self.params_ = Parameters(robot)

    def to_spec(self):
        p = self.params_
        s = capi.Spec()
        check(lib.twb_spec_default(C.byref(s), self.model_))
        s.terrain = int(self.terrain_)
        s.n_ee = p.GetEECount()
        if s.n_ee > capi.MAX_EE or len(self.initial_ee_W_) != s.n_ee:
            raise ValueError("initial_ee_W_ / ee_in_contact_at_start_ size mismatch")
        for ee in range(s.n_ee):
            d = p.ee_phase_durations_[ee]
            if len(d) > capi.MAX_PHASES:
                raise ValueError("too many phases")
            s.n_phases[ee] = len(d)
            for i, v in enumerate(d):
                s.phase_durations[ee][i] = v
            s.in_contact_at_start[ee] = int(bool(p.ee_in_contact_at_start_[ee]))
            for k in range(3):
                s.initial_ee_W[ee][k] = float(self.initial_ee_W_[ee][k])
        for k in range(3):
            s.initial_base_lin_pos[k] = float(self.initial_base_.lin.p[k])
            s.initial_base_lin_vel[k] = float(self.initial_base_.lin.v[k])
            s.initial_base_ang_pos[k] = float(self.initial_base_.ang.p[k])
            s.initial_base_ang_vel[k] = float(self.initial_base_.ang.v[k])
            s.final_base_lin_pos[k] = float(self.final_base_.lin.p[k])
            s.final_base_lin_vel[k] = float(self.final_base_.lin.v[k])
            s.final_base_ang_pos[k] = float(self.final_base_.ang.p[k])
            s.final_base_ang_vel[k] = float(self.final_base_.ang.v[k])
            s.bounds_final_lin_pos[k] = int(k in p.bounds_final_lin_pos_)
            s.bounds_final_lin_vel[k] = int(k in p.bounds_final_lin_vel_)
            s.bounds_final_ang_pos[k] = int(k in p.bounds_final_ang_pos_)
            s.bounds_final_ang_vel[k] = int(k in p.bounds_final_ang_vel_)
        s.duration_base_polynomial = p.duration_base_polynomial_
        s.force_polynomials_per_stance_phase = p.force_polynomials_per_stance_phase_
        s.ee_polynomials_per_swing_phase = p.ee_polynomials_per_swing_phase_
        s.force_limit_in_normal_direction = p.force_limit_in_normal_direction_
        s.dt_constraint_range_of_motion = p.dt_constraint_range_of_motion_
        s.dt_constraint_dynamic = p.dt_constraint_dynamic_
        s.dt_constraint_base_motion = p.dt_constraint_base_motion_
        s.bound_phase_duration_min, s.bound_phase_duration_max = p.bound_phase_duration_
        s.n_constraints = len(p.constraints_)
        for i, c in enumerate(p.constraints_):
            s.constraints[i] = int(c)
        s.n_costs = len(p.costs_)
        for i, (cid, w) in enumerate(p.costs_):
            s.cost_ids[i] = int(cid)
            s.cost_weights[i] = float(w)
        return s

    def state_record(self):
        """initial_base_, final_base_ and initial_ee_W_ of this formulation as one (STATE_DOUBLES,) state record."""
        return pack_states([self.initial_base_], [self.final_base_], [self.initial_ee_W_])[0]


def pack_states(initial_bases, final_bases, initial_ee_W):
    """Per-instance start / goal states as the C ABI takes them (TWB_STATE_DOUBLES): a (B, 36) float64 array from B
    initial BaseStates, B final BaseStates and B lists of foot positions (initial_ee_W_, at most MAX_EE feet of 3 values):
    initial lin p, v, ang p, v | final lin p, v, ang p, v | feet [MAX_EE][3] (feet beyond the list stay 0)."""
    B = len(initial_bases)
    if len(final_bases) != B or len(initial_ee_W) != B:
        raise ValueError("initial_bases, final_bases and initial_ee_W must have one entry per instance")
    out = np.zeros((B, capi.STATE_DOUBLES))
    for b in range(B):
        i, f = initial_bases[b], final_bases[b]
        out[b, :24] = np.concatenate([i.lin.p, i.lin.v, i.ang.p, i.ang.v, f.lin.p, f.lin.v, f.ang.p, f.ang.v])
        feet = np.asarray(initial_ee_W[b], np.float64).reshape(-1, 3)
        if len(feet) > capi.MAX_EE:
            raise ValueError("more than MAX_EE feet")
        out[b, 24:24 + 3 * len(feet)] = feet.ravel()
    return out


class Problem:
    """One structure class: what ifopt::Problem exposes besides evaluation."""

    def __init__(self, spec):
        self.spec = spec
        self._h = C.c_void_p()
        check(lib.twb_problem_create(C.byref(spec), C.byref(self._h)))
        n, m, nnz = C.c_int(), C.c_int(), C.c_int()
        check(lib.twb_problem_dims(self._h, C.byref(n), C.byref(m), C.byref(nnz)))
        self.n, self.m, self.nnz = n.value, m.value, nnz.value

    def __del__(self):
        if getattr(self, "_h", None):
            lib.twb_problem_destroy(self._h)
            self._h = None

    # ifopt::Problem::GetNumberOfOptimizationVariables / GetNumberOfConstraints
    def GetNumberOfOptimizationVariables(self):
        return self.n

    def GetNumberOfConstraints(self):
        return self.m

    def structure(self):
        """(iRow, jCol) as IpoptAdapter reads them from GetJacobianOfConstraints()."""
        r = np.empty(self.nnz, np.int32)
        c = np.empty(self.nnz, np.int32)
        ip = C.POINTER(C.c_int)
        check(lib.twb_problem_structure(self._h, r.ctypes.data_as(ip), c.ctypes.data_as(ip)))
        return r, c

    def row_ptr(self):
        rp = np.empty(self.m + 1, np.int32)
        check(lib.twb_problem_row_ptr(self._h, rp.ctypes.data_as(C.POINTER(C.c_int))))
        return rp

    def bounds(self):
        """GetBoundsOnOptimizationVariables / GetBoundsOnConstraints -> xl, xu, gl, gu."""
        dp = C.POINTER(C.c_double)
        xl, xu = np.empty(self.n), np.empty(self.n)
        gl, gu = np.empty(self.m), np.empty(self.m)
        check(lib.twb_problem_bounds(self._h, xl.ctypes.data_as(dp), xu.ctypes.data_as(dp),
                                     gl.ctypes.data_as(dp), gu.ctypes.data_as(dp)))
        return xl, xu, gl, gu

    def GetVariableValues(self):
        x0 = np.empty(self.n)
        check(lib.twb_problem_x0(self._h, x0.ctypes.data_as(C.POINTER(C.c_double))))
        return x0

    def goal_instances(self, goals):
        """x0, x_lower, x_upper (each (G, n)) of instances that differ from the spec only in their goal pose;
        goals: (G, 6) = final base x, y, z, roll, pitch, yaw (NlpFormulation::final_base_)."""
        goals = np.ascontiguousarray(goals, np.float64)
        assert goals.ndim == 2 and goals.shape[1] == 6
        G = goals.shape[0]
        x0, xl, xu = np.empty((G, self.n)), np.empty((G, self.n)), np.empty((G, self.n))
        dp = C.POINTER(C.c_double)
        check(lib.twb_problem_goal_instances(self._h, G, goals.ctypes.data_as(dp), x0.ctypes.data_as(dp),
                                             xl.ctypes.data_as(dp), xu.ctypes.data_as(dp)))
        return x0, xl, xu

    def state_instances(self, states):
        """x0, x_lower, x_upper (each (S, n)) and g_lower, g_upper (each (S, m)) of instances with their own start and goal
        states; states: (S, 36) state records (pack_states).  Only the BaseMotionConstraint LZ rows of the constraint bounds
        differ between instances."""
        states = np.ascontiguousarray(states, np.float64)
        assert states.ndim == 2 and states.shape[1] == capi.STATE_DOUBLES
        S = states.shape[0]
        x0, xl, xu = np.empty((S, self.n)), np.empty((S, self.n)), np.empty((S, self.n))
        gl, gu = np.empty((S, self.m)), np.empty((S, self.m))
        dp = C.POINTER(C.c_double)
        check(lib.twb_problem_state_instances(self._h, S, states.ctypes.data_as(dp), x0.ctypes.data_as(dp), xl.ctypes.data_as(dp),
                                              xu.ctypes.data_as(dp), gl.ctypes.data_as(dp), gu.ctypes.data_as(dp)))
        return x0, xl, xu, gl, gu

    def _components(self, count_fn, get_fn):
        out = []
        buf = C.create_string_buffer(64)
        for i in range(count_fn(self._h)):
            a, b = C.c_int(), C.c_int()
            check(get_fn(self._h, i, buf, 64, C.byref(a), C.byref(b)))
            out.append((buf.value.decode(), a.value, b.value))
        return out

    def variable_sets(self):
        return self._components(lib.twb_layout_num_variable_sets, lib.twb_layout_variable_set)

    def constraint_sets(self):
        return self._components(lib.twb_layout_num_constraint_sets, lib.twb_layout_constraint_set)

    def batch(self, batch_size, device=0):
        return Batch(self, batch_size, device)


def pack_polygons(polygons):
    """A list of (k_i, 2) vertex arrays (world x, y of the planar regions' boundaries) as the C ABI takes them:
    (poly_offsets int32 (n_polys + 1,), vertices float64 (total, 2)); polygon k owns vertices[offs[k]:offs[k + 1]]."""
    offs = np.zeros(len(polygons) + 1, np.int32)
    offs[1:] = np.cumsum([len(q) for q in polygons])
    verts = np.ascontiguousarray(np.concatenate([np.asarray(q, np.float64).reshape(-1, 2) for q in polygons]) if polygons else np.zeros((0, 2)))
    return offs, verts


def pack_polygon_sets(polygon_sets):
    """One list of polygons per instance (each as pack_polygons takes it) as one shared list: (poly_offsets, vertices,
    poly_ranges int32 (n_sets, 2)); instance b's polygons are poly_ranges[b, 0] .. poly_ranges[b, 0] + poly_ranges[b, 1] - 1."""
    counts = np.array([len(s) for s in polygon_sets], np.int64)
    ranges = np.zeros((len(polygon_sets), 2), np.int32)
    ranges[:, 1] = counts
    ranges[1:, 0] = np.cumsum(counts)[:-1]
    offs, verts = pack_polygons([q for s in polygon_sets for q in s])
    return offs, verts, ranges


def _stream_ptr(stream, tensor):
    import torch
    return C.c_void_p((torch.cuda.current_stream(tensor.device) if stream is None else stream).cuda_stream)


def _check_tensor(t, dtype, shape, what):
    assert t.is_cuda and t.dtype == dtype and t.is_contiguous() and tuple(t.shape) == tuple(shape), \
        f"{what}: expected a contiguous CUDA {dtype} tensor of shape {tuple(shape)}"


class Batch:
    """B instances of one Problem resident on one GPU."""

    def __init__(self, problem, batch_size, device=0):
        self.problem = problem
        self.B = int(batch_size)
        self.device = device
        self._h = C.c_void_p()
        check(lib.twb_batch_create(problem._h, self.B, device, C.byref(self._h)))

    def __del__(self):
        if getattr(self, "_h", None):
            lib.twb_batch_destroy(self._h)
            self._h = None

    def sample_trajectory(self, x, dt):
        """fpowr::GetTrajectory for every instance: (B, n_samples, 19 + 13 n_ee) — see include/towr_b200.h."""
        p = self.problem
        x = np.ascontiguousarray(x, np.float64)
        assert x.shape == (self.B, p.n)
        ns, nv = C.c_int(), C.c_int()
        check(lib.twb_problem_trajectory_dims(p._h, float(dt), C.byref(ns), C.byref(nv)))
        out = np.empty((self.B, ns.value, nv.value))
        check(lib.twb_batch_sample_trajectory_host(self._h, x.ctypes.data_as(C.c_void_p), float(dt), out.ctypes.data_as(C.c_void_p)))
        return out

    def initial_guesses(self, x, times):
        """fpowr::ExtractInitialGuesses for every instance: (B, n_times, 49) = time | state[12] | controls[36]."""
        p = self.problem
        x = np.ascontiguousarray(x, np.float64)
        times = np.ascontiguousarray(times, np.float64)
        assert x.shape == (self.B, p.n)
        out = np.empty((self.B, times.size, 49))
        check(lib.twb_batch_initial_guess_host(self._h, x.ctypes.data_as(C.c_void_p), times.ctypes.data_as(C.c_void_p),
                                               int(times.size), out.ctypes.data_as(C.c_void_p)))
        return out

    def footstep_plans(self, x, time_horizon):
        """fpowr::ExtractFootstepPlan for every instance (without the nearest-plane lookup): list of (n_states_b,
        2 + 4 n_ee) arrays — t_global | duration | per foot: contact flag, ee position."""
        p = self.problem
        x = np.ascontiguousarray(x, np.float64)
        assert x.shape == (self.B, p.n)
        ms, nv = C.c_int(), C.c_int()
        check(lib.twb_problem_footstep_plan_dims(p._h, C.byref(ms), C.byref(nv)))
        out = np.empty((self.B, ms.value, nv.value))
        count = np.empty(self.B, np.int32)
        check(lib.twb_batch_footstep_plan_host(self._h, x.ctypes.data_as(C.c_void_p), float(time_horizon),
                                               count.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)))
        assert count.max() <= ms.value
        return [out[b, :count[b]] for b in range(self.B)]

    def footstep_contact_sets(self, x, time_horizon, polygons):
        """fpowr::ExtractFootstepPlan including the nearest-plane lookup: `polygons` is a list of (k_i, 2) vertex arrays
        (world x, y of the planar regions' boundaries).  Returns (plans, contact_sets): per instance the footstep states
        (see footstep_plans) and an (n_states_b, n_ee) int array — polygon index under every foot in contact, -1 in the air."""
        offs, verts = pack_polygons(polygons)
        return self._footstep_contact_sets(x, time_horizon, offs, verts, None)

    def footstep_contact_sets_per_instance(self, x, time_horizon, polygon_sets):
        """footstep_contact_sets where every instance has its own planar regions: polygon_sets[b] is instance b's list of
        (k_i, 2) vertex arrays, and its contact sets index into that list."""
        assert len(polygon_sets) == self.B, "one polygon list per instance"
        offs, verts, ranges = pack_polygon_sets(polygon_sets)
        return self._footstep_contact_sets(x, time_horizon, offs, verts, ranges)

    def _footstep_contact_sets(self, x, time_horizon, offs, verts, ranges):
        p = self.problem
        x = np.ascontiguousarray(x, np.float64)
        ms, nv = C.c_int(), C.c_int()
        check(lib.twb_problem_footstep_plan_dims(p._h, C.byref(ms), C.byref(nv)))
        n_ee = (nv.value - 2) // 4
        out = np.zeros((self.B, ms.value, nv.value))
        count = np.empty(self.B, np.int32)
        check(lib.twb_batch_footstep_plan_host(self._h, x.ctypes.data_as(C.c_void_p), float(time_horizon),
                                               count.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)))
        cs = np.empty((self.B, ms.value, n_ee), np.int32)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)
        if ranges is None:
            check(lib.twb_batch_nearest_planes_host(self._h, ptr(out), ptr(count), ptr(offs), len(offs) - 1, ptr(verts), ptr(cs)))
        else:
            check(lib.twb_batch_nearest_planes_ranges_host(self._h, ptr(out), ptr(count), ptr(ranges), ptr(offs), len(offs) - 1,
                                                           ptr(verts), ptr(cs)))
        return [out[b, :count[b]] for b in range(self.B)], [cs[b, :count[b]] for b in range(self.B)]

    # ---- device-pointer variants: torch CUDA tensors in and out, only enqueued on `stream` (default: the current one) ----
    # The first call with a given dt / sample-time list builds and uploads the sample tables (blocking); the later ones can
    # be captured in a CUDA graph.

    def sample_trajectory_device(self, x, dt, out=None, stream=None):
        """sample_trajectory on the device: x (B, n) CUDA float64 -> (B, n_samples, 19 + 13 n_ee) CUDA float64."""
        import torch
        p = self.problem
        _check_tensor(x, torch.float64, (self.B, p.n), "x")
        ns, nv = C.c_int(), C.c_int()
        check(lib.twb_problem_trajectory_dims(p._h, float(dt), C.byref(ns), C.byref(nv)))
        if out is None:
            out = torch.empty((self.B, ns.value, nv.value), dtype=torch.float64, device=x.device)
        _check_tensor(out, torch.float64, (self.B, ns.value, nv.value), "out")
        check(lib.twb_batch_sample_trajectory_device(self._h, C.c_void_p(x.data_ptr()), float(dt), C.c_void_p(out.data_ptr()),
                                                     _stream_ptr(stream, x)))
        return out

    def initial_guesses_device(self, x, times, out=None, stream=None):
        """initial_guesses on the device: x (B, n) CUDA float64, times a host sequence -> (B, n_times, 49) CUDA float64."""
        import torch
        p = self.problem
        _check_tensor(x, torch.float64, (self.B, p.n), "x")
        times = np.ascontiguousarray(times, np.float64)
        if out is None:
            out = torch.empty((self.B, times.size, 49), dtype=torch.float64, device=x.device)
        _check_tensor(out, torch.float64, (self.B, times.size, 49), "out")
        check(lib.twb_batch_initial_guess_device(self._h, C.c_void_p(x.data_ptr()), times.ctypes.data_as(C.c_void_p), int(times.size),
                                                 C.c_void_p(out.data_ptr()), _stream_ptr(stream, x)))
        return out

    def footstep_plan_dims(self):
        ms, nv = C.c_int(), C.c_int()
        check(lib.twb_problem_footstep_plan_dims(self.problem._h, C.byref(ms), C.byref(nv)))
        return ms.value, nv.value

    def footstep_plans_device(self, x, time_horizon, out=None, stream=None):
        """footstep_plans on the device: x (B, n) CUDA float64 -> (plans (B, max_states, 2 + 4 n_ee) CUDA float64, rows past
        n_states[b] are 0; n_states (B,) CUDA int32).  `out`: an optional (plans, n_states) pair to write into."""
        import torch
        p = self.problem
        _check_tensor(x, torch.float64, (self.B, p.n), "x")
        ms, nv = self.footstep_plan_dims()
        if out is None:
            out = (torch.empty((self.B, ms, nv), dtype=torch.float64, device=x.device), torch.empty(self.B, dtype=torch.int32, device=x.device))
        plans, count = out
        _check_tensor(plans, torch.float64, (self.B, ms, nv), "plans")
        _check_tensor(count, torch.int32, (self.B,), "n_states")
        check(lib.twb_batch_footstep_plan_device(self._h, C.c_void_p(x.data_ptr()), float(time_horizon), C.c_void_p(count.data_ptr()),
                                                 C.c_void_p(plans.data_ptr()), _stream_ptr(stream, x)))
        return plans, count

    def nearest_planes_device(self, plans, n_states, poly_offsets, vertices, out=None, stream=None):
        """The nearest-plane lookup of footstep_contact_sets on the device: plans / n_states as footstep_plans_device returns
        them, poly_offsets (n_polys + 1,) CUDA int32 and vertices (total, 2) CUDA float64 (pack_polygons, then moved to the
        device) -> contact sets (B, max_states, n_ee) CUDA int32: polygon index under every foot in contact, -1 in the air
        and for unused states.  Offsets must ascend: a polygon with a negative vertex count is treated as empty."""
        import torch
        ms, nv = self.footstep_plan_dims()
        n_ee = (nv - 2) // 4
        _check_tensor(plans, torch.float64, (self.B, ms, nv), "plans")
        _check_tensor(n_states, torch.int32, (self.B,), "n_states")
        assert poly_offsets.ndim == 1 and poly_offsets.numel() >= 1, "poly_offsets: (n_polys + 1,)"
        _check_tensor(poly_offsets, torch.int32, (poly_offsets.numel(),), "poly_offsets")
        _check_tensor(vertices, torch.float64, (vertices.shape[0], 2), "vertices")
        if out is None:
            out = torch.empty((self.B, ms, n_ee), dtype=torch.int32, device=plans.device)
        _check_tensor(out, torch.int32, (self.B, ms, n_ee), "out")
        check(lib.twb_batch_nearest_planes_device(self._h, C.c_void_p(plans.data_ptr()), C.c_void_p(n_states.data_ptr()),
                                                  C.c_void_p(poly_offsets.data_ptr()), poly_offsets.numel() - 1,
                                                  C.c_void_p(vertices.data_ptr()), C.c_void_p(out.data_ptr()), _stream_ptr(stream, plans)))
        return out

    def nearest_planes_ranges_device(self, plans, n_states, poly_ranges, poly_offsets, vertices, out=None, stream=None):
        """nearest_planes_device where instance b looks only at its own polygons: poly_ranges (B, 2) CUDA int32 = (first
        polygon, count) of instance b in the shared list (pack_polygon_sets, then moved to the device); the contact sets hold
        the index relative to that first polygon.  Ranges outside the list are clamped to it (the device cannot check them)."""
        import torch
        ms, nv = self.footstep_plan_dims()
        n_ee = (nv - 2) // 4
        _check_tensor(plans, torch.float64, (self.B, ms, nv), "plans")
        _check_tensor(n_states, torch.int32, (self.B,), "n_states")
        _check_tensor(poly_ranges, torch.int32, (self.B, 2), "poly_ranges")
        assert poly_offsets.ndim == 1 and poly_offsets.numel() >= 1, "poly_offsets: (n_polys + 1,)"
        _check_tensor(poly_offsets, torch.int32, (poly_offsets.numel(),), "poly_offsets")
        _check_tensor(vertices, torch.float64, (vertices.shape[0], 2), "vertices")
        if out is None:
            out = torch.empty((self.B, ms, n_ee), dtype=torch.int32, device=plans.device)
        _check_tensor(out, torch.int32, (self.B, ms, n_ee), "out")
        check(lib.twb_batch_nearest_planes_ranges_device(self._h, C.c_void_p(plans.data_ptr()), C.c_void_p(n_states.data_ptr()),
                                                         C.c_void_p(poly_ranges.data_ptr()), C.c_void_p(poly_offsets.data_ptr()),
                                                         poly_offsets.numel() - 1, C.c_void_p(vertices.data_ptr()),
                                                         C.c_void_p(out.data_ptr()), _stream_ptr(stream, plans)))
        return out

    def linear_equality(self, x, var_set, M):
        """towr::LinearEqualityConstraint::GetValues for every instance: (B, rows) = M x_set; var_set is a set name."""
        p = self.problem
        names = [n for n, _, _ in p.variable_sets()]
        x = np.ascontiguousarray(x, np.float64); M = np.ascontiguousarray(M, np.float64)
        assert x.shape == (self.B, p.n) and M.shape[1] == p.variable_sets()[names.index(var_set)][2]
        g = np.empty((self.B, M.shape[0]))
        check(lib.twb_batch_linear_equality_host(self._h, x.ctypes.data_as(C.c_void_p), names.index(var_set), M.ctypes.data_as(C.c_void_p),
                                                 M.shape[0], g.ctypes.data_as(C.c_void_p)))
        return g

    def soft_constraint(self, constraint_set, weights=None):
        """towr::SoftConstraint around a constraint set (by name), from the last eval_host(G | JAC): (cost (B,), grad (B, n))."""
        p = self.problem
        names = [n for n, _, _ in p.constraint_sets()]
        cost = np.empty(self.B); grad = np.empty((self.B, p.n))
        w = None if weights is None else np.ascontiguousarray(weights, np.float64)
        check(lib.twb_batch_soft_constraint_host(self._h, names.index(constraint_set), None if w is None else w.ctypes.data_as(C.c_void_p),
                                                 cost.ctypes.data_as(C.c_void_p), grad.ctypes.data_as(C.c_void_p)))
        return cost, grad

    def set_terrains(self, terrain_ids):
        if terrain_ids is None:
            check(lib.twb_batch_set_terrains(self._h, None))
            return
        t = np.ascontiguousarray(terrain_ids, np.int32)
        assert t.shape == (self.B,)
        check(lib.twb_batch_set_terrains(self._h, t.ctypes.data_as(C.POINTER(C.c_int))))

    def set_grid_terrain(self, heights):
        """heights[y_cell, x_cell] (2-D float64, cells of 0.17 m) of the GRID_CSV terrain; None removes it."""
        if heights is None:
            check(lib.twb_batch_set_grid_terrain(self._h, None, 0, 0))
            return
        h = np.ascontiguousarray(heights, np.float64)
        assert h.ndim == 2
        check(lib.twb_batch_set_grid_terrain(self._h, h.ctypes.data_as(C.POINTER(C.c_double)), h.shape[0], h.shape[1]))

    def set_grid_map(self, heights, resolution, position=(0.0, 0.0)):
        """heights[ix, iy] (2-D float32) = the "elevation" layer of a grid_map::GridMap centred at `position` with
        `resolution` metres per cell (index 0 = largest coordinate), for the GRID_MAP terrain; None removes it."""
        if heights is None:
            check(lib.twb_batch_set_grid_map(self._h, None, 0, 0, 1.0, 0.0, 0.0))
            return
        h = np.ascontiguousarray(heights, np.float32)
        assert h.ndim == 2
        check(lib.twb_batch_set_grid_map(self._h, h.ctypes.data_as(C.POINTER(C.c_float)), h.shape[0], h.shape[1], float(resolution),
                                         float(position[0]), float(position[1])))

    def set_grid_maps(self, maps, map_of_instance=None):
        """Several GRID_MAP layers for this batch: maps is a list of (heights[ix, iy], resolution, position) tuples as
        set_grid_map takes them; instance b uses maps[map_of_instance[b]] (None: every instance uses maps[0]).  An empty
        list removes every map."""
        if not maps:
            check(lib.twb_batch_set_grid_maps(self._h, 0, None, None, None, None))
            return
        layers = [np.ascontiguousarray(h, np.float32) for h, _, _ in maps]
        assert all(h.ndim == 2 for h in layers), "heights: 2-D arrays"
        heights = np.ascontiguousarray(np.concatenate([h.ravel() for h in layers]))
        sizes = np.array([h.shape for h in layers], np.int32)
        geometry = np.array([(float(res), float(pos[0]), float(pos[1])) for _, res, pos in maps], np.float64)
        idx = None
        if map_of_instance is not None:
            idx = np.ascontiguousarray(map_of_instance, np.int32)
            assert idx.shape == (self.B,), "map_of_instance: one map index per instance"
        check(lib.twb_batch_set_grid_maps(self._h, len(layers), heights.ctypes.data_as(C.POINTER(C.c_float)),
                                          sizes.ctypes.data_as(C.POINTER(C.c_int)), geometry.ctypes.data_as(C.POINTER(C.c_double)),
                                          None if idx is None else idx.ctypes.data_as(C.POINTER(C.c_int))))

    def launches_per_eval(self, flags=capi.EVAL_ALL):
        return lib.twb_batch_launches_per_eval(self._h, flags)

    def eval_host(self, x, flags=capi.EVAL_G | capi.EVAL_JAC, out=None):
        """x: (B, n) float64 numpy (pinned or pageable). Returns dict of numpy arrays."""
        p = self.problem
        x = np.ascontiguousarray(x, np.float64)
        assert x.shape == (self.B, p.n)
        out = out or {}
        g = out.get("g") if flags & capi.EVAL_G else None
        jac = out.get("jac") if flags & capi.EVAL_JAC else None
        if flags & capi.EVAL_G and g is None:
            g = np.empty((self.B, p.m))
        if flags & capi.EVAL_JAC and jac is None:
            jac = np.empty((self.B, p.nnz))
        cost = grad = None
        if flags & capi.EVAL_COST:
            cost = out.get("cost", np.empty(self.B))
            grad = out.get("grad", np.empty((self.B, p.n)))
        status = out.get("status", np.empty(self.B, np.int32))
        ptr = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        check(lib.twb_batch_eval_host(self._h, ptr(x), ptr(g), ptr(jac), ptr(cost), ptr(grad), ptr(status), flags))
        return dict(g=g, jac=jac, cost=cost, grad=grad, status=status)

    def goal_instances_device(self, goals, want_bounds=True, stream=None):
        """Batched setup on the device: goals (B, 6) torch CUDA float64 = final base position + final base Euler angles of
        every instance.  Returns (x0, x_lower, x_upper) CUDA tensors of shape (B, n) (bounds None if not wanted).  The terrain
        under each goal is the instance's own (set_terrains / grids)."""
        import torch
        p = self.problem
        assert goals.is_cuda and goals.dtype == torch.float64 and goals.is_contiguous() and tuple(goals.shape) == (self.B, 6)
        if stream is None:
            stream = torch.cuda.current_stream(goals.device)
        x0 = torch.empty((self.B, p.n), dtype=torch.float64, device=goals.device)
        lo = torch.empty_like(x0) if want_bounds else None
        up = torch.empty_like(x0) if want_bounds else None
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        check(lib.twb_batch_goal_instances_device(self._h, ptr(goals), ptr(x0), ptr(lo), ptr(up), C.c_void_p(stream.cuda_stream)))
        return x0, lo, up

    def state_instances_device(self, states, want_bounds=True, want_g_bounds=False, stream=None):
        """Batched setup on the device from per-instance start and goal states: states (B, 36) torch CUDA float64 state
        records (pack_states).  Returns (x0, x_lower, x_upper) of shape (B, n) and (g_lower, g_upper) of shape (B, m) as CUDA
        tensors (None where not wanted).  The terrain under each goal is the instance's own (set_terrains / grids)."""
        import torch
        p = self.problem
        assert states.is_cuda and states.dtype == torch.float64 and states.is_contiguous() and tuple(states.shape) == (self.B, capi.STATE_DOUBLES)
        if stream is None:
            stream = torch.cuda.current_stream(states.device)
        x0 = torch.empty((self.B, p.n), dtype=torch.float64, device=states.device)
        lo = torch.empty_like(x0) if want_bounds else None
        up = torch.empty_like(x0) if want_bounds else None
        gl = torch.empty((self.B, p.m), dtype=torch.float64, device=states.device) if want_g_bounds else None
        gu = torch.empty_like(gl) if want_g_bounds else None
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        check(lib.twb_batch_state_instances_device(self._h, ptr(states), ptr(x0), ptr(lo), ptr(up), ptr(gl), ptr(gu),
                                                   C.c_void_p(stream.cuda_stream)))
        return x0, lo, up, gl, gu

    def lm_step_device(self, x, g, jac, x_lower=None, x_upper=None, mu=1e-2, cap=0.1, cg_iters=25, violation=None, stream=None,
                       g_lower=None, g_upper=None):
        """twb_batch_lm_step_device: one Levenberg-Marquardt feasibility step for every instance on the outputs of
        eval_device; x (B, n) is updated in place.  All arguments are torch CUDA float64 tensors (bounds: (B, n) or None).
        g_lower / g_upper: per-instance constraint bounds, (B, m) each (e.g. from state_instances_device(...,
        want_g_bounds=True)), stepped against with twb_batch_lm_step_bounds_device; None: the problem's own."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(x.device)
        p = self.problem
        for t, count in ((x, self.B * p.n), (g, self.B * p.m), (jac, self.B * p.nnz), (x_lower, self.B * p.n), (x_upper, self.B * p.n),
                         (violation, self.B)):
            assert t is None or (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous() and t.numel() == count), "bad tensor"
        for t in (g_lower, g_upper):
            assert t is None or (torch.is_tensor(t) and t.is_cuda and t.device == x.device and t.dtype == torch.float64 and t.is_contiguous()
                                 and tuple(t.shape) == (self.B, p.m)), "bad constraint bounds: (B, m) contiguous CUDA float64"
        assert (g_lower is None) == (g_upper is None), "g_lower and g_upper: both or neither"
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        if g_lower is None:
            check(lib.twb_batch_lm_step_device(self._h, ptr(x), ptr(g), ptr(jac), ptr(x_lower), ptr(x_upper), float(mu), float(cap),
                                               int(cg_iters), ptr(violation), C.c_void_p(stream.cuda_stream)))
        else:
            check(lib.twb_batch_lm_step_bounds_device(self._h, ptr(x), ptr(g), ptr(jac), ptr(x_lower), ptr(x_upper), ptr(g_lower),
                                                      ptr(g_upper), float(mu), float(cap), int(cg_iters), ptr(violation),
                                                      C.c_void_p(stream.cuda_stream)))

    def _check_lm_tensors(self, x, specs, g_lower, g_upper):
        import torch
        p = self.problem
        sizes = {"n": p.n, "m": p.m, "nnz": p.nnz, "1": 1}
        for t, dt, per in specs:
            assert t is None or (torch.is_tensor(t) and t.is_cuda and t.device == x.device and t.dtype == dt and t.is_contiguous()
                                 and t.numel() == self.B * sizes[per]), "bad tensor"
        for t in (g_lower, g_upper):
            assert t is None or (torch.is_tensor(t) and t.is_cuda and t.device == x.device and t.dtype == torch.float64 and t.is_contiguous()
                                 and tuple(t.shape) == (self.B, p.m)), "bad constraint bounds: (B, m) contiguous CUDA float64"
        assert (g_lower is None) == (g_upper is None), "g_lower and g_upper: both or neither"

    def lm_trial_device(self, x, g, jac, mu, solve_status, x_trial, row_scale, merit, predicted, x_lower=None, x_upper=None,
                        g_lower=None, g_upper=None, cap=0.1, cg_iters=25, tol=1e-6, violation=None, stream=None):
        """twb_batch_lm_trial_device: the trial step of a solve iteration.  Reads x (B, n), g, jac, mu (B,) and solve_status
        (B,) int32; writes x_trial (B, n), row_scale (B, m), merit, predicted and violation (B,) for the RUNNING instances and
        sets their status to LM_CONVERGED or LM_NONFINITE where that applies.  torch CUDA tensors; only enqueues."""
        import torch
        f64, i32 = torch.float64, torch.int32
        self._check_lm_tensors(x, ((x, f64, "n"), (g, f64, "m"), (jac, f64, "nnz"), (mu, f64, "1"), (solve_status, i32, "1"),
                                   (x_trial, f64, "n"), (row_scale, f64, "m"), (merit, f64, "1"), (predicted, f64, "1"),
                                   (x_lower, f64, "n"), (x_upper, f64, "n"), (violation, f64, "1")), g_lower, g_upper)
        if stream is None:
            stream = torch.cuda.current_stream(x.device)
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        check(lib.twb_batch_lm_trial_device(self._h, ptr(x), ptr(g), ptr(jac), ptr(x_lower), ptr(x_upper), ptr(g_lower), ptr(g_upper),
                                            ptr(mu), float(cap), int(cg_iters), float(tol), ptr(solve_status), ptr(x_trial),
                                            ptr(row_scale), ptr(merit), ptr(predicted), ptr(violation), C.c_void_p(stream.cuda_stream)))

    def lm_accept_device(self, x, x_trial, g_trial, row_scale, merit, predicted, mu, nu, solve_status, iterations, g_lower=None,
                         g_upper=None, eta=1e-4, mu_min=1e-12, mu_max=1e10, stream=None):
        """twb_batch_lm_accept_device: the gain-ratio decision of a solve iteration for the RUNNING instances, on g_trial (B, m)
        evaluated at x_trial.  Updates x (accepted: x_trial), mu, nu, solve_status and iterations (B,) int32 in place.  torch
        CUDA tensors; only enqueues."""
        import torch
        f64, i32 = torch.float64, torch.int32
        self._check_lm_tensors(x, ((x, f64, "n"), (x_trial, f64, "n"), (g_trial, f64, "m"), (row_scale, f64, "m"), (merit, f64, "1"),
                                   (predicted, f64, "1"), (mu, f64, "1"), (nu, f64, "1"), (solve_status, i32, "1"),
                                   (iterations, i32, "1")), g_lower, g_upper)
        if stream is None:
            stream = torch.cuda.current_stream(x.device)
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        check(lib.twb_batch_lm_accept_device(self._h, ptr(x), ptr(x_trial), ptr(g_trial), ptr(g_lower), ptr(g_upper), ptr(row_scale),
                                             ptr(merit), ptr(predicted), ptr(mu), ptr(nu), ptr(solve_status), ptr(iterations),
                                             float(eta), float(mu_min), float(mu_max), C.c_void_p(stream.cuda_stream)))

    def lm_solve_device(self, x, x_lower=None, x_upper=None, g_lower=None, g_upper=None, max_iters=60, tol=1e-6, mu0=1e-2, cap=0.1,
                        cg_iters=25, eta=1e-4, mu_min=1e-12, mu_max=1e10, step_rule="cap", radius_max=1e3, out=None, stream=None):
        """twb_batch_lm_solve_device: a whole solve in one call that only enqueues — the loop of BatchedLevenbergMarquardt.solve
        run on the device, stopping at the iteration after which no instance is RUNNING.  x (B, n) is updated in place;
        x_lower / x_upper (B, n) and g_lower / g_upper (B, m): per-instance bounds or None (the problem's own).  Returns
        (status, iterations, violation, mu, counts, loop_count): (B,) int32, (B,) int32, (B,) float64, (B,) float64, (4,) int32
        instances per LM_* status and (1,) int32 loop iterations run, all CUDA tensors.  `out`: those six tensors from an
        earlier call to write into instead; with the same tensors and arguments the call replays the batch's cached graph.
        step_rule: "cap" (max |dx| <= cap, then clipped to the bounds) or "trust" (a trust radius per instance that starts at
        cap, adapts to the gain ratio up to radius_max, with CG on the variables not held at a bound; include/towr_b200.h)."""
        import torch
        f64, i32 = torch.float64, torch.int32
        self._check_lm_tensors(x, ((x, f64, "n"), (x_lower, f64, "n"), (x_upper, f64, "n")), g_lower, g_upper)
        if out is None:
            dev = x.device
            out = (torch.empty(self.B, dtype=i32, device=dev), torch.empty(self.B, dtype=i32, device=dev),
                   torch.empty(self.B, dtype=f64, device=dev), torch.empty(self.B, dtype=f64, device=dev),
                   torch.empty(4, dtype=i32, device=dev), torch.empty(1, dtype=i32, device=dev))
        status, iterations, violation, mu, counts, loop_count = out
        self._check_lm_tensors(x, ((status, i32, "1"), (iterations, i32, "1"), (violation, f64, "1"), (mu, f64, "1")), None, None)
        assert counts.is_cuda and counts.dtype == i32 and counts.numel() == 4 and loop_count.is_cuda and loop_count.dtype == i32 \
            and loop_count.numel() == 1, "bad counts / loop_count"
        rules = {"cap": capi.LM_STEP_CAP, "trust": capi.LM_STEP_TRUST}
        assert step_rule in rules, f"step_rule must be one of {sorted(rules)}"
        opt = capi.LmSolveOptions(float(mu0), float(cap), float(tol), float(eta), float(mu_min), float(mu_max), int(cg_iters), int(max_iters),
                                  rules[step_rule], float(radius_max))
        if stream is None:
            stream = torch.cuda.current_stream(x.device)
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        check(lib.twb_batch_lm_solve_device(self._h, ptr(x), ptr(x_lower), ptr(x_upper), ptr(g_lower), ptr(g_upper), C.byref(opt),
                                            ptr(status), ptr(iterations), ptr(violation), ptr(mu), ptr(counts), ptr(loop_count),
                                            C.c_void_p(stream.cuda_stream)))
        return out

    def lm_solve_radius(self):
        """(radius, step_norm) as (B,) float64 numpy arrays after the batch's last trust-region solve, whose stream the caller
        has synchronised (twb_batch_lm_solve_radius)."""
        radius, step_norm = np.empty(self.B), np.empty(self.B)
        check(lib.twb_batch_lm_solve_radius(self._h, radius.ctypes.data_as(C.POINTER(C.c_double)),
                                            step_norm.ctypes.data_as(C.POINTER(C.c_double))))
        return radius, step_norm

    def lm_solve_graphs_instantiated(self):
        """The solve graphs this batch has instantiated so far (twb_batch_lm_solve_graph_stats)."""
        n = C.c_int()
        check(lib.twb_batch_lm_solve_graph_stats(self._h, C.byref(n)))
        return n.value

    def eval_device(self, x, g=None, jac=None, cost=None, grad=None, status=None,
                    flags=capi.EVAL_G | capi.EVAL_JAC, stream=None):
        """Device-pointer variant. Arguments are torch CUDA float64 tensors (or None);
        `stream` a torch.cuda.Stream (default: current). Only enqueues."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(x.device)
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        p = self.problem
        assert x.is_cuda and x.dtype == torch.float64 and x.is_contiguous() and x.numel() == self.B * p.n
        for t, dt, count in ((g, torch.float64, self.B * p.m), (jac, torch.float64, self.B * p.nnz), (cost, torch.float64, self.B),
                             (grad, torch.float64, self.B * p.n), (status, torch.int32, self.B)):
            assert t is None or (t.is_cuda and t.dtype == dt and t.is_contiguous() and t.numel() == count), "bad output tensor"
        check(lib.twb_batch_eval_device(self._h, ptr(x), ptr(g), ptr(jac), ptr(cost), ptr(grad), ptr(status),
                                        flags, C.c_void_p(stream.cuda_stream)))
