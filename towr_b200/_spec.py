"""struct twb_spec and the enums of include/towr_b200.h as ctypes definitions.  Pure data: importing this module does NOT
load libtowr_b200.so (bench.py's reference arm and the fixture scripts load it by file path, without the package)."""
import ctypes as C

MAX_EE, MAX_PHASES, MAX_CONSTRAINTS, MAX_COSTS = 4, 32, 16, 8
STATE_DOUBLES = 36   # TWB_STATE_DOUBLES: per-instance state record (formulation.pack_states)

OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_NO_DEVICE = 0, 1, 2, 3, 4
EVAL_G, EVAL_JAC, EVAL_COST, EVAL_ALL = 1, 2, 4, 7
# solve status of an instance (twb_batch_lm_trial_device / twb_batch_lm_accept_device)
LM_RUNNING, LM_CONVERGED, LM_STALLED, LM_NONFINITE = 0, 1, 2, 3
LM_STEP_CAP, LM_STEP_TRUST = 0, 1

# towr::RobotModel::Robot (robot_model.h:70-75)
MONOPED, BIPED, HYQ, ANYMAL, GO1 = range(5)
# towr::HeightMap::TerrainID (height_map.h:79-86)
FLAT, BLOCK, STAIRS, GAP, SLOPE, CHIMNEY, CHIMNEY_LR = range(7)
GRID_CSV = 7   # towr::HeightMapFromCSV; grid data per batch (Batch.set_grid_terrain)
GRID_MAP = 8   # towr Grid (grid_height_map.h): grid_map elevation layer per batch (Batch.set_grid_map) or per instance (Batch.set_grid_maps)
# towr::Parameters::ConstraintName (parameters.h:139-147)
C_DYNAMIC, C_EE_ROM, C_TOTAL_TIME, C_TERRAIN, C_FORCE, C_SWING, C_BASE_ROM, C_BASE_ACC = range(8)
# towr::Parameters::CostName
COST_FORCES, COST_EE_MOTION = range(2)


class Spec(C.Structure):
    """struct twb_spec"""
    _fields_ = [
        ("robot", C.c_int), ("terrain", C.c_int), ("n_ee", C.c_int),
        ("n_phases", C.c_int * MAX_EE),
        ("phase_durations", (C.c_double * MAX_PHASES) * MAX_EE),
        ("in_contact_at_start", C.c_int * MAX_EE),
        ("initial_base_lin_pos", C.c_double * 3), ("initial_base_lin_vel", C.c_double * 3),
        ("initial_base_ang_pos", C.c_double * 3), ("initial_base_ang_vel", C.c_double * 3),
        ("final_base_lin_pos", C.c_double * 3), ("final_base_lin_vel", C.c_double * 3),
        ("final_base_ang_pos", C.c_double * 3), ("final_base_ang_vel", C.c_double * 3),
        ("initial_ee_W", (C.c_double * 3) * MAX_EE),
        ("duration_base_polynomial", C.c_double),
        ("force_polynomials_per_stance_phase", C.c_int),
        ("ee_polynomials_per_swing_phase", C.c_int),
        ("force_limit_in_normal_direction", C.c_double),
        ("dt_constraint_range_of_motion", C.c_double),
        ("dt_constraint_dynamic", C.c_double),
        ("dt_constraint_base_motion", C.c_double),
        ("bound_phase_duration_min", C.c_double), ("bound_phase_duration_max", C.c_double),
        ("n_constraints", C.c_int), ("constraints", C.c_int * MAX_CONSTRAINTS),
        ("n_costs", C.c_int), ("cost_ids", C.c_int * MAX_COSTS), ("cost_weights", C.c_double * MAX_COSTS),
        ("bounds_final_lin_pos", C.c_int * 3), ("bounds_final_lin_vel", C.c_int * 3),
        ("bounds_final_ang_pos", C.c_int * 3), ("bounds_final_ang_vel", C.c_int * 3),
    ]




def motion_velocity_mask(spec, ee):
    """True for the velocity variables of the phase-based set ee-motion_<ee>, in variable order
    (nodes_variables_phase_based.cc:190-253: a swing node holds px, vx, py, vy, pz; the two nodes of a stance phase share
    px, py, pz and have no velocity variables).  Pure Python on the spec: bench.py's reference arm uses it without the library."""
    polys = []                      # True: polynomial of a constant (stance) phase
    const = bool(spec.in_contact_at_start[ee])
    for _ in range(spec.n_phases[ee]):
        polys += [True] if const else [False] * spec.ee_polynomials_per_swing_phase
        const = not const
    n_nodes = len(polys) + 1

    def const_node(i):
        if i == 0:
            return polys[0]
        if i == n_nodes - 1:
            return polys[-1]
        return polys[i - 1] or polys[i]

    mask, nd = [], 0
    while nd < n_nodes:
        if const_node(nd):
            mask += [False, False, False]
            nd += 2
        else:
            mask += [False, True, False, True, False]
            nd += 1
    return mask
