/* towr_b200.h — C ABI of the B200-native NLP-evaluation path for towr.
 *
 * This is the drop-in boundary (DESIGN.md §2): everything below replaces, for
 * a whole batch of independent problem instances at once, what the reference
 * serves one instance at a time through ifopt::Problem:
 *
 *   ifopt::Problem::GetNumberOfOptimizationVariables / GetNumberOfConstraints
 *   ifopt::Problem::GetJacobianOfConstraints  (structure: rows then ascending cols)
 *   ifopt::Problem::GetBoundsOnOptimizationVariables / GetBoundsOnConstraints
 *   ifopt::Problem::GetVariableValues          (initial guess)
 *   ifopt::Problem::EvaluateConstraints / EvalNonzerosOfJacobian
 *   ifopt::Problem::EvaluateCostFunction / EvaluateCostFunctionGradient
 *
 * assembled from the reference's
 *   towr/src/nlp_formulation.cc:63-376   (variable sets, constraint sets, costs)
 *   towr/src/parameters.cc:40-135        (towr::Parameters defaults)
 * The per-set views (ifopt Component API: GetValues / GetBounds /
 * FillJacobianBlock, reference headers towr/include/towr/constraints/) are
 * served by twb_layout_* + slices of the flat arrays; see INTEGRATION.md.
 *
 * Plain C: opaque handles, caller-allocated arrays, int status returns
 * (0 = TWB_OK), never throws across the boundary.  All reals are fp64, all
 * indices 32-bit int, 0-based.
 */
#ifndef TOWR_B200_H_
#define TOWR_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define TWB_MAX_EE 4
#define TWB_MAX_PHASES 32
#define TWB_MAX_CONSTRAINTS 16
#define TWB_MAX_COSTS 8

/* status codes */
enum {
  TWB_OK = 0,
  TWB_ERR_INVALID = 1,     /* bad argument / spec */
  TWB_ERR_UNSUPPORTED = 2, /* valid towr configuration the device path does not serve yet */
  TWB_ERR_CUDA = 3,        /* CUDA runtime error; see twb_last_error() */
  TWB_ERR_NO_DEVICE = 4    /* no CUDA device: there is NO CPU fallback */
};

/* towr::RobotModel::Robot, towr/include/towr/models/robot_model.h:70-75 */
enum { TWB_MONOPED = 0, TWB_BIPED = 1, TWB_HYQ = 2, TWB_ANYMAL = 3, TWB_GO1 = 4 };

/* towr::HeightMap::TerrainID, towr/include/towr/terrain/height_map.h:79-86 */
enum { TWB_FLAT = 0, TWB_BLOCK = 1, TWB_STAIRS = 2, TWB_GAP = 3, TWB_SLOPE = 4,
       TWB_CHIMNEY = 5, TWB_CHIMNEY_LR = 6, TWB_TERRAIN_COUNT = 7,
       /* towr::HeightMapFromCSV (towr/include/towr/terrain/height_map_from_csv.h:29-111): a cell-constant height grid
        * with one-sided edge slopes; the grid is per-batch data (twb_batch_set_grid_terrain), usable as a per-instance
        * terrain id in twb_batch_set_terrains but not as twb_spec.terrain */
       TWB_GRID_CSV = 7,
       /* towr `Grid` (towr/include/towr/terrain/grid_height_map.h:16-59, what fpowr's footstep_plan_server.cc:155 plans on):
        * a grid_map elevation layer, bilinear height in float, FLT_MAX outside the map, central-difference slopes with
        * eps = resolution / 6; per-batch data (twb_batch_set_grid_map), per-instance terrain id like TWB_GRID_CSV */
       TWB_GRID_MAP = 8 };

/* towr::Parameters::ConstraintName, towr/include/towr/parameters.h:139-147 */
enum { TWB_C_DYNAMIC = 0, TWB_C_EE_ROM = 1, TWB_C_TOTAL_TIME = 2, TWB_C_TERRAIN = 3,
       TWB_C_FORCE = 4, TWB_C_SWING = 5, TWB_C_BASE_ROM = 6, TWB_C_BASE_ACC = 7 };

/* towr::Parameters::CostName, towr/include/towr/parameters.h:148-150 */
enum { TWB_COST_FORCES = 0, TWB_COST_EE_MOTION = 1 };

/* One NLP "structure class" + the instance data of NlpFormulation's public
 * fields (towr/include/towr/nlp_formulation.h:100-105) and towr::Parameters
 * (towr/include/towr/parameters.h:152-214). */
typedef struct twb_spec {
  int robot;                              /* TWB_MONOPED.. */
  int terrain;                            /* default terrain for every instance of a batch */
  int n_ee;                               /* params_.ee_in_contact_at_start_.size() */
  int n_phases[TWB_MAX_EE];               /* params_.ee_phase_durations_.at(ee).size() */
  double phase_durations[TWB_MAX_EE][TWB_MAX_PHASES];
  int in_contact_at_start[TWB_MAX_EE];

  double initial_base_lin_pos[3], initial_base_lin_vel[3];   /* initial_base_.lin */
  double initial_base_ang_pos[3], initial_base_ang_vel[3];   /* initial_base_.ang */
  double final_base_lin_pos[3], final_base_lin_vel[3];       /* final_base_.lin   */
  double final_base_ang_pos[3], final_base_ang_vel[3];       /* final_base_.ang   */
  double initial_ee_W[TWB_MAX_EE][3];                        /* initial_ee_W_     */

  double duration_base_polynomial;        /* parameters.cc:43 */
  int force_polynomials_per_stance_phase; /* :44 */
  int ee_polynomials_per_swing_phase;     /* :45 */
  double force_limit_in_normal_direction; /* :48 */
  double dt_constraint_range_of_motion;   /* :49 */
  double dt_constraint_dynamic;           /* :50 */
  double dt_constraint_base_motion;       /* :51 */
  double bound_phase_duration_min, bound_phase_duration_max; /* :52 */

  int n_constraints;                      /* params_.constraints_ in order */
  int constraints[TWB_MAX_CONSTRAINTS];
  int n_costs;                            /* params_.costs_ in order */
  int cost_ids[TWB_MAX_COSTS];
  double cost_weights[TWB_MAX_COSTS];

  int bounds_final_lin_pos[3];            /* 1 if that dimension is bounded, parameters.cc:66-69 */
  int bounds_final_lin_vel[3];
  int bounds_final_ang_pos[3];
  int bounds_final_ang_vel[3];
} twb_spec;

typedef struct twb_problem twb_problem; /* host-side structure class (+ bounds, x0) */
typedef struct twb_batch twb_batch;     /* B instances of one problem resident on one GPU */

/* ---- setup helpers (host only) ------------------------------------------------ */

/* Parameters::Parameters() defaults (parameters.cc:40-73) + the robot; zero
 * states; no phases. */
int twb_spec_default(twb_spec* spec, int robot);

/* Parameters::OptimizePhaseDurations (parameters.cc:77-80): appends TotalTime. */
int twb_spec_optimize_phase_durations(twb_spec* spec);

/* GaitGenerator::MakeGaitGenerator(n_ee)->SetCombo(combo) then, per foot,
 * GetPhaseDurations(t_total, ee) / IsInContactAtStart(ee)
 * (gait_generator.cc:54-105, {monoped,biped,quadruped}_gait_generator.cc).
 * Fills spec->n_ee, n_phases, phase_durations, in_contact_at_start. */
int twb_spec_set_gait(twb_spec* spec, int n_ee, int combo, double t_total);

/* KinematicModel::GetNominalStanceInBase / GetMaximumDeviationFromNominal and
 * the SRBD constants of the robot (models/examples/(robot)_model.h). */
int twb_robot_info(int robot, int* n_ee, double* mass, double inertia6[6],
                   double nominal_stance[TWB_MAX_EE][3], double max_dev[3]);

/* HeightMap::GetHeight of the analytic terrains (height_map_examples.cc). */
double twb_terrain_height(int terrain, double x, double y);

/* ---- structure class ---------------------------------------------------------- */

int twb_problem_create(const twb_spec* spec, twb_problem** out);
void twb_problem_destroy(twb_problem* p);

/* n = #variables, m = #constraint rows, nnz = #Jacobian non-zeros */
int twb_problem_dims(const twb_problem* p, int* n, int* m, int* nnz);

/* Jacobian structure exactly as IpoptAdapter reads it from
 * GetJacobianOfConstraints(): row-major, ascending column inside a row. */
int twb_problem_structure(const twb_problem* p, int* iRow, int* jCol);
/* CSR row pointer, m+1 entries */
int twb_problem_row_ptr(const twb_problem* p, int* row_ptr);

/* Bounds (ifopt::Bounds, inf = 1e20) and initial guess. */
int twb_problem_bounds(const twb_problem* p, double* x_lower, double* x_upper,
                       double* g_lower, double* g_upper);
/* 1 if the formulation has cost terms (ifopt::Problem::HasCostTerms; params_.costs_ non-empty), else 0 */
int twb_problem_has_cost(const twb_problem* p);
int twb_problem_x0(const twb_problem* p, double* x0);

/* Goal-randomised instances of one structure class (BASELINE configs[2]: "randomized goal/initial-guess instances"):
 * initial guess and variable bounds NlpFormulation::GetVariableSets (nlp_formulation.cc:95-181) produces when only
 * final_base_.lin.p / final_base_.ang.p differ from the spec.  `goals` holds n_goals x {x, y, z, roll, pitch, yaw};
 * x0 / x_lower / x_upper receive n_goals rows of n values (any of them may be NULL).  Structure, constraint bounds
 * and dimensions do not depend on the goal. */
int twb_problem_goal_instances(const twb_problem* p, int n_goals, const double* goals, double* x0, double* x_lower,
                               double* x_upper);

/* Component layout: variable sets (column ranges) and constraint sets (row
 * ranges) in ifopt's Add*Set order; names are the reference's
 * ("base-lin", "ee-motion_0", "dynamic", "rangeofmotion-1", ...). */
int twb_layout_num_variable_sets(const twb_problem* p);
int twb_layout_variable_set(const twb_problem* p, int i, char* name, int name_cap,
                            int* col_start, int* n_cols);
int twb_layout_num_constraint_sets(const twb_problem* p);
int twb_layout_constraint_set(const twb_problem* p, int i, char* name, int name_cap,
                              int* row_start, int* n_rows);

/* ---- batched evaluation on a B200 --------------------------------------------- */

/* Allocates device state for `batch_size` instances on CUDA device `device`.
 * Fails with TWB_ERR_NO_DEVICE when there is none (no CPU fallback). */
int twb_batch_create(const twb_problem* p, int batch_size, int device, twb_batch** out);
void twb_batch_destroy(twb_batch* b);

/* Per-instance terrain ids (host array of batch_size ints). The structure does
 * not depend on the terrain, so one batch may mix terrains. */
int twb_batch_set_terrains(twb_batch* b, const int* terrain_ids);

/* The height grid of TWB_GRID_CSV for this batch: heights[y_cell * cols + x_cell] in metres, cells of 0.17 m
 * (HeightMapFromCSV::res_m_p_cell_), uploaded to the device.  NULL removes it (every height is then 0). */
int twb_batch_set_grid_terrain(twb_batch* b, const double* heights, int rows, int cols);

/* The elevation layer of TWB_GRID_MAP for this batch: heights[ix * size_y + iy] (float, metres) = layer(ix, iy) of a
 * grid_map::GridMap with `resolution` metres per cell centred at (pos_x, pos_y); index 0 is the cell with the LARGEST
 * coordinate (grid_map convention), buffer start index (0, 0).  NULL removes it. */
int twb_batch_set_grid_map(twb_batch* b, const float* heights, int size_x, int size_y, double resolution,
                           double pos_x, double pos_y);

/* Batched setup on the device (no host loop): twb_problem_goal_instances for the B instances of the batch.  goals: device
 * [B][6]; x0 / x_lower / x_upper: device [B][n] (any may be NULL).  The terrain under each goal is the INSTANCE's terrain
 * (twb_batch_set_terrains, height grids included; else twb_spec.terrain).  The call only enqueues on `stream`. */
int twb_batch_goal_instances_device(twb_batch* b, const double* goals, double* x0, double* x_lower, double* x_upper, void* stream);

#define TWB_EVAL_G 1u     /* constraint values        (Problem::EvaluateConstraints)       */
#define TWB_EVAL_JAC 2u   /* Jacobian values          (Problem::EvalNonzerosOfJacobian)    */
#define TWB_EVAL_COST 4u  /* cost + gradient          (EvaluateCostFunction[Gradient])     */
#define TWB_EVAL_ALL 7u

/* Device-pointer variant: all arrays live on the batch's device.
 *   x    [B][n]    in
 *   g    [B][m]    out (may be NULL if !(flags&TWB_EVAL_G))
 *   jac  [B][nnz]  out (CSR value order of twb_problem_structure)
 *   cost [B]       out, grad [B][n] out (only written when the problem has cost terms)
 *   status [B]     out, bit0: non-finite value produced, bit1: sum of phase durations >= T
 * `stream` is a cudaStream_t (NULL = default stream); the call only enqueues.
 * jac must be 16-byte aligned (cudaMalloc'ed arrays are; an odd-offset view of one is not): TWB_ERR_INVALID otherwise.
 * A batch serves ONE evaluation / post-processing call at a time: its staging matrices and fork / join events are shared,
 * so a second call on another stream must be ordered after the first by the caller.
 * The kernels of an evaluation are captured once per argument set (pointers + flags) and replayed as a CUDA graph launched
 * into `stream` (up to 16 sets cached per batch; environment TWB_GRAPH=0: plain launches). */
int twb_batch_eval_device(twb_batch* b, const double* x, double* g, double* jac,
                          double* cost, double* grad, int* status,
                          unsigned flags, void* stream);

/* One step of a device-resident multi-start solver loop on the outputs of twb_batch_eval_device — the stand-in for the IPOPT
 * solves of the reference's drivers (towr/test/hopper_example.cc:77-93, fpowr/src/footstep_plan_server.cc:222-236; IPOPT is
 * not part of this library): a Levenberg-Marquardt FEASIBILITY step for every instance,
 *   r = violation of g against the constraint bounds, Js = diag(s) J with s_i = 1 / max(1, max_k |J_ik|),
 *   (Js^T Js + mu I) dx = -Js^T (s r) by `cg_iters` conjugate-gradient iterations, x <- clip(x + dx min(1, cap / max|dx|)).
 * x [B][n] in / out, g [B][m] and jac [B][nnz] as written by twb_batch_eval_device, x_lower / x_upper [B][n] per-instance
 * variable bounds (both NULL: the problem's own), violation [B] out = max |s r| before the step (may be NULL).  All device
 * pointers; the call only enqueues on `stream`.  Deterministic (fixed summation orders, no atomics). */
int twb_batch_lm_step_device(twb_batch* b, double* x, const double* g, const double* jac, const double* x_lower,
                             const double* x_upper, double mu, double cap, int cg_iters, double* violation, void* stream);

/* Host-pointer variant: copies x up, evaluates, copies the requested outputs
 * back and synchronises. Pinned host memory makes the copies asynchronous. */
int twb_batch_eval_host(twb_batch* b, const double* x, double* g, double* jac,
                        double* cost, double* grad, int* status, unsigned flags);

/* ---- solution post-processing: fpowr::GetTrajectory (fpowr/include/fpowr/footstep_plan_extractor.h:19-53) --------
 * The splines of every instance sampled at t = 0, dt, 2 dt, ... <= T + 1e-5.  Per sample n_values = 19 + 13 n_ee
 * doubles: base lin p, v, a (9) | base orientation quaternion w, x, y, z (4) | angular velocity (3) | angular
 * acceleration (3) | per foot: contact flag 0/1, ee-motion p, v, a (9), ee-force (3). */
int twb_problem_trajectory_dims(const twb_problem* p, double dt, int* n_samples, int* n_values);
/* x: host [B][n] (e.g. converged solutions); out: host [B][n_samples][n_values] */
int twb_batch_sample_trajectory_host(twb_batch* b, const double* x, double dt, double* out);

/* fpowr::ExtractInitialGuess (fpowr/include/fpowr/initial_guess_extractor.h:17-34) for every instance at the caller's
 * sample times (FootstepPlanGoal::state_sample_times).  Per time 49 doubles: time | state[12] = base lin p, base ang p
 * (Euler angles), base lin v, base ang v | controls[36] = ee-motion accelerations (3 per foot, 12), joint torques = 0
 * (12), ee-forces (3 per foot, 12); feet beyond n_ee stay 0 (the reference's layout is sized for four feet).
 * x: host [B][n]; times: host [n_times]; out: host [B][n_times][49] */
int twb_batch_initial_guess_host(twb_batch* b, const double* x, const double* times, int n_times, double* out);

/* fpowr::ExtractFootstepPlan (fpowr/include/fpowr/footstep_plan_extractor.h:55-133) for every instance, without the
 * nearest-plane lookup (boost::geometry over a ROS PlanarTerrain message: stays with the caller, who gets the contact
 * positions): the trajectory sampled every 0.01 s is scanned for changes of the contact set; the first state and every
 * change are footstep states.  (One fused kernel: only the contact flags are walked and the feet's positions evaluated at
 * the changes — bit-identical to sampling the trajectory and scanning it, without the sampled trajectory in memory.)  Per footstep state n_values = 2 + 4 n_ee doubles: t_global | duration (to the next
 * footstep state; the last one up to time_horizon) | per foot: contact flag 0/1, ee position (3).
 * max_states = 1 + sum over feet of (phases - 1) bounds the number of footstep states. */
int twb_problem_footstep_plan_dims(const twb_problem* p, int* max_states, int* n_values);
/* x: host [B][n]; n_states: host [B]; out: host [B][max_states][n_values] (unused states are 0) */
int twb_batch_footstep_plan_host(twb_batch* b, const double* x, double time_horizon, int* n_states, double* out);

/* fpowr::NearestPlaneLookup::GetNearestPlaneIndex (fpowr/include/fpowr/nearest_plane_lookup.h:62-84) for every foot of every
 * footstep state of a plan returned by twb_batch_footstep_plan_host: contact_set[b][state][foot] = index of the polygon
 * nearest to the foot's (x, y) — boost::geometry::distance(point, polygon): 0 inside / on the ring, else the distance to the
 * nearest ring segment; the first polygon wins ties — or -1 for a foot in the air and for unused states
 * (footstep_plan_extractor.h:106-116).  Polygons are plain arrays (what PlanarRegionsToPolygons, :24-55, produces from the
 * PlanarTerrain message): polygon k owns vertices[poly_offsets[k] .. poly_offsets[k+1]-1][2]; like bg::model::polygon's
 * default (closed) ring, the closing segment exists only if the first vertex is repeated at the end.
 * plan: host [B][max_states][2 + 4 n_ee]; n_states: host [B]; contact_set: host [B][max_states][n_ee]. */
int twb_batch_nearest_planes_host(twb_batch* b, const double* plan, const int* n_states, const int* poly_offsets, int n_polys,
                                  const double* vertices, int* contact_set);

/* Device-pointer variants of the four post-processing calls above: the same outputs in the same layouts, computed by the
 * same kernels, for arrays that live on the batch's device (e.g. the iterates of a device-resident solver loop), so that
 * only the results the caller asks for cross PCIe.  `stream` is a cudaStream_t (NULL = default stream).
 *   x [B][n]; out as for the _host twin; n_states [B]; plan [B][max_states][2 + 4 n_ee]; contact_set [B][max_states][n_ee];
 *   poly_offsets [n_polys + 1] and vertices [poly_offsets[n_polys]][2] are device arrays too; `times` stays a HOST array
 *   [n_times] (it selects the sample tables).
 * The footstep plan's rows past n_states[b] are written as 0 by the call (no memset needed).  The offsets cannot be checked
 * on the host here: a polygon with a negative vertex count (poly_offsets[k + 1] < poly_offsets[k]) counts as empty and is
 * never the nearest.  Errors: null required pointers, dt <= 0, n_times <= 0, n_polys < 0: TWB_ERR_INVALID; n_ee > 4 for
 * initial guesses: TWB_ERR_UNSUPPORTED; a failed launch: TWB_ERR_CUDA.  Nothing is enqueued when a call fails its checks.
 * A call only enqueues on `stream` (no host synchronisation, no device allocation) — except the FIRST call with a given
 * table key (trajectory dt; footstep plan; the contents of `times`): it builds the sample tables on the host and uploads
 * them with a blocking copy into a per-batch cache (8 keys, least recently used replaced, freed by twb_batch_destroy).
 * After that first call the same call can be captured into a CUDA graph; the graph stays valid while its key is cached.
 * Like twb_batch_eval_device these calls stage the iterates in the batch's shared transposed matrix: a batch serves ONE
 * evaluation / post-processing call at a time, so a second call on another stream must be ordered after the first by the
 * caller. */
int twb_batch_sample_trajectory_device(twb_batch* b, const double* x, double dt, double* out, void* stream);
int twb_batch_initial_guess_device(twb_batch* b, const double* x, const double* times, int n_times, double* out, void* stream);
int twb_batch_footstep_plan_device(twb_batch* b, const double* x, double time_horizon, int* n_states, double* out, void* stream);
int twb_batch_nearest_planes_device(twb_batch* b, const double* plan, const int* n_states, const int* poly_offsets, int n_polys,
                                    const double* vertices, int* contact_set, void* stream);

/* ---- the two ifopt components of towr that no Parameters::ConstraintName / CostName reaches ---------------------------
 * towr::LinearEqualityConstraint (towr/src/linear_constraint.cc:35-73) on variable set `var_set` (index of
 * twb_layout_variable_set): g[b][rows] = M x_set for every instance (M: host [rows][n_cols], row-major, n_cols = size of
 * the set); its bounds are -v[i] on both sides and its Jacobian block is M.sparseView(): the non-zeros of M, constant.
 * x: host [B][n]; g: host [B][rows]. */
int twb_batch_linear_equality_host(twb_batch* b, const double* x, int var_set, const double* M, int rows, double* g);
/* towr::SoftConstraint (towr/src/soft_constraint.cc:34-72) around constraint set `constraint_set` (index of
 * twb_layout_constraint_set): cost[b] = 0.5 (g - b)^T W (g - b) with b = (upper + lower) / 2 of the set's bounds and
 * grad[b][n] = J^T W (g - b), from the g / Jacobian values of the LAST twb_batch_eval_host(TWB_EVAL_G | TWB_EVAL_JAC) of this
 * batch (they are still on the device).  weights: host [rows of the set] or NULL (ones, the reference's default). */
int twb_batch_soft_constraint_host(twb_batch* b, int constraint_set, const double* weights, double* cost, double* grad);

/* number of kernel launches one twb_batch_eval_device(flags) enqueues */
int twb_batch_launches_per_eval(const twb_batch* b, unsigned flags);

const char* twb_last_error(void);
const char* twb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* TOWR_B200_H_ */
