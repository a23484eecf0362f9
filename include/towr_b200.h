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
        * eps = resolution / 6; per-batch data (twb_batch_set_grid_map, or one map per instance with
        * twb_batch_set_grid_maps), per-instance terrain id like TWB_GRID_CSV */
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

/* Per-instance start AND goal states: one fixed-stride record per instance that mirrors NlpFormulation's three state fields
 * (towr/include/towr/nlp_formulation.h:100-105), with the meaning they have in twb_spec. */
#define TWB_STATE_DOUBLES 36
/* per instance, in this order:
 *   initial_base_: lin p[3], lin v[3], ang p[3] (Euler, as twb_spec), ang v[3]      doubles  0..11
 *   final_base_:   lin p[3], lin v[3], ang p[3], ang v[3]                            doubles 12..23
 *   initial_ee_W_: [TWB_MAX_EE][3]; feet beyond n_ee are ignored                     doubles 24..35
 * The final base z only enters the final-position bound (bounds_final_lin_pos); the initial guess ends at the terrain height
 * minus the nominal z, as for the spec.  The final velocities only enter the bounds bounds_final_*_vel selects.  The initial
 * feet are taken as given (not projected onto the terrain). */
/* Initial guess, variable bounds AND constraint bounds of n_states such instances of one structure class.  states: host
 * [n_states][TWB_STATE_DOUBLES]; x0 / x_lower / x_upper: [n_states][n]; g_lower / g_upper: [n_states][m]; any output may be
 * NULL.  The constraint bounds are twb_problem_bounds' except the BaseMotionConstraint (TWB_C_BASE_ROM) LZ rows, which are
 * [z_init - 0.02, z_init + 0.1] around the instance's initial base z (base_motion_constraint.cc:51-54); without
 * TWB_C_BASE_ROM every instance has the problem's constraint bounds.  Errors: NULL states, n_states <= 0: TWB_ERR_INVALID. */
int twb_problem_state_instances(const twb_problem* p, int n_states, const double* states, double* x0, double* x_lower,
                                double* x_upper, double* g_lower, double* g_upper);

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
 * coordinate (grid_map convention), buffer start index (0, 0).  NULL removes it (and every map of twb_batch_set_grid_maps).
 * The same as twb_batch_set_grid_maps(b, 1, heights, {size_x, size_y}, {resolution, pos_x, pos_y}, NULL). */
int twb_batch_set_grid_map(twb_batch* b, const float* heights, int size_x, int size_y, double resolution,
                           double pos_x, double pos_y);

/* n_maps grid_map elevation layers for this batch, so that instances standing on different maps (e.g. the requests of a plan
 * server, each with its own perception) share one batch; instance b uses map map_of_instance[b] wherever its terrain id is
 * TWB_GRID_MAP.  heights: the layers back to back, layer k = [sizes[k][0]][sizes[k][1]] floats, laid out as for
 * twb_batch_set_grid_map; sizes: [n_maps][2] (size_x, size_y); geometry: [n_maps][3] (resolution, pos_x, pos_y);
 * map_of_instance: host [B], each in [0, n_maps), or NULL = every instance uses map 0.  heights NULL or n_maps == 0
 * removes every map (TWB_GRID_MAP instances are then outside the map everywhere: heights FLT_MAX).  The last call of this
 * and twb_batch_set_grid_map wins; the terrain ids of twb_batch_set_terrains are kept, in either call order.
 * Errors: n_maps < 0 or > 2^27, a map with a bad size (at most 2^28 cells) or a resolution / position that is not finite
 * (resolution > 0), an index out of range: TWB_ERR_INVALID, and the previous maps and indices stay in place.
 * Like the other terrain setters, the call drops the batch's cached evaluation graphs. */
int twb_batch_set_grid_maps(twb_batch* b, int n_maps, const float* heights, const int* sizes, const double* geometry,
                            const int* map_of_instance);

/* Batched setup on the device (no host loop): twb_problem_goal_instances for the B instances of the batch.  goals: device
 * [B][6]; x0 / x_lower / x_upper: device [B][n] (any may be NULL).  The terrain under each goal is the INSTANCE's terrain
 * (twb_batch_set_terrains, height grids included; else twb_spec.terrain).  The call only enqueues on `stream`. */
int twb_batch_goal_instances_device(twb_batch* b, const double* goals, double* x0, double* x_lower, double* x_upper, void* stream);

/* Batched setup on the device: twb_problem_state_instances for the B instances of the batch, so that a device-resident
 * pipeline can start every instance from its own measured state.  states: device [B][TWB_STATE_DOUBLES]; x0 / x_lower /
 * x_upper: device [B][n]; g_lower / g_upper: device [B][m]; any output may be NULL, but not all of them.  The terrain under
 * each goal is the instance's own, as for twb_batch_goal_instances_device.  The call only enqueues on `stream` (no host
 * synchronisation, no allocation), so it can be captured in a CUDA graph.  Errors: NULL states, every output NULL:
 * TWB_ERR_INVALID, nothing enqueued.
 * Only the BaseMotionConstraint LZ rows of g_lower / g_upper differ per instance, and only when TWB_C_BASE_ROM is among the
 * constraints (the default list has no such rows).  twb_batch_lm_step_bounds_device steps every instance against its own
 * rows of these outputs; twb_batch_lm_step_device steps against the problem's own constraint bounds. */
int twb_batch_state_instances_device(twb_batch* b, const double* states, double* x0, double* x_lower, double* x_upper,
                                     double* g_lower, double* g_upper, void* stream);

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
 * pointers.  Deterministic (fixed summation orders, no atomics).
 * An instance whose x, g or jac holds a non-finite entry (NaN or +-Inf, e.g. status bit0 of the evaluation) is not stepped:
 * its x is left exactly as it was and violation[b] is NaN.  The other instances of the batch are not affected.
 * The call only enqueues on `stream` (no host synchronisation) — except the FIRST call on a batch: it builds the pattern's
 * transpose on the host and uploads it with cudaMalloc and blocking copies.  After that first call the step can be captured
 * into a CUDA graph.  Errors: NULL b / x / g / jac, only one of x_lower / x_upper NULL, mu < 0, cap <= 0 (or NaN), cg_iters
 * outside [0, 10000]: TWB_ERR_INVALID; solver vectors over 200 KiB of shared memory (8 (2 m + 4 n + 32) bytes):
 * TWB_ERR_UNSUPPORTED.  Nothing is enqueued when a call fails its checks. */
int twb_batch_lm_step_device(twb_batch* b, double* x, const double* g, const double* jac, const double* x_lower,
                             const double* x_upper, double mu, double cap, int cg_iters, double* violation, void* stream);

/* twb_batch_lm_step_device with per-instance CONSTRAINT bounds: instance b's violation r is measured against
 * [g_lower[b][i], g_upper[b][i]] (device [B][m] each, e.g. the g_lower / g_upper of twb_batch_state_instances_device, whose
 * BaseMotionConstraint rows follow each instance's initial base height).  Both NULL: the problem's own constraint bounds,
 * exactly twb_batch_lm_step_device.  -Inf / +Inf (like +-1e20) mean unbounded; a NaN bound counts like a non-finite g entry
 * (the instance is not stepped, violation[b] is NaN); with lower > upper the lower bound wins (g < lower is tested first).
 * Everything else — the other arguments, the first call's upload, graph capture after it, determinism, the errors — as for
 * twb_batch_lm_step_device; in addition only one of g_lower / g_upper NULL is TWB_ERR_INVALID.  Nothing is enqueued when a
 * call fails its checks. */
int twb_batch_lm_step_bounds_device(twb_batch* b, double* x, const double* g, const double* jac, const double* x_lower,
                                    const double* x_upper, const double* g_lower, const double* g_upper, double mu, double cap,
                                    int cg_iters, double* violation, void* stream);

/* ---- solving to a tolerance: trial step, gain-ratio acceptance, damping per instance ----------------------------------
 * One solve iteration for every instance of the batch in lock step is four calls, all of which only enqueue on `stream`:
 *   twb_batch_eval_device(x -> g, jac, flags TWB_EVAL_G | TWB_EVAL_JAC)
 *   twb_batch_lm_trial_device(x, g, jac -> x_trial, row_scale, merit, predicted, violation; sets converged / non-finite)
 *   twb_batch_eval_device(x_trial -> g_trial, flags TWB_EVAL_G)
 *   twb_batch_lm_accept_device(x_trial, g_trial -> x, mu, nu, solve_status, iterations)
 * The host decides how many iterations run (nothing loops on the device) and may stop once no instance is RUNNING.  The
 * caller initialises, per instance, mu [B] > 0 (e.g. 1e-2), nu [B] = 2, solve_status [B] = TWB_LM_RUNNING and
 * iterations [B] = 0, all device arrays.  An instance that is still RUNNING when the host's budget ends has hit the iteration
 * limit.  All other arrays are device pointers as for twb_batch_lm_step_device; x_trial must not overlap x. */
#define TWB_LM_RUNNING 0     /* still being stepped                                                                      */
#define TWB_LM_CONVERGED 1   /* max |s r| <= tol at x                                                                    */
#define TWB_LM_STALLED 2     /* mu grew past mu_max on rejected trials                                                   */
#define TWB_LM_NONFINITE 3   /* x, g, jac or a constraint bound holds a non-finite entry (a NaN bound); violation[b] NaN */

/* Trial step: twb_batch_lm_step_bounds_device's arithmetic with mu[b] per instance, written to x_trial [B][n] instead of x
 * (x is not changed).  For every instance whose solve_status is RUNNING when the call starts:
 *   row_scale [B][m] = s at x;  merit [B] = phi0 = 1/2 ||s r(g)||^2;  violation [B] = max |s r(g)| (may be NULL);
 *   predicted [B] = phi0 - 1/2 ||s r(g + J d)||^2, d = x_trial - x (the step after the cap and the projection): the decrease of
 *   the linearised violation, with the rows' bounds taken into account.
 * If max |s r| <= tol the status becomes TWB_LM_CONVERGED; if x, g, jac or a constraint bound is non-finite (as for
 * twb_batch_lm_step_device) it becomes TWB_LM_NONFINITE with violation NaN and merit NaN.  In both cases x_trial = x and
 * predicted = 0.  An instance that is not RUNNING when the call starts only gets x_trial = x; nothing else of it is written.
 * With mu[b] = mu for every instance, x_trial and violation are bit for bit what twb_batch_lm_step_device (or _bounds_device)
 * writes into x and violation, for every instance left RUNNING.  g_lower / g_upper: per-instance constraint bounds [B][m] (both
 * NULL: the problem's own).  Errors: those of twb_batch_lm_step_bounds_device except the mu check, NULL mu / solve_status /
 * x_trial / row_scale / merit / predicted, tol < 0 or NaN: TWB_ERR_INVALID; nothing is enqueued when a call fails its checks.
 * The first call of the step family on a batch (this, the two step calls, twb_batch_lm_accept_device) uploads
 * the pattern; after it, the calls can be captured into a CUDA graph. */
int twb_batch_lm_trial_device(twb_batch* b, const double* x, const double* g, const double* jac, const double* x_lower,
                              const double* x_upper, const double* g_lower, const double* g_upper, const double* mu, double cap,
                              int cg_iters, double tol, int* solve_status, double* x_trial, double* row_scale, double* merit,
                              double* predicted, double* violation, void* stream);

/* Acceptance, for every instance whose solve_status is RUNNING (the others are not touched): g_trial [B][m] is g at x_trial
 * (twb_batch_eval_device with TWB_EVAL_G), phi_t = 1/2 ||row_scale r(g_trial)||^2 with the row scales of x, and
 * rho = (merit - phi_t) / predicted.
 *   accept if predicted > 0, every g_trial entry and phi_t are finite and rho > eta:
 *     x <- x_trial, mu <- max(mu_min, mu max(1/3, 1 - (2 rho - 1)^3)), nu <- 2
 *   reject otherwise (a non-finite g_trial included; x keeps its bits): mu <- mu nu, nu <- 2 nu, and the status becomes
 *     TWB_LM_STALLED if the new mu > mu_max
 *   iterations[b] += 1 either way.
 * g_lower / g_upper as for the trial call (they must be the same).  Errors: NULL b or a required pointer, only one of g_lower /
 * g_upper NULL, eta outside [0, 1), not 0 < mu_min <= mu_max: TWB_ERR_INVALID, nothing enqueued. */
int twb_batch_lm_accept_device(twb_batch* b, double* x, const double* x_trial, const double* g_trial, const double* g_lower,
                               const double* g_upper, const double* row_scale, const double* merit, const double* predicted, double* mu,
                               double* nu, int* solve_status, int* iterations, double eta, double mu_min, double mu_max, void* stream);

/* ---- a whole solve in one call: the loop of the four calls above runs on the device ------------------------------------
 * The stand-in for ipopt.Solve(nlp) (towr/test/hopper_example.cc:93).  Enqueues on `stream` one CUDA graph:
 *   start: mu = mu0, nu = 2, status RUNNING, iterations 0 per instance
 *   WHILE (an instance is RUNNING and fewer than max_iters loop iterations ran) {
 *     eval (g, jac at x); trial; eval (g at x_trial); accept; count the instances per status }
 *   tail: eval (g, jac at x); trial with cg_iters = 0 (so that status and violation describe the returned x); count
 * The loop's exit test is a kernel: the loop stops at the iteration after which no instance is RUNNING, with no host round
 * trip.  The outputs equal, bit for bit, what BatchedLevenbergMarquardt.solve (towr_b200/solver.py) returns for the same
 * inputs — the four-call loop with its host-side early exit — since a finished instance does not move in further iterations.
 *   x [B][n] in / out; x_lower / x_upper [B][n] (both NULL: the problem's own variable bounds); g_lower / g_upper [B][m] (both
 *   NULL: the problem's own constraint bounds; exactly one NULL is TWB_ERR_INVALID); solve_status [B], iterations [B] (trials
 *   taken), violation [B] (max |s r| at the returned x; NaN for TWB_LM_NONFINITE), mu [B] (the final damping) out;
 *   status_counts [4] (instances per TWB_LM_* status after the tail; may be NULL) and loop_count [1] (loop iterations run; may
 *   be NULL) out.  All device pointers of the batch's device, in the layouts of the trial and accept calls.
 * The batch owns the work arrays (g, jac, x_trial, g_trial, row scales, merit, predicted, nu): allocated by the first solve
 * call, freed by twb_batch_destroy.  The first call with an argument set (the pointers and the options) also uploads the
 * pattern (as the step family's first call does) and builds and instantiates the graph; it is cached per argument set (up to
 * 16 per batch, least recently used replaced, dropped when terrains or grids change).  After that a call only launches the
 * graph into `stream`: no host synchronisation, no allocation.
 * A batch serves ONE evaluation or solve at a time (the work arrays and the staging matrix are shared): a second call on
 * another stream must be ordered after the first by the caller.
 * Errors, with nothing enqueued and no output touched: NULL b / x / opt / solve_status / iterations / violation / mu, one of
 * x_lower / x_upper or of g_lower / g_upper NULL, max_iters < 0, tol < 0 or NaN, eta outside [0, 1), not
 * 0 < mu_min <= mu_max, mu0 <= 0 or NaN, cap <= 0 or NaN, cg_iters outside [0, 10000], a step_rule other than the two
 * below, and with TWB_LM_STEP_TRUST radius_max < cap or NaN: TWB_ERR_INVALID; a stream that is being captured (a solve
 * cannot be captured into the caller's graph), TWB_PROFILE set, or solver vectors over 200 KiB of shared memory (as for
 * twb_batch_lm_step_device): TWB_ERR_UNSUPPORTED.
 *
 * Step rules (twb_lm_solve_options.step_rule):
 *   TWB_LM_STEP_CAP (the default): the trial step of twb_batch_lm_trial_device — the CG step scaled to max |dx| <= cap, then
 *     projected onto the variable bounds.  radius_max is ignored.
 *   TWB_LM_STEP_TRUST: a trust region of radius Delta[b] per instance, Delta = cap at the start.  Per trial:
 *     free set: with gamma = Js^T s r, variable j is frozen if x_lower[j] == x_upper[j], or x_j <= x_lower[j] and
 *       gamma_j > 0, or x_j >= x_upper[j] and gamma_j < 0 (the descent direction leaves the box); every other is free.  CG runs
 *       on the free set only (a frozen j keeps dx_j = 0);
 *     dx scaled to max |dx| <= Delta, then projected onto the bounds; predicted is computed from d = x_trial - x as for the cap
 *       rule, and step_norm = max |d|.
 *   Acceptance, rho and the mu update are those of twb_batch_lm_accept_device; after them
 *     rho < 0.25 or rejected:                   Delta <- 0.25 step_norm
 *     rho > 0.75 and step_norm >= 0.99 Delta:   Delta <- min(2 Delta, radius_max)
 *     otherwise Delta is kept, and an instance whose Delta < 1e-12 max(1, max |x|) becomes TWB_LM_STALLED.
 *   (0.25, 0.75, 2 and 0.99 are the textbook constants; they are not options.)  The batch allocates Delta and step_norm on its
 *   first trust-region solve and frees them in twb_batch_destroy.  Each rule gets its own cached graph. */
#define TWB_LM_STEP_CAP 0
#define TWB_LM_STEP_TRUST 1
typedef struct twb_lm_solve_options {
  double mu0;        /* initial damping (> 0)                                      */
  double cap;        /* largest step entry, as for twb_batch_lm_step_device; the    */
                     /* first trust radius with TWB_LM_STEP_TRUST                   */
  double tol;        /* CONVERGED when max |s r| <= tol                             */
  double eta;        /* accept when the gain ratio rho > eta, eta in [0, 1)         */
  double mu_min;     /* damping floor after an accepted trial                       */
  double mu_max;     /* STALLED once a rejected trial raises mu past mu_max         */
  int cg_iters;      /* conjugate-gradient iterations per trial                     */
  int max_iters;     /* iteration budget (>= 0)                                     */
  int step_rule;     /* TWB_LM_STEP_CAP or TWB_LM_STEP_TRUST                        */
  double radius_max; /* largest trust radius (>= cap; TWB_LM_STEP_TRUST only)       */
} twb_lm_solve_options;

/* the defaults of BatchedLevenbergMarquardt.solve: mu0 1e-2, cap 0.1, tol 1e-6, eta 1e-4, mu_min 1e-12, mu_max 1e10,
 * cg_iters 25, max_iters 60; step_rule TWB_LM_STEP_CAP, radius_max 1e3 */
void twb_lm_solve_options_default(twb_lm_solve_options* o);

int twb_batch_lm_solve_device(twb_batch* b, double* x, const double* x_lower, const double* x_upper, const double* g_lower,
                              const double* g_upper, const twb_lm_solve_options* opt, int* solve_status, int* iterations,
                              double* violation, double* mu, int* status_counts, int* loop_count, void* stream);

/* Host-pointer twin of twb_batch_lm_solve_device, for callers without the CUDA runtime (BatchedProblem::Solve in
 * towr_b200_ifopt.hpp): copies x and the bounds given into buffers of the batch, runs the same solve graph on the batch's
 * stream, copies x and the outputs back and synchronises.  Arguments and errors as for the device call, all host arrays. */
int twb_batch_lm_solve_host(twb_batch* b, double* x, const double* x_lower, const double* x_upper, const double* g_lower,
                            const double* g_upper, const twb_lm_solve_options* opt, int* solve_status, int* iterations,
                            double* violation, double* mu, int* status_counts, int* loop_count);

/* For tests: the solve graphs this batch has instantiated so far (a call that reuses a cached graph adds none). */
int twb_batch_lm_solve_graph_stats(const twb_batch* b, int* instantiations);

/* For tests and diagnostics: the trust radius Delta [B] and step_norm [B] of the last trial an instance took in the loop
 * (0 if it took none) (host arrays) of the batch's last TWB_LM_STEP_TRUST solve, copied after that solve's stream has been synchronised by the caller (the batch's own stream is
 * synchronised here).  TWB_ERR_INVALID with NULL arguments or before the batch's first trust-region solve. */
int twb_batch_lm_solve_radius(const twb_batch* b, double* radius, double* step_norm);

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

/* twb_batch_nearest_planes_* where instance b looks only at polygons poly_ranges[b][0] .. poly_ranges[b][0] + poly_ranges[b][1] - 1
 * of the shared list, and contact_set holds the index RELATIVE to that first polygon (what NearestPlaneLookup built from
 * that request's own PlanarTerrain returns), -1 in the air / for unused states / for an empty range.  So one call serves a
 * batch whose instances each have their own planar regions: pack every instance's polygons into one list.
 * poly_ranges: [B][2] (first polygon, count), a host array for _ranges_host, a device array for _ranges_device.
 * _ranges_host rejects a range outside [0, n_polys) (first < 0, count < 0, first + count > n_polys) with TWB_ERR_INVALID.
 * _ranges_device cannot check the ranges: it clamps each to [0, n_polys) (it never reads outside the list) and counts the
 * index from the first polygon of the clamped range.  Otherwise as the calls above. */
int twb_batch_nearest_planes_ranges_host(twb_batch* b, const double* plan, const int* n_states, const int* poly_ranges,
                                         const int* poly_offsets, int n_polys, const double* vertices, int* contact_set);
int twb_batch_nearest_planes_ranges_device(twb_batch* b, const double* plan, const int* n_states, const int* poly_ranges,
                                           const int* poly_offsets, int n_polys, const double* vertices, int* contact_set,
                                           void* stream);

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
