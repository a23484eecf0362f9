// device_tables.h — plain-old-data tables the host builder (formulation.cc)
// uploads once per structure class and the CUDA kernels (kernels.cu) read on
// every evaluation.  Nothing in here depends on the iterate x.
#ifndef TOWR_B200_DEVICE_TABLES_H_
#define TOWR_B200_DEVICE_TABLES_H_

#include <cstdint>

namespace twb {

constexpr int kMaxEE = 4;

// One spline evaluated at one constraint sample when phase durations are
// fixed: the active polynomial (Spline::GetSegmentID, spline.cc:48-63), its
// local time (Spline::GetLocalTime, spline.cc:66-78) and where its two
// boundary nodes live in x.  `xi` holds x indices of p0[3], v0[3], p1[3],
// v1[3]; node values that are not optimised (always 0 in towr) point at the
// zero slot, index n.
struct alignas(16) SplineSample {   // 96 bytes = six 16-byte loads
  double T, T2, T3;   // polynomial duration and std::pow(T,2), std::pow(T,3)
  double rT2, rT3;    // correctly rounded 1/T2, 1/T3 (seed of the exact division on the device)
  double t, t2, t3;   // local time and std::pow(t,2), std::pow(t,3)
  int16_t xi[12];
  int16_t pad[4];
};

// ---- phase-duration optimisation (Parameters::OptimizePhaseDurations) --------------------------------
// With "ee-schedule" variable sets the foot splines are PhaseSplines (phase_spline.cc): their polynomial
// durations, hence the active polynomial and the local time of every constraint sample, depend on the
// iterate.  A SplineSample with xi[0] == kPhaseMarker refers to such a spline: xi[1] = index into
// Plan::phase_defs, T = the GLOBAL sample time.
constexpr uint16_t kPhaseMarker = 0xFFFFu;
struct PhasePoly {       // one polynomial of a phase-based node set (nodes_variables_phase_based.cc:38-89)
  int16_t xi[12];        // x indices of p0[3], v0[3], p1[3], v1[3] (zero slot if not optimised)
  int16_t phase, n_in_phase, k_in_phase, pad;
};
struct PhaseSplineDef {
  int32_t poly0, n_polys;     // range in Plan::phase_polys
  int32_t sched0, n_phases;   // x index of the foot's first duration variable; number of phases (variables: n_phases - 1)
  double t_total;
};
// Work item of the PhaseJac kernel: the TotalDurationConstraint rows (total_duration_constraint.cc:36-72) — value, the
// constant Jacobian entries and status bit 1.  (The PhaseSpline entries of the dynamic and range-of-motion rows are
// "phase elements" of the output lists, see PhaseExt below.)
enum PhaseUnitKind : int32_t { kPhaseTotal = 2 };
struct PhaseUnit {
  int32_t kind;
  int32_t pad;
  int32_t rows[kMaxEE];       // the foot's constraint row
  int32_t slot0[kMaxEE];      // CSR slot of the row's first entry (its entries are the foot's duration columns, ascending)
};

// ---- output lists -------------------------------------------------------------
// Every value a unit produces — a CSR Jacobian value or a constraint value — is
//     out[instance][off + h] = state[d_h][instance] * c_h,     h = 0, 1
// where `state` is the unit's local state block (row 0 holds the constant 1) and (off, off + 1) is a
// 16-byte aligned pair of elements of the instance's output row, so that one lane issues one 16-byte store
// per instance and a warp covers 512 contiguous bytes.
//
// HBM only sustains its write bandwidth for whole 32-byte sectors (a partially written sector that has left
// the L2 costs a read-modify-write), so the Jacobian values are written by whole CTAs: after the CTA barrier all
// threads walk ONE list of pairs that covers the output of the CTA's consecutive units (`d` = row in the CTA's
// shared memory = warp * block rows + local row).  The lists are built sector by sector: a sector is written, whole,
// by the CTA that owns its last element; only sectors shared with another CTA fall back to 8-byte single-element
// stores.  The alignment of an instance's row inside its sectors depends on (instance * row length) mod 4, so a
// list exists per alignment class q = instance mod n_classes (n_classes = 1 when the row length is a multiple of 4).
// The constraint values are written by the CTAs as well (kernels.cu: StoreValuesDirect).
constexpr int kMaxClasses = 4;
// ---- phase elements (optimised phase durations) ----------------------------------------------------------------------
// With PhaseSplines a constraint sample's row is structurally dense in ALL node variables of the foot's set
// (phase_spline.cc:45-51) and in the foot's duration variables, but which of those entries are non-zero depends on the
// polynomial the sample falls into — on the iterate.  Such an element is written by the same CTA-wide pair loop as every
// other element (coalesced, whole sectors).  The compute phase leaves, for every PhaseSpline of the sample, an "info block"
// of kInfoRows state rows:
//   +0   32-bit integers: [0..31] active polynomial P per instance | [32], [33] min / max of P over the tile
//        | [34..65] current phase per instance | [66], [67] its min / max
//   +1   Z, a row of zeros
//   +2.. WINDOW form (P differs by at most 2 over the tile — the normal case): the weight of node pmin + s, s = 0..3, for
//        node derivative 0 / 1 in row +2 + 2 s + deriv:  B[0][deriv] where P == node, B[1][deriv] where P == node - 1, else 0
//        (NodeSpline::FillJacobianWrtNodes, node_spline.cc:85-112).  An element of node a then is, for EVERY instance of the
//        tile, out = (state[d] * c) * state[w], w = the row of node a (a shared stance position: the sum of the rows of a and
//        a + 1), or zero when a is outside the window — no per-instance selection in the store loop.
//        TABLE form (wider spread): Z B1[0] B0[0] Z B1[1] B0[1] Z B1[0] B0[0]+B1[0] B0[0] Z from +1 on, walked per instance
//        with the clamped index P - a + 2.
// Duration columns (PhaseDurations::GetJacobianOfPos, phase_durations.cc:122-154): column ph is U (state rows d ..) where
// ph < current phase, V where ph == current phase, else 0.  Rows: U | X.  Window form (current phase differs by less than
// `dwin` over the tile): X holds the finished columns cmin, cmin + 1, .. (row d + v_off (1 + ph - cmin)); columns before cmin
// are U, columns after cmax zero, for every instance.  Otherwise X starts with V and the store loop selects per instance.
// One 32-bit word per element, parallel to the pair / single entries: kind (bits 0-1), deriv (bit 2), shared (bit 3),
// a or ph (bits 8-15), first row of the info block in the CTA's shared memory (bits 16-31).
enum PhaseElemKind : uint32_t { kElemPlain = 0, kElemNode = 1, kElemDuration = 2 };
struct PhaseExt { uint32_t e0, e1; };
constexpr int kInfoRows = 12;
constexpr int kDynDurWin = 2, kRomDurWin = 2;   // duration columns finished per instance (window form) in DynTailOut / RomBody
// state rows of one foot in the DynTailOut kernel: 0: 1 | 1..3: f_e | 4..6: c - p_e | 7..18: info block of ee-motion_e |
// 19..30: info block of ee-force_e | 31..36: U | 37..54: X   (duration columns of the sample's 6 rows)
constexpr int kTailRows = 7 + 2 * kInfoRows + 6 + 6 * kDynDurWin;
struct OutPair { int32_t off; uint16_t d0, d1; };       // pair: element index of the first half; single / value entry: element index / g row, d0 = state row
struct alignas(16) OutCoef { double c0, c1; };
struct OutRange { int32_t first, count; };
// A run of iterate-independent Jacobian values (state row 0 = the constant 1 on every element: spline-acc and swing rows
// with fixed durations, ...), whole sectors, at least kConstRunMin elements: not part of any CTA list — a "constant CTA"
// loads the run's values (the same for every instance) into shared memory with one TMA bulk copy and writes them to the
// 32 instances of its tile with one cp.async.bulk per instance (SASS UBLKCP.S.G / UBLKCP.G.S), no LSU work at all.
struct ConstRun { int32_t off, len, src, pad; };   // element offset in the instance's CSR row, elements (multiple of 4), first value in Plan::const_vals
constexpr int kConstRunMin = 128, kConstRunMax = 2048;   // elements per run piece (1 KB .. 16 KB)
struct OutList {                        // per alignment class
  OutRange pairs[kMaxClasses];          // whole sectors, two pairs each
  OutRange singles[kMaxClasses];        // single elements (lane = instance)
  OutRange phase[kMaxClasses];          // whole sectors that hold at least one phase element (same layout as `pairs`, with Plan::exts)
};
// Range-of-motion state block: [0]=1 | R^T (9) | two buffers of { D_e (9) | g_e (3) } used by the feet in turn (one CTA
// barrier and one list per foot).  With optimised phase durations a foot's buffer is D_e (9) | info block of its PhaseSpline
// (kInfoRows) | U (3) | X (3 kRomDurWin).
#define RomBufRows(phase) ((phase) ? 9 + kInfoRows + 3 + 3 * kRomDurWin : 12)
#define RomBufferP(e, phase) (RomBufRows(phase) * ((e) & 1))   /* first row of foot e's buffer, relative to row 10 */
#define RomBlockRowsP(n_ee, phase) (10 + RomBufRows(phase) * 2)

// The constraint values leave the output kernels straight into g[B][m]: after the CTA barrier all threads write the CTA's
// consecutive rows (24 per dynamic CTA, 12 per range-of-motion CTA and foot) with consecutive threads = consecutive rows of
// one instance.  The dynamic unit keeps its 6 values in 6 more state rows.
#define DynBlockRows(n_ee) (46 + 6 * (n_ee))   /* 1 | 3 | 36 | 6 per foot | 6 values */

// warps per CTA of the output kernels = consecutive units whose output ranges are chained through carry rows.  The
// range-of-motion and node CTAs of a tile run in ONE kernel (RomNodeOut) and need equal CTA sizes.
constexpr int kDynWarps = 4;    // consecutive dynamic samples per CTA (one instance tile)
constexpr int kRomWarps = 4;    // consecutive range-of-motion samples per CTA
constexpr int kNodeWarps = 4;   // consecutive node groups per CTA

// TerrainConstraint row (terrain_constraint.cc:59-108): one ee-motion node.
// local state: [base + 0] = -dh/dx, [base + 1] = -dh/dy, g at [g_base]
struct TerrainUnit { int16_t xi[3]; int16_t pad; };
// ForceConstraint node (force_constraint.cc:64-171): 5 rows.  local state: 25 values [row][{d/dpx,d/dpy,d/dfx,d/dfy,d/dfz}]
struct ForceUnit { int16_t xf[3]; int16_t xp[3]; int16_t pad[2]; };
// SwingConstraint node (swing_constraint.cc:57-83): 4 rows (values only; the Jacobian is constant)
struct SwingUnit { int16_t xc_p[2], xc_v[2]; int16_t xprev[2], xnext[2]; };
// SplineAccConstraint junction (spline_acc_constraint.cc:49-65), fixed durations (values only)
struct AccUnit {
  double Tp, Tp2, Tp3, rTp2, rTp3;  // previous polynomial duration, pow 2, pow 3, reciprocals
  double Tn, Tn2, rTn2;             // next polynomial
  int32_t x0;           // x index of node j, dim 0 position (NodesVariablesAll layout)
  int32_t pad;
};
// BaseMotionConstraint sample (base_motion_constraint.cc:56-66): values only, 6 rows
struct BaseMotionUnit { int32_t sample_lin, sample_ang; };

// A dynamic sample (6 rows): 2 + 2 n_ee spline samples starting at `sample0`
// (base-lin, base-ang, ee-motion.., ee-force..) and its output lists.
struct DynUnit { int32_t sample0; int32_t g_row0; };   // g_row0: first of the sample's 6 constraint rows
// A range-of-motion sample (3 rows for every foot): 2 + n_ee spline samples (base-lin, base-ang, ee-motion..);
// the feet are evaluated and written one after the other.
struct RomUnit { int32_t sample0; };

// Node-wise work of one warp: `count` consecutive units of one kind evaluated into one state block,
// then one pass over the group's output lists.
enum NodeKind : int32_t { kGroupForce = 0, kGroupTerrain = 1, kGroupSwing = 2, kGroupAcc = 3, kGroupConst = 4, kGroupBaseMotion = 5 };
// g_row0 >= 0: the group's constraint values are the consecutive rows g_row0 .. g_row0 + g_n - 1 taken from the
// consecutive state rows g_d0 ..: written without a table (no dependent loads); otherwise the `values` entries are used.
struct NodeGroup { int32_t kind, first, count, g_row0; OutRange values; int32_t g_d0, g_n; };
constexpr int kNodeStateRowsMax = 64;   // upper bound of the local state rows of a node group (row 0 = 1); Plan::node_rows is the actual maximum

// NodeCost term (node_cost.cc:53-76) flattened: one entry per node value that
// enters the cost; var >= 0 when the value is an optimisation variable.
struct CostEntry {
  int16_t xi;        // x index holding the node value (zero slot if fixed)
  int16_t grad_col;  // column of the gradient this node contributes to, or -1
  int32_t pad;       // 1: first entry of a cost term
  double weight;
};

// ---- batched setup: NlpFormulation::GetVariableSets' initial guess and variable bounds (nlp_formulation.cc:95-181) as a
// per-variable recipe, so that goal-randomised instances of one structure class are set up by a kernel:
//   position variable: x0 = a[dim] + frac * (b[dim] - a[dim])   (NodesVariables::SetByLinearInterpolation, nodes_variables.cc:126-150;
//                      frac = node / (n_nodes - 1) of the LAST node the variable belongs to)
//   velocity variable: x0 = (b[dim] - a[dim]) / T
// with (a, b) = (initial, final) of the variable's set: base-lin (final z = terrain height - nominal z), base-ang, ee-motion_e
// (final = goal base + yaw-rotated nominal stance, z on the terrain), ee-force_e (a = b = (0, 0, m g / n_ee)); ee-schedule
// variables are constants.  Bounds: free, a constant on both sides, the goal's own base position / angle, or a constant pair.
// The start-state recipe (Plan::state_vars, StateInstanceKernel) is the same recipe with the endpoints taken from a per-instance
// state record (TWB_STATE_DOUBLES, layout below) and every bound that copies a spec field turned into kBoundState: both sides
// = record[src].  Only the state recipe holds kBoundState; goal_vars keeps the four goal-recipe modes.
enum GoalBound : int8_t { kBoundFree = 0, kBoundConst = 1, kBoundGoalLin = 2, kBoundGoalAng = 3, kBoundPair = 4, kBoundState = 5 };
enum GoalKind : int8_t { kGoalLin = 0, kGoalAng = 1, kGoalMotion = 2, kGoalForce = 3, kGoalConst = 4 };
struct GoalVar {
  int8_t kind, ee, deriv, dim;   // GoalKind, foot (motion / force), 0 position / 1 velocity, dimension
  int8_t bound, src, pad[2];     // GoalBound; kBoundState: index into the state record
  double frac;                   // node fraction (positions); constant x0 (kGoalConst)
  double c0, c1;                 // bound constants
};
struct GoalSetup {                // goal-independent inputs of the recipe (twb_spec + robot)
  double initial_lin[3], initial_ang[3], initial_ee[kMaxEE][3], nominal[kMaxEE][3];
  double t_total, f_stance_z;
};
// per-instance state record (include/towr_b200.h: TWB_STATE_DOUBLES): offsets of NlpFormulation's three state fields
constexpr int kStateDoubles = 36;
enum StateField : int8_t { kStInitLinPos = 0, kStInitLinVel = 3, kStInitAngPos = 6, kStInitAngVel = 9, kStFinalLinPos = 12, kStFinalLinVel = 15,
                           kStFinalAngPos = 18, kStFinalAngVel = 21, kStInitEE = 24 };

// ---- per-instance terrain word (twb_batch::d_terrain): the terrain id, and for TWB_GRID_MAP (8) instances the index of the
// instance's map in Plan::gmaps above the low four bits.  Every other id is stored as it is, so the analytic terrains see
// their raw id; words of 7 and above are decoded only in the out-of-line grid path (kernels.cu: EvalGridTerrain).
#ifdef __CUDACC__
#define TWB_HOST_DEVICE __host__ __device__
#else
#define TWB_HOST_DEVICE
#endif
constexpr int kTerrainGridMap = 8;
constexpr int kMaxGridMaps = 1 << 27;   // map << 4 stays a positive int
inline TWB_HOST_DEVICE int TerrainWord(int id, int map) { return id == kTerrainGridMap ? id | (map << 4) : id; }
inline TWB_HOST_DEVICE int TerrainWordId(int word) { return word & 15; }
inline TWB_HOST_DEVICE int TerrainWordMap(int word) { return word >> 4; }
// one grid_map elevation layer of a batch: layer(ix, iy) = pool[offset + ix * sy + iy], `res` metres per cell, centred at (px, py)
struct GridMapDesc { long long offset; int sx, sy; double res, px, py; };

struct Plan {
  int n, m, nnz, n_ee;
  int n_dyn, n_rom, n_groups, n_cost;
  int node_rows, dyn_rows, rom_rows;   // state rows of one unit's block: node groups (largest), dynamic samples, range-of-motion samples
  int nc_jac;         // alignment classes of the Jacobian-value rows (length nnz)
  int dyn_list0, rom_list0, node_list0;   // first entry of cta_lists of the dynamic CTAs, (rom CTA, foot) pairs, node CTAs
  int tail_list0;                         // optimised durations: list of dynamic sample k's PhaseSpline columns (DynTailOut) = tail_list0 + k
  int rom_row0[kMaxEE];                   // first constraint row of foot e's range-of-motion set (sample k owns rows rom_row0[e] + 3k ..+2)
  // robot
  double mass, gravity;
  double I_b[9];
  double mu;
  // tables (device pointers)
  const SplineSample* samples;
  const DynUnit* dyn;
  const RomUnit* rom;
  const NodeGroup* groups;
  const TerrainUnit* terr;
  const ForceUnit* force;
  const SwingUnit* swing;
  const AccUnit* acc;
  const BaseMotionUnit* base_motion;
  const CostEntry* cost;
  const double* dyn_ang_basis;  // [n_dyn][12]: base-ang basis of the active polynomial, {pos, vel, acc} x {p0, v0, p1, v1}
  const OutPair* pairs;
  const OutCoef* coefs;
  const OutList* cta_lists;
  const PhaseExt* exts;                 // parallel to pairs / coefs (optimised durations only, else null)
  // height grid of the TWB_GRID_CSV terrain (per batch; null: heights 0)
  const double* grid;
  int grid_rows, grid_cols;
  // elevation layers of the TWB_GRID_MAP terrain (per batch): instance b reads gmaps[TerrainWordMap(word_b)]; an index
  // >= n_gmaps (no maps) puts every position outside the map
  const float* gmap_pool;
  const GridMapDesc* gmaps;
  int n_gmaps;
  const GoalVar* goal_vars;             // [n] recipe of x0 / bounds per variable
  const GoalVar* state_vars;            // [n] the same recipe for per-instance start states (bounds from the state record)
  const double* g_lower;                // [m] the problem's constraint bounds (per-instance setup copies them)
  const double* g_upper;
  const int32_t* base_z_rows;           // BaseMotionConstraint LZ rows, bounds [z_init - 0.02, z_init + 0.1] (none without TWB_C_BASE_ROM)
  int n_base_z_rows;
  int n_const_runs;                     // constant runs (TMA-written; fixed durations, row length a multiple of 4)
  const ConstRun* const_runs;
  const double* const_vals;
  // phase-duration optimisation (all null / 0 otherwise)
  int n_phase_units, n_phase_defs;
  const PhaseSplineDef* phase_defs;   // [2 * n_ee]: ee-motion_e at 2e, ee-force_e at 2e + 1
  const PhasePoly* phase_polys;
  const PhaseUnit* phase_units;
};

}  // namespace twb
#endif
