// formulation.cc — builds one NLP structure class on the host.
//
// What the reference obtains implicitly by running Eigen sparse algebra once
// (IpoptAdapter reads the pattern of the first GetJacobianOfConstraints()),
// this builder derives explicitly: every Jacobian entry is *emitted* as
//     (row, col)  ->  S[a] * coef            (or a 3-term variant)
// where S is the small per-instance state vector the kernels compute per
// iterate and `coef` is an iterate-independent constant (a Hermite basis value
// at a fixed sample time, a sign, the mass, ...).  Sorting the emitted entries
// row-major / ascending column gives the CSR pattern; the sorted (a, coef)
// pairs are the slot descriptors the fill kernel walks.
//
// Reference behaviour restated here (cited per function):
//   towr/src/nlp_formulation.cc:63-376, parameters.cc:82-135,
//   nodes_variables*.cc, spline.cc:48-78, polynomial.cc:106-234,
//   time_discretization_constraint.cc:37-51 and the *_constraint.cc files.
#include "formulation.h"

#include <algorithm>
#include <cmath>
#include <map>
#include <numeric>

namespace twb {
namespace {

constexpr double kInf = 1e20;  // ifopt::inf
enum { kPos = 0, kVel = 1, kAcc = 2 };
enum { X = 0, Y = 1, Z = 2 };

// ---- node parameterisations ------------------------------------------------
struct NodeSet {
  std::string name;
  int offset = 0, n_vars = 0, n_nodes = 0;
  std::vector<std::array<int, 6>> var;  // [node][deriv*3+dim] -> local variable index or -1 (fixed 0)
  std::vector<double> x0, lo, up;
  struct Poly { int phase, k_in_phase, n_in_phase; bool constant; };
  std::vector<Poly> poly;  // phase-based sets only

  int Var(int node, int deriv, int dim) const { return var[node][deriv * 3 + dim]; }
  bool ConstNode(int id) const {  // nodes_variables_phase_based.cc:104-116,156-172
    if (id == 0) return poly.front().constant;
    if (id == n_nodes - 1) return poly.back().constant;
    return poly[id - 1].constant || poly[id].constant;
  }
  void Alloc(int nodes) { n_nodes = nodes; var.assign(nodes, {-1, -1, -1, -1, -1, -1}); }
  void Finish() { x0.assign(n_vars, 0.0); lo.assign(n_vars, -kInf); up.assign(n_vars, +kInf); }
  // NodesVariables::SetByLinearInterpolation, nodes_variables.cc:126-150; a variable shared by two
  // nodes ends up holding the later node's value (NodesVariables::GetValues, :53-61)
  void Interpolate(const double a[3], const double b[3], double t_total) {
    for (int node = 0; node < n_nodes; ++node)
      for (int dim = 0; dim < 3; ++dim) {
        double dp = b[dim] - a[dim];
        int vp = Var(node, kPos, dim), vv = Var(node, kVel, dim);
        if (vp >= 0) x0[vp] = a[dim] + node / static_cast<double>(n_nodes - 1) * dp;
        if (vv >= 0) x0[vv] = dp / t_total;
      }
  }
  void Fix(int node, int deriv, int dim, double val) {  // NodesVariables::AddBound, :161-168
    int v = Var(node, deriv, dim);
    if (v >= 0) { lo[v] = val; up[v] = val; }
  }
};

NodeSet MakeBaseSet(const std::string& name, int nodes) {  // nodes_variables_all.cc:34-61
  NodeSet s; s.name = name; s.Alloc(nodes);
  for (int nd = 0; nd < nodes; ++nd) for (int k = 0; k < 6; ++k) s.var[nd][k] = nd * 6 + k;
  s.n_vars = nodes * 6; s.Finish();
  return s;
}
void BuildPolys(NodeSet* s, int phases, bool first_constant, int polys_in_changing) {  // nodes_variables_phase_based.cc:38-76
  bool c = first_constant;
  for (int ph = 0; ph < phases; ++ph) {
    if (c) s->poly.push_back({ph, 0, 1, true});
    else for (int j = 0; j < polys_in_changing; ++j) s->poly.push_back({ph, j, polys_in_changing, false});
    c = !c;
  }
  s->Alloc((int)s->poly.size() + 1);
}
NodeSet MakeMotionSet(const std::string& name, int phases, bool contact_at_start, int polys_per_swing) {  // :190-253
  NodeSet s; s.name = name; BuildPolys(&s, phases, contact_at_start, polys_per_swing);
  int idx = 0;
  for (int nd = 0; nd < s.n_nodes; ++nd) {
    if (!s.ConstNode(nd)) {  // swing node: px, vx, py, vy, pz
      for (int dim = 0; dim < 3; ++dim) { s.var[nd][dim] = idx++; if (dim != Z) s.var[nd][3 + dim] = idx++; }
    } else {                 // stance pair shares one position
      for (int dim = 0; dim < 3; ++dim) { s.var[nd][dim] = idx; s.var[nd + 1][dim] = idx; ++idx; }
      ++nd;
    }
  }
  s.n_vars = idx; s.Finish();
  return s;
}
NodeSet MakeForceSet(const std::string& name, int phases, bool contact_at_start, int polys_per_stance) {  // :255-298
  NodeSet s; s.name = name; BuildPolys(&s, phases, !contact_at_start, polys_per_stance);
  int idx = 0;
  for (int nd = 0; nd < s.n_nodes; ++nd) {
    if (!s.ConstNode(nd)) { for (int dim = 0; dim < 3; ++dim) { s.var[nd][dim] = idx++; s.var[nd][3 + dim] = idx++; } }
    else ++nd;  // swing pair: all zeros, not optimised
  }
  s.n_vars = idx; s.Finish();
  return s;
}

// ---- splines at fixed durations --------------------------------------------
struct SplineDef { const NodeSet* set; std::vector<double> T; };

int SegmentID(double t_global, const std::vector<double>& T) {  // spline.cc:48-63
  const double eps = 1e-10; double t = 0; int i = 0;
  for (double d : T) { t += d; if (t >= t_global - eps) return i; ++i; }
  return (int)T.size() - 1;
}
void Locate(const SplineDef& s, double t_global, int* poly, double* t_local) {  // spline.cc:66-78
  *poly = SegmentID(t_global, s.T);
  double tl = t_global; for (int i = 0; i < *poly; ++i) tl -= s.T[i];
  *t_local = tl;
}
// d(value derivative dxdt at local time t)/d(node value): polynomial.cc:106-234
double NodeBasis(int side, int dxdt, int node_deriv, double t, double T) {
  double t2 = std::pow(t, 2), t3 = std::pow(t, 3), T2 = std::pow(T, 2), T3 = std::pow(T, 3);
  if (side == 0) {
    if (dxdt == kPos) return node_deriv == kPos ? (2 * t3) / T3 - (3 * t2) / T2 + 1 : t - (2 * t2) / T + t3 / T2;
    if (dxdt == kVel) return node_deriv == kPos ? (6 * t2) / T3 - (6 * t) / T2 : (3 * t2) / T2 - (4 * t) / T + 1;
    return node_deriv == kPos ? (12 * t) / T3 - 6 / T2 : (6 * t) / T2 - 4 / T;
  }
  if (dxdt == kPos) return node_deriv == kPos ? (3 * t2) / T2 - (2 * t3) / T3 : t3 / T2 - t2 / T;
  if (dxdt == kVel) return node_deriv == kPos ? (6 * t) / T2 - (6 * t2) / T3 : (3 * t2) / T2 - (2 * t) / T;
  return node_deriv == kPos ? 6 / T2 - (12 * t) / T3 : (6 * t) / T2 - 2 / T;
}
struct BasisEntry { int dim, var; double val; };
// NodeSpline::FillJacobianWrtNodes, node_spline.cc:85-112: which variables of the set move
// the spline value (derivative dxdt) of polynomial `poly` at local time tl, and by how much.
std::vector<BasisEntry> Basis(const SplineDef& s, int poly, double tl, int dxdt) {
  std::map<int, BasisEntry> acc;  // keyed by variable -> ascending column order
  for (int side = 0; side < 2; ++side)
    for (int deriv = 0; deriv < 2; ++deriv)
      for (int dim = 0; dim < 3; ++dim) {
        int v = s.set->Var(poly + side, deriv, dim);
        if (v < 0) continue;
        double b = NodeBasis(side, dxdt, deriv, tl, s.T[poly]);
        auto it = acc.find(v);
        if (it == acc.end()) acc[v] = BasisEntry{dim, v, 0.0 + b};
        else it->second.val += b;  // stance position shared by both boundary nodes
      }
  std::vector<BasisEntry> out;
  for (auto& kv : acc) out.push_back(kv.second);
  return out;
}
int16_t XIndex(const NodeSet& set, int node, int deriv, int dim, int zero_slot) {
  int v = set.Var(node, deriv, dim);
  return (int16_t)(v < 0 ? zero_slot : set.offset + v);
}
SplineSample MakeSample(const SplineDef& s, double t_global, int zero_slot) {
  SplineSample o{};
  int p; double tl; Locate(s, t_global, &p, &tl);
  o.T = s.T[p]; o.T2 = std::pow(o.T, 2); o.T3 = std::pow(o.T, 3);
  o.rT2 = 1.0 / o.T2; o.rT3 = 1.0 / o.T3;
  o.t = tl; o.t2 = std::pow(tl, 2); o.t3 = std::pow(tl, 3);
  for (int side = 0; side < 2; ++side) for (int deriv = 0; deriv < 2; ++deriv) for (int dim = 0; dim < 3; ++dim)
    o.xi[side * 6 + deriv * 3 + dim] = XIndex(*s.set, p + side, deriv, dim, zero_slot);
  return o;
}

std::vector<double> SampleTimes(double T, double dt) {  // time_discretization_constraint.cc:37-51
  double t = 0.0; std::vector<double> v = {t};
  for (int i = 0; i < std::floor(T / dt); ++i) { t += dt; v.push_back(t); }
  v.push_back(T);
  return v;
}
std::vector<double> BasePolyDurations(double T, double dt) {  // parameters.cc:82-98
  std::vector<double> v; double left = T; const double eps = 1e-10;
  while (left > eps) { v.push_back(left > dt ? dt : left); left -= dt; }
  return v;
}

// a: local state row of the owning unit (0 = the constant 1); ext: phase-element word (device_tables.h: PhaseExt) with the
// info row local to the unit as well; tail >= 0: element of dynamic sample `tail` written by the DynTailOut kernel (a and
// the info row are then rows of that kernel's CTA)
struct Emit { int row, col; uint32_t a; double c0; uint32_t ext = 0; int tail = -1; };
uint32_t PackExt(uint32_t kind, int deriv, bool shared, int a_or_ph, uint32_t info_row) {
  return kind | ((uint32_t)deriv << 2) | ((uint32_t)(shared ? 1 : 0) << 3) | ((uint32_t)a_or_ph << 8) | (info_row << 16);
}

// Who computes a constraint row: a dynamic sample, a range-of-motion sample (all feet) or a node unit.
enum OwnerKind { kOwnDyn, kOwnRom, kOwnNode, kOwnPhase };   // kOwnPhase: rows written by the PhaseJac kernel (total duration)
struct RowOwner { int kind = -1, index = -1; uint32_t g_local = 0; };   // g_local: state row of a node unit's value inside the unit
// node unit before grouping: kind, index into its table, rows of local state / values it needs
struct NodeUnitRef { int kind, index, n_state, n_g, set_id; };

// sign/component of Cross(v)[i][d] (single_rigid_body_dynamics.cc:46-57): value = sign * v[comp]
void CrossEntry(int i, int d, int* comp, double* sign) {
  static const int c[3][3] = {{-1, 2, 1}, {2, -1, 0}, {1, 0, -1}};
  static const double s[3][3] = {{0, -1, +1}, {+1, 0, -1}, {-1, +1, 0}};
  *comp = c[i][d]; *sign = s[i][d];
}

// NlpFormulation::GetVariableSets' initial guess and bounds (nlp_formulation.cc:95-181) for the goal / initial state in
// `sp`; `sets` supplies the variable maps and receives the per-set x0 / bounds.
void InitialGuessAndBounds(const twb_spec& sp, const RobotConst& rb, double T, bool optimize_timings, std::vector<NodeSet>* sets_io,
                           std::vector<double>* x0_out, std::vector<double>* lo_out, std::vector<double>* up_out) {
  std::vector<NodeSet>& sets = *sets_io;
  const int n_ee = sp.n_ee;
  NodeSet& lin = sets[0]; NodeSet& ang = sets[1];
  auto motion = [&](int e) -> NodeSet& { return sets[2 + e]; };
  auto force = [&](int e) -> NodeSet& { return sets[2 + n_ee + e]; };
  for (auto& s : sets) s.Finish();
  std::vector<double>& x0 = *x0_out; std::vector<double>& x_lower = *lo_out; std::vector<double>& x_upper = *up_out;
  {
    double fx = sp.final_base_lin_pos[0], fy = sp.final_base_lin_pos[1];
    double fz = TerrainHeight(sp.terrain, fx, fy) - rb.nominal[0][2];
    double final_pos[3] = {fx, fy, fz};
    lin.Interpolate(sp.initial_base_lin_pos, final_pos, T);
    ang.Interpolate(sp.initial_base_ang_pos, sp.final_base_ang_pos, T);
    const int last = lin.n_nodes - 1;
    for (int d = 0; d < 3; ++d) {
      lin.Fix(0, kPos, d, sp.initial_base_lin_pos[d]); lin.Fix(0, kVel, d, sp.initial_base_lin_vel[d]);
      ang.Fix(0, kPos, d, sp.initial_base_ang_pos[d]); ang.Fix(0, kVel, d, sp.initial_base_ang_vel[d]);
      if (sp.bounds_final_lin_pos[d]) lin.Fix(last, kPos, d, sp.final_base_lin_pos[d]);
      if (sp.bounds_final_lin_vel[d]) lin.Fix(last, kVel, d, sp.final_base_lin_vel[d]);
      if (sp.bounds_final_ang_pos[d]) ang.Fix(last, kPos, d, sp.final_base_ang_pos[d]);
      if (sp.bounds_final_ang_vel[d]) ang.Fix(last, kVel, d, sp.final_base_ang_vel[d]);
    }
    // yaw-only rotation of the nominal stance (EulerConverter::GetRotationMatrixBaseToWorld with x=y=0)
    double yaw = sp.final_base_ang_pos[2];
    double x = 0.0, y = 0.0, z = yaw;
    double R[3][3] = {{cos(y) * cos(z), cos(z) * sin(x) * sin(y) - cos(x) * sin(z), sin(x) * sin(z) + cos(x) * cos(z) * sin(y)},
                      {cos(y) * sin(z), cos(x) * cos(z) + sin(x) * sin(y) * sin(z), cos(x) * sin(y) * sin(z) - cos(z) * sin(x)},
                      {-sin(y), cos(y) * sin(x), cos(x) * cos(y)}};
    for (int e = 0; e < n_ee; ++e) {
      const double* nom = rb.nominal[e];
      double w[3];
      for (int i = 0; i < 3; ++i) w[i] = sp.final_base_lin_pos[i] + (R[i][0] * nom[0] + R[i][1] * nom[1] + R[i][2] * nom[2]);
      double goal[3] = {w[0], w[1], TerrainHeight(sp.terrain, w[0], w[1])};
      motion(e).Interpolate(sp.initial_ee_W[e], goal, T);
      for (int d = 0; d < 3; ++d) motion(e).Fix(0, kPos, d, sp.initial_ee_W[e][d]);
      double f_stance[3] = {0.0, 0.0, rb.mass * 9.80665 / n_ee};
      force(e).Interpolate(f_stance, f_stance, T);
    }
  }
  x0.clear(); x_lower.clear(); x_upper.clear();
  for (auto& s : sets) {
    x0.insert(x0.end(), s.x0.begin(), s.x0.end());
    x_lower.insert(x_lower.end(), s.lo.begin(), s.lo.end());
    x_upper.insert(x_upper.end(), s.up.begin(), s.up.end());
  }
  if (optimize_timings)   // PhaseDurations::GetValues / GetBounds, phase_durations.cc:68-77, 102-110
    for (int e = 0; e < n_ee; ++e)
      for (int i = 0; i + 1 < sp.n_phases[e]; ++i) {
        x0.push_back(sp.phase_durations[e][i]); x_lower.push_back(sp.bound_phase_duration_min); x_upper.push_back(sp.bound_phase_duration_max);
      }

}

}  // namespace

struct SetsHolder { std::vector<NodeSet> sets; RobotConst robot; double T = 0.0; std::vector<double> base_T; };

int Formulation::TrajectoryTables(double dt, std::vector<double>* times, std::vector<SplineSample>* samples, std::vector<int>* contact) const {
  if (!holder || !(dt > 0.0)) return TWB_ERR_INVALID;
  // Spline::GetTotalTime of the base spline (sum of its polynomial durations), then t += dt while t <= T + 1e-5
  double T = 0.0; for (double d : holder->base_T) T += d;
  times->clear();
  for (double t = 0.0; t <= T + 1e-5; t += dt) times->push_back(t);
  return SampleTables(*times, samples, contact);
}

int Formulation::SampleTables(const std::vector<double>& at, std::vector<SplineSample>* samples, std::vector<int>* contact) const {
  if (!holder) return TWB_ERR_INVALID;
  const std::vector<double>* times = &at;
  const std::vector<NodeSet>& sets = holder->sets;
  const int n_ee = spec.n_ee, zero_slot = n;
  samples->clear(); contact->clear();
  auto poly_durations = [&](const NodeSet& s, int e) {
    std::vector<double> d; for (auto& p : s.poly) d.push_back(spec.phase_durations[e][p.phase] / p.n_in_phase); return d;
  };
  SplineDef lin{&sets[0], holder->base_T}, ang{&sets[1], holder->base_T};
  std::vector<SplineDef> mo, fo;
  for (int e = 0; e < n_ee; ++e) { mo.push_back({&sets[2 + e], poly_durations(sets[2 + e], e)}); fo.push_back({&sets[2 + n_ee + e], poly_durations(sets[2 + n_ee + e], e)}); }
  auto foot = [&](int e, int kind, double t) {
    if (!optimize_timings) return MakeSample(kind == 0 ? mo[e] : fo[e], t, zero_slot);
    SplineSample o{}; o.T = t; o.xi[0] = (int16_t)kPhaseMarker; o.xi[1] = (int16_t)(2 * e + kind); return o;
  };
  for (double t : *times) {
    samples->push_back(MakeSample(lin, t, zero_slot));
    samples->push_back(MakeSample(ang, t, zero_slot));
    for (int e = 0; e < n_ee; ++e) samples->push_back(foot(e, 0, t));
    for (int e = 0; e < n_ee; ++e) samples->push_back(foot(e, 1, t));
    if (!optimize_timings)
      for (int e = 0; e < n_ee; ++e) {   // PhaseDurations::IsContactPhase, phase_durations.cc:120-124
        std::vector<double> ph(spec.phase_durations[e], spec.phase_durations[e] + spec.n_phases[e]);
        const int phase = SegmentID(t, ph);
        const bool first = spec.in_contact_at_start[e] != 0;
        contact->push_back((phase % 2 == 0 ? first : !first) ? 1 : 0);
      }
  }
  return TWB_OK;
}

// x0 and variable bounds of an instance that differs from the spec only in its goal pose (NlpFormulation::final_base_)
int Formulation::GoalInstance(const double final_lin_pos[3], const double final_ang_pos[3], double* x0_out, double* lo_out, double* up_out) const {
  if (!holder) return TWB_ERR_INVALID;
  twb_spec sp = spec;
  for (int k = 0; k < 3; ++k) { sp.final_base_lin_pos[k] = final_lin_pos[k]; sp.final_base_ang_pos[k] = final_ang_pos[k]; }
  std::vector<NodeSet> sets = holder->sets;
  std::vector<double> a, b, c;
  InitialGuessAndBounds(sp, holder->robot, holder->T, optimize_timings, &sets, &a, &b, &c);
  if (x0_out) std::copy(a.begin(), a.end(), x0_out);
  if (lo_out) std::copy(b.begin(), b.end(), lo_out);
  if (up_out) std::copy(c.begin(), c.end(), up_out);
  return TWB_OK;
}

// x0, variable bounds and constraint bounds of an instance whose NlpFormulation::initial_base_, final_base_ and initial_ee_W_
// are the state record `st` (TWB_STATE_DOUBLES): the constraint bounds are the problem's except the BaseMotionConstraint LZ
// rows, whose z_init is the instance's own initial guess of base-lin node 0 (base_motion_constraint.cc:51-54)
int Formulation::StateInstance(const double* st, double* x0_out, double* lo_out, double* up_out, double* gl_out, double* gu_out) const {
  if (!holder || !st) return TWB_ERR_INVALID;
  twb_spec sp = spec;
  for (int k = 0; k < 3; ++k) {
    sp.initial_base_lin_pos[k] = st[kStInitLinPos + k]; sp.initial_base_lin_vel[k] = st[kStInitLinVel + k];
    sp.initial_base_ang_pos[k] = st[kStInitAngPos + k]; sp.initial_base_ang_vel[k] = st[kStInitAngVel + k];
    sp.final_base_lin_pos[k] = st[kStFinalLinPos + k]; sp.final_base_lin_vel[k] = st[kStFinalLinVel + k];
    sp.final_base_ang_pos[k] = st[kStFinalAngPos + k]; sp.final_base_ang_vel[k] = st[kStFinalAngVel + k];
  }
  for (int e = 0; e < spec.n_ee; ++e) for (int k = 0; k < 3; ++k) sp.initial_ee_W[e][k] = st[kStInitEE + 3 * e + k];
  std::vector<NodeSet> sets = holder->sets;
  std::vector<double> a, b, c;
  InitialGuessAndBounds(sp, holder->robot, holder->T, optimize_timings, &sets, &a, &b, &c);
  if (x0_out) std::copy(a.begin(), a.end(), x0_out);
  if (lo_out) std::copy(b.begin(), b.end(), lo_out);
  if (up_out) std::copy(c.begin(), c.end(), up_out);
  const double z_init = sets[0].x0[sets[0].Var(0, kPos, Z)];
  if (gl_out) { std::copy(g_lower.begin(), g_lower.end(), gl_out); for (int r : tables.base_z_rows) gl_out[r] = z_init - 0.02; }
  if (gu_out) { std::copy(g_upper.begin(), g_upper.end(), gu_out); for (int r : tables.base_z_rows) gu_out[r] = z_init + 0.1; }
  return TWB_OK;
}

int Formulation::Build(const twb_spec& sp, std::string* err) {
  auto fail = [&](int code, const char* why) { if (err) *err = why; return code; };
  spec = sp;
  RobotConst rb;
  if (!GetRobot(sp.robot, &rb)) return fail(TWB_ERR_INVALID, "unknown robot");
  if (sp.n_ee != rb.n_ee) return fail(TWB_ERR_INVALID, "n_ee does not match the robot model");
  if (sp.terrain < 0 || sp.terrain >= TWB_TERRAIN_COUNT) return fail(TWB_ERR_INVALID, "unknown terrain");
  const int n_ee = sp.n_ee;
  for (int e = 0; e < n_ee; ++e)
    if (sp.n_phases[e] < 1 || sp.n_phases[e] > TWB_MAX_PHASES) return fail(TWB_ERR_INVALID, "bad phase count");
  if (sp.n_constraints < 0 || sp.n_constraints > TWB_MAX_CONSTRAINTS || sp.n_costs < 0 || sp.n_costs > TWB_MAX_COSTS)
    return fail(TWB_ERR_INVALID, "bad constraint/cost count");
  // numeric fields that drive loops and allocations (a zero-initialised or corrupted spec must fail here, not hang,
  // overflow or silently change m / nnz)
  auto pos_finite = [](double v) { return std::isfinite(v) && v > 0.0; };
  if (!pos_finite(sp.duration_base_polynomial) || !pos_finite(sp.dt_constraint_dynamic) || !pos_finite(sp.dt_constraint_range_of_motion) ||
      !pos_finite(sp.dt_constraint_base_motion))
    return fail(TWB_ERR_INVALID, "duration_base_polynomial and dt_constraint_* must be finite and > 0");
  if (sp.ee_polynomials_per_swing_phase < 1 || sp.ee_polynomials_per_swing_phase > 16 || sp.force_polynomials_per_stance_phase < 1 ||
      sp.force_polynomials_per_stance_phase > 16)
    return fail(TWB_ERR_INVALID, "polynomials per phase must be in 1..16");
  for (int e = 0; e < n_ee; ++e)
    for (int i = 0; i < sp.n_phases[e]; ++i)
      if (!pos_finite(sp.phase_durations[e][i])) return fail(TWB_ERR_INVALID, "phase durations must be finite and > 0");
  if (!std::isfinite(sp.force_limit_in_normal_direction) || !std::isfinite(sp.bound_phase_duration_min) || !std::isfinite(sp.bound_phase_duration_max))
    return fail(TWB_ERR_INVALID, "non-finite parameter");
  optimize_timings = false;
  for (int i = 0; i < sp.n_constraints; ++i) {
    if (sp.constraints[i] == TWB_C_TOTAL_TIME) optimize_timings = true;  // parameters.cc:128-135
    if (sp.constraints[i] < 0 || sp.constraints[i] > TWB_C_BASE_ACC) return fail(TWB_ERR_INVALID, "constraint not defined!");
  }

  // Parameters::GetTotalTime, parameters.cc:112-126
  double T = 0.0; for (int i = 0; i < sp.n_phases[0]; ++i) T += sp.phase_durations[0][i];
  for (int e = 1; e < n_ee; ++e) {
    double Te = 0.0; for (int i = 0; i < sp.n_phases[e]; ++i) Te += sp.phase_durations[e][i];
    if (std::fabs(Te - T) >= 1e-6) return fail(TWB_ERR_INVALID, "feet phase durations do not sum to the same total time");
  }
  if (!(T > 0.0)) return fail(TWB_ERR_INVALID, "total time must be positive");
  {   // bound the sample / polynomial counts (T / dt) before anything is allocated
    const double smallest = std::min(std::min(sp.duration_base_polynomial, sp.dt_constraint_dynamic), std::min(sp.dt_constraint_range_of_motion, sp.dt_constraint_base_motion));
    if (T / smallest > 4096.0) return fail(TWB_ERR_INVALID, "more than 4096 samples or base polynomials (T / dt)");
  }
  const std::vector<double> base_T = BasePolyDurations(T, sp.duration_base_polynomial);

  // ---- variable sets in AddVariableSet order (nlp_formulation.cc:63-93)
  std::vector<NodeSet> sets;
  sets.reserve(2 + 2 * n_ee);
  sets.push_back(MakeBaseSet("base-lin", (int)base_T.size() + 1));
  sets.push_back(MakeBaseSet("base-ang", (int)base_T.size() + 1));
  for (int e = 0; e < n_ee; ++e)
    sets.push_back(MakeMotionSet("ee-motion_" + std::to_string(e), sp.n_phases[e], sp.in_contact_at_start[e] != 0, sp.ee_polynomials_per_swing_phase));
  for (int e = 0; e < n_ee; ++e)
    sets.push_back(MakeForceSet("ee-force_" + std::to_string(e), sp.n_phases[e], sp.in_contact_at_start[e] != 0, sp.force_polynomials_per_stance_phase));
  n = 0; var_sets.clear();
  for (auto& s : sets) { s.offset = n; var_sets.push_back({s.name, n, s.n_vars}); n += s.n_vars; }
  // MakeContactScheduleVariables (nlp_formulation.cc:183-198): PhaseDurations sets "ee-schedule<ee>" hold all but the last phase
  std::vector<int> sched0(n_ee, -1);
  if (optimize_timings)
    for (int e = 0; e < n_ee; ++e) { sched0[e] = n; var_sets.push_back({"ee-schedule" + std::to_string(e), n, sp.n_phases[e] - 1}); n += sp.n_phases[e] - 1; }
  if (n + 1 > 32767) return fail(TWB_ERR_UNSUPPORTED, "more than 32766 variables");
  const int zero_slot = n;
  NodeSet& lin = sets[0]; NodeSet& ang = sets[1];
  auto motion = [&](int e) -> NodeSet& { return sets[2 + e]; };
  auto force = [&](int e) -> NodeSet& { return sets[2 + n_ee + e]; };

  // ---- initial guess and variable bounds (nlp_formulation.cc:95-181)
  InitialGuessAndBounds(sp, rb, T, optimize_timings, &sets, &x0, &x_lower, &x_upper);
  holder = std::make_shared<SetsHolder>(); holder->sets = sets; holder->robot = rb; holder->T = T; holder->base_T = base_T;

  // ---- the same initial guess / bounds as a per-variable recipe for the device (GoalInstanceKernel): mirrors
  // InitialGuessAndBounds above line by line; tests compare the kernel with Formulation::GoalInstance
  {
    tables = HostTables{};
    std::vector<GoalVar>& gv = tables.goal_vars; gv.assign(n, GoalVar{});
    auto fill_set = [&](const NodeSet& ns, int kind, int ee) {
      for (int node = 0; node < ns.n_nodes; ++node)
        for (int k = 0; k < 6; ++k) {
          const int v = ns.var[node][k];
          if (v < 0) continue;
          GoalVar& g = gv[ns.offset + v];
          g.kind = (int8_t)kind; g.ee = (int8_t)ee; g.deriv = (int8_t)(k / 3); g.dim = (int8_t)(k % 3);
          g.frac = node / static_cast<double>(ns.n_nodes - 1);   // the later node of a shared variable wins, like the reference's loop
          g.bound = kBoundFree;
        }
    };
    auto fix = [&](const NodeSet& ns, int node, int deriv, int dim, int8_t mode, double c) {
      const int v = ns.Var(node, deriv, dim);
      if (v >= 0) { gv[ns.offset + v].bound = mode; gv[ns.offset + v].c0 = c; gv[ns.offset + v].c1 = c; }
    };
    fill_set(lin, kGoalLin, 0); fill_set(ang, kGoalAng, 0);
    for (int e = 0; e < n_ee; ++e) { fill_set(motion(e), kGoalMotion, e); fill_set(force(e), kGoalForce, e); }
    const int last = lin.n_nodes - 1;
    for (int d = 0; d < 3; ++d) {
      fix(lin, 0, kPos, d, kBoundConst, sp.initial_base_lin_pos[d]); fix(lin, 0, kVel, d, kBoundConst, sp.initial_base_lin_vel[d]);
      fix(ang, 0, kPos, d, kBoundConst, sp.initial_base_ang_pos[d]); fix(ang, 0, kVel, d, kBoundConst, sp.initial_base_ang_vel[d]);
      if (sp.bounds_final_lin_pos[d]) fix(lin, last, kPos, d, kBoundGoalLin, 0.0);
      if (sp.bounds_final_lin_vel[d]) fix(lin, last, kVel, d, kBoundConst, sp.final_base_lin_vel[d]);
      if (sp.bounds_final_ang_pos[d]) fix(ang, last, kPos, d, kBoundGoalAng, 0.0);
      if (sp.bounds_final_ang_vel[d]) fix(ang, last, kVel, d, kBoundConst, sp.final_base_ang_vel[d]);
      for (int e = 0; e < n_ee; ++e) fix(motion(e), 0, kPos, d, kBoundConst, sp.initial_ee_W[e][d]);
    }
    if (optimize_timings)
      for (int e = 0; e < n_ee; ++e)
        for (int i = 0; i + 1 < sp.n_phases[e]; ++i) {
          GoalVar& g = gv[sched0[e] + i];
          g.kind = kGoalConst; g.frac = sp.phase_durations[e][i]; g.bound = kBoundPair; g.c0 = sp.bound_phase_duration_min; g.c1 = sp.bound_phase_duration_max;
        }
    // the start-state recipe: every bound above that copies a twb_spec state field reads the instance's state record instead
    // (the same Fix calls in the same order, so that a later Fix of the same variable still wins)
    std::vector<GoalVar>& sv = tables.state_vars; sv = gv;
    auto fix_state = [&](const NodeSet& ns, int node, int deriv, int dim, int src) {
      const int v = ns.Var(node, deriv, dim);
      if (v >= 0) { GoalVar& g = sv[ns.offset + v]; g.bound = kBoundState; g.src = (int8_t)src; g.c0 = g.c1 = 0.0; }
    };
    for (int d = 0; d < 3; ++d) {
      fix_state(lin, 0, kPos, d, kStInitLinPos + d); fix_state(lin, 0, kVel, d, kStInitLinVel + d);
      fix_state(ang, 0, kPos, d, kStInitAngPos + d); fix_state(ang, 0, kVel, d, kStInitAngVel + d);
      if (sp.bounds_final_lin_pos[d]) fix_state(lin, last, kPos, d, kStFinalLinPos + d);
      if (sp.bounds_final_lin_vel[d]) fix_state(lin, last, kVel, d, kStFinalLinVel + d);
      if (sp.bounds_final_ang_pos[d]) fix_state(ang, last, kPos, d, kStFinalAngPos + d);
      if (sp.bounds_final_ang_vel[d]) fix_state(ang, last, kVel, d, kStFinalAngVel + d);
      for (int e = 0; e < n_ee; ++e) fix_state(motion(e), 0, kPos, d, kStInitEE + 3 * e + d);
    }
    GoalSetup& gs = tables.goal_setup; gs = GoalSetup{};
    for (int d = 0; d < 3; ++d) { gs.initial_lin[d] = sp.initial_base_lin_pos[d]; gs.initial_ang[d] = sp.initial_base_ang_pos[d]; }
    for (int e = 0; e < n_ee; ++e) for (int d = 0; d < 3; ++d) { gs.initial_ee[e][d] = sp.initial_ee_W[e][d]; gs.nominal[e][d] = rb.nominal[e][d]; }
    gs.t_total = T; gs.f_stance_z = rb.mass * 9.80665 / n_ee;
  }

  // ---- splines (spline_holder.cc:35-61, fixed durations)
  auto poly_durations = [&](const NodeSet& s, int e) {  // nodes_variables_phase_based.cc:78-89
    std::vector<double> d;
    for (auto& p : s.poly) d.push_back(sp.phase_durations[e][p.phase] / p.n_in_phase);
    return d;
  };
  SplineDef sp_lin{&lin, base_T}, sp_ang{&ang, base_T};
  std::vector<SplineDef> sp_motion, sp_force;
  for (int e = 0; e < n_ee; ++e) { sp_motion.push_back({&motion(e), poly_durations(motion(e), e)}); sp_force.push_back({&force(e), poly_durations(force(e), e)}); }

  // ---- units and their Jacobian entries
  HostTables& tb = tables;
  // foot splines: fixed-duration samples, or a reference to the PhaseSpline when the durations are optimised
  auto foot_sample = [&](int e, int kind, double t) {   // kind 0: ee-motion, 1: ee-force
    if (!optimize_timings) return MakeSample(kind == 0 ? sp_motion[e] : sp_force[e], t, zero_slot);
    SplineSample o{};
    o.T = t; o.xi[0] = (int16_t)kPhaseMarker; o.xi[1] = (int16_t)(2 * e + kind);
    return o;
  };
  if (optimize_timings) {
    for (int e = 0; e < n_ee; ++e)
      for (int kind = 0; kind < 2; ++kind) {
        const NodeSet& ns = kind == 0 ? motion(e) : force(e);
        PhaseSplineDef def{}; def.poly0 = (int32_t)tb.phase_polys.size(); def.n_polys = (int32_t)ns.poly.size();
        def.sched0 = sched0[e]; def.n_phases = sp.n_phases[e];
        def.t_total = 0.0; for (int i = 0; i < sp.n_phases[e]; ++i) def.t_total += sp.phase_durations[e][i];   // std::accumulate, phase_durations.cc:47
        for (int p = 0; p < (int)ns.poly.size(); ++p) {
          PhasePoly pp{};
          for (int side = 0; side < 2; ++side) for (int deriv = 0; deriv < 2; ++deriv) for (int dim = 0; dim < 3; ++dim)
            pp.xi[side * 6 + deriv * 3 + dim] = XIndex(ns, p + side, deriv, dim, zero_slot);
          pp.phase = (int16_t)ns.poly[p].phase; pp.n_in_phase = (int16_t)ns.poly[p].n_in_phase; pp.k_in_phase = (int16_t)ns.poly[p].k_in_phase;
          tb.phase_polys.push_back(pp);
        }
        tb.phase_defs.push_back(def);
      }
  }
  // PhaseSpline pattern (phase_spline.cc:45-51): every variable of the set is structurally non-zero in the row of its dimension.
  // Per variable: column, dimension, node derivative, first node holding it and whether the next node shares it (stance
  // position of a phase-based ee-motion set) — what decides, per instance, which Hermite basis value multiplies it.
  struct VarInfo { int col = -1, dim = -1, deriv = -1, a = -1, count = 0; bool ok = true; };
  auto all_vars = [&](const NodeSet& ns) {
    std::vector<VarInfo> v(ns.n_vars);
    for (int nd = 0; nd < ns.n_nodes; ++nd) for (int k = 0; k < 6; ++k) {
      const int var = ns.var[nd][k];
      if (var < 0) continue;
      VarInfo& vi = v[var];
      if (vi.count == 0) { vi.col = ns.offset + var; vi.dim = k % 3; vi.deriv = k / 3; vi.a = nd; vi.count = 1; }
      else { if (vi.dim != k % 3 || vi.deriv != k / 3 || nd != vi.a + vi.count || vi.count >= 2) vi.ok = false; vi.count++; }
    }
    return v;
  };
  if (optimize_timings)
    for (int e = 0; e < n_ee; ++e) for (int kind = 0; kind < 2; ++kind) {
      const NodeSet& ns = kind == 0 ? motion(e) : force(e);
      if (ns.n_nodes > 255) return fail(TWB_ERR_UNSUPPORTED, "more than 255 nodes in a phase-based set");
      for (auto& vi : all_vars(ns)) if (!vi.ok || vi.count < 1 || (vi.count == 2 && vi.deriv != kPos)) return fail(TWB_ERR_UNSUPPORTED, "node variable shared by more than two adjacent nodes");
    }
  Plan& pl = tb.plan;
  const uint32_t S_ONE = 0;      // local row 0 of every unit's state block is the constant 1

  std::vector<Emit> em;
  auto emit1 = [&](int row, int col, uint32_t a, double c) { em.push_back({row, col, a, c}); };
  auto emit_phase = [&](int row, int col, uint32_t a, double c, uint32_t ext, int tail) { Emit e{row, col, a, c}; e.ext = ext; e.tail = tail; em.push_back(e); };
  std::vector<RowOwner> owner;         // per constraint row
  std::vector<NodeUnitRef> node_units; // node-wise units in row order
  int set_counter = 0;

  m = 0; con_sets.clear(); g_lower.clear(); g_upper.clear();
  auto add_set = [&](const std::string& name, int rows) {
    con_sets.push_back({name, m, rows}); int r0 = m; m += rows;
    g_lower.resize(m, 0.0); g_upper.resize(m, 0.0); owner.resize(m); ++set_counter;
    return r0;
  };
  auto bound = [&](int row, double lo, double up) { g_lower[row] = lo; g_upper[row] = up; };
  auto own = [&](int row, int kind, int index, uint32_t g_local) { owner[row].kind = kind; owner[row].index = index; owner[row].g_local = g_local; };
  // node unit `index` of table `kind` owns `n_g` rows starting at `row`; returns its id
  auto add_node_unit = [&](int kind, int index, int n_state, int n_g, int row) {
    const int id = (int)node_units.size();
    node_units.push_back({kind, index, n_state, n_g, set_counter});
    for (int r = 0; r < n_g; ++r) own(row + r, kOwnNode, id, (uint32_t)r);
    return id;
  };

  pl.n_dyn = pl.n_rom = 0;
  bool have_dyn = false, have_rom = false, have_base_motion = false;

  for (int ci = 0; ci < sp.n_constraints; ++ci) {
    switch (sp.constraints[ci]) {
      case TWB_C_DYNAMIC: {  // dynamic_constraint.cc + single_rigid_body_dynamics.cc:103-192
        if (have_dyn) return fail(TWB_ERR_UNSUPPORTED, "constraint listed twice");
        have_dyn = true;
        std::vector<double> ts = SampleTimes(T, sp.dt_constraint_dynamic);
        int r0 = add_set("dynamic", (int)ts.size() * 6);
        pl.n_dyn = (int)ts.size();
        // local state: [0]=1 | sum f (3) | base-ang block (36) | f_e, c-p_e (6 per foot) | the 6 constraint values
        for (int k = 0; k < pl.n_dyn; ++k) {
          const double t = ts[k];
          const int row = r0 + 6 * k;
          const uint32_t sb = 1;
          DynUnit du{}; du.sample0 = (int32_t)tb.samples.size(); du.g_row0 = row;
          tb.dyn.push_back(du);
          for (int r = 0; r < 6; ++r) { bound(row + r, 0.0, 0.0); own(row + r, kOwnDyn, k, 0); }
          // spline samples: base-lin, base-ang, ee-motion.., ee-force..
          tb.samples.push_back(MakeSample(sp_lin, t, zero_slot));
          tb.samples.push_back(MakeSample(sp_ang, t, zero_slot));
          for (int e = 0; e < n_ee; ++e) tb.samples.push_back(foot_sample(e, 0, t));
          for (int e = 0; e < n_ee; ++e) tb.samples.push_back(foot_sample(e, 1, t));
          int p; double tl;
          // base-lin: angular rows = -sum_e [f_e]x dc ; linear rows = m * d(acc)
          Locate(sp_lin, t, &p, &tl);
          for (auto& b : Basis(sp_lin, p, tl, kPos))
            for (int i = 0; i < 3; ++i) if (i != b.dim) {
              int comp; double sg; CrossEntry(i, b.dim, &comp, &sg);
              emit1(row + i, lin.offset + b.var, sb + comp, -sg * b.val);
            }
          for (auto& b : Basis(sp_lin, p, tl, kAcc)) emit1(row + 3 + b.dim, lin.offset + b.var, S_ONE, rb.mass * b.val);
          // base-ang: angular rows = A*dtheta + B*dtheta_dot + C*dtheta_ddot, contracted with the
          // basis by the dynamic unit itself: S holds the 3 x 12 finished values
          Locate(sp_ang, t, &p, &tl);
          {
            auto bp = Basis(sp_ang, p, tl, kPos), bv = Basis(sp_ang, p, tl, kVel), ba = Basis(sp_ang, p, tl, kAcc);
            if (bp.size() != 12) return fail(TWB_ERR_UNSUPPORTED, "base-ang basis layout");
            for (int j = 0; j < 12; ++j) {
              if (bp[j].dim != j % 3 || bp[j].var != p * 6 + j) return fail(TWB_ERR_UNSUPPORTED, "base-ang basis layout");
              for (int i = 0; i < 3; ++i) emit1(row + i, ang.offset + bp[j].var, sb + 3 + i * 12 + j, 1.0);
            }
            for (int q = 0; q < 4; ++q) tb.dyn_ang_basis.push_back(bp[3 * q].val);
            for (int q = 0; q < 4; ++q) tb.dyn_ang_basis.push_back(bv[3 * q].val);
            for (int q = 0; q < 4; ++q) tb.dyn_ang_basis.push_back(ba[3 * q].val);
          }
          for (int e = 0; e < n_ee && optimize_timings; ++e) {
            // PhaseSpline columns (dynamic_constraint.cc:91-113, single_rigid_body_dynamics.cc:167-192): phase elements written by
            // the DynTailOut kernel, CTA = sample, warp = foot; rows of the foot's state block (kTailRows):
            // 0: 1 | 1..3: f_e | 4..6: c - p_e | 7..18: info block of ee-motion | 19..30: info block of ee-force | 31..36: U | 37..: X
            const uint32_t tb0 = (uint32_t)e * kTailRows, F = tb0 + 1, Rr = tb0 + 4, info_mo = tb0 + 7, info_fo = tb0 + 7 + kInfoRows, cur = info_mo, U0 = tb0 + 7 + 2 * kInfoRows;
            for (auto& vi : all_vars(motion(e)))   // angular rows: [f_e]x d(p_e)
              for (int i = 0; i < 3; ++i) if (i != vi.dim) {
                int comp; double sg; CrossEntry(i, vi.dim, &comp, &sg);
                emit_phase(row + i, vi.col, F + comp, sg, PackExt(kElemNode, vi.deriv, vi.count == 2, vi.a, info_mo), k);
              }
            for (auto& vi : all_vars(force(e))) {   // angular rows: [c - p_e]x d(f_e); linear rows: -d(f_e)
              for (int i = 0; i < 3; ++i) if (i != vi.dim) {
                int comp; double sg; CrossEntry(i, vi.dim, &comp, &sg);
                emit_phase(row + i, vi.col, Rr + comp, sg, PackExt(kElemNode, vi.deriv, vi.count == 2, vi.a, info_fo), k);
              }
              emit_phase(row + 3 + vi.dim, vi.col, tb0, -1.0, PackExt(kElemNode, vi.deriv, vi.count == 2, vi.a, info_fo), k);
            }
            // ee-schedule: JacWrtForce + JacWrtEEPos of the dense 3 x (P-1) duration Jacobians (dynamic_constraint.cc:106-112)
            for (int ph = 0; ph + 1 < sp.n_phases[e]; ++ph)
              for (int r = 0; r < 6; ++r) emit_phase(row + r, sched0[e] + ph, U0 + r, 1.0, PackExt(kElemDuration, 0, false, ph, cur), k);
          }
          for (int e = 0; e < n_ee && !optimize_timings; ++e) {
            // ee-motion: angular rows = [f_e]x dp_e
            Locate(sp_motion[e], t, &p, &tl);
            for (auto& b : Basis(sp_motion[e], p, tl, kPos))
              for (int i = 0; i < 3; ++i) if (i != b.dim) {
                int comp; double sg; CrossEntry(i, b.dim, &comp, &sg);
                emit1(row + i, motion(e).offset + b.var, sb + 39 + e * 6 + comp, sg * b.val);
              }
            // ee-force: angular rows = [c - p_e]x df_e ; linear rows = -df_e
            Locate(sp_force[e], t, &p, &tl);
            for (auto& b : Basis(sp_force[e], p, tl, kPos)) {
              for (int i = 0; i < 3; ++i) if (i != b.dim) {
                int comp; double sg; CrossEntry(i, b.dim, &comp, &sg);
                emit1(row + i, force(e).offset + b.var, sb + 39 + e * 6 + 3 + comp, sg * b.val);
              }
              emit1(row + 3 + b.dim, force(e).offset + b.var, S_ONE, -b.val);
            }
          }
        }
        break;
      }
      case TWB_C_EE_ROM: {  // range_of_motion_constraint.cc
        if (have_rom) return fail(TWB_ERR_UNSUPPORTED, "constraint listed twice");
        have_rom = true;
        std::vector<double> ts = SampleTimes(T, sp.dt_constraint_range_of_motion);
        pl.n_rom = (int)ts.size();
        // local state: [0]=1 | R^T (9) | two buffers of D_e (9) + g_e (3) used by the feet in turn (foot e: buffer e & 1)
        for (int k = 0; k < pl.n_rom; ++k) {  // spline samples: base-lin, base-ang, ee-motion..
          RomUnit ru{}; ru.sample0 = (int32_t)tb.samples.size();
          tb.rom.push_back(ru);
          tb.samples.push_back(MakeSample(sp_lin, ts[k], zero_slot));
          tb.samples.push_back(MakeSample(sp_ang, ts[k], zero_slot));
          for (int e = 0; e < n_ee; ++e) tb.samples.push_back(foot_sample(e, 0, ts[k]));
        }
        for (int e = 0; e < n_ee; ++e) {
          int r0 = add_set("rangeofmotion-" + std::to_string(e), pl.n_rom * 3);
          pl.rom_row0[e] = r0;
          for (int k = 0; k < pl.n_rom; ++k) {
            const double t = ts[k]; const int row = r0 + 3 * k;
            const uint32_t sb = 1, sd = 10 + RomBufferP(e, optimize_timings);
            for (int d = 0; d < 3; ++d) {
              bound(row + d, (0.0 + rb.nominal[e][d]) - rb.max_dev[d], (0.0 + rb.nominal[e][d]) + rb.max_dev[d]);
              own(row + d, kOwnRom, k * n_ee + e, 0);
            }
            int p; double tl;
            Locate(sp_lin, t, &p, &tl);   // -R^T dc
            for (auto& b : Basis(sp_lin, p, tl, kPos)) for (int i = 0; i < 3; ++i) emit1(row + i, lin.offset + b.var, sb + i * 3 + b.dim, -b.val);
            Locate(sp_ang, t, &p, &tl);   // d(R^T r)/dtheta ; row X does not depend on roll
            for (auto& b : Basis(sp_ang, p, tl, kPos)) for (int i = 0; i < 3; ++i)
              if (!(i == 0 && b.dim == 0)) emit1(row + i, ang.offset + b.var, sd + i * 3 + b.dim, b.val);
            if (optimize_timings) {
              // PhaseSpline columns (range_of_motion_constraint.cc:83-109): phase elements of the foot's own list; the foot's
              // buffer continues with the info block (sd + 9 .. sd + 20) | sd + 21..23: U | sd + 24..: X
              const uint32_t info = sd + 9, cur = info, U0 = sd + 9 + kInfoRows;
              for (auto& vi : all_vars(motion(e)))   // R^T d(p_e)
                for (int i = 0; i < 3; ++i) emit_phase(row + i, vi.col, sb + i * 3 + vi.dim, 1.0, PackExt(kElemNode, vi.deriv, vi.count == 2, vi.a, info), -1);
              for (int ph = 0; ph + 1 < sp.n_phases[e]; ++ph)
                for (int i = 0; i < 3; ++i) emit_phase(row + i, sched0[e] + ph, U0 + i, 1.0, PackExt(kElemDuration, 0, false, ph, cur), -1);
              continue;
            }
            Locate(sp_motion[e], t, &p, &tl);  // R^T dp_e
            for (auto& b : Basis(sp_motion[e], p, tl, kPos)) for (int i = 0; i < 3; ++i) emit1(row + i, motion(e).offset + b.var, sb + i * 3 + b.dim, b.val);
          }
        }
        break;
      }
      case TWB_C_BASE_ROM: {  // base_motion_constraint.cc:38-91
        if (have_base_motion) return fail(TWB_ERR_UNSUPPORTED, "constraint listed twice");
        have_base_motion = true;
        std::vector<double> ts = SampleTimes(T, sp.dt_constraint_base_motion);
        int r0 = add_set("baseMotion", (int)ts.size() * 6);
        const double dev_rad = 0.05;
        // z_init = base_linear_->GetPoint(0.0).p().z() at construction (:51): polynomial 0 of the initial guess at t = 0
        const double z_init = lin.x0[lin.Var(0, kPos, Z)];
        for (int k = 0; k < (int)ts.size(); ++k) {
          const int row = r0 + 6 * k;   // rows AX, AY, AZ, LX, LY, LZ
          BaseMotionUnit u{}; u.sample_lin = (int32_t)tb.samples.size(); u.sample_ang = u.sample_lin + 1;
          tb.samples.push_back(MakeSample(sp_lin, ts[k], zero_slot));
          tb.samples.push_back(MakeSample(sp_ang, ts[k], zero_slot));
          tb.base_motion.push_back(u);
          add_node_unit(kGroupBaseMotion, (int)tb.base_motion.size() - 1, 0, 6, row);
          bound(row + 0, -dev_rad, dev_rad); bound(row + 1, -dev_rad, dev_rad); bound(row + 2, -kInf, +kInf);
          bound(row + 3, -kInf, +kInf); bound(row + 4, -kInf, +kInf); bound(row + 5, z_init - 0.02, z_init + 0.1);
          tb.base_z_rows.push_back(row + 5);   // the only constraint bounds that depend on the start state (StateInstance)
          int p; double tl;
          Locate(sp_ang, ts[k], &p, &tl);
          for (auto& b : Basis(sp_ang, p, tl, kPos)) emit1(row + b.dim, ang.offset + b.var, S_ONE, b.val);
          Locate(sp_lin, ts[k], &p, &tl);
          for (auto& b : Basis(sp_lin, p, tl, kPos)) emit1(row + 3 + b.dim, lin.offset + b.var, S_ONE, b.val);
        }
        break;
      }
      case TWB_C_TERRAIN: {  // terrain_constraint.cc
        for (int e = 0; e < n_ee; ++e) {
          const NodeSet& mo = motion(e);
          int r0 = add_set("terrain-ee-motion_" + std::to_string(e), mo.n_nodes - 1);
          for (int nd = 1; nd < mo.n_nodes; ++nd) {
            int row = r0 + nd - 1;
            if (mo.ConstNode(nd)) bound(row, 0.0, 0.0); else bound(row, 0.0, 1e20);
            TerrainUnit u{}; for (int d = 0; d < 3; ++d) u.xi[d] = XIndex(mo, nd, kPos, d, zero_slot);
            tb.terr.push_back(u);
            add_node_unit(kGroupTerrain, (int)tb.terr.size() - 1, 2, 1, row);   // unit state: -dh/dx | -dh/dy
            emit1(row, mo.offset + mo.Var(nd, kPos, X), 1, 1.0);
            emit1(row, mo.offset + mo.Var(nd, kPos, Y), 2, 1.0);
            emit1(row, mo.offset + mo.Var(nd, kPos, Z), S_ONE, 1.0);
          }
        }
        break;
      }
      case TWB_C_FORCE: {  // force_constraint.cc
        for (int e = 0; e < n_ee; ++e) {
          const NodeSet& fo = force(e); const NodeSet& mo = motion(e);
          std::vector<int> ids; for (int nd = 0; nd < fo.n_nodes; ++nd) if (!fo.ConstNode(nd)) ids.push_back(nd);
          int r0 = add_set("force-ee-force_" + std::to_string(e), (int)ids.size() * 5);
          int row = r0;
          for (int nd : ids) {
            // NodesVariablesPhaseBased::GetPhase (:136-143) and GetNodeIDAtStartOfPhase (:145-168)
            int phase = fo.poly[nd == 0 ? 0 : (nd == fo.n_nodes - 1 ? nd - 1 : nd - 1)].phase;
            int mnode = 0; for (int i = 0; i < (int)mo.poly.size(); ++i) if (mo.poly[i].phase == phase) { mnode = i; break; }
            ForceUnit u{};
            for (int d = 0; d < 3; ++d) { u.xf[d] = XIndex(fo, nd, kPos, d, zero_slot); u.xp[d] = XIndex(mo, mnode, kPos, d, zero_slot); }
            tb.force.push_back(u);
            add_node_unit(kGroupForce, (int)tb.force.size() - 1, 25, 5, row);   // unit state: 25 values [row][{d/dpx,d/dpy,d/dfx,d/dfy,d/dfz}]
            bound(row + 0, 0.0, sp.force_limit_in_normal_direction);
            bound(row + 1, -kInf, 0.0); bound(row + 2, 0.0, +kInf); bound(row + 3, -kInf, 0.0); bound(row + 4, 0.0, +kInf);
            for (int r = 0; r < 5; ++r) {
              for (int d = 0; d < 2; ++d) emit1(row + r, mo.offset + mo.Var(mnode, kPos, d), 1 + r * 5 + d, 1.0);
              for (int d = 0; d < 3; ++d) emit1(row + r, fo.offset + fo.Var(nd, kPos, d), 1 + r * 5 + 2 + d, 1.0);
            }
            row += 5;
          }
        }
        break;
      }
      case TWB_C_SWING: {  // swing_constraint.cc
        const double t_swing_avg = 0.3;  // swing_constraint.h:68
        for (int e = 0; e < n_ee; ++e) {
          const NodeSet& mo = motion(e);
          std::vector<int> ids; for (int nd = 0; nd < mo.n_nodes; ++nd) if (!mo.ConstNode(nd)) ids.push_back(nd);
          int r0 = add_set("swing-ee-motion_" + std::to_string(e), (int)ids.size() * 4);
          int row = r0;
          for (int nd : ids) {
            if (nd == 0 || nd == mo.n_nodes - 1) return fail(TWB_ERR_UNSUPPORTED, "swing node at the spline boundary");
            SwingUnit u{};
            for (int d = 0; d < 2; ++d) {
              u.xc_p[d] = XIndex(mo, nd, kPos, d, zero_slot); u.xc_v[d] = XIndex(mo, nd, kVel, d, zero_slot);
              u.xprev[d] = XIndex(mo, nd - 1, kPos, d, zero_slot); u.xnext[d] = XIndex(mo, nd + 1, kPos, d, zero_slot);
            }
            tb.swing.push_back(u);
            add_node_unit(kGroupSwing, (int)tb.swing.size() - 1, 0, 4, row);
            for (int d = 0; d < 2; ++d) {
              bound(row, 0.0, 0.0);
              emit1(row, mo.offset + mo.Var(nd, kPos, d), S_ONE, 1.0);
              emit1(row, mo.offset + mo.Var(nd + 1, kPos, d), S_ONE, -0.5);
              emit1(row, mo.offset + mo.Var(nd - 1, kPos, d), S_ONE, -0.5);
              ++row;
              bound(row, 0.0, 0.0);
              emit1(row, mo.offset + mo.Var(nd, kVel, d), S_ONE, 1.0);
              emit1(row, mo.offset + mo.Var(nd + 1, kPos, d), S_ONE, -1.0 / t_swing_avg);
              emit1(row, mo.offset + mo.Var(nd - 1, kPos, d), S_ONE, +1.0 / t_swing_avg);
              ++row;
            }
          }
        }
        break;
      }
      case TWB_C_BASE_ACC: {  // spline_acc_constraint.cc
        for (int which = 0; which < 2; ++which) {
          const SplineDef& s = which == 0 ? sp_lin : sp_ang;
          const NodeSet& ns = *s.set;
          int nj = (int)s.T.size() - 1;
          int r0 = add_set("splineacc-" + ns.name, 3 * nj);
          for (int j = 0; j < nj; ++j) {
            AccUnit u{};
            u.Tp = s.T[j]; u.Tp2 = std::pow(u.Tp, 2); u.Tp3 = std::pow(u.Tp, 3); u.rTp2 = 1.0 / u.Tp2; u.rTp3 = 1.0 / u.Tp3;
            u.Tn = s.T[j + 1]; u.Tn2 = std::pow(u.Tn, 2); u.rTn2 = 1.0 / u.Tn2;
            u.x0 = ns.offset + j * 6;
            tb.acc.push_back(u);
            add_node_unit(kGroupAcc, (int)tb.acc.size() - 1, 0, 3, r0 + 3 * j);
            // acc_prev - acc_next with the union of both patterns (:67-80)
            std::map<int, std::pair<int, double>> u_map;  // var -> (dim, value)
            for (auto& b : Basis(s, j, s.T[j], kAcc)) u_map[b.var] = {b.dim, b.val};
            for (auto& b : Basis(s, j + 1, 0.0, kAcc)) {
              auto it = u_map.find(b.var);
              if (it == u_map.end()) u_map[b.var] = {b.dim, 0.0 - b.val}; else it->second.second = it->second.second - b.val;
            }
            for (auto& kv : u_map) emit1(r0 + 3 * j + kv.second.first, ns.offset + kv.first, S_ONE, kv.second.second);
            for (int d = 0; d < 3; ++d) bound(r0 + 3 * j + d, 0.0, 0.0);
          }
        }
        break;
      }
      case TWB_C_TOTAL_TIME: {  // total_duration_constraint.cc:36-72 — written by the PhaseJac kernel
        PhaseUnit pu{}; pu.kind = kPhaseTotal;
        for (int e = 0; e < n_ee; ++e) {
          int row = add_set("totalduration-" + std::to_string(e), 1);
          bound(row, 0.1, T - 0.2);
          own(row, kOwnPhase, e, 0);
          pu.rows[e] = row;
          for (int ph = 0; ph + 1 < sp.n_phases[e]; ++ph) emit1(row, sched0[e] + ph, S_ONE, 1.0);
        }
        tb.phase_units.push_back(pu);
        break;
      }
      default: return fail(TWB_ERR_INVALID, "constraint not defined!");
    }
  }
  if (tb.samples.size() > 0x7FFFFFFFu) return fail(TWB_ERR_UNSUPPORTED, "too many spline samples");

  // ---- CSR assembly: row-major, ascending column (what setFromTriplets yields)
  std::stable_sort(em.begin(), em.end(), [](const Emit& a, const Emit& b) { return a.row != b.row ? a.row < b.row : a.col < b.col; });
  for (size_t i = 1; i < em.size(); ++i)
    if (em[i].row == em[i - 1].row && em[i].col == em[i - 1].col) return fail(TWB_ERR_UNSUPPORTED, "duplicate Jacobian entry emitted");
  nnz = (int)em.size();
  row_ptr.assign(m + 1, 0); col_idx.resize(nnz);
  for (int s = 0; s < nnz; ++s) { row_ptr[em[s].row + 1]++; col_idx[s] = em[s].col; }
  for (int r = 0; r < m; ++r) row_ptr[r + 1] += row_ptr[r];

  for (auto& pu : tb.phase_units) for (int e = 0; e < n_ee; ++e) pu.slot0[e] = row_ptr[pu.rows[e]];

  // ---- node groups: consecutive units of one kind and one constraint set share a warp's state block
  struct GroupBuild { int kind, first, count; std::vector<int> unit_ids; };
  std::vector<GroupBuild> groups;
  std::vector<int> unit_group(node_units.size(), -1), unit_state0(node_units.size(), 0), unit_g0(node_units.size(), 0);
  {
    auto cap = [&](int kind) { return kind == kGroupForce ? 1 : kind == kGroupTerrain ? 10 : kind == kGroupSwing ? 7 : kind == kGroupAcc ? 10 : 5; };
    for (size_t u = 0; u < node_units.size(); ++u) {
      const NodeUnitRef& nu = node_units[u];
      bool open = !groups.empty() && groups.back().kind == nu.kind && groups.back().count < cap(nu.kind) &&
                  node_units[groups.back().unit_ids.back()].set_id == nu.set_id && groups.back().first + groups.back().count == nu.index;
      if (!open) groups.push_back({nu.kind, nu.index, 0, {}});
      groups.back().count++; groups.back().unit_ids.push_back((int)u);
      unit_group[u] = (int)groups.size() - 1;
    }
    pl.node_rows = 1;
    for (auto& gb : groups) {   // state block: [0]=1 | unit states | unit values
      int top = 1;
      for (int u : gb.unit_ids) { unit_state0[u] = top; top += node_units[u].n_state; }
      for (int u : gb.unit_ids) { unit_g0[u] = top; top += node_units[u].n_g; }
      if (top > kNodeStateRowsMax) return fail(TWB_ERR_UNSUPPORTED, "node group state block too large");
      pl.node_rows = std::max(pl.node_rows, top);
    }
  }

  // ---- output lists (device_tables.h).  The Jacobian values are written by CTAs: a CTA holds the state blocks of
  // kDynWarps / kRomWarps / kNodeWarps consecutive units (one per warp) and, after its barrier, ALL its threads walk one
  // combined list of 16-byte pairs (`d` = row in the CTA's shared memory = warp * block_rows + local row).  Every
  // 32-byte sector is written whole by the list that owns its last element; only sectors shared with another CTA (or a
  // row of the PhaseJac kernel, or the ends of the row) fall back to single-element stores.  The constraint values
  // are written from the units' state rows (kernels.cu: StoreValuesDirect); only a node group's rows that are not
  // consecutive state rows need a table (NodeGroup::values).
  const int n_rom_blocks = pl.n_rom * n_ee, n_blocks = pl.n_dyn + n_rom_blocks + (int)groups.size();
  auto block_id = [&](const RowOwner& o) {   // global block number: dynamic samples | (rom sample, foot) | node groups; -1: not an output-kernel row
    if (o.kind == kOwnPhase) return -1;
    if (o.kind == kOwnDyn) return o.index;
    if (o.kind == kOwnRom) return pl.n_dyn + o.index;
    return pl.n_dyn + n_rom_blocks + unit_group[o.index];
  };
  const int n_dyn_ctas = (pl.n_dyn + kDynWarps - 1) / kDynWarps, n_rom_ctas = (pl.n_rom + kRomWarps - 1) / kRomWarps;
  const int n_node_ctas = ((int)groups.size() + kNodeWarps - 1) / kNodeWarps;
  const int tail_list0 = n_dyn_ctas + n_rom_ctas * n_ee + n_node_ctas;
  const int n_lists = tail_list0 + (optimize_timings ? pl.n_dyn : 0);   // dynamic CTAs | (rom CTA, foot) | node CTAs | PhaseSpline columns of dynamic sample k
  pl.tail_list0 = tail_list0;
  pl.dyn_rows = DynBlockRows(n_ee); pl.rom_rows = RomBlockRowsP(n_ee, optimize_timings);
  std::vector<int> list_of(n_blocks, -1), row_base(n_blocks, 0);   // list a block's elements belong to; first row of the block inside its CTA
  for (int k = 0; k < pl.n_dyn; ++k) { list_of[k] = k / kDynWarps; row_base[k] = (k % kDynWarps) * pl.dyn_rows; }
  for (int k = 0; k < pl.n_rom; ++k) for (int e = 0; e < n_ee; ++e) {
    const int b = pl.n_dyn + k * n_ee + e;
    list_of[b] = n_dyn_ctas + (k / kRomWarps) * n_ee + e; row_base[b] = (k % kRomWarps) * pl.rom_rows;
  }
  for (int gi = 0; gi < (int)groups.size(); ++gi) {
    const int b = pl.n_dyn + n_rom_blocks + gi;
    list_of[b] = n_dyn_ctas + n_rom_ctas * n_ee + gi / kNodeWarps; row_base[b] = (gi % kNodeWarps) * pl.node_rows;
  }
  struct Elem { int list; uint16_t d; double c; uint32_t ext; };
  std::vector<Elem> elems(nnz);
  struct Entry { OutPair p; OutCoef c; PhaseExt x{0, 0}; };
  std::vector<std::vector<Entry>> values(groups.size());   // constraint values of a node group: (g row, local state row, 1)
  for (int r = 0; r < m; ++r) {
    const RowOwner& o = owner[r];
    if (o.kind < 0) return fail(TWB_ERR_UNSUPPORTED, "constraint row without an owner");
    uint32_t state0 = 1;
    if (o.kind == kOwnNode) {
      state0 = unit_state0[o.index];
      values[unit_group[o.index]].push_back({OutPair{r, (uint16_t)(unit_g0[o.index] + o.g_local), 0}, OutCoef{1.0, 0.0}});
    }
    const int blk = block_id(o);
    for (int s = row_ptr[r]; s < row_ptr[r + 1]; ++s) {
      uint32_t a = em[s].a;
      if (em[s].tail >= 0) { elems[s] = Elem{tail_list0 + em[s].tail, (uint16_t)a, em[s].c0, em[s].ext}; continue; }   // rows of the tail kernel's CTA
      if (o.kind == kOwnNode && a != S_ONE) a = state0 + (a - 1);
      uint32_t ext = em[s].ext;
      if (blk >= 0 && (ext & 3u)) ext += (uint32_t)row_base[blk] << 16;   // info row: unit-local -> row of the CTA's shared memory
      elems[s] = blk >= 0 ? Elem{list_of[blk], (uint16_t)(row_base[blk] + a), em[s].c0, ext} : Elem{-1, 0, 0.0, 0};
    }
  }
  // lists[list][class][0: pairs, 1: singles, 2: pairs of sectors with a phase element]
  std::vector<std::array<std::array<std::vector<Entry>, 3>, kMaxClasses>> lists(n_lists);
  const int NC = (nnz % 4 == 0) ? 1 : (nnz % 2 == 0) ? 2 : 4;
  pl.nc_jac = NC;
  // ---- constant runs (device_tables.h: ConstRun): whole sectors whose elements all multiply the constant-1 state row.
  // Only with one alignment class (every instance's row starts on a sector) and without PhaseJac overwrites.
  std::vector<char> is_const_run(nnz, 0);
  if (NC == 1 && !optimize_timings) {   // (the constant CTAs live in RomNodeOut's grid)
    auto constant = [&](int i) {
      if (elems[i].list < 0) return false;
      const int kind_rows = elems[i].list < n_dyn_ctas ? pl.dyn_rows : elems[i].list < n_dyn_ctas + n_rom_ctas * n_ee ? pl.rom_rows : pl.node_rows;
      return elems[i].d % kind_rows == 0;   // row 0 of a warp's state block
    };
    int i = 0;
    while (i + 3 < nnz) {
      if (i % 4 != 0 || !(constant(i) && constant(i + 1) && constant(i + 2) && constant(i + 3))) { i += (i % 4) ? (4 - i % 4) : 4; continue; }
      int j = i;
      while (j + 3 < nnz && constant(j) && constant(j + 1) && constant(j + 2) && constant(j + 3)) j += 4;
      if (j - i >= kConstRunMin) {
        for (int a = i; a < j; a += kConstRunMax) {
          const int len = std::min(kConstRunMax, j - a);
          if (len < 4) break;
          tb.const_runs.push_back(ConstRun{a, len, (int32_t)tb.const_vals.size(), 0});
          for (int k = a; k < a + len; ++k) { tb.const_vals.push_back(elems[k].c); is_const_run[k] = 1; elems[k].list = -2; }
        }
      }
      i = j;
    }
  }
  pl.n_const_runs = (int)tb.const_runs.size();
  for (int q = 0; q < NC; ++q) {
    const int L = nnz, c = (int)(((long long)q * L) % 4);   // position of the row's first element inside its sector
    std::vector<int> hits(L, 0);
    for (int S = 0; 4 * S < c + L; ++S) {
      const int first = std::max(0, 4 * S - c), last = std::min(L - 1, 4 * S + 3 - c);
      const int writer = elems[last].list;
      bool full = (4 * S - c >= 0) && (4 * S + 3 - c <= L - 1) && writer >= 0;
      for (int i = first; i <= last && full; ++i) if (elems[i].list != writer) full = false;
      if (!full) {
        for (int i = first; i <= last; ++i) if (elems[i].list >= 0) { lists[elems[i].list][q][1].push_back({OutPair{i, elems[i].d, 0}, OutCoef{elems[i].c, 0.0}, PhaseExt{elems[i].ext, 0}}); hits[i]++; }
        continue;
      }
      const int cat = ((elems[first].ext | elems[first + 1].ext | elems[first + 2].ext | elems[first + 3].ext) & 3u) ? 2 : 0;
      lists[writer][q][cat].push_back({OutPair{first, elems[first].d, elems[first + 1].d}, OutCoef{elems[first].c, elems[first + 1].c}, PhaseExt{elems[first].ext, elems[first + 1].ext}});
      lists[writer][q][cat].push_back({OutPair{first + 2, elems[first + 2].d, elems[first + 3].d}, OutCoef{elems[first + 2].c, elems[first + 3].c}, PhaseExt{elems[first + 2].ext, elems[first + 3].ext}});
      for (int i = first; i <= last; ++i) hits[i]++;
    }
    // self-check: every element of an output-kernel row is written exactly once
    for (int i = 0; i < L; ++i) if (hits[i] != (elems[i].list >= 0 ? 1 : 0)) return fail(TWB_ERR_UNSUPPORTED, "output lists do not cover every element exactly once");
    for (int i = 0; i < L; ++i) if (is_const_run[i] && hits[i] != 0) return fail(TWB_ERR_UNSUPPORTED, "constant run also written by a list");
  }
  auto flush_list = [&](int list) {
    OutList out{};
    for (int q = 0; q < NC; ++q) {
      OutRange* dst[3] = {&out.pairs[q], &out.singles[q], &out.phase[q]};
      for (int w = 0; w < 3; ++w) {
        const auto& v = lists[list][q][w];
        dst[w]->first = (int32_t)tb.pairs.size(); dst[w]->count = (int32_t)v.size();
        for (const Entry& en : v) { tb.pairs.push_back(en.p); tb.coefs.push_back(en.c); if (optimize_timings) tb.exts.push_back(en.x); }
      }
    }
    return out;
  };
  for (int i = 0; i < n_lists; ++i) tb.cta_lists.push_back(flush_list(i));
  for (size_t gi = 0; gi < groups.size(); ++gi) {
    NodeGroup ng{}; ng.kind = groups[gi].kind; ng.first = groups[gi].first; ng.count = groups[gi].count;
    const auto& vals = values[gi];
    bool consecutive = !vals.empty();
    for (size_t i = 1; i < vals.size() && consecutive; ++i)
      consecutive = vals[i].p.off == vals[0].p.off + (int)i && vals[i].p.d0 == vals[0].p.d0 + (int)i;
    ng.g_row0 = consecutive ? vals[0].p.off : -1; ng.g_d0 = consecutive ? vals[0].p.d0 : 0; ng.g_n = consecutive ? (int32_t)vals.size() : 0;
    ng.values = OutRange{(int32_t)tb.pairs.size(), (int32_t)vals.size()};
    for (const Entry& en : vals) { tb.pairs.push_back(en.p); tb.coefs.push_back(en.c); if (optimize_timings) tb.exts.push_back(en.x); }
    tb.groups.push_back(ng);
  }
  pl.dyn_list0 = 0; pl.rom_list0 = n_dyn_ctas; pl.node_list0 = n_dyn_ctas + n_rom_ctas * n_ee;

  // ---- costs (nlp_formulation.cc:333-376, node_cost.cc:53-76)
  has_cost = false;
  for (int i = 0; i < sp.n_costs; ++i) {
    auto add_term = [&](const NodeSet& ns, int deriv, int dim, double w) {
      bool first = true;
      for (int nd = 0; nd < ns.n_nodes; ++nd) {
        int v = ns.Var(nd, deriv, dim);
        CostEntry c{}; c.xi = (int16_t)(v < 0 ? zero_slot : ns.offset + v); c.grad_col = (int16_t)(v < 0 ? -1 : ns.offset + v);
        c.pad = first ? 1 : 0; c.weight = w; first = false;
        tb.cost.push_back(c);
      }
    };
    if (sp.cost_ids[i] == TWB_COST_FORCES) for (int e = 0; e < n_ee; ++e) add_term(force(e), kPos, Z, sp.cost_weights[i]);
    else if (sp.cost_ids[i] == TWB_COST_EE_MOTION) for (int e = 0; e < n_ee; ++e) { add_term(motion(e), kVel, X, sp.cost_weights[i]); add_term(motion(e), kVel, Y, sp.cost_weights[i]); }
    else return fail(TWB_ERR_INVALID, "cost not defined!");
    has_cost = true;
  }

  pl.n_phase_units = (int)tb.phase_units.size(); pl.n_phase_defs = (int)tb.phase_defs.size();
  // ---- plan scalars
  pl.n = n; pl.m = m; pl.nnz = nnz; pl.n_ee = n_ee;
  pl.n_groups = (int)tb.groups.size(); pl.n_cost = (int)tb.cost.size();
  pl.n_base_z_rows = (int)tb.base_z_rows.size();
  pl.mass = rb.mass; pl.gravity = 9.80665;  // dynamic_model.cc:37
  const double* I = rb.inertia;             // single_rigid_body_dynamics.cc:36-44
  double Ib[9] = {I[0], -I[3], -I[4], -I[3], I[1], -I[5], -I[4], -I[5], I[2]};
  for (int i = 0; i < 9; ++i) pl.I_b[i] = Ib[i];
  pl.mu = 0.5;  // height_map.h:136
  return TWB_OK;
}

}  // namespace twb
