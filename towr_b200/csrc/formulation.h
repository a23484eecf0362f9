// formulation.h — host-side structure builder.  Turns a twb_spec (the public
// fields of towr::NlpFormulation + towr::Parameters) into everything that does
// not depend on the iterate: dimensions, the CSR pattern of the constraint
// Jacobian, bounds, the initial guess, the component layout, and the tables
// the CUDA kernels consume (device_tables.h).
#ifndef TOWR_B200_FORMULATION_H_
#define TOWR_B200_FORMULATION_H_

#include <array>
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "../../include/towr_b200.h"
#include "device_tables.h"

namespace twb {

struct RobotConst {
  int n_ee;
  double mass;
  double inertia[6];  // Ixx, Iyy, Izz, Ixy, Ixz, Iyz
  double nominal[kMaxEE][3];
  double max_dev[3];
};
bool GetRobot(int id, RobotConst* r);
double TerrainHeight(int id, double x, double y);
bool GaitPhases(int n_ee, int combo, double t_total, std::vector<std::vector<double>>* durations,
                std::vector<bool>* contact_at_start);

struct Component { std::string name; int start; int count; };
struct SetsHolder;   // variable maps of the node sets (formulation.cc)

// Everything the kernels need, still on the host (capi.cc uploads it).
struct HostTables {
  Plan plan{};  // pointer members are filled in after upload
  std::vector<SplineSample> samples;
  std::vector<DynUnit> dyn;
  std::vector<RomUnit> rom;
  std::vector<NodeGroup> groups;
  std::vector<TerrainUnit> terr;
  std::vector<ForceUnit> force;
  std::vector<SwingUnit> swing;
  std::vector<AccUnit> acc;
  std::vector<BaseMotionUnit> base_motion;
  std::vector<CostEntry> cost;
  std::vector<OutPair> pairs;
  std::vector<OutCoef> coefs;
  std::vector<OutList> cta_lists;
  std::vector<double> dyn_ang_basis;
  std::vector<PhaseSplineDef> phase_defs;
  std::vector<PhasePoly> phase_polys;
  std::vector<PhaseUnit> phase_units;
  std::vector<PhaseExt> exts;
  std::vector<GoalVar> goal_vars;
  std::vector<GoalVar> state_vars;    // goal_vars with the bounds of the start / goal state read from a state record
  std::vector<int32_t> base_z_rows;   // BaseMotionConstraint LZ rows (their bounds follow the instance's initial base z)
  std::vector<ConstRun> const_runs;
  std::vector<double> const_vals;
  GoalSetup goal_setup{};
};

class Formulation {
 public:
  // returns TWB_OK / TWB_ERR_*; `err` gets a one-line reason on failure
  int Build(const twb_spec& spec, std::string* err);
  // NlpFormulation::GetVariableSets with another final_base_: x0 / bounds of a goal-randomised instance (n values each)
  // time grid and spline samples of fpowr::GetTrajectory(dt): per time step 2 + 2 n_ee samples (base-lin, base-ang,
  // ee-motion.., ee-force..); contact[step][foot] (fixed durations) or empty (durations optimised: per instance on the device)
  int TrajectoryTables(double dt, std::vector<double>* times, std::vector<SplineSample>* samples, std::vector<int>* contact) const;
  // the same tables at caller-given times (fpowr::ExtractInitialGuess)
  int SampleTables(const std::vector<double>& times, std::vector<SplineSample>* samples, std::vector<int>* contact) const;
  int GoalInstance(const double final_lin_pos[3], const double final_ang_pos[3], double* x0, double* x_lower, double* x_upper) const;
  // the same with the whole state record (TWB_STATE_DOUBLES: initial_base_, final_base_, initial_ee_W_), plus the m
  // constraint bounds of that instance; any output may be null
  int StateInstance(const double* state, double* x0, double* x_lower, double* x_upper, double* g_lower, double* g_upper) const;

  int n = 0, m = 0, nnz = 0;
  std::vector<int> row_ptr, col_idx;
  std::vector<double> x_lower, x_upper, g_lower, g_upper, x0;
  std::vector<Component> var_sets, con_sets;
  bool has_cost = false;
  bool optimize_timings = false;
  twb_spec spec{};
  HostTables tables;
  std::shared_ptr<SetsHolder> holder;
};

}  // namespace twb
#endif
