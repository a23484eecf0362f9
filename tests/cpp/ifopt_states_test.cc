// Per-instance start states in include/towr_b200_ifopt.hpp: BatchedProblem::SetStates, then the ifopt::Problem view of each
// instance (GpuProblem) serves that instance's initial guess, variable bounds and constraint bounds.  Structure-only
// (no device batch): SetStates runs on the host.  The recipe is the Python `anymal_trot_block_base_rom`
// (towr_b200/configs.py): Anymal trot on the block terrain with BaseMotionConstraint, whose LZ rows follow each instance's
// initial base height.  Prints, in C99 hex floats, the state records and per instance the values and bounds the views
// serve; tests/test_ifopt_states.py checks them against twb_problem_state_instances through the Python binding.
//   ./ifopt_states_test
#include <cmath>
#include <cstdio>
#include <vector>

#include "../../include/towr_b200_ifopt.hpp"

#define REQUIRE(cond) do { if (!(cond)) { std::printf("FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); return 1; } } while (0)

using namespace towr_b200;

static void PrintVec(const char* key, int b, const std::vector<double>& v) {
  std::printf("%s %d", key, b);
  for (double d : v) std::printf(" %a", d);
  std::printf("\n");
}

// x0, variable bounds and constraint bounds of GpuProblem(p, b), as IpoptAdapter reads them
static void PrintInstance(const char* tag, BatchedProblem& p, int b) {
  GpuProblem ip(p, b);
  std::vector<double> x0, xl, xu, gl, gu;
  for (double v : ip.GetVariableValues()) x0.push_back(v);
  for (auto& bd : ip.GetBoundsOnOptimizationVariables()) { xl.push_back(bd.lower_); xu.push_back(bd.upper_); }
  for (auto& bd : ip.GetBoundsOnConstraints()) { gl.push_back(bd.lower_); gu.push_back(bd.upper_); }
  char key[64];
  const char* names[5] = {"x0", "xl", "xu", "gl", "gu"};
  const std::vector<double>* vals[5] = {&x0, &xl, &xu, &gl, &gu};
  for (int k = 0; k < 5; ++k) { std::snprintf(key, sizeof key, "%s_%s", tag, names[k]); PrintVec(key, b, *vals[k]); }
}

int main() {
  NlpFormulation f(TWB_ANYMAL, TWB_BLOCK);
  int n_ee = 0; double mass = 0, inertia[6], nominal[TWB_MAX_EE][3], max_dev[3];
  Check(twb_robot_info(TWB_ANYMAL, &n_ee, &mass, inertia, nominal, max_dev), "twb_robot_info");
  const double z0 = -nominal[0][2];
  f.initial_base_.lin.p[2] = z0;
  for (int e = 0; e < n_ee; ++e) f.initial_ee_W_.push_back({nominal[e][0], nominal[e][1], 0.0});
  f.final_base_.lin.p[0] = 1.5; f.final_base_.lin.p[2] = z0;
  f.SetGait(n_ee, 1, 2.0);
  // params_.constraints_.insert(2, BaseRom)
  twb_spec& s = f.params_;
  for (int i = s.n_constraints; i > 2; --i) s.constraints[i] = s.constraints[i - 1];
  s.constraints[2] = TWB_C_BASE_ROM; s.n_constraints++;
  const twb_spec spec = f.ToSpec();

  const int B = 4, S = 3;                       // instance 3 gets no state record
  std::vector<double> states((size_t)S * TWB_STATE_DOUBLES, 0.0);
  for (int k = 0; k < S; ++k) {
    double* r = states.data() + (size_t)k * TWB_STATE_DOUBLES;
    for (int d = 0; d < 3; ++d) {
      r[0 + d] = spec.initial_base_lin_pos[d]; r[3 + d] = spec.initial_base_lin_vel[d];
      r[6 + d] = spec.initial_base_ang_pos[d]; r[9 + d] = spec.initial_base_ang_vel[d];
      r[12 + d] = spec.final_base_lin_pos[d]; r[15 + d] = spec.final_base_lin_vel[d];
      r[18 + d] = spec.final_base_ang_pos[d]; r[21 + d] = spec.final_base_ang_vel[d];
    }
    for (int e = 0; e < n_ee; ++e) for (int d = 0; d < 3; ++d) r[24 + 3 * e + d] = spec.initial_ee_W[e][d];
    const double z_off[S] = {-0.04, 0.0, 0.035};
    r[0] += 0.1 * k; r[1] -= 0.05 * k; r[2] += z_off[k];                // initial base position
    r[3] = 0.2 * k; r[8] = 0.1 * (k - 1); r[11] = -0.1 * k;              // initial velocity, yaw, yaw rate
    r[12] += 0.3 * k; r[13] = 0.1 * (1 - k); r[14] += 0.02 * k;         // goal position
    r[20] = 0.15 * k;                                                    // goal yaw
    for (int e = 0; e < n_ee; ++e) { r[24 + 3 * e] += 0.1 * k; r[24 + 3 * e + 1] += 0.01 * (e - k); }
  }
  for (int k = 0; k < S; ++k)
    PrintVec("state", k, std::vector<double>(states.begin() + (size_t)k * TWB_STATE_DOUBLES, states.begin() + (size_t)(k + 1) * TWB_STATE_DOUBLES));

  BatchedProblem plain(spec, B, 0, false);          // no SetStates: every instance is the problem
  PrintInstance("spec", plain, 1);
  std::vector<double> px0(plain.X.begin(), plain.X.begin() + plain.GetNumberOfOptimizationVariables());
  PrintVec("problem_x0", 0, px0);
  PrintVec("problem_gl", 0, plain.g_lower());

  BatchedProblem nlp(spec, B, 0, false);
  bool threw = false;
  try { nlp.SetStates(states.data(), B + 1); } catch (const std::runtime_error&) { threw = true; }
  REQUIRE(threw);
  nlp.SetStates(states.data(), S);
  for (int b = 0; b < B; ++b) PrintInstance("inst", nlp, b);
  // the no-argument accessors keep serving the problem's bounds; instances differ from each other and from the problem
  REQUIRE(nlp.g_lower() == plain.g_lower() && nlp.x_lower() == plain.x_lower());
  const int m = nlp.GetNumberOfConstraints();
  int differ = 0;
  for (int i = 0; i < m; ++i) differ += nlp.g_lower(0)[i] != nlp.g_lower(2)[i];
  REQUIRE(differ > 0);
  for (int i = 0; i < m; ++i) REQUIRE(nlp.g_lower(3)[i] == plain.g_lower()[i] && nlp.g_upper(3)[i] == plain.g_upper()[i]);
  std::printf("dims %d %d\n", nlp.GetNumberOfOptimizationVariables(), m);
  std::printf("ok\n");
  return 0;
}
