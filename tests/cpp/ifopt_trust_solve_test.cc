// BatchedProblem::Solve (include/towr_b200_ifopt.hpp) with the trust-region step rule: the options go through as given.
// The instances are those of ifopt_solve_test.cc (the Python `anymal_trot_block_base_rom` recipe, per-instance start states).
//   ./ifopt_trust_solve_test    checks the two option errors of the rule (TWB_ERR_INVALID, X untouched), then prints, in C99
//                               hex floats, the state records and per instance the solved x, status, iterations, violation
//                               and mu; tests/test_lm_trust_region.py repeats the solve through the C call
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "../../include/towr_b200_ifopt.hpp"

#define REQUIRE(cond) do { if (!(cond)) { std::printf("FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); return 1; } } while (0)

using namespace towr_b200;

static void PrintVec(const char* key, int b, const std::vector<double>& v) {
  std::printf("%s %d", key, b);
  for (double d : v) std::printf(" %a", d);
  std::printf("\n");
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
  twb_spec& s = f.params_;   // params_.constraints_.insert(2, BaseRom)
  for (int i = s.n_constraints; i > 2; --i) s.constraints[i] = s.constraints[i - 1];
  s.constraints[2] = TWB_C_BASE_ROM; s.n_constraints++;
  const twb_spec spec = f.ToSpec();

  const int B = 4;
  std::vector<double> states((size_t)B * TWB_STATE_DOUBLES, 0.0);
  for (int k = 0; k < B; ++k) {
    double* r = states.data() + (size_t)k * TWB_STATE_DOUBLES;
    for (int d = 0; d < 3; ++d) {
      r[0 + d] = spec.initial_base_lin_pos[d]; r[3 + d] = spec.initial_base_lin_vel[d];
      r[6 + d] = spec.initial_base_ang_pos[d]; r[9 + d] = spec.initial_base_ang_vel[d];
      r[12 + d] = spec.final_base_lin_pos[d]; r[15 + d] = spec.final_base_lin_vel[d];
      r[18 + d] = spec.final_base_ang_pos[d]; r[21 + d] = spec.final_base_ang_vel[d];
    }
    for (int e = 0; e < n_ee; ++e) for (int d = 0; d < 3; ++d) r[24 + 3 * e + d] = spec.initial_ee_W[e][d];
    r[0] += 0.1 * k; r[2] += 0.02 * (k - 1);              // initial base position
    r[12] += 0.25 * k; r[13] = 0.05 * (1 - k);           // goal position
    r[20] = 0.1 * k;                                     // goal yaw
  }
  twb_lm_solve_options opt;
  twb_lm_solve_options_default(&opt);
  opt.tol = 1e-2; opt.max_iters = 30;
  opt.step_rule = TWB_LM_STEP_TRUST; opt.radius_max = 50.0;

  for (int k = 0; k < B; ++k)
    PrintVec("state", k, std::vector<double>(states.begin() + (size_t)k * TWB_STATE_DOUBLES, states.begin() + (size_t)(k + 1) * TWB_STATE_DOUBLES));
  BatchedProblem nlp(spec, B, 0);
  nlp.SetStates(states.data(), B);
  const int n = nlp.GetNumberOfOptimizationVariables();
  const std::vector<double> x_before = nlp.X;
  twb_lm_solve_options bad = opt;
  bad.step_rule = 2;
  REQUIRE(nlp.Solve(bad) == TWB_ERR_INVALID);
  bad = opt;
  bad.radius_max = 0.5 * opt.cap;
  REQUIRE(nlp.Solve(bad) == TWB_ERR_INVALID);
  REQUIRE(nlp.X == x_before);
  const int rc = nlp.Solve(opt);
  if (rc != TWB_OK) { std::printf("FAILED Solve: %d %s\n", rc, twb_last_error()); return 1; }
  REQUIRE(nlp.X != x_before);
  for (int b = 0; b < B; ++b) {
    std::vector<double> x;
    for (double v : GpuProblem(nlp, b).GetVariableValues()) x.push_back(v);
    REQUIRE((int)x.size() == n);
    PrintVec("x", b, x);
    std::printf("result %d %d %d %a %a\n", b, nlp.solve_status(b), nlp.solve_iterations(b), nlp.solve_violation(b), nlp.SOLVE_MU[b]);
  }
  std::printf("ok\n");
  return 0;
}
