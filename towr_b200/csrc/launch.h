// launch.h — host entry point of kernels.cu
#ifndef TOWR_B200_LAUNCH_H_
#define TOWR_B200_LAUNCH_H_
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

#include "device_tables.h"

namespace twb {

// profiling hook: when set, called after every kernel launch (label "begin" starts a group) and all
// kernels are serialised on one stream
extern void (*g_after_launch)(const char* label, cudaStream_t stream);

// fpowr::GetTrajectory for `nb` instances: x -> XT, then out[b][step][19 + 13 n_ee]; `samples` / `contact` are the device
// copies of Formulation::TrajectoryTables (contact null when the durations are optimised)
int LaunchTrajectory(const Plan& P, const double* x, double* XT, const SplineSample* samples, const int* contact, int n_steps,
                     double* out, int nb, cudaStream_t s);
// fpowr::ExtractInitialGuess at `n_times` caller-given times: x -> XT, then out[b][time][49]; `samples` as for the trajectory
int LaunchInitialGuess(const Plan& P, const double* x, double* XT, const SplineSample* samples, const double* times, int n_times,
                       double* out, int nb, cudaStream_t s);
// fpowr::ExtractFootstepPlan without the nearest-plane lookup, fused (no sampled trajectory): x -> XT, then
// out[b][max_states][2 + 4 n_ee] (rows past n_states[b] written as 0) and n_states[b].  samples / times: the tables of
// Formulation::TrajectoryTables(0.01); fixed durations: codes[n_codes] = (step << 4) | contact mask of the first step and of
// every change of the contact set, contact unused; optimised durations: contact = in_contact_at_start per foot, codes unused
int LaunchFootstepPlan(const Plan& P, const double* x, double* XT, const SplineSample* samples, const double* times, const int* contact,
                       const int* codes, int n_codes, int n_steps, double time_horizon, int max_states, int* n_states, double* out, int nb,
                       cudaStream_t s);
// fpowr::NearestPlaneLookup for every (instance, footstep state, foot) of a footstep plan: out[b][state][foot] = index of
// the nearest polygon (polygon k = vertices poly_offset[k] .. poly_offset[k+1]-1 of verts[][2]) or -1 (foot in the air);
// ranges [nb][2] (first, count; may be null = all polygons): instance b's own polygons, index relative to the first of them
int LaunchNearestPlanes(const double* plan, const int* n_states, int max_states, int n_ee, const int* poly_offset, int n_polys,
                        const int* ranges, const double* verts, int* out, int nb, cudaStream_t s);
// towr::LinearEqualityConstraint values g[b][rows] = M x_set (x -> XT first); towr::SoftConstraint cost / gradient of one
// constraint set from device-resident g / jac
int LaunchLinearEquality(const Plan& P, const double* x, double* XT, int col0, int n_cols, const double* M, int rows, double* g, int nb, cudaStream_t s);
int LaunchSoftConstraint(const Plan& P, const double* g, const double* jac, const int* row_ptr, const int* col_idx, int row0, int n_rows,
                         const double* b_avg, const double* w, double* cost, double* grad, int nb, cudaStream_t s);
// x0 / variable bounds of `nb` goal-randomised instances (goals[b][6] = final base position, final base Euler angles)
int LaunchGoalInstances(const Plan& P, const GoalSetup& S, const double* goals, const int* terrain_ids, int default_terrain, double* x0, double* lo,
                        double* up, int nb, cudaStream_t s);
// x0 / variable bounds [nb][n] and constraint bounds [nb][m] of `nb` instances with their own start / goal states
// (states[b][kStateDoubles]); any output may be null
int LaunchStateInstances(const Plan& P, const GoalSetup& S, const double* states, const int* terrain_ids, int default_terrain, double* x0, double* lo,
                         double* up, double* gl, double* gu, int nb, cudaStream_t s);
// ---- device-resident solver step (lm_kernel.cu): the shared sparsity pattern and its transpose, constraint bounds (device pointers)
struct LmPattern {
  const int* row_ptr;   // [m + 1]
  const int* col_idx;   // [nnz]
  const int* col_ptr;   // [n + 1]  transpose: entries of column j, ascending row
  const int* slot_t;    // [nnz]    CSR slot of the transposed entry
  const int* row_t;     // [nnz]    its row
  const double* g_lower;
  const double* g_upper;   // [m] the problem's constraint bounds (what twb_batch_lm_step_device steps against)
  const int* row_order;    // [m] rows in descending length (balanced warps in the row pass)
  const int* col_order;    // [n] columns in descending length
  const uint16_t *col_idx16, *slot_t16, *row_t16;   // the same index arrays in 16 bits when n, m, nnz < 65 536 (else null)
};
size_t LmSharedBytes(int n, int m);
// solve status of an instance (include/towr_b200.h: TWB_LM_*)
enum LmStatus : int { kLmRunning = 0, kLmConverged = 1, kLmStalled = 2, kLmNonFinite = 3 };
// the trial variant of the step (twb_batch_lm_trial_device): damping mu[b] per instance, x left unchanged and the step
// written to x_trial; only instances whose status is kLmRunning are stepped
struct LmTrialArgs {
  const double* mu;     // [nb]
  double tol;           // status kLmConverged when max |s r| <= tol
  int* status;          // [nb] in / out
  double* x_trial;      // [nb][n]
  double* row_scale;    // [nb][m] s at x
  double* merit;        // [nb] 1/2 ||s r(g)||^2
  double* predicted;    // [nb] merit - 1/2 ||s r(g + J d)||^2, d = x_trial - x
  double* radius;       // [nb] trust-region rule: max |dx| <= radius[b] instead of cap, CG on the free set; null: the cap rule
  double* step_norm;    // [nb] max |d| (trust-region rule only)
};
// one Levenberg-Marquardt feasibility step for nb instances (CTA = instance): x[b][n] in / out, g[b][m], jac[b][nnz] in,
// variable bounds x_lower / x_upper at b * bound_stride and constraint bounds g_lower / g_upper at b * g_bound_stride (0: the
// same bounds for every instance), violation[b] out (may be null).  trial non-null: the trial variant (x is only read, mu unused)
int LaunchLmStep(const LmPattern& pat, int n, int m, int nnz, double* x, const double* g, const double* jac, const double* x_lower,
                 const double* x_upper, size_t bound_stride, const double* g_lower, const double* g_upper, size_t g_bound_stride, double mu,
                 double cap, int cg_iters, double* violation, const LmTrialArgs* trial, int nb, cudaStream_t s);
// the gain-ratio decision after a trial step for nb instances (CTA = instance, kLmRunning ones only): accept x <- x_trial and
// lower mu, or keep x and raise mu (kLmStalled past mu_max); g_trial[b][m] is g at x_trial.  radius non-null: the
// trust-region update of radius[b] from rho and step_norm[b] (clamped to radius_max; kLmStalled once it collapses)
int LaunchLmAccept(int n, int m, double* x, const double* x_trial, const double* g_trial, const double* g_lower, const double* g_upper,
                   size_t g_bound_stride, const double* row_scale, const double* merit, const double* predicted, double* mu, double* nu,
                   int* status, int* iterations, double eta, double mu_min, double mu_max, double* radius, const double* step_norm,
                   double radius_max, int nb, cudaStream_t s);
// the device-side solve loop (twb_batch_lm_solve_device).  loop: kLoopInts device ints of loop state (iterations run, the
// counts being added up); cond: the WHILE node's handle in the graph these kernels are captured into.
constexpr int kLoopInts = 6;
// per instance mu = mu0, nu = 2, status RUNNING, iterations 0 (and radius = radius0, step_norm = 0 when radius is non-null);
// the loop state cleared; the condition = max_iters > 0
int LaunchLmSolveInit(int nb, double mu0, double* mu, double* nu, int* status, int* iterations, double radius0, double* radius,
                      double* step_norm, int* loop, int max_iters, cudaGraphConditionalHandle cond, cudaStream_t s);
// instances per status.  loop_step: iterations run += 1, condition = (RUNNING > 0 && iterations run < max_iters); else
// status_counts[4] / loop_count[1] (each may be null) receive the counts and the iterations run, the condition is not touched
int LaunchLmCount(int nb, const int* status, int* loop, int max_iters, cudaGraphConditionalHandle cond, bool loop_step, int* status_counts,
                  int* loop_count, cudaStream_t s);
// number of output kernels one evaluation launches for this plan
int OutKernelsPerEval(const Plan& P, unsigned flags);
// One batched evaluation of `nb` instances.  XT is [tiles][n+1][32] (zero-initialised once; row n stays 0; tile = 32
// instances).  x, g, jac, cost, grad, status and terrain_ids point at the first instance.  `flags` are the TWB_EVAL_* bits.
// Work is enqueued on `s` and on two auxiliary streams that are forked from / joined back into `s` with ev[0..2].
// FS: scratch of the feet's positions / forces per dynamic sample, [tiles][n_dyn][6 n_ee][32] (optimised durations only, else null)
int LaunchEval(const Plan& P, const double* x, double* XT, double* FS, double* g, double* jac, double* cost, double* grad,
               int* status, const int* terrain_ids, int default_terrain, int nb, unsigned flags, cudaStream_t s,
               cudaStream_t aux0, cudaStream_t aux1, cudaEvent_t* ev, int* launches);

}  // namespace twb
#endif
