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

// One batched evaluation of `nb` instances.  XT is [tiles][n+1][32] (zero-initialised once; row n stays 0;
// tile = 32 consecutive instances), GT is [tiles][m][32] (staging of the constraint values).  x, g, jac, cost, grad, status and terrain_ids point at the first
// instance.  `flags` are the TWB_EVAL_* bits.  Work is enqueued on `s` and on two auxiliary streams that
// are forked from / joined back into `s` with ev[0..2].
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
// the nearest polygon (polygon k = vertices poly_offset[k] .. poly_offset[k+1]-1 of verts[][2]) or -1 (foot in the air)
int LaunchNearestPlanes(const double* plan, const int* n_states, int max_states, int n_ee, const int* poly_offset, int n_polys,
                        const double* verts, int* out, int nb, cudaStream_t s);
// towr::LinearEqualityConstraint values g[b][rows] = M x_set (x -> XT first); towr::SoftConstraint cost / gradient of one
// constraint set from device-resident g / jac
int LaunchLinearEquality(const Plan& P, const double* x, double* XT, int col0, int n_cols, const double* M, int rows, double* g, int nb, cudaStream_t s);
int LaunchSoftConstraint(const Plan& P, const double* g, const double* jac, const int* row_ptr, const int* col_idx, int row0, int n_rows,
                         const double* b_avg, const double* w, double* cost, double* grad, int nb, cudaStream_t s);
// x0 / variable bounds of `nb` goal-randomised instances (goals[b][6] = final base position, final base Euler angles)
int LaunchGoalInstances(const Plan& P, const GoalSetup& S, const double* goals, const int* terrain_ids, int default_terrain, double* x0, double* lo,
                        double* up, int nb, cudaStream_t s);
// ---- device-resident solver step (lm_kernel.cu): the shared sparsity pattern and its transpose, constraint bounds (device pointers)
struct LmPattern {
  const int* row_ptr;   // [m + 1]
  const int* col_idx;   // [nnz]
  const int* col_ptr;   // [n + 1]  transpose: entries of column j, ascending row
  const int* slot_t;    // [nnz]    CSR slot of the transposed entry
  const int* row_t;     // [nnz]    its row
  const double* g_lower;
  const double* g_upper;   // [m]
  const int* row_order;    // [m] rows in descending length (balanced warps in the row pass)
  const int* col_order;    // [n] columns in descending length
  const uint16_t *col_idx16, *slot_t16, *row_t16;   // the same index arrays in 16 bits when n, m, nnz < 65 536 (else null)
};
size_t LmSharedBytes(int n, int m);
// one Levenberg-Marquardt feasibility step for nb instances (CTA = instance): x[b][n] in / out, g[b][m], jac[b][nnz] in,
// bounds x_lower / x_upper at b * bound_stride (0: the same bounds for every instance), violation[b] out (may be null)
int LaunchLmStep(const LmPattern& pat, int n, int m, int nnz, double* x, const double* g, const double* jac, const double* x_lower,
                 const double* x_upper, size_t bound_stride, double mu, double cap, int cg_iters, double* violation, int nb, cudaStream_t s);
// L2 access-policy window applied to the evaluation kernels launched by this thread (null: none)
void SetL2Window(const cudaAccessPolicyWindow* w);
// number of output kernels one evaluation launches for this plan
int OutKernelsPerEval(const Plan& P, unsigned flags);
int TransposeOutPerEval(const Plan& P);
// FS: scratch of the feet's positions / forces per dynamic sample, [tiles][n_dyn][6 n_ee][32] (optimised durations only, else null)
// TD: one zero-initialised counter per tile (the output CTAs count themselves; the last one of a tile drops the tile's XT lines)
int LaunchEval(const Plan& P, const double* x, double* XT, double* GT, double* FS, int* TD, double* g, double* jac, double* cost, double* grad,
               int* status, const int* terrain_ids, int default_terrain, int nb, unsigned flags, cudaStream_t s,
               cudaStream_t aux0, cudaStream_t aux1, cudaEvent_t* ev, int* launches);

}  // namespace twb
#endif
