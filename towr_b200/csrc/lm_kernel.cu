// lm_kernel.cu — one Levenberg-Marquardt feasibility step for every instance of a batch, entirely on the device.
//
// The stand-in for the IPOPT solves BASELINE configs[0] / [4] name (hopper_example.cc:77-93, footstep_plan_server.cc:222-236;
// neither IPOPT nor ifopt exists in this image): what towr_b200/solver.py documents and tests/test_solver_loop.py walks a
// second time on the CPU —
//     r  = violation of g(x) against [g_lower, g_upper]    (the problem's bounds, or one row of bounds per instance)
//     Js = diag(s) J,  rs = s r,   s_i = 1 / max(1, max_k |J_ik|)
//     (Js^T Js + mu I) dx = -Js^T rs          cg_iters conjugate-gradient iterations, matrix-free
//     x <- clip(x + dx min(1, cap / max|dx|), x_lower, x_upper)
// CTA = instance.  When they fit (config 2: 120 KB of 227 KB), the instance's row-scaled CSR values Js are kept in shared
// memory for the whole step — one pass over global memory, then 2 x cg_iters sparse products on chip (512 threads, one CTA
// per SM); larger patterns (config 4: 436 KB) are re-read from global memory / the L2 in every product (256 threads, several
// CTAs per SM).  All solver vectors live in shared memory.  Both products walk the ONE sparsity pattern of the structure class:
// Js p row by row (thread = row), Js^T u column by column through the pattern's transpose (thread = column) — fixed
// summation orders, no atomics, bit-reproducible.
// The trial variant (kTrial, twb_batch_lm_trial_device) is the same step with mu[b] per instance; it writes the step to x_trial
// and leaves x alone, sets the instance's solve status (converged: max |s r| <= tol, non-finite), and writes the row scales s,
// the merit phi0 = 1/2 ||s r(g)||^2 and the decrease of the linear model, phi0 - 1/2 ||s r(g + J d)||^2 with d = x_trial - x
// (one more row pass over Js, with d in pd and Js d in u).  LmAcceptKernel then decides on g at x_trial with the same row
// scales: accept when rho = (phi0 - phi_t) / predicted > eta, else keep x and raise mu.
// An instance with a non-finite x, g or J entry, or a NaN constraint bound, keeps its x and reports violation NaN.  Left to the
// step, such an entry would be dropped by fmax (row scale, violation) and a NaN step turned into a bound by the projection:
// the instance would jump to its bounds and report a finite violation (a NaN bound would silently mean "unbounded").
// +-Inf constraint bounds mean unbounded, like the 1e20 convention.  With lower > upper the lower bound wins (g < lo is
// tested first).
// The trust-region rule (LmTrialArgs::radius non-null; the one-call solve with TWB_LM_STEP_TRUST) changes the trial step in
// two places.  Free set: gamma = Js^T rs (the column pass that forms -b); variable j is frozen when x_lower[j] == x_upper[j],
// or x_j <= x_lower[j] with gamma_j > 0, or x_j >= x_upper[j] with gamma_j < 0 — a frozen j starts CG with res_j = pd_j = 0
// and its column product is skipped (ap_j = 0), so dx_j stays 0 and CG runs on the free variables only.  The frozen flags of
// a thread's columns sit in one 32-bit register (bit k: its k-th column in col_order; n <= 32 x threads, which the 200 KiB
// vector limit implies).  Radius: the cap becomes radius[b]; the trial also writes step_norm[b] = max |x_trial - x|.
// LmAcceptKernel then updates the radius from the gain ratio (kTr* below) and stalls an instance whose radius collapsed.
// The solve loop on the device (twb_batch_lm_solve_device) adds two small kernels: LmSolveInitKernel starts a solve (mu, nu,
// status, iterations per instance; the loop counter; the WHILE condition of the solve graph) and LmCountKernel counts the
// instances per status — at the end of every loop iteration it sets the condition, after the loop it reports the counts.
#include <cuda_runtime.h>
#include <math_constants.h>

#include <algorithm>
#include <cstdint>

#include "launch.h"

namespace twb {
namespace {

// the trust-region update (textbook constants): shrink to kTrShrink x step_norm when rho < kTrLow or the trial is rejected;
// grow to min(kTrGrow x radius, radius_max) when rho > kTrHigh and step_norm >= kTrEdge x radius; stalled once
// radius < kTrCollapse x max(1, max |x|)
constexpr double kTrShrink = 0.25, kTrLow = 0.25, kTrHigh = 0.75, kTrGrow = 2.0, kTrEdge = 0.99, kTrCollapse = 1e-12;

// sum / max over the CTA, result broadcast to every thread (fixed tree: deterministic)
__device__ __forceinline__ double BlockSum(double v, double* scratch) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += scratch[w];
  return t;
}
__device__ __forceinline__ double BlockMax(double v, double* scratch) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = scratch[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) t = fmax(t, scratch[w]);
  return t;
}

// kTrust (with kTrial; LmTrialArgs::radius non-null): the trust-region rule, a separate instantiation so that the cap
// rule's kernels stay as they were.  Its minimum of one CTA per SM lets ptxas use 95-115 registers: without it ptxas held
// these kernels to 40-64 registers and spilled (the cap rule's kernels keep their unchanged launch bound).
// kSmemJ: the scaled values Js live in shared memory (after the vectors); else they are formed on the fly from global memory.
// Idx: the pattern's index arrays as 16-bit (n, m, nnz < 65 536: 90 KB instead of 180 KB, so that they stay in the L1 beside
// one CTA's shared memory — with 32-bit indices every index load was an L2 round trip: 14.6 instead of 10.5 ms per step) or 32-bit.
// thread = row (Js p) / thread = column (Js^T u): measured faster than 16 lanes per row with shuffle trees (25.4 vs 14.6 ms).
template <bool kSmemJ, class Idx, bool kTrial, bool kTrust>
__global__ void __launch_bounds__(512, kTrust ? 1 : 0) LmStepKernel(LmPattern pat, const Idx* __restrict__ col_idx, const Idx* __restrict__ slot_t,
                                                    const Idx* __restrict__ row_t, int n, int m, int nnz, double* __restrict__ X,
                                                    const double* __restrict__ G, const double* __restrict__ JAC, const double* __restrict__ x_lower,
                                                    const double* __restrict__ x_upper, size_t bound_stride,
                                                    const double* __restrict__ g_lower, const double* __restrict__ g_upper, size_t g_bound_stride,
                                                    double mu, double cap, int cg_iters, double* __restrict__ violation, LmTrialArgs tr) {
  extern __shared__ __align__(16) double sm[];
  double* s = sm;             // [m] row scales
  double* u = s + m;          // [m] row vector (rs, then Js p)
  double* dx = u + m;         // [n]
  double* res = dx + n;       // [n]
  double* pd = res + n;       // [n]
  double* ap = pd + n;        // [n]
  double* scratch = ap + n;   // [32]
  double* Js = scratch + 32;  // [nnz] (kSmemJ)
  const int b = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
  const double* __restrict__ J = JAC + (size_t)b * nnz;
  const double* __restrict__ g = G + (size_t)b * m;
  const double* __restrict__ gl = g_lower + (size_t)b * g_bound_stride;
  const double* __restrict__ gu = g_upper + (size_t)b * g_bound_stride;
  if constexpr (kTrial) {
    if (tr.status[b] != kLmRunning) {    // finished before this call: x_trial = x and nothing else (uniform over the CTA)
      for (int j = tid; j < n; j += nt) tr.x_trial[(size_t)b * n + j] = X[(size_t)b * n + j];
      return;
    }
    mu = tr.mu[b];
    if constexpr (kTrust) cap = tr.radius[b];
  }
  // row scales, the scaled values and the scaled violation
  double vmax = 0.0, phi = 0.0;               // phi: sum of (s r)^2 (kTrial)
  double chk = 0.0;                           // fma(v, 0, chk): NaN once a v that is not finite has been seen
  for (int q = tid; q < m; q += nt) {
    const int i = __ldg(pat.row_order + q);   // rows in descending length: the lanes of a warp walk rows of similar length
    const int k0 = __ldg(pat.row_ptr + i), k1 = __ldg(pat.row_ptr + i + 1);
    double big = 0.0;
    for (int k = k0; k < k1; ++k) { const double v = J[k]; big = fmax(big, fabs(v)); chk = fma(v, 0.0, chk); }
    const double si = 1.0 / fmax(big, 1.0);
    if (kSmemJ) for (int k = k0; k < k1; ++k) Js[k] = J[k] * si;
    const double gi = g[i], lo = __ldg(gl + i), up = __ldg(gu + i);
    const double r = gi < lo ? gi - lo : gi > up ? gi - up : 0.0;
    chk = fma(gi, 0.0, chk);
    if (lo != lo || up != up) chk = CUDART_NAN;   // a NaN bound (an infinite one is a valid "unbounded")
    s[i] = si;
    if constexpr (kTrial) tr.row_scale[(size_t)b * m + i] = si;
    const double rs = si * r;
    u[i] = rs;
    vmax = fmax(vmax, fabs(rs));
    if constexpr (kTrial) phi += rs * rs;
  }
  vmax = BlockMax(vmax, scratch);        // (also orders the writes of s, u, Js)
  const bool finite_gj = BlockMax(chk != chk ? 1.0 : 0.0, scratch) == 0.0;
  if constexpr (kTrial) {                // converged or non-finite: no step (uniform over the CTA)
    double chk_x = 0.0;
    for (int j = tid; j < n; j += nt) chk_x = fma(X[(size_t)b * n + j], 0.0, chk_x);
    const bool finite = BlockMax(chk_x != chk_x ? 1.0 : 0.0, scratch) == 0.0 && finite_gj;
    phi = 0.5 * BlockSum(phi, scratch);
    if (!finite || vmax <= tr.tol) {
      for (int j = tid; j < n; j += nt) tr.x_trial[(size_t)b * n + j] = X[(size_t)b * n + j];
      if (tid == 0) {
        tr.status[b] = finite ? kLmConverged : kLmNonFinite;
        tr.merit[b] = finite ? phi : CUDART_NAN;
        tr.predicted[b] = 0.0;
        if (violation) violation[b] = finite ? vmax : CUDART_NAN;
      }
      return;
    }
  }
  auto row_dot = [&](int i) {            // (Js p)_i
    double acc = 0.0;
    const int k0 = __ldg(pat.row_ptr + i), k1 = __ldg(pat.row_ptr + i + 1);
    if (kSmemJ) { for (int k = k0; k < k1; ++k) acc += Js[k] * pd[__ldg(col_idx + k)]; }
    else { const double si = s[i]; for (int k = k0; k < k1; ++k) acc += (J[k] * si) * pd[__ldg(col_idx + k)]; }
    return acc;
  };
  auto col_dot = [&](int j) {            // (Js^T u)_j
    double acc = 0.0;
    const int k0 = __ldg(pat.col_ptr + j), k1 = __ldg(pat.col_ptr + j + 1);
    for (int k = k0; k < k1; ++k) {
      const int r = __ldg(row_t + k), slot = __ldg(slot_t + k);
      acc += (kSmemJ ? Js[slot] : J[slot] * s[r]) * u[r];
    }
    return acc;
  };
  // b = -Js^T rs; the trust-region rule freezes j (bit k of `frozen` for this thread's k-th column) and zeroes its b_j
  uint32_t frozen = 0;
  double rr = 0.0;
  for (int q = tid, k = 0; q < n; q += nt, ++k) {
    const int j = __ldg(pat.col_order + q);
    double bj = -col_dot(j);
    if constexpr (kTrust) {
      const double xj = X[(size_t)b * n + j], lj = x_lower[(size_t)b * bound_stride + j], uj = x_upper[(size_t)b * bound_stride + j];
      if (lj == uj || (xj <= lj && bj < 0.0) || (xj >= uj && bj > 0.0)) { frozen |= 1u << k; bj = 0.0; }
    }
    dx[j] = 0.0; res[j] = bj; pd[j] = bj;
    rr += bj * bj;
  }
  rr = BlockSum(rr, scratch);
  for (int it = 0; it < cg_iters; ++it) {
    for (int q = tid; q < m; q += nt) { const int i = __ldg(pat.row_order + q); u[i] = row_dot(i); }
    __syncthreads();
    double pap = 0.0;
    for (int q = tid, k = 0; q < n; q += nt, ++k) {   // ap = Js^T (Js p) + mu p (0 for a frozen j)
      const int j = __ldg(pat.col_order + q);
      const double a = kTrust && ((frozen >> k) & 1u) ? 0.0 : col_dot(j) + mu * pd[j];
      ap[j] = a;
      pap += pd[j] * a;
    }
    pap = BlockSum(pap, scratch);
    const double alpha = pap > 0.0 ? rr / pap : 0.0;
    double rr_new = 0.0;
    for (int j = tid; j < n; j += nt) {
      dx[j] += alpha * pd[j];
      const double rj = res[j] - alpha * ap[j];
      res[j] = rj;
      rr_new += rj * rj;
    }
    rr_new = BlockSum(rr_new, scratch);
    const double beta = rr > 0.0 ? rr_new / rr : 0.0;
    for (int j = tid; j < n; j += nt) pd[j] = res[j] + beta * pd[j];
    rr = rr_new;
    __syncthreads();
  }
  double big = 0.0, chk_x = 0.0;
  for (int j = tid; j < n; j += nt) { big = fmax(big, fabs(dx[j])); if (!kTrial) chk_x = fma(X[(size_t)b * n + j], 0.0, chk_x); }
  big = BlockMax(big, scratch);
  const bool finite = kTrial || (BlockMax(chk_x != chk_x ? 1.0 : 0.0, scratch) == 0.0 && finite_gj);
  const double scale = big > cap ? cap / big : 1.0;
  double* x = X + (size_t)b * n;
  const double* lo = x_lower + (size_t)b * bound_stride;
  const double* up = x_upper + (size_t)b * bound_stride;
  if constexpr (kTrial) {
    double* xt = tr.x_trial + (size_t)b * n;
    double dmax = 0.0;
    for (int j = tid; j < n; j += nt) {
      const double xj = x[j], v = fmin(fmax(xj + dx[j] * scale, lo[j]), up[j]);
      xt[j] = v;
      pd[j] = v - xj;                    // d: the step after cap and projection
      if constexpr (kTrust) dmax = fmax(dmax, fabs(pd[j]));
    }
    if constexpr (kTrust) {              // (also orders the writes of pd)
      dmax = BlockMax(dmax, scratch);
      if (tid == 0) tr.step_norm[b] = dmax;
    } else {
      __syncthreads();
    }
    double phi_lin = 0.0;                // sum of (s r(g + J d))^2, J d = (Js d) / s
    for (int q = tid; q < m; q += nt) {
      const int i = __ldg(pat.row_order + q);
      const double si = s[i];
      const double gi = g[i] + row_dot(i) / si, lo_i = __ldg(gl + i), up_i = __ldg(gu + i);
      const double rs = si * (gi < lo_i ? gi - lo_i : gi > up_i ? gi - up_i : 0.0);
      phi_lin += rs * rs;
    }
    phi_lin = 0.5 * BlockSum(phi_lin, scratch);
    if (tid == 0) {
      tr.merit[b] = phi;
      tr.predicted[b] = phi - phi_lin;
      if (violation) violation[b] = vmax;
    }
    return;
  }
  if (finite)
    for (int j = tid; j < n; j += nt) x[j] = fmin(fmax(x[j] + dx[j] * scale, lo[j]), up[j]);
  if (tid == 0 && violation) violation[b] = finite ? vmax : CUDART_NAN;
}

template <bool kSmemJ, class Idx, bool kTrial, bool kTrust>
int LaunchLmKernel(const LmPattern& pat, const Idx* col_idx, const Idx* slot_t, const Idx* row_t, int threads, size_t smem, int n, int m, int nnz,
                   double* x, const double* g, const double* jac, const double* xl, const double* xu, size_t bound_stride, const double* gl,
                   const double* gu, size_t g_bound_stride, double mu, double cap, int cg_iters, double* violation, const LmTrialArgs& tr, int nb,
                   cudaStream_t s) {
  cudaError_t e = cudaFuncSetAttribute(LmStepKernel<kSmemJ, Idx, kTrial, kTrust>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  LmStepKernel<kSmemJ, Idx, kTrial, kTrust><<<nb, threads, smem, s>>>(pat, col_idx, slot_t, row_t, n, m, nnz, x, g, jac, xl, xu, bound_stride, gl, gu,
                                                              g_bound_stride, mu, cap, cg_iters, violation, tr);
  return (int)cudaGetLastError();
}

template <bool kSmemJ, class Idx>
int LaunchLm(const LmPattern& pat, const Idx* col_idx, const Idx* slot_t, const Idx* row_t, int threads, size_t smem, int n, int m, int nnz, double* x,
             const double* g, const double* jac, const double* xl, const double* xu, size_t bound_stride, const double* gl, const double* gu,
             size_t g_bound_stride, double mu, double cap, int cg_iters, double* violation, const LmTrialArgs* trial, int nb, cudaStream_t s) {
  if (trial && trial->radius)
    return LaunchLmKernel<kSmemJ, Idx, true, true>(pat, col_idx, slot_t, row_t, threads, smem, n, m, nnz, x, g, jac, xl, xu, bound_stride, gl, gu,
                                                   g_bound_stride, mu, cap, cg_iters, violation, *trial, nb, s);
  if (trial)
    return LaunchLmKernel<kSmemJ, Idx, true, false>(pat, col_idx, slot_t, row_t, threads, smem, n, m, nnz, x, g, jac, xl, xu, bound_stride, gl, gu,
                                             g_bound_stride, mu, cap, cg_iters, violation, *trial, nb, s);
  return LaunchLmKernel<kSmemJ, Idx, false, false>(pat, col_idx, slot_t, row_t, threads, smem, n, m, nnz, x, g, jac, xl, xu, bound_stride, gl, gu,
                                            g_bound_stride, mu, cap, cg_iters, violation, LmTrialArgs{}, nb, s);
}

// CTA = instance, RUNNING instances only.  phi_t = 1/2 ||row_scale r(g_trial)||^2 (fixed summation order), rho = (phi0 - phi_t) /
// predicted; accept when predicted > 0, every g_trial entry is finite (an infinite g against an infinite bound would count as
// no violation) and rho > eta.  Every thread takes the same decision from the broadcast sums; thread 0 updates the scalars.
__global__ void __launch_bounds__(256) LmAcceptKernel(int n, int m, double* __restrict__ X, const double* __restrict__ x_trial,
                                                      const double* __restrict__ g_trial, const double* __restrict__ g_lower,
                                                      const double* __restrict__ g_upper, size_t g_bound_stride,
                                                      const double* __restrict__ row_scale, const double* __restrict__ merit,
                                                      const double* __restrict__ predicted, double* __restrict__ mu, double* __restrict__ nu,
                                                      int* __restrict__ status, int* __restrict__ iterations, double eta, double mu_min,
                                                      double mu_max, double* __restrict__ radius, const double* __restrict__ step_norm,
                                                      double radius_max) {
  __shared__ double scratch[32];
  const int b = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
  if (status[b] != kLmRunning) return;
  const double* __restrict__ g = g_trial + (size_t)b * m;
  const double* __restrict__ s = row_scale + (size_t)b * m;
  const double* __restrict__ gl = g_lower + (size_t)b * g_bound_stride;
  const double* __restrict__ gu = g_upper + (size_t)b * g_bound_stride;
  double phi = 0.0, chk = 0.0;
  for (int i = tid; i < m; i += nt) {
    const double gi = g[i], lo = __ldg(gl + i), up = __ldg(gu + i);
    const double rs = s[i] * (gi < lo ? gi - lo : gi > up ? gi - up : 0.0);
    phi += rs * rs;
    chk = fma(gi, 0.0, chk);
  }
  phi = 0.5 * BlockSum(phi, scratch);
  const bool finite = BlockMax(chk != chk ? 1.0 : 0.0, scratch) == 0.0 && isfinite(phi);
  const double pred = predicted[b];
  const double rho = (merit[b] - phi) / pred;
  const bool accept = pred > 0.0 && finite && rho > eta;
  if (accept)
    for (int j = tid; j < n; j += nt) X[(size_t)b * n + j] = x_trial[(size_t)b * n + j];
  double xmax = 0.0;                     // max |x| after the decision (the trust-region rule's collapse test)
  if (radius) {
    const double* __restrict__ xn = (accept ? x_trial : X) + (size_t)b * n;
    for (int j = tid; j < n; j += nt) xmax = fmax(xmax, fabs(xn[j]));
    xmax = BlockMax(xmax, scratch);
  }
  if (tid == 0) {
    if (accept) {                        // mu <- max(mu_min, mu max(1/3, 1 - (2 rho - 1)^3)), nu <- 2
      const double t = 2.0 * rho - 1.0;
      mu[b] = fmax(mu_min, mu[b] * fmax(1.0 / 3.0, 1.0 - t * t * t));
      nu[b] = 2.0;
    } else {                             // mu <- mu nu, nu <- 2 nu; past mu_max: stalled
      const double mu_new = mu[b] * nu[b];
      mu[b] = mu_new;
      nu[b] = 2.0 * nu[b];
      if (mu_new > mu_max) status[b] = kLmStalled;
    }
    if (radius) {
      const double sn = step_norm[b];
      double r = radius[b];
      if (!accept || rho < kTrLow) r = kTrShrink * sn;
      else if (rho > kTrHigh && sn >= kTrEdge * r) r = fmin(kTrGrow * r, radius_max);
      radius[b] = r;
      if (r < kTrCollapse * fmax(1.0, xmax)) status[b] = kLmStalled;
    }
    iterations[b] += 1;
  }
}

// ---- the device-side solve loop (twb_batch_lm_solve_device): the start of a solve and the loop's exit test
// loop[kLoopIter] = iterations the loop has run, loop[kLoopCount + s] = instances with status s (accumulated over the CTAs of
// one count), loop[kLoopTicket] = CTAs of the current count that have added theirs
constexpr int kLoopIter = 0, kLoopCount = 1, kLoopTicket = 5;
constexpr int kCountThreads = 256, kCountPerThread = 4;

__global__ void __launch_bounds__(256) LmSolveInitKernel(int nb, double mu0, double* __restrict__ mu, double* __restrict__ nu,
                                                         int* __restrict__ status, int* __restrict__ iterations, double radius0,
                                                         double* __restrict__ radius, double* __restrict__ step_norm,
                                                         int* __restrict__ loop, int max_iters,
                                                         cudaGraphConditionalHandle cond) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < nb) {
    mu[b] = mu0; nu[b] = 2.0; status[b] = kLmRunning; iterations[b] = 0;
    if (radius) { radius[b] = radius0; step_norm[b] = 0.0; }
  }
  if (b == 0) {
    for (int k = 0; k < kLoopInts; ++k) loop[k] = 0;
    cudaGraphSetConditional(cond, max_iters > 0 ? 1u : 0u);
  }
}

// Instances per status, one CTA per chunk of kCountThreads * kCountPerThread instances: integer counts per CTA, added up with
// integer atomics (exact, so the result does not depend on the order of the CTAs); the last CTA to finish reads the totals.
// loop_step: the last kernel of the loop body — loop[kLoopIter] += 1 and the WHILE condition becomes "an instance is RUNNING
// and the budget is not spent".  Otherwise (after the tail): the counts and the loop's iterations go to the caller's
// status_counts[4] / loop_count[1] when given.
__global__ void __launch_bounds__(kCountThreads) LmCountKernel(int nb, const int* __restrict__ status, int* __restrict__ loop, int max_iters,
                                                               cudaGraphConditionalHandle cond, bool loop_step, int* __restrict__ status_counts,
                                                               int* __restrict__ loop_count) {
  __shared__ int part[kCountThreads / 32][4];
  __shared__ bool last;
  int c[4] = {0, 0, 0, 0};
  const int b0 = blockIdx.x * kCountThreads * kCountPerThread;
  for (int k = 0; k < kCountPerThread; ++k) {
    const int b = b0 + k * kCountThreads + threadIdx.x;
    if (b < nb) {
      const int s = status[b];
      for (int q = 0; q < 4; ++q) c[q] += s == q;
    }
  }
  for (int q = 0; q < 4; ++q) c[q] = __reduce_add_sync(0xffffffffu, c[q]);
  if ((threadIdx.x & 31) == 0) for (int q = 0; q < 4; ++q) part[threadIdx.x >> 5][q] = c[q];
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int q = 0; q < 4; ++q) {
      int t = 0;
      for (int w = 0; w < kCountThreads / 32; ++w) t += part[w][q];
      if (t) atomicAdd(loop + kLoopCount + q, t);
    }
    __threadfence();
    last = atomicAdd(loop + kLoopTicket, 1) == (int)gridDim.x - 1;
  }
  __syncthreads();
  if (!last || threadIdx.x != 0) return;
  __threadfence();
  int total[4];
  for (int q = 0; q < 4; ++q) { total[q] = atomicExch(loop + kLoopCount + q, 0); }
  loop[kLoopTicket] = 0;
  if (loop_step) {
    const int it = loop[kLoopIter] + 1;
    loop[kLoopIter] = it;
    cudaGraphSetConditional(cond, (total[kLmRunning] > 0 && it < max_iters) ? 1u : 0u);
  } else {
    if (status_counts) for (int q = 0; q < 4; ++q) status_counts[q] = total[q];
    if (loop_count) *loop_count = loop[kLoopIter];
  }
}

}  // namespace

size_t LmSharedBytes(int n, int m) { return sizeof(double) * ((size_t)2 * m + 4 * (size_t)n + 32); }

int LaunchLmStep(const LmPattern& pat, int n, int m, int nnz, double* x, const double* g, const double* jac, const double* x_lower,
                 const double* x_upper, size_t bound_stride, const double* g_lower, const double* g_upper, size_t g_bound_stride, double mu,
                 double cap, int cg_iters, double* violation, const LmTrialArgs* trial, int nb, cudaStream_t s) {
  if (nb <= 0) return 0;
  const size_t vec = LmSharedBytes(n, m), with_j = vec + sizeof(double) * (size_t)nnz;
  const bool smem_j = with_j <= 220 * 1024;   // the scaled values fit beside the vectors: one CTA of 512 threads per SM
  const int threads = smem_j ? 512 : 256;
  if (trial && trial->radius && n > 32 * threads) return (int)cudaErrorInvalidValue;   // one frozen bit per column and thread
  const size_t smem = smem_j ? with_j : vec;
  if (pat.col_idx16) {
    return smem_j ? LaunchLm<true>(pat, pat.col_idx16, pat.slot_t16, pat.row_t16, threads, smem, n, m, nnz, x, g, jac, x_lower, x_upper, bound_stride, g_lower, g_upper, g_bound_stride, mu, cap, cg_iters, violation, trial, nb, s)
                  : LaunchLm<false>(pat, pat.col_idx16, pat.slot_t16, pat.row_t16, threads, smem, n, m, nnz, x, g, jac, x_lower, x_upper, bound_stride, g_lower, g_upper, g_bound_stride, mu, cap, cg_iters, violation, trial, nb, s);
  }
  // 32-bit indices mean n, m or nnz >= 65 536, so with_j >= 8 * 65 536 bytes > 220 KiB: never the shared-memory Js path
  return LaunchLm<false>(pat, pat.col_idx, pat.slot_t, pat.row_t, threads, smem, n, m, nnz, x, g, jac, x_lower, x_upper, bound_stride, g_lower, g_upper, g_bound_stride, mu, cap, cg_iters, violation, trial, nb, s);
}

int LaunchLmAccept(int n, int m, double* x, const double* x_trial, const double* g_trial, const double* g_lower, const double* g_upper,
                   size_t g_bound_stride, const double* row_scale, const double* merit, const double* predicted, double* mu, double* nu,
                   int* status, int* iterations, double eta, double mu_min, double mu_max, double* radius, const double* step_norm,
                   double radius_max, int nb, cudaStream_t s) {
  if (nb <= 0) return 0;
  LmAcceptKernel<<<nb, 256, 0, s>>>(n, m, x, x_trial, g_trial, g_lower, g_upper, g_bound_stride, row_scale, merit, predicted, mu, nu, status,
                                    iterations, eta, mu_min, mu_max, radius, step_norm, radius_max);
  return (int)cudaGetLastError();
}

int LaunchLmSolveInit(int nb, double mu0, double* mu, double* nu, int* status, int* iterations, double radius0, double* radius,
                      double* step_norm, int* loop, int max_iters, cudaGraphConditionalHandle cond, cudaStream_t s) {
  LmSolveInitKernel<<<(std::max(nb, 1) + 255) / 256, 256, 0, s>>>(nb, mu0, mu, nu, status, iterations, radius0, radius, step_norm, loop,
                                                                  max_iters, cond);
  return (int)cudaGetLastError();
}

int LaunchLmCount(int nb, const int* status, int* loop, int max_iters, cudaGraphConditionalHandle cond, bool loop_step, int* status_counts,
                  int* loop_count, cudaStream_t s) {
  const int per_cta = kCountThreads * kCountPerThread;
  LmCountKernel<<<(std::max(nb, 1) + per_cta - 1) / per_cta, kCountThreads, 0, s>>>(nb, status, loop, max_iters, cond, loop_step,
                                                                                    status_counts, loop_count);
  return (int)cudaGetLastError();
}

}  // namespace twb
