// kernels.cu — sm_100a kernels of the batched NLP evaluation (fp64).
//
// Everything is a data-parallel map with LANE = PROBLEM INSTANCE.  The iterates are first brought into
// an instance-tiled matrix XT[tile][n+1][32] (tile = 32 instances of one alignment class, lane = instance), so that
// every read of a node value by a warp is one 256-byte row segment:
//
//   TransposeInP  x[B][n]   -> XT[tile][n+1][32]   (row n stays 0: "not optimised" node values; persistent CTAs)
//   DynOut        XT        -> CSR values + constraint values of the dynamic constraint (warp = sample x tile)
//   RomNodeOut    XT        -> CSR values + constraint values of the range-of-motion constraints (warp = sample x
//                              tile, all feet) and of the node-wise sets: terrain, force, swing, spline-acc,
//                              base-motion (warp = group of consecutive nodes x tile); the CTAs of a tile in row order;
//                              constant runs of the CSR rows by TMA bulk copies (ConstRunBody)
//   DynTailOut    (optimised phase durations only) the PhaseSpline columns of the dynamic rows (warp = foot)
//   PhaseJac      (optimised phase durations only) the TotalDurationConstraint rows
//   CostKernel    XT        -> cost + gradient (only when the formulation has cost terms)
//   (TransposeOut GT[tile][m][32] -> g[B][m]: only in the -DTWB_GDIRECT=0 variants; the output CTAs write g themselves)
//
// In the output kernels a warp owns one unit of 32 instances: each lane evaluates the splines its unit needs
// (reference operation order) and computes its instance's unit state into a padded shared-memory block (row =
// state slot, column = lane).  After the CTA barrier ALL threads of the CTA switch roles — thread = 16-byte pair
// of output elements — and stream
//     out[instance][off + h] = state[d_h][instance] * c_h
// for the 32 instances from ONE list that covers the CTA's consecutive units (adjacent CSR rows): every store
// instruction covers 512 contiguous bytes of one instance's CSR value row, whole 32-byte sectors only.  The
// state never leaves the SM; HBM sees x once and g / jac exactly once.  DynOut runs beside RomNodeOut on a
// second stream; twb_batch_eval_device replays the whole evaluation as one CUDA graph.
//
// Reference math restated per device function (file:line cited there).  This translation unit is
// compiled with -fmad=false: plain * and + round like the reference's scalar C++; fused
// multiply-adds are written explicitly (fma) where the algebra is re-associated anyway.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstdio>

#include "device_tables.h"
#include "launch.h"

namespace twb {
void (*g_after_launch)(const char* label, cudaStream_t stream) = nullptr;   // profiling hook (capi.cc, TWB_PROFILE=1)
#define TWB_MARK(label, stream) do { if (g_after_launch) g_after_launch(label, stream); } while (0)
// L2 access-policy window of the evaluation kernels (capi.cc sets it per call): the two staging matrices XT / GT are marked
// persisting, so that the 524 MB of streaming output per step cannot push them out of the L2 before their readers run
// (ncu, round 2: 38 MB of XT were re-fetched from HBM by the output kernels and all 29 MB of GT by TransposeOut).
thread_local const cudaAccessPolicyWindow* t_l2_window = nullptr;
void SetL2Window(const cudaAccessPolicyWindow* w) { t_l2_window = w; }
namespace {

#ifndef TWB_TOUT_LD
#define TWB_TOUT_LD 0    // cache operator of TransposeOut's loads of GT: 0 .cs, 1 .cg, 2 default, 3 .lu
#endif
#ifndef TWB_DISCARD
#define TWB_DISCARD 1    // TransposeOut drops the dead L2 lines of GT and XT (discard.global.L2) instead of letting them be written back
#endif
#ifndef TWB_PDL
#define TWB_PDL 1        // 1: RomNodeOut is launched with programmatic stream serialization behind TransposeIn (138.9 vs 144.6 us per step on config 2)
#endif
#if TWB_FUSED
#ifndef TWB_CTAS
#define TWB_CTAS 2   // CTAs per SM the fused output kernel is compiled for (bounds its registers)
#endif
#else
#ifndef TWB_DYN_CTAS
#define TWB_DYN_CTAS 2
#endif
#ifndef TWB_ROM_CTAS
#define TWB_ROM_CTAS 4
#endif
#ifndef TWB_NODE_CTAS
#define TWB_NODE_CTAS 3
#endif
#endif
#ifndef TWB_TMA
#define TWB_TMA 0        // 1: the Jacobian values of a CTA list leave the SM as cp.async.bulk.global.shared::cta copies of contiguous row segments assembled in shared memory; 0 (ships): 16-byte st.global.cs from the pair loop.  Measured (profiles/README.md, round 2): parity green, but 192 us per step instead of 139 us on config 2 — the extra pass through shared memory costs more than the better DRAM pattern gains
#endif
#ifndef TWB_CONST_WAIT_ALL
#define TWB_CONST_WAIT_ALL 0
#endif
#ifndef TWB_ST_HINT
#define TWB_ST_HINT 0    // cache operator of the Jacobian-value stores: 0 .cs (evict-first), 1 default (.wb), 2 .wt
#endif
#ifndef TWB_XT_EVICT_LAST
#define TWB_XT_EVICT_LAST 0   // 1: TransposeIn writes XT with an L2 evict_last policy (experiment)
#endif
#ifndef TWB_ST256
#define TWB_ST256 0     // 1: thread = whole sector (two consecutive pairs of the list), 256-bit stores, items of 8 instances
#endif
#ifndef TWB_TMA_DYN
#define TWB_TMA_DYN TWB_TMA   // per-kernel switches of the TMA store path (tuning)
#endif
#ifndef TWB_TMA_ROM
#define TWB_TMA_ROM TWB_TMA
#endif
#ifndef TWB_TMA_G
#define TWB_TMA_G 2      // instances assembled per staging step (2: 16-byte reads of the state rows)
#endif
#ifndef TWB_TMA_BUF
#define TWB_TMA_BUF 1    // staging buffers per warp (ring)
#endif
constexpr int kLD = 34;                      // leading dimension of a state block: 32 instances, padded; even keeps rows 16-byte aligned

// output stores: streaming (evict-first) — the values are consumed by the host / a solver, not by these kernels
__device__ __forceinline__ void StoreOut(double* p, double v) { __stcs(p, v); }
__device__ __forceinline__ void StoreOut2(double* p, double a, double b) {
#if TWB_ST_HINT == 1
  asm volatile("st.global.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(a), "d"(b) : "memory");
#elif TWB_ST_HINT == 2
  asm volatile("st.global.wt.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(a), "d"(b) : "memory");
#else
  asm volatile("st.global.cs.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(a), "d"(b) : "memory");
#endif
}

// 256-bit store (sm_100: SASS STG.E.256): a thread writes a whole 32-byte sector
__device__ __forceinline__ void StoreOut4(double* p, double a, double b, double c, double d) {
  asm volatile("st.global.cs.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}
// column `b` of a row-major [rows][ld] matrix: element r lives at p[r * ld]
struct Col {
  double* p;
  size_t ld;
  __device__ __forceinline__ double& operator[](int r) const { return p[(size_t)r * ld]; }
};
struct ConstCol {
  const double* __restrict__ p;
  __device__ __forceinline__ double operator[](int r) const { return __ldg(p + (size_t)r * 32); }
};

// ---- cubic Hermite evaluation ------------------------------------------------
// a / b, correctly rounded, from y = RN(1/b) (Markstein): two residual corrections with exact
// FMA residuals.  Replaces the ~35-instruction IEEE division sequence; the divisors (T^2, T^3)
// are structure-class constants whose reciprocals come with the sample table.
__device__ __forceinline__ double DivExact(double a, double b, double y) {
  double q = a * y;
  double r = fma(-b, q, a);
  q = fma(r, y, q);
  r = fma(-b, q, a);
  return fma(r, y, q);
}
// CubicHermitePolynomial::UpdateCoeff (polynomial.cc:97-104) followed by
// Polynomial::GetPoint (polynomial.cc:47-61): sum_c d^k/dt^k(t^c) * coeff_c, c = A..D, in the
// reference's operation order (this translation unit is compiled with -fmad=false, so the
// products and sums below round exactly like the reference's scalar code).
struct SampleRegs { double T, T2, T3, rT2, rT3, t, t2, t3; int xi[12]; };
__device__ __forceinline__ SampleRegs LoadSample(const SplineSample* __restrict__ p) {
  const double2* d = reinterpret_cast<const double2*>(p);
  const double2 a = __ldg(d), b = __ldg(d + 1), c = __ldg(d + 2), e = __ldg(d + 3);
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(p) + 4);
  const uint2 w = __ldg(reinterpret_cast<const uint2*>(p) + 10);
  SampleRegs r;
  r.T = a.x; r.T2 = a.y; r.T3 = b.x; r.rT2 = b.y; r.rT3 = c.x; r.t = c.y; r.t2 = e.x; r.t3 = e.y;
  const uint32_t v[6] = {u.x, u.y, u.z, u.w, w.x, w.y};
#pragma unroll
  for (int i = 0; i < 6; ++i) { r.xi[2 * i] = (int)(v[i] & 0xFFFFu); r.xi[2 * i + 1] = (int)(v[i] >> 16); }
  return r;
}
// std::pow(x, 3) and std::pow(x, 4) of the reference (polynomial.cc:47-61, 236-257; glibc's pow is correctly rounded
// apart from a handful of hard cases): x*x*x rounds twice and is up to 1 ulp off, which the division by T^3 / T^4 in front
// of cancelling sums amplifies past 1e-12.  Here: the square with its exact FMA error term, then one rounding of the
// compensated product — the correctly rounded power (x^2 itself is a single rounding in both).
__device__ __forceinline__ double Pow3(double x) {
  const double x2 = x * x, e2 = fma(x, x, -x2);       // x^2 = x2 + e2 exactly
  const double hi = x2 * x, lo = fma(x2, x, -hi);     // x2 * x = hi + lo exactly
  return hi + fma(e2, x, lo);
}
__device__ __forceinline__ double Pow4(double x) {
  const double x2 = x * x, e2 = fma(x, x, -x2);
  const double hi = x2 * x2, lo = fma(x2, x2, -hi);
  return hi + fma(2.0 * x2, e2, lo);
}
// ---- PhaseSpline (phase_spline.cc, phase_durations.cc): polynomial durations are functions of the iterate ----
// Active polynomial and local time of global time t: PhaseDurations::SetVariables (phase_durations.cc:79-100),
// NodesVariablesPhaseBased::ConvertPhaseToPolyDurations (nodes_variables_phase_based.cc:78-89),
// Spline::GetSegmentID / GetLocalTime (spline.cc:48-78) — same operations in the same order, per instance.
// One pass over the foot's phases (their polynomials are consecutive in Plan::phase_polys, every phase has at least one):
// the sum of the optimised durations and the last phase's duration (phase_durations.cc:92-98), the phase the time falls
// into (GetSegmentID over the phase durations), and the polynomial / local time (GetSegmentID / GetLocalTime over the
// polynomial durations phase / n) — every accumulation in the reference's order.  d / n is a plain copy for n = 1 and an
// exact scaling for n = 2 (both are the correctly rounded quotient); other n divide.
struct PhaseLoc { int poly, cur; double tl, T, last; };
__device__ __forceinline__ PhaseLoc LocatePhasePoly(const Plan& P, const PhaseSplineDef& def, double t, const ConstCol xs) {
  PhaseLoc o; o.poly = def.n_polys - 1; o.cur = def.n_phases - 1; o.tl = t; o.T = 0.0; o.last = def.t_total;
  const double eps = 1e-10, thr = t - eps;
  double sum = 0.0, acc = 0.0, acc_ph = 0.0, tl_run = t; bool found = false, found_ph = false;
  const PhasePoly* pp = P.phase_polys + def.poly0;
  int p = 0;
  for (int ph = 0; ph < def.n_phases; ++ph) {
    double d;
    if (ph == def.n_phases - 1) { d = def.t_total - sum; o.last = d; }
    else { d = xs[def.sched0 + ph]; sum += d; }
    acc_ph += d;
    if (!found_ph && acc_ph >= thr) { found_ph = true; o.cur = ph; }
    const int n = pp[p].n_in_phase;
    const double Tp = n == 1 ? d : n == 2 ? d * 0.5 : d / (double)n;
    for (int k = 0; k < n; ++k, ++p) {
      acc += Tp;
      if (!found) {
        if (acc >= thr || p == def.n_polys - 1) { found = true; o.poly = p; o.T = Tp; o.tl = tl_run; }
        tl_run -= Tp;
      }
    }
  }
  return o;
}
// kWant: 0 position; 1 position + acceleration; 2 position + velocity + acceleration
// kPhase: the sample may refer to a PhaseSpline (only in kernels instantiated for duration-optimised problems, so
// that the fixed-duration kernels carry neither the branch nor the code)
template <int kWant, bool kPhase = false>
__device__ __forceinline__ void EvalSpline(const Plan& P, const SplineSample* __restrict__ sp, const ConstCol xs, double pos[3], double vel[3], double acc[3]) {
  const SampleRegs s = LoadSample(sp);
  if (kPhase && s.xi[0] == (int)kPhaseMarker) {   // PhaseSpline: s.T holds the global sample time (warp-uniform branch)
    const PhaseSplineDef def = P.phase_defs[s.xi[1]];
    const PhaseLoc L = LocatePhasePoly(P, def, s.T, xs);
    const PhasePoly* pp = P.phase_polys + def.poly0 + L.poly;
    const double T = L.T, T2 = T * T, T3 = Pow3(T), t = L.tl, t2 = t * t, t3 = Pow3(t);   // std::pow(x, 2), std::pow(x, 3)
    const double rT2 = 1.0 / T2, rT3 = 1.0 / T3;   // the quotients below: exact (Markstein) divisions seeded with these
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const double p0 = xs[pp->xi[d]], v0 = xs[pp->xi[3 + d]], p1 = xs[pp->xi[6 + d]], v1 = xs[pp->xi[9 + d]];
      const double C = DivExact(-(3 * (p0 - p1) + T * (2 * v0 + v1)), T2, rT2);
      const double D = DivExact(2 * (p0 - p1) + T * (v0 + v1), T3, rT3);
      pos[d] = ((p0 + t * v0) + t2 * C) + t3 * D;
      if (kWant == 2) vel[d] = (v0 + (2 * t) * C) + (3 * t2) * D;
      if (kWant >= 1) acc[d] = 2 * C + (6 * t) * D;
    }
    return;
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const double p0 = xs[s.xi[d]], v0 = xs[s.xi[3 + d]], p1 = xs[s.xi[6 + d]], v1 = xs[s.xi[9 + d]];
    const double C = DivExact(-(3 * (p0 - p1) + s.T * (2 * v0 + v1)), s.T2, s.rT2);
    const double D = DivExact(2 * (p0 - p1) + s.T * (v0 + v1), s.T3, s.rT3);
    pos[d] = ((p0 + s.t * v0) + s.t2 * C) + s.t3 * D;
    if (kWant == 2) vel[d] = (v0 + (2 * s.t) * C) + (3 * s.t2) * D;
    if (kWant >= 1) acc[d] = 2 * C + (6 * s.t) * D;
  }
}

// ---- Euler angles (roll x, pitch y, yaw z; applied Z-Y'-X'') -------------------
struct Trig { double sx, cx, sy, cy, sz, cz; };
__device__ __forceinline__ Trig MakeTrig(const double th[3]) {
  Trig t; sincos(th[0], &t.sx, &t.cx); sincos(th[1], &t.sy, &t.cy); sincos(th[2], &t.sz, &t.cz); return t;
}
// EulerConverter::GetRotationMatrixBaseToWorld, euler_converter.cc:207-221
__device__ __forceinline__ void RotationMatrix(const Trig& t, double R[3][3]) {
  R[0][0] = t.cy * t.cz; R[0][1] = t.cz * t.sx * t.sy - t.cx * t.sz; R[0][2] = t.sx * t.sz + t.cx * t.cz * t.sy;
  R[1][0] = t.cy * t.sz; R[1][1] = t.cx * t.cz + t.sx * t.sy * t.sz; R[1][2] = t.cx * t.sy * t.sz - t.cz * t.sx;
  R[2][0] = -t.sy;       R[2][1] = t.cy * t.sx;                      R[2][2] = t.cx * t.cy;
}
// d(R_ij)/d(theta_d): coefficients of jac_x / jac_y / jac_z in
// EulerConverter::GetDerivativeOfRotationMatrixWrtNodes, euler_converter.cc:241-268
__device__ __forceinline__ void RotationDerivative(const Trig& t, double dR[3][3][3]) {
  const double sx = t.sx, cx = t.cx, sy = t.sy, cy = t.cy, sz = t.sz, cz = t.cz;
  dR[0][0][0] = 0.0;                         dR[0][0][1] = -cz * sy;      dR[0][0][2] = -cy * sz;
  dR[0][1][0] = sx * sz + cx * cz * sy;      dR[0][1][1] = cy * cz * sx;  dR[0][1][2] = -cx * cz - sx * sy * sz;
  dR[0][2][0] = cx * sz - cz * sx * sy;      dR[0][2][1] = cx * cy * cz;  dR[0][2][2] = cz * sx - cx * sy * sz;
  dR[1][0][0] = 0.0;                         dR[1][0][1] = -sy * sz;      dR[1][0][2] = cy * cz;
  dR[1][1][0] = cx * sy * sz - cz * sx;      dR[1][1][1] = cy * sx * sz;  dR[1][1][2] = -cx * sz + cz * sx * sy;
  dR[1][2][0] = -cx * cz - sx * sy * sz;     dR[1][2][1] = cx * cy * sz;  dR[1][2][2] = sx * sz + cx * cz * sy;
  dR[2][0][0] = 0.0;                         dR[2][0][1] = -cy;           dR[2][0][2] = 0.0;
  dR[2][1][0] = cx * cy;                     dR[2][1][1] = -sx * sy;      dR[2][1][2] = 0.0;
  dR[2][2][0] = -cy * sx;                    dR[2][2][1] = -cx * sy;      dR[2][2][2] = 0.0;
}
// EulerConverter::DerivOfRotVecMult (euler_converter.cc:223-239) as a dense 3x3:
// D[row][d] = sum_col v[col] * d(R or R^T)[row][col] / d(theta_d)
template <bool kInverse>
__device__ __forceinline__ void RotVecDerivative(const double dR[3][3][3], const double v[3], double D[3][3]) {
#pragma unroll
  for (int row = 0; row < 3; ++row)
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      double s = 0.0;
#pragma unroll
      for (int col = 0; col < 3; ++col) s = fma(v[col], kInverse ? dR[col][row][d] : dR[row][col][d], s);
      D[row][d] = s;
    }
}
__device__ __forceinline__ void Mul33(const double A[3][3], const double B[3][3], double C[3][3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) C[i][j] = fma(A[i][2], B[2][j], fma(A[i][1], B[1][j], A[i][0] * B[0][j]));
}
__device__ __forceinline__ void MulVec(const double A[3][3], const double v[3], double o[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) o[i] = A[i][0] * v[0] + A[i][1] * v[1] + A[i][2] * v[2];
}
// C = [w]x * A  (Cross(), single_rigid_body_dynamics.cc:46-57)
__device__ __forceinline__ void CrossMul(const double w[3], const double A[3][3], double C[3][3]) {
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    C[0][j] = fma(w[1], A[2][j], -w[2] * A[1][j]);
    C[1][j] = fma(w[2], A[0][j], -w[0] * A[2][j]);
    C[2][j] = fma(w[0], A[1][j], -w[1] * A[0][j]);
  }
}

// ---- DynamicConstraint sample ------------------------------------------------
// Values: DynamicConstraint::UpdateModel (dynamic_constraint.cc:119-137) +
//   SingleRigidBodyDynamics::GetDynamicViolation (single_rigid_body_dynamics.cc:76-101).
// Jacobian state: the 3x3 maps A, B, C with
//   d(angular rows)/d(base-ang nodes) = A*dtheta + B*dtheta_dot + C*dtheta_ddot
//   restating SingleRigidBodyDynamics::GetJacobianWrtBaseAng (:123-165) with
//   EulerConverter::GetDerivOfAng{Vel,Acc}WrtEulerNodes (euler_converter.cc:85-131),
//   GetDerivMwrtNodes (:168-198), GetDerivMdotwrtNodes (:270-304);
//   sum of forces, per-foot force and lever arm for the other blocks (:103-121, :167-192).
// Sk: local state rows 1.. (Sk[0..2] sum f, Sk[3..38] base-ang block, Sk[39 + 6e ..] f_e, c - p_e);
// gk: the 6 constraint values
// feet: with optimised durations and a Jacobian evaluation the DynTailOut kernel has already evaluated the feet's PhaseSplines
// of this sample; their values come from its scratch rows (6 per foot: p_e, f_e; lane = instance) instead of a second evaluation
template <int kNEE, bool kPhase>
__device__ __forceinline__ void DynamicUnit(const Plan& P, int k, const SplineSample* __restrict__ sp, const ConstCol xs,
                                            const Col Sk, const Col gk, const double* __restrict__ feet) {
  double c[3], cdd[3], th[3], thd[3], thdd[3], unused[3];
  EvalSpline<1>(P, sp + 0, xs, c, unused, cdd);
  EvalSpline<2>(P, sp + 1, xs, th, thd, thdd);

  // feet
  double fsum[3] = {0, 0, 0}, tau[3] = {0, 0, 0};
#pragma unroll
  for (int e = 0; e < kNEE; ++e) {
    double pe[3], f[3];
    if (kPhase && feet) {
#pragma unroll
      for (int d = 0; d < 3; ++d) { pe[d] = __ldcg(feet + (e * 6 + d) * 32); f[d] = __ldcg(feet + (e * 6 + 3 + d) * 32); }
    } else {
      EvalSpline<0, kPhase>(P, sp + 2 + e, xs, pe, unused, unused);
      EvalSpline<0, kPhase>(P, sp + 2 + kNEE + e, xs, f, unused, unused);
    }
    const double r[3] = {c[0] - pe[0], c[1] - pe[1], c[2] - pe[2]};
    tau[0] += f[1] * r[2] - f[2] * r[1];
    tau[1] += f[2] * r[0] - f[0] * r[2];
    tau[2] += f[0] * r[1] - f[1] * r[0];
#pragma unroll
    for (int d = 0; d < 3; ++d) { fsum[d] += f[d]; Sk[39 + e * 6 + d] = f[d]; Sk[39 + e * 6 + 3 + d] = r[d]; }
  }
  Sk[0] = fsum[0]; Sk[1] = fsum[1]; Sk[2] = fsum[2];

  const Trig tr = MakeTrig(th);
  const double sy = tr.sy, cy = tr.cy, sz = tr.sz, cz = tr.cz;
  double R[3][3]; RotationMatrix(tr, R);
  const double yd = thd[1], zd = thd[2];
  // EulerConverter::GetM (:133-148) and GetMdot (:150-166)
  double M[3][3] = {{cy * cz, -sz, 0.0}, {cy * sz, cz, 0.0}, {-sy, 0.0, 1.0}};
  double Md[3][3] = {{-cz * sy * yd - cy * sz * zd, -cz * zd, 0.0}, {cy * cz * zd - sy * sz * yd, -sz * zd, 0.0}, {-cy * yd, 0.0, 0.0}};
  double om[3], omd[3];
  om[0] = M[0][0] * thd[0] + M[0][1] * thd[1];
  om[1] = M[1][0] * thd[0] + M[1][1] * thd[1];
  om[2] = M[2][0] * thd[0] + thd[2];
  omd[0] = (Md[0][0] * thd[0] + Md[0][1] * thd[1]) + (M[0][0] * thdd[0] + M[0][1] * thdd[1]);
  omd[1] = (Md[1][0] * thd[0] + Md[1][1] * thd[1]) + (M[1][0] * thdd[0] + M[1][1] * thdd[1]);
  omd[2] = (Md[2][0] * thd[0]) + (M[2][0] * thdd[0] + thdd[2]);

  // I_w = R I_b R^T
  double Ib[3][3], RIb[3][3], Rt[3][3], Iw[3][3];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) { Ib[i][j] = P.I_b[i * 3 + j]; Rt[i][j] = R[j][i]; }
  Mul33(R, Ib, RIb); Mul33(RIb, Rt, Iw);

  double Iw_om[3], Iw_omd[3];
  MulVec(Iw, om, Iw_om); MulVec(Iw, omd, Iw_omd);
  {
    const double wx[3] = {om[1] * Iw_om[2] - om[2] * Iw_om[1], om[2] * Iw_om[0] - om[0] * Iw_om[2], om[0] * Iw_om[1] - om[1] * Iw_om[0]};
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      gk[d] = Iw_omd[d] + wx[d] - tau[d];
      const double grav = (d == 2) ? -P.mass * P.gravity : 0.0;
      gk[3 + d] = P.mass * cdd[d] - fsum[d] - grav;
    }
  }

  // ---- base-angular Jacobian maps
  double dR[3][3][3]; RotationDerivative(tr, dR);
  // d(omega)/d(theta) (GetDerivMwrtNodes contracted with theta_dot) ; d(omega)/d(theta_dot) = M
  double Jw[3][3] = {{0.0, thd[0] * (-cz * sy), thd[0] * (-cy * sz) + thd[1] * (-cz)},
                     {0.0, thd[0] * (-sy * sz), thd[0] * (cy * cz) + thd[1] * (-sz)},
                     {0.0, thd[0] * (-cy), 0.0}};
  // d(omega_dot)/d(theta): theta_dot * dMdot/dtheta + theta_ddot * dM/dtheta
  double Jwd_th[3][3] = {
      {0.0, thd[0] * (-cy * cz * yd + sy * sz * zd) + thdd[0] * (-cz * sy),
            (thd[0] * (sy * sz * yd - cy * cz * zd) + thd[1] * (sz * zd)) + (thdd[0] * (-cy * sz) + thdd[1] * (-cz))},
      {0.0, thd[0] * (-cy * sz * yd - cz * sy * zd) + thdd[0] * (-sy * sz),
            (thd[0] * (-cz * sy * yd - cy * sz * zd) + thd[1] * (-cz * zd)) + (thdd[0] * (cy * cz) + thdd[1] * (-sz))},
      {0.0, thd[0] * (sy * yd) + thdd[0] * (-cy), 0.0}};
  // d(omega_dot)/d(theta_dot): theta_dot * dMdot/dtheta_dot + Mdot
  double Jwd_thd[3][3] = {{Md[0][0], thd[0] * (-cz * sy) + Md[0][1], thd[0] * (-cy * sz) + thd[1] * (-cz)},
                          {Md[1][0], thd[0] * (-sy * sz) + Md[1][1], thd[0] * (cy * cz) + thd[1] * (-sz)},
                          {Md[2][0], thd[0] * (-cy), 0.0}};

  double v11[3], v21[3], tmp[3];
  MulVec(Rt, omd, tmp); MulVec(Ib, tmp, v11);   // I_b R^T omega_dot
  MulVec(Rt, om, tmp);  MulVec(Ib, tmp, v21);   // I_b R^T omega
  double D11[3][3], D12[3][3], D21[3][3], D22[3][3], T1[3][3], T2[3][3];
  RotVecDerivative<false>(dR, v11, D11); RotVecDerivative<true>(dR, omd, D12);
  RotVecDerivative<false>(dR, v21, D21); RotVecDerivative<true>(dR, om, D22);

  double A[3][3], Bm[3][3], C[3][3];
  // jac1 = D11 + R I_b D12 + I_w d(omega_dot)
  Mul33(RIb, D12, T1); Mul33(Iw, Jwd_th, T2);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int d = 0; d < 3; ++d) A[i][d] = (D11[i][d] + T1[i][d]) + T2[i][d];
  Mul33(Iw, Jwd_thd, Bm);
  Mul33(Iw, M, C);
  // jac2 = [omega]x (D21 + R I_b D22 + I_w d(omega)) - [I_w omega]x d(omega)
  double Gth[3][3], X1[3][3], X2[3][3];
  Mul33(RIb, D22, T1); Mul33(Iw, Jw, T2);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int d = 0; d < 3; ++d) Gth[i][d] = (D21[i][d] + T1[i][d]) + T2[i][d];
  CrossMul(om, Gth, X1); CrossMul(Iw_om, Jw, X2);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int d = 0; d < 3; ++d) A[i][d] += X1[i][d] - X2[i][d];
  CrossMul(om, C, X1); CrossMul(Iw_om, M, X2);   // I_w d(omega)/d(theta_dot) = I_w M = C
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int d = 0; d < 3; ++d) Bm[i][d] += X1[i][d] - X2[i][d];
  // contract with the Hermite basis of the active base-ang polynomial: 3 rows x 12 node values
  const double* bb = P.dyn_ang_basis + 12 * k;
  double bpv[4], bvv[4], bav[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) { bpv[q] = __ldg(bb + q); bvv[q] = __ldg(bb + 4 + q); bav[q] = __ldg(bb + 8 + q); }
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 12; ++j) {
      const int d = j % 3, q = j / 3;
      Sk[3 + i * 12 + j] = fma(C[i][d], bav[q], fma(Bm[i][d], bvv[q], A[i][d] * bpv[q]));
    }
}

// ---- analytic terrains: height_map_examples.cc:35-211 ------------------------
struct TerrainPoint { double h, hx, hy, hxx; };
// HeightMapFromCSV (height_map_from_csv.h:29-111): cell-constant heights, cells of 0.17 m; slope diff/eps on the last
// eps = res/50 before a rising edge and the first eps after a falling edge, 0 elsewhere; outside the grid everything is 0
// (static_cast<size_t>(x / res), :31-32, truncates toward zero: a quotient in (-1, 0) is cell 0, inside the grid; a quotient
// <= -1 or NaN converts to a huge cell index, i.e. "outside").
// the height grids of a batch, by value: the grid terrains are evaluated out of line (EvalGridTerrain), so that their code —
// five bilinear look-ups per point for the grid_map layer — exists once per kernel instead of once per inlined call site
// (RomNodeOut shrank from 12 952 to 8 456 SASS instructions; the step time did not change)
struct GridArgs {
  const double* grid; int grid_rows, grid_cols;
  const float* gmap; int gmap_sx, gmap_sy; double gmap_res, gmap_px, gmap_py;
};
__device__ __forceinline__ bool GridCell(const GridArgs& P, double x, double y, long long* xc, long long* yc) {
  const double res = 0.17;
  const double fx = x / res, fy = y / res;
  if (!(fx > -1.0) || !(fy > -1.0) || !P.grid) return false;
  *xc = (long long)fx; *yc = (long long)fy;
  return *xc < P.grid_cols && *yc < P.grid_rows;
}
__device__ __forceinline__ double GridEdgeSlope(const GridArgs& P, long long c, long long o, bool along_x, double coord) {
  const double res = 0.17, eps = res / 50;
  const long long n = along_x ? P.grid_cols : P.grid_rows;
  auto at = [&](long long k) { return along_x ? __ldg(P.grid + o * P.grid_cols + k) : __ldg(P.grid + k * P.grid_cols + o); };
  if (c + 1 < n) {   // next cell higher: slope just before it
    const double diff_end = at(c + 1) - at(c), end = (double)(c + 1) * res;
    if (diff_end > 0 && coord <= end && coord >= end - eps) return diff_end / eps;
  }
  if (c - 1 >= 0) {  // previous cell higher: slope just after it
    const double diff_start = at(c) - at(c - 1), start = (double)c * res;
    if (diff_start < 0 && coord >= start && coord <= start + eps) return diff_start / eps;
  }
  return 0.0;
}
// towr `Grid` (grid_height_map.h:16-59) over grid_map::GridMap::atPosition(layer, p, INTER_LINEAR) (grid_map_core, restated;
// un-vendored dependency): bilinear over the four cell centres around p with double weights stored to FLOAT, nearest cell
// when one of the four is outside, FLT_MAX outside the map; cell (ix, iy) is centred at pos + L/2 - res/2 - res * (ix, iy).
__device__ __forceinline__ void GridMapCentre(const GridArgs& P, int ix, int iy, double* x, double* y) {
  *x = P.gmap_px + (0.5 * (P.gmap_sx * P.gmap_res) - 0.5 * P.gmap_res) + P.gmap_res * (double)(-ix);
  *y = P.gmap_py + (0.5 * (P.gmap_sy * P.gmap_res) - 0.5 * P.gmap_res) + P.gmap_res * (double)(-iy);
}
__device__ __noinline__ float GridMapHeight(const GridArgs& P, double x, double y) {
  const float outside = 3.402823466e+38f;   // std::numeric_limits<float>::max(), grid_height_map.h:43
  if (!P.gmap) return outside;
  const double Lx = P.gmap_sx * P.gmap_res, Ly = P.gmap_sy * P.gmap_res;
  const int ix0 = (int)(-((x - 0.5 * Lx - P.gmap_px) / P.gmap_res)), iy0 = (int)(-((y - 0.5 * Ly - P.gmap_py) / P.gmap_res));
  double cx, cy; GridMapCentre(P, ix0, iy0, &cx, &cy);
  const bool dir = x >= cx, up = y >= cy;
  const int ix1 = dir ? ix0 - 1 : ix0 + 1, iy2 = up ? iy0 - 1 : iy0 + 1;
  // the four cells in grid_map's order after idxShift: f[0] = cell with the smaller x / y centre ... (GridMap.cpp, atPositionLinearInterpolated)
  const int cxs[4] = {ix0, ix1, ix0, ix1}, cys[4] = {iy0, iy0, iy2, iy2};
  int sh[4];
  if (up) { if (dir) { sh[0] = 0; sh[1] = 1; sh[2] = 2; sh[3] = 3; } else { sh[0] = 1; sh[1] = 0; sh[2] = 3; sh[3] = 2; } }
  else    { if (dir) { sh[0] = 2; sh[1] = 3; sh[2] = 0; sh[3] = 1; } else { sh[0] = 3; sh[1] = 2; sh[2] = 1; sh[3] = 0; } }
  const unsigned long long buffer = (unsigned long long)P.gmap_sx * P.gmap_sy;
  float f[4]; bool ok = true;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const unsigned long long lin = (unsigned long long)((long long)cys[sh[i]] * P.gmap_sx + cxs[sh[i]]);   // column-major linear index in size_t, as grid_map
    if (lin >= buffer) { ok = false; f[i] = 0.0f; }
    else f[i] = __ldg(P.gmap + (lin % (unsigned long long)P.gmap_sx) * P.gmap_sy + lin / (unsigned long long)P.gmap_sx);
  }
  if (ok) {
    GridMapCentre(P, cxs[sh[0]], cys[sh[0]], &cx, &cy);
    const double rx = (x - cx) / P.gmap_res, ry = (y - cy) / P.gmap_res, fx = 1.0 - rx, fy = 1.0 - ry;
    return (float)(f[0] * fx * fy + f[1] * rx * fy + f[2] * fx * ry + f[3] * rx * ry);
  }
  const double tx = -(x - P.gmap_px - 0.5 * Lx), ty = -(y - P.gmap_py - 0.5 * Ly);   // checkIfPositionWithinMap + checkIfIndexInRange
  if (tx >= 0.0 && ty >= 0.0 && tx < Lx && ty < Ly && ix0 >= 0 && iy0 >= 0 && ix0 < P.gmap_sx && iy0 < P.gmap_sy)
    return __ldg(P.gmap + (size_t)ix0 * P.gmap_sy + iy0);
  return outside;
}
__device__ __noinline__ TerrainPoint EvalGridTerrain(const GridArgs P, int id, double x, double y) {
  TerrainPoint o{0.0, 0.0, 0.0, 0.0};
  switch (id) {
    case 8: {  // Grid (grid_map elevation layer), grid_height_map.h:29-60: float heights, central differences with eps = res / 6
      const double eps = P.gmap_res / 6.0;
      o.h = (double)GridMapHeight(P, x, y);
      o.hx = (double)(GridMapHeight(P, x + eps, y) - GridMapHeight(P, x - eps, y)) / (2 * eps);
      o.hy = (double)(GridMapHeight(P, x, y + eps) - GridMapHeight(P, x, y - eps)) / (2 * eps);
      break; }
    case 7: {  // Grid (CSV)
      long long xc, yc;
      if (GridCell(P, x, y, &xc, &yc)) {
        o.h = __ldg(P.grid + yc * P.grid_cols + xc);
        o.hx = GridEdgeSlope(P, xc, yc, true, x);
        o.hy = GridEdgeSlope(P, yc, xc, false, y);
      }
      break; }
    default: break;
  }
  return o;
}
__device__ __forceinline__ TerrainPoint EvalTerrain(const Plan& P, int id, double x, double y) {
  if (id >= 7) return EvalGridTerrain(GridArgs{P.grid, P.grid_rows, P.grid_cols, P.gmap, P.gmap_sx, P.gmap_sy, P.gmap_res, P.gmap_px, P.gmap_py}, id, x, y);
  TerrainPoint o{0.0, 0.0, 0.0, 0.0};
  switch (id) {
    case 1: {  // Block
      const double start = 0.7, eps = 0.03, len = 3.5, height = 0.5; const double slope = height / eps;
      if (start <= x && x <= start + eps) { o.h = slope * (x - start); o.hx = slope; }
      if (start + eps <= x && x <= start + len) o.h = height;
      break; }
    case 2:  // Stairs
      if (x >= 1.0) o.h = 0.2;
      if (x >= 1.0 + 0.4) o.h = 0.4;
      if (x >= 1.0 + 0.4 + 1.0) o.h = 0.0;
      break;
    case 3: {  // Gap
      const double gs = 1.0, w = 0.5, hh = 1.5; const double xc = gs + w / 2.0;
      const double a = (4 * hh) / (w * w), b = -(8 * hh * xc) / (w * w), c = -(hh * (w - 2 * xc) * (w + 2 * xc)) / (w * w);
      if (gs <= x && x <= gs + w) { o.h = a * x * x + b * x + c; o.hx = 2 * a * x + b; o.hxx = 2 * a; }
      break; }
    case 4: {  // Slope
      const double s0 = 1.0, up = 1.0, down = 1.0, hc = 0.7; const double slope = hc / up;
      if (x >= s0) { o.h = slope * (x - s0); o.hx = slope; }
      if (x >= s0 + up) { o.h = hc - slope * (x - (s0 + up)); o.hx = -slope; }
      if (x >= (s0 + up) + down) { o.h = 0.0; o.hx = 0.0; }
      break; }
    case 5:  // Chimney
      if (1.0 <= x && x <= 1.0 + 1.5) { o.h = 3.0 * (y - 0.5); o.hy = 3.0; }
      break;
    case 6:  // ChimneyLR
      if (0.5 <= x && x <= 0.5 + 1.0) { o.h = 2.0 * (y - 0.5); o.hy = 2.0; }
      if (0.5 + 1.0 <= x && x <= 0.5 + 2 * 1.0) { o.h = -2.0 * (y + 0.5); o.hy = -2.0; }
      break;
    default: break;  // FlatGround(0.0)
  }
  return o;
}

// TerrainConstraint, terrain_constraint.cc:59-108.  Sk: {-dh/dx, -dh/dy}; gk: the constraint value
__device__ __forceinline__ void TerrainUnitEval(const Plan& P, const TerrainUnit& u, int terrain, const ConstCol xs, const Col Sk, const Col gk) {
  const double px = xs[u.xi[0]], py = xs[u.xi[1]], pz = xs[u.xi[2]];
  const TerrainPoint tp = EvalTerrain(P, terrain, px, py);
  gk[0] = pz - tp.h;
  Sk[0] = -tp.hx; Sk[1] = -tp.hy;
}

// normalised vector and HeightMap::GetDerivativeOfNormalizedBasisWrt (height_map.cc:62-91,140-146):
// out[i] = (1/|v|^2 * (|v| * delta(i,dim) - v[dim] * v_hat[i])) * dv[i]   (element-wise, as the reference)
__device__ __forceinline__ void Normalize(const double v[3], double vh[3], double* sn, double* nrm) {
  *sn = v[0] * v[0] + v[1] * v[1] + v[2] * v[2]; *nrm = sqrt(*sn);
  vh[0] = v[0] / *nrm; vh[1] = v[1] / *nrm; vh[2] = v[2] / *nrm;
}
__device__ __forceinline__ void NormalizedDeriv(const double v[3], const double vh[3], double sn, double nrm, int dim,
                                                const double dv[3], double out[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double unit = (i == dim) ? 1.0 : 0.0;
    out[i] = (1 / sn * (nrm * unit - v[dim] * vh[i])) * dv[i];
  }
}
__device__ __forceinline__ double Dot3(const double a[3], const double b[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

// ForceConstraint, force_constraint.cc:64-171.  Su: 25 Jacobian values; gr: the 5 constraint values
__device__ __forceinline__ void ForceUnitEval(const Plan& P, const ForceUnit& u, int terrain, const ConstCol xs, const Col Su, const Col gr) {
  const double mu = P.mu;
  const double px = xs[u.xp[0]], py = xs[u.xp[1]];
  const double f[3] = {xs[u.xf[0]], xs[u.xf[1]], xs[u.xf[2]]};
  const TerrainPoint tp = EvalTerrain(P, terrain, px, py);
  // HeightMap::GetNormal / GetTangent1 / GetTangent2, height_map.cc:93-138
  const double vn[3] = {-tp.hx, -tp.hy, 1.0}, vt1[3] = {1.0, 0.0, tp.hx}, vt2[3] = {0.0, 1.0, tp.hy};
  double n[3], t1[3], t2[3], sn_n, nr_n, sn_1, nr_1, sn_2, nr_2;
  Normalize(vn, n, &sn_n, &nr_n); Normalize(vt1, t1, &sn_1, &nr_1); Normalize(vt2, t2, &sn_2, &nr_2);
  double a1[3], b1[3], a2[3], b2[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    a1[d] = t1[d] - mu * n[d]; b1[d] = t1[d] + mu * n[d];
    a2[d] = t2[d] - mu * n[d]; b2[d] = t2[d] + mu * n[d];
  }
  gr[0] = Dot3(f, n); gr[1] = Dot3(f, a1); gr[2] = Dot3(f, b1); gr[3] = Dot3(f, a2); gr[4] = Dot3(f, b2);
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    Su[0 * 5 + 2 + d] = n[d]; Su[1 * 5 + 2 + d] = a1[d]; Su[2 * 5 + 2 + d] = b1[d];
    Su[3 * 5 + 2 + d] = a2[d]; Su[4 * 5 + 2 + d] = b2[d];
  }
  // second derivatives of the height: only d2h/dx2 exists in the analytic terrains
#pragma unroll
  for (int dim = 0; dim < 2; ++dim) {
    const double hxd = (dim == 0) ? tp.hxx : 0.0;   // d2h/(dx ddim)
    const double hyd = 0.0;                          // d2h/(dy ddim)
    const double dvn[3] = {-hxd, -hyd, 0.0}, dvt1[3] = {0.0, 0.0, hxd}, dvt2[3] = {0.0, 0.0, hyd};
    double dn[3], dt1[3], dt2[3];
    NormalizedDeriv(vn, n, sn_n, nr_n, dim, dvn, dn);
    NormalizedDeriv(vt1, t1, sn_1, nr_1, dim, dvt1, dt1);
    NormalizedDeriv(vt2, t2, sn_2, nr_2, dim, dvt2, dt2);
    double m1[3], p1[3], m2[3], p2[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      m1[d] = dt1[d] - mu * dn[d]; p1[d] = dt1[d] + mu * dn[d];
      m2[d] = dt2[d] - mu * dn[d]; p2[d] = dt2[d] + mu * dn[d];
    }
    Su[0 * 5 + dim] = Dot3(f, dn); Su[1 * 5 + dim] = Dot3(f, m1); Su[2 * 5 + dim] = Dot3(f, p1);
    Su[3 * 5 + dim] = Dot3(f, m2); Su[4 * 5 + dim] = Dot3(f, p2);
  }
}

// SwingConstraint::GetValues, swing_constraint.cc:57-83 (Jacobian is constant)
__device__ __forceinline__ void SwingUnitEval(const SwingUnit& u, const ConstCol xs, const Col gk) {
  const double t_swing_avg = 0.3;
#pragma unroll
  for (int d = 0; d < 2; ++d) {
    const double prev = xs[u.xprev[d]], next = xs[u.xnext[d]];
    const double dist = next - prev;
    const double center = prev + 0.5 * dist;
    const double des_vel = dist / t_swing_avg;
    gk[2 * d] = xs[u.xc_p[d]] - center;
    gk[2 * d + 1] = xs[u.xc_v[d]] - des_vel;
  }
}

// SplineAccConstraint::GetValues, spline_acc_constraint.cc:49-65 (Jacobian constant for fixed durations)
__device__ __forceinline__ void AccUnitEval(const AccUnit& u, const ConstCol xs, const Col gk) {
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const double p0 = xs[u.x0 + d], v0 = xs[u.x0 + 3 + d], p1 = xs[u.x0 + 6 + d], v1 = xs[u.x0 + 9 + d];
    const double p2 = xs[u.x0 + 12 + d], v2 = xs[u.x0 + 15 + d];
    const double Cp = DivExact(-(3 * (p0 - p1) + u.Tp * (2 * v0 + v1)), u.Tp2, u.rTp2);
    const double Dp = DivExact(2 * (p0 - p1) + u.Tp * (v0 + v1), u.Tp3, u.rTp3);
    const double Cn = DivExact(-(3 * (p1 - p2) + u.Tn * (2 * v1 + v2)), u.Tn2, u.rTn2);
    const double a_prev = 2 * Cp + (6 * u.Tp) * Dp;
    const double a_next = 2 * Cn;
    gk[d] = a_prev - a_next;
  }
}

// BaseMotionConstraint::UpdateConstraintAtInstance, base_motion_constraint.cc:56-66: rows AX.. = base-ang, LX.. = base-lin position
__device__ __forceinline__ void BaseMotionUnitEval(const Plan& P, const BaseMotionUnit& u, const ConstCol xs, const Col gk) {
  double lin[3], ang[3], unused[3];
  EvalSpline<0>(P, P.samples + u.sample_lin, xs, lin, unused, unused);
  EvalSpline<0>(P, P.samples + u.sample_ang, xs, ang, unused, unused);
#pragma unroll
  for (int d = 0; d < 3; ++d) { gk[d] = ang[d]; gk[3 + d] = lin[d]; }
}

// ---- PhaseSplines: what the Jacobian needs beyond the value (optimised phase durations only) ------------------
// Everything a PhaseSpline contributes at one sample: value, velocity, the four Hermite basis values of the active
// polynomial (polynomial.cc:106-234), d(pos)/d(phase duration) (polynomial.cc:236-257, phase_spline.cc:77-93) and
// the phase the sample falls into (phase_durations.cc:122-154).
struct PhaseFull {
  const PhasePoly* pp;
  double B[2][2];          // [side][node derivative]: d(pos)/d(node value)
  double pos[3], vel[3], dxdT[3];
  int cur, n_phases;       // current phase, number of phases
  int poly;                // active polynomial
};
__device__ __forceinline__ PhaseFull EvalPhaseFull(const Plan& P, int def_index, double tg, const ConstCol xs) {
  const PhaseSplineDef def = P.phase_defs[def_index];
  const PhaseLoc L = LocatePhasePoly(P, def, tg, xs);
  PhaseFull o; o.pp = P.phase_polys + def.poly0 + L.poly; o.n_phases = def.n_phases; o.poly = L.poly;
  const double T = L.T, T2 = T * T, T3 = Pow3(T), T4 = Pow4(T), t = L.tl, t2 = t * t, t3 = Pow3(t);
  // every x / T^k below is the correctly rounded quotient: DivExact seeded with the correctly rounded reciprocal
  const double rT = 1.0 / T, rT2 = 1.0 / T2, rT3 = 1.0 / T3, rT4 = 1.0 / T4;
  const double q23 = DivExact(2 * t3, T3, rT3), q32 = DivExact(3 * t2, T2, rT2), q32b = DivExact(t3, T2, rT2);
  o.B[0][0] = q23 - q32 + 1; o.B[0][1] = t - DivExact(2 * t2, T, rT) + q32b;
  o.B[1][0] = q32 - q23;     o.B[1][1] = q32b - DivExact(t2, T, rT);
  const double inner = 1. / (double)o.pp->n_in_phase, prev = (double)o.pp->k_in_phase;
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const double x0 = xs[o.pp->xi[d]], v0 = xs[o.pp->xi[3 + d]], x1 = xs[o.pp->xi[6 + d]], v1 = xs[o.pp->xi[9 + d]];
    const double C = DivExact(-(3 * (x0 - x1) + T * (2 * v0 + v1)), T2, rT2);
    const double D = DivExact(2 * (x0 - x1) + T * (v0 + v1), T3, rT3);
    o.pos[d] = ((x0 + t * v0) + t2 * C) + t3 * D;
    o.vel[d] = (v0 + (2 * t) * C) + (3 * t2) * D;
    const double dT = DivExact(t3 * (v0 + v1), T3, rT3) - DivExact(t2 * (2 * v0 + v1), T2, rT2) -
                      DivExact(3 * t3 * (2 * x0 - 2 * x1 + T * v0 + T * v1), T4, rT4) +
                      DivExact(2 * t2 * (3 * x0 - 3 * x1 + 2 * T * v0 + T * v1), T3, rT3);
    o.dxdT[d] = inner * (dT - prev * o.vel[d]);
  }
  o.cur = L.cur;   // Spline::GetSegmentID over the PHASE durations
  return o;
}
// column `ph` of PhaseDurations::GetJacobianOfPos (phase_durations.cc:122-154)
__device__ __forceinline__ void DurationColumn(const PhaseFull& f, int ph, double col[3]) {
  const bool in_last = f.cur == f.n_phases - 1;
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    double v = 0.0;
    if (!in_last && ph == f.cur) v = f.dxdT[d];
    else if (ph < f.cur) { v = -1 * f.vel[d]; if (in_last) v = v - f.dxdT[d]; }
    col[d] = v;
  }
}
// The two non-zero shapes of a duration column (DurationColumn above): U for the columns of earlier phases (ph < cur),
// V for the column of the current phase (zero when the sample lies in the last phase)
__device__ __forceinline__ void DurationVectors(const PhaseFull& f, double U[3], double V[3]) {
  if (f.cur >= 1) DurationColumn(f, f.cur - 1, U); else { U[0] = U[1] = U[2] = 0.0; }
  DurationColumn(f, f.cur, V);
}
// info block of a PhaseSpline at one sample (device_tables.h: PhaseExt), rows `info`..`info + kInfoRows - 1` of the warp's
// state block `t`; called by all 32 lanes (lane = instance)
__device__ __forceinline__ void StorePhaseInfo(const PhaseFull& f, double* t, int info, int lane) {
  int* pi = reinterpret_cast<int*>(t + info * kLD);
  pi[lane] = f.poly;
  const int pmin = __reduce_min_sync(0xffffffffu, f.poly), pmax = __reduce_max_sync(0xffffffffu, f.poly);
  if (lane == 0) { pi[32] = pmin; pi[33] = pmax; }
  double* r = t + (info + 1) * kLD + lane;
  const double b00 = f.B[0][0], b01 = f.B[0][1], b10 = f.B[1][0], b11 = f.B[1][1];
  if (pmax - pmin <= 2) {   // window form: weights of the nodes pmin .. pmin + 3
#pragma unroll
    for (int k = 0; k < 9; ++k) r[k * kLD] = 0.0;
    double* w = r + (1 + 2 * (f.poly - pmin)) * kLD;   // this instance's polynomial joins the nodes P (side 0) and P + 1 (side 1)
    w[0] = b00; w[kLD] = b01; w[2 * kLD] = b10; w[3 * kLD] = b11;
  } else {                  // table form
    r[0] = 0.0; r[kLD] = b10; r[2 * kLD] = b00; r[3 * kLD] = 0.0; r[4 * kLD] = b11; r[5 * kLD] = b01; r[6 * kLD] = 0.0;
    r[7 * kLD] = b10; r[8 * kLD] = b00 + b10; r[9 * kLD] = b00; r[10 * kLD] = 0.0;
  }
}
// Current phase of the foot (the same for its ee-motion and ee-force splines: integers 34.. of the ee-motion info block's
// first row) and the duration columns of `kRows` constraint rows: U (columns of earlier phases) into rows u0 .., then X —
// window form (the current phase differs by less than kWin over the tile): the finished columns cmin, cmin + 1, ..; else V.
template <int kRows, int kWin>
__device__ __forceinline__ void StorePhaseDurations(int cur, const double* U, const double* V, double* t, int info, int u0, int lane) {
  int* pi = reinterpret_cast<int*>(t + info * kLD);
  pi[34 + lane] = cur;
  const int cmin = __reduce_min_sync(0xffffffffu, cur), cmax = __reduce_max_sync(0xffffffffu, cur);
  if (lane == 0) { pi[66] = cmin; pi[67] = cmax; }
#pragma unroll
  for (int r = 0; r < kRows; ++r) t[(u0 + r) * kLD + lane] = U[r];
  if (cmax - cmin < kWin) {
#pragma unroll
    for (int w = 0; w < kWin; ++w) {
      const int ph = cmin + w;
#pragma unroll
      for (int r = 0; r < kRows; ++r) t[(u0 + kRows * (1 + w) + r) * kLD + lane] = ph < cur ? U[r] : ph == cur ? V[r] : 0.0;
    }
  } else {
#pragma unroll
    for (int r = 0; r < kRows; ++r) t[(u0 + kRows + r) * kLD + lane] = V[r];
  }
}
// C = Cross(v) of single_rigid_body_dynamics.cc:46-57
__device__ __forceinline__ void CrossMatrix(const double v[3], double C[3][3]) {
  C[0][0] = 0.0;   C[0][1] = -v[2]; C[0][2] = v[1];
  C[1][0] = v[2];  C[1][1] = 0.0;   C[1][2] = -v[0];
  C[2][0] = -v[1]; C[2][1] = v[0];  C[2][2] = 0.0;
}

// ---- kernels ---------------------------------------------------------------------
// ---- instances <-> (tile, lane) ----------------------------------------------------------------------------------------
// A tile is the set of 32 instances one warp serves (lane = instance).  When the Jacobian-value row length is not a multiple
// of 4 doubles, the rows of consecutive instances start at different offsets inside their 32-byte sectors: nc = 2 or 4
// alignment classes, instance b belongs to class b mod nc.  The tiles are then INTERLEAVED: tile nc G + q holds the
// instances 32 nc G + nc lane + q, i.e. 32 instances of ONE class, so that a whole tile is written from one pair list
// (one sector layout) with the same store loop as an aligned problem — the instance stride is nc rows.  nc = 1: tile t =
// instances 32 t .. 32 t + 31.  XT, GT and the scratch matrices are indexed by (tile, lane).
__device__ __forceinline__ int TileInstance(int nc, int tile, int lane) {
  return nc == 1 ? tile * 32 + lane : (tile / nc) * (32 * nc) + lane * nc + tile % nc;
}
__device__ __forceinline__ int TileCount(int nc, int tile, int nb) {   // valid lanes of the tile (a prefix)
  if (nc == 1) return max(0, min(32, nb - tile * 32));
  const int first = TileInstance(nc, tile, 0);
  return first >= nb ? 0 : min(32, (nb - first + nc - 1) / nc);
}
// column (tile, lane) of a tiled matrix with `rows` rows: element r lives at base[(tile * rows + r) * 32 + lane]
__device__ __forceinline__ ConstCol TileCol(const double* base, int tile, int lane, int rows) {
  return ConstCol{base + ((size_t)tile * rows) * 32 + lane};
}
// the same for instance b (kernels that are not organised by tiles)
__device__ __forceinline__ ConstCol TiledCol(const double* base, int b, int rows, int nc) {
  const int grp = b / (32 * nc), rem = b - grp * (32 * nc);
  return TileCol(base, grp * nc + rem % nc, rem / nc, rows);
}

// x[b][i] -> XT[tile][i][lane]: 32x32 tiles through shared memory, coalesced on both sides; clears status.  A CTA moves
// kTinTiles consecutive column tiles: all their loads are issued before the barrier (more bytes in flight per thread, fewer
// waves of CTAs for this short, latency-bound kernel that everything else waits for).
#ifndef TWB_TIN_TILES
#define TWB_TIN_TILES 1
#endif
constexpr int kTinTiles = TWB_TIN_TILES;
__global__ void __launch_bounds__(256) TransposeIn(const double* __restrict__ x, double* __restrict__ XT,
                                                   int* __restrict__ status, int n, int nb, int nc) {
  __shared__ double tile[kTinTiles][32][33];
#if TWB_PDL
  asm volatile("griddepcontrol.launch_dependents;");   // the dependent output kernel may become resident while this grid drains
#endif
  if (status && blockIdx.x == 0 && threadIdx.y == 0 && TileInstance(nc, blockIdx.y, threadIdx.x) < nb) status[TileInstance(nc, blockIdx.y, threadIdx.x)] = 0;
#pragma unroll
  for (int c = 0; c < kTinTiles; ++c) {
    const int i0 = (blockIdx.x * kTinTiles + c) * 32;
#pragma unroll
    for (int r = threadIdx.y; r < 32; r += 8) {
      const int b = TileInstance(nc, blockIdx.y, r), i = i0 + threadIdx.x;
      if (b < nb && i < n) tile[c][r][threadIdx.x] = __ldcs(x + (size_t)b * n + i);
    }
  }
  __syncthreads();
  double* dst = XT + ((size_t)blockIdx.y * (n + 1)) * 32;
  const int b = TileInstance(nc, blockIdx.y, threadIdx.x);
#pragma unroll
  for (int c = 0; c < kTinTiles; ++c) {
    const int i0 = (blockIdx.x * kTinTiles + c) * 32;
#pragma unroll
    for (int r = threadIdx.y; r < 32; r += 8) {
      const int i = i0 + r;
#if TWB_XT_EVICT_LAST
      if (b < nb && i < n) {
        unsigned long long pol;
        asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
        asm volatile("st.global.L2::cache_hint.f64 [%0], %1, %2;" ::"l"(dst + (size_t)i * 32 + threadIdx.x), "d"(tile[c][threadIdx.x][r]), "l"(pol) : "memory");
      }
#else
      if (b < nb && i < n) dst[(size_t)i * 32 + threadIdx.x] = tile[c][threadIdx.x][r];
#endif
    }
  }
}

// Persistent variant (TWB_TIN_PERSIST = CTAs per SM, 0 = the kernel above): a fixed grid of 148 x 8 CTAs walks the 32 x 32 tiles; the
// loads of a CTA's next tile are issued before the stores of the current one, and no CTA launch sits between the two.  Measured
// (config 2, one box): 8.2 us instead of 12.3 us for the kernel, 127.1 instead of 131.5 us per step (6 / 4 CTAs per SM: 127.7 / 128.8 us).
#ifndef TWB_TIN_PERSIST
#define TWB_TIN_PERSIST 8
#endif
__global__ void __launch_bounds__(256) TransposeInP(const double* __restrict__ x, double* __restrict__ XT, int* __restrict__ status, int n, int nb,
                                                    int nc, int n_ctiles, int total) {
  __shared__ double tile[32][33];
#if TWB_PDL
  asm volatile("griddepcontrol.launch_dependents;");
#endif
  const int tx = threadIdx.x, ty = threadIdx.y;
  double v[4];
  auto load = [&](int t) {
    const int it = t / n_ctiles, ct = t - it * n_ctiles, i = ct * 32 + tx;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int b = TileInstance(nc, it, ty + 8 * k);
      v[k] = (b < nb && i < n) ? __ldcs(x + (size_t)b * n + i) : 0.0;
    }
  };
  int t = blockIdx.x;
  if (t < total) load(t);
  for (; t < total; t += gridDim.x) {
    const int it = t / n_ctiles, ct = t - it * n_ctiles;
    const int b = TileInstance(nc, it, tx);
    if (status && ct == 0 && ty == 0 && b < nb) status[b] = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) tile[ty + 8 * k][tx] = v[k];
    __syncthreads();
    if (t + (int)gridDim.x < total) load(t + gridDim.x);
    double* dst = XT + ((size_t)it * (n + 1)) * 32;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = ct * 32 + ty + 8 * k;
      if (b < nb && i < n) dst[(size_t)i * 32 + tx] = tile[tx][ty + 8 * k];
    }
    __syncthreads();
  }
}

// GT[b/32][r][b%32] -> g[b][r]: 32x32 tiles through shared memory, coalesced on both sides
// TWB_DISCARD: GT is dead once it has been read, and so is XT (rows 0 .. n-1; row n is the permanent zero row) — both
// are still dirty in the L2; `discard.global.L2` drops the lines instead of writing them back to HBM (50 MB per step
// on config 2, 9 % of the step's DRAM writes).  Both matrices are rewritten by the next evaluation before they are read.
__device__ __forceinline__ void DiscardLine(const void* p) { asm volatile("discard.global.L2 [%0], 128;" ::"l"(p) : "memory"); }
// Experiment (TWB_XT_DROP=1): without TransposeOut (direct constraint values) the LAST output CTA of a tile drops the tile's XT lines: every output CTA
// counts itself on the tile's counter when it is done; the one that completes the count discards rows 0 .. n-1 (row n is the
// permanent zero row; a ragged tile keeps its lines: its padded lanes are never rewritten) and resets the counter.
// Measured (config 2, one box): 137.3 us per step with the counters against 132.1 us without — the atomics and the extra CTA
// barriers cost more than the 21 MB of XT write-back they save.  Off.
#ifndef TWB_XT_DROP
#define TWB_XT_DROP 0
#endif
__device__ __forceinline__ void TileDone(int* __restrict__ tile_done, int total, const double* __restrict__ XT, int n, int nc, int tile, int nb) {
#if TWB_XT_DROP
  if (!tile_done) return;
  __shared__ int last;
  __syncthreads();   // every thread of the CTA is past its reads of XT
  if (threadIdx.x == 0) last = (atomicAdd(tile_done + tile, 1) == total - 1);
  __syncthreads();
  if (!last) return;
  if (threadIdx.x == 0) tile_done[tile] = 0;
  if (TileCount(nc, tile, nb) != 32) return;
  const double* xt = XT + ((size_t)tile * (n + 1)) * 32;
  for (int l = threadIdx.x; l < 2 * n; l += blockDim.x) DiscardLine(xt + (size_t)l * 16);
#endif
}
__global__ void __launch_bounds__(256) TransposeOut(const double* __restrict__ GT, double* __restrict__ g, int m, int nb,
                                                    const double* __restrict__ XT, int n, int nc) {
  __shared__ double tile[32][33];
  const int r0 = blockIdx.x * 32;
  const double* src = GT + ((size_t)blockIdx.y * m) * 32;
#pragma unroll
  for (int q = threadIdx.y; q < 32; q += 8) {
    const int r = r0 + q;
#if TWB_TOUT_LD == 1
    if (r < m) tile[q][threadIdx.x] = __ldcg(src + (size_t)r * 32 + threadIdx.x);
#elif TWB_TOUT_LD == 2
    if (r < m) tile[q][threadIdx.x] = src[(size_t)r * 32 + threadIdx.x];
#elif TWB_TOUT_LD == 3
    if (r < m) tile[q][threadIdx.x] = __ldlu(src + (size_t)r * 32 + threadIdx.x);
#else
    if (r < m) tile[q][threadIdx.x] = __ldcs(src + (size_t)r * 32 + threadIdx.x);
#endif
  }
  __syncthreads();
#if TWB_DISCARD
  {
    const int tid = threadIdx.y * 32 + threadIdx.x;
    if (tid < 64) {                       // the 32 GT rows of this CTA: two 128-byte lines each
      const int r = r0 + (tid >> 1);
      if (r < m) DiscardLine(src + (size_t)r * 32 + (tid & 1) * 16);
    } else if (XT && tid < 128 && TileCount(nc, blockIdx.y, nb) == 32) {   // XT rows of this tile, 32 per CTA of the tile (CTAs wrap around when m < n); a ragged last tile keeps its lines: its padded lanes are never rewritten
      const double* xt = XT + ((size_t)blockIdx.y * (n + 1)) * 32;
      for (int r = r0 + ((tid - 64) >> 1); r < n; r += gridDim.x * 32) DiscardLine(xt + (size_t)r * 32 + (tid & 1) * 16);
    }
  }
#endif
#pragma unroll
  for (int q = threadIdx.y; q < 32; q += 8) {
    const int b = TileInstance(nc, blockIdx.y, q), r = r0 + threadIdx.x;
    if (b < nb && r < m) StoreOut(g + (size_t)b * m + r, tile[threadIdx.x][q]);
  }
}

// ---- CTA-collective output: threads switch from "instance" to "pair of output elements" ----------------------
// out[j][off + h] = t[d_h][j] * c_h for the lanes j < n_inst of the tile; `t` is the CTA's shared memory (all state
// blocks), `out` points at element 0 of the tile's first instance, `stride` is the distance between the rows of consecutive
// lanes (nc rows of nnz elements).  The list holds whole 32-byte sectors (two consecutive pairs = two adjacent lanes); thread `tid` of
// `n_threads` takes the pairs tid, tid + n_threads, ..
__device__ __forceinline__ void LoadPair(const OutPair* __restrict__ pairs, const OutCoef* __restrict__ coefs, int i, int n,
                                         int* off, int* d0, int* d1, double* c0, double* c1) {
  if (i < n) {
    const uint2 raw = __ldg(reinterpret_cast<const uint2*>(pairs) + i);
    const double2 c = __ldg(reinterpret_cast<const double2*>(coefs) + i);
    *off = (int)raw.x; *d0 = (int)(raw.y & 0xFFFFu); *d1 = (int)(raw.y >> 16); *c0 = c.x; *c1 = c.y;
  }
}
__device__ __forceinline__ void StorePairs(const double* t, const OutPair* __restrict__ pairs, const OutCoef* __restrict__ coefs,
                                           int n_pairs, double* __restrict__ out, size_t stride, int n_inst,
                                           int tid, int n_threads) {
#if TWB_ST256
  if (n_inst == 32 && (reinterpret_cast<uintptr_t>(out) & 31) == 0 && (stride & 3) == 0) {
    // thread = whole 32-byte sector (the list holds two consecutive pairs per sector), item = (sector, quarter of the tile's
    // instances): one 256-bit store per instance, a warp instruction covers 1 KB of the instance's row
    const int n_sec = n_pairs >> 1, n_items = 4 * n_sec;
    for (int i = tid; i < n_items; i += n_threads) {
      const int qd = i / n_sec, k = i - qd * n_sec;
      int off = 0, d0 = 0, d1 = 0, off2 = 0, d2 = 0, d3 = 0; double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
      LoadPair(pairs, coefs, 2 * k, n_pairs, &off, &d0, &d1, &c0, &c1);
      LoadPair(pairs, coefs, 2 * k + 1, n_pairs, &off2, &d2, &d3, &c2, &c3);
      const int jb = 8 * qd;
      double* o = out + off + (size_t)jb * stride;
      const double* r0 = t + d0 * kLD + jb; const double* r1 = t + d1 * kLD + jb;
      const double* r2 = t + d2 * kLD + jb; const double* r3 = t + d3 * kLD + jb;
#pragma unroll
      for (int j = 0; j < 8; j += 2) {
        const double2 a = *reinterpret_cast<const double2*>(r0 + j), b = *reinterpret_cast<const double2*>(r1 + j);
        const double2 c = *reinterpret_cast<const double2*>(r2 + j), d = *reinterpret_cast<const double2*>(r3 + j);
        StoreOut4(o, a.x * c0, b.x * c1, c.x * c2, d.x * c3); o += stride;
        StoreOut4(o, a.y * c0, b.y * c1, c.y * c2, d.y * c3); o += stride;
      }
    }
    return;
  }
#endif
  if (n_inst == 32) {
    // Work items are (pair, half of the tile's instances): twice as many items as pairs keep the threads of a CTA
    // evenly busy when a list is only 1 - 2 pairs per thread long.  Items 0 .. n_pairs-1 are the first 16 instances,
    // n_pairs .. 2 n_pairs-1 the last 16, so consecutive threads still hold consecutive pairs (whole sectors).
    const int n_items = 2 * n_pairs;
    if (tid >= n_items) return;
    int off = 0, d0 = 0, d1 = 0; double c0 = 0.0, c1 = 0.0;
    LoadPair(pairs, coefs, tid < n_pairs ? tid : tid - n_pairs, n_pairs, &off, &d0, &d1, &c0, &c1);
    for (int i = tid; i < n_items; i += n_threads) {
      // prefetch the next entry of this thread under the stores of the current one
      int noff = 0, nd0 = 0, nd1 = 0; double nc0 = 0.0, nc1 = 0.0;
      const int ni = i + n_threads;
      if (ni < n_items) LoadPair(pairs, coefs, ni < n_pairs ? ni : ni - n_pairs, n_pairs, &noff, &nd0, &nd1, &nc0, &nc1);
      const int jb = i < n_pairs ? 0 : 16;
      double* o = out + off + (size_t)jb * stride;
      const double* r0 = t + d0 * kLD + jb; const double* r1 = t + d1 * kLD + jb;   // rows are 16-byte aligned (kLD even)
#pragma unroll
      for (int j = 0; j < 16; j += 2) {
        const double2 a = *reinterpret_cast<const double2*>(r0 + j), b = *reinterpret_cast<const double2*>(r1 + j);
        StoreOut2(o, a.x * c0, b.x * c1); o += stride;
        StoreOut2(o, a.y * c0, b.y * c1); o += stride;
      }
      off = noff; d0 = nd0; d1 = nd1; c0 = nc0; c1 = nc1;
    }
    return;
  }
  if (tid >= n_pairs) return;
  int off = 0, d0 = 0, d1 = 0; double c0 = 0.0, c1 = 0.0;
  LoadPair(pairs, coefs, tid, n_pairs, &off, &d0, &d1, &c0, &c1);
  for (int i = tid; i < n_pairs; i += n_threads) {
    int noff = 0, nd0 = 0, nd1 = 0; double nc0 = 0.0, nc1 = 0.0;
    LoadPair(pairs, coefs, i + n_threads, n_pairs, &noff, &nd0, &nd1, &nc0, &nc1);
    double* o = out + off;
    const double* r0 = t + d0 * kLD; const double* r1 = t + d1 * kLD;
#pragma unroll 4
    for (int j = 0; j < n_inst; ++j) StoreOut2(o + j * stride, r0[j] * c0, r1[j] * c1);   // ragged last tile
    off = noff; d0 = nd0; d1 = nd1; c0 = nc0; c1 = nc1;
  }
}

// ---- TMA store path ---------------------------------------------------------------------------------------------
// A CTA list whose pairs form one contiguous run of the CSR value row (OutList::run_off) is written per instance as ONE
// bulk copy shared -> global (SASS UBLKCP): every warp owns 32 / W instances of the tile, assembles the run of kG of them
// in its staging rows in OUTPUT ORDER (thread = pair: 16-byte shared stores, conflict-free), makes the writes visible to
// the async proxy and lets lane 0 issue the copies.  The TMA engine drains the staging rows while the warp goes on
// (next instances, then the evaluation of the next unit); a row is only refilled after its copy has finished reading.
__device__ __forceinline__ unsigned SmemAddr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void BulkStore(void* gdst, const void* ssrc, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(SmemAddr(ssrc)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void BulkCommit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void BulkWaitRead() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void BulkWaitAll() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void FenceProxyAsync() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
struct Stage { double* base; int cap; };   // staging rows of the CTA (after the state blocks): W x kBuf x kG rows of `cap` doubles (cap even)

__device__ __forceinline__ void StorePairsTma(const double* t, const OutPair* __restrict__ pairs, const OutCoef* __restrict__ coefs, int n_pairs,
                                              int run_off, double* __restrict__ out, size_t stride, int q, int nc, int n_inst, const Stage st) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, W = blockDim.x >> 5, per = 32 / W;
  const int j_end = min(n_inst, (warp + 1) * per);
  double* rows = st.base + (size_t)warp * (TWB_TMA_BUF * TWB_TMA_G) * st.cap;
  const unsigned bytes = (unsigned)n_pairs * 16u;
  if (lane == 0) BulkWaitRead<0>();   // copies of the previous list (issued before the evaluation of this unit) have long finished reading
  __syncwarp();
  int it = 0;
  if (TWB_TMA_G == 2 && nc == 1) {
    for (int j = warp * per; j < j_end; j += 2, ++it) {
      double* b0 = rows + (size_t)(it % TWB_TMA_BUF) * 2 * st.cap; double* b1 = b0 + st.cap;
      if (it >= TWB_TMA_BUF) { if (lane == 0) BulkWaitRead<TWB_TMA_BUF - 1>(); __syncwarp(); }
      for (int i = lane; i < n_pairs; i += 32) {
        int off = 0, d0 = 0, d1 = 0; double c0 = 0.0, c1 = 0.0;
        LoadPair(pairs, coefs, i, n_pairs, &off, &d0, &d1, &c0, &c1);
        const double2 a = *reinterpret_cast<const double2*>(t + d0 * kLD + j), b = *reinterpret_cast<const double2*>(t + d1 * kLD + j);
        const int o = off - run_off;
        *reinterpret_cast<double2*>(b0 + o) = make_double2(a.x * c0, b.x * c1);
        *reinterpret_cast<double2*>(b1 + o) = make_double2(a.y * c0, b.y * c1);
      }
      FenceProxyAsync();
      __syncwarp();
      if (lane == 0) {
        BulkStore(out + (size_t)j * stride + run_off, b0, bytes);
        if (j + 1 < j_end) BulkStore(out + (size_t)(j + 1) * stride + run_off, b1, bytes);
        BulkCommit();
      }
    }
    return;
  }
  constexpr int kSlots = TWB_TMA_BUF * TWB_TMA_G;
  for (int j = warp * per; j < j_end; ++j) {
    if (j % nc != q) continue;
    double* b0 = rows + (size_t)(it % kSlots) * st.cap;
    if (it >= kSlots) { if (lane == 0) BulkWaitRead<kSlots - 1>(); __syncwarp(); }
    ++it;
    for (int i = lane; i < n_pairs; i += 32) {
      int off = 0, d0 = 0, d1 = 0; double c0 = 0.0, c1 = 0.0;
      LoadPair(pairs, coefs, i, n_pairs, &off, &d0, &d1, &c0, &c1);
      *reinterpret_cast<double2*>(b0 + (off - run_off)) = make_double2(t[d0 * kLD + j] * c0, t[d1 * kLD + j] * c1);
    }
    FenceProxyAsync();
    __syncwarp();
    if (lane == 0) { BulkStore(out + (size_t)j * stride + run_off, b0, bytes); BulkCommit(); }
  }
}
// ---- phase elements (device_tables.h: PhaseExt) --------------------------------------------------------------------
// per-instance value of one element whose info block is in TABLE form / whose duration columns are not finished:
// `x` is the element's PhaseExt word, d / c its state row and coefficient
__device__ __forceinline__ double PhaseVal(const double* t, int j, unsigned x, int d, double c, int v_off) {
  const int a = (int)((x >> 8) & 0xFFu), info = (int)(x >> 16);
  const int* pi = reinterpret_cast<const int*>(t + info * kLD);
  if ((x & 3u) == kElemNode) {   // NodeSpline::FillJacobianWrtNodes (node_spline.cc:85-112) for the instance's active polynomial
    const int shared = (int)((x >> 3) & 1u);
    const int tbl = info + (shared ? 7 : 1 + 3 * (int)((x >> 2) & 1u));
    const int idx = min(max(pi[j] - a + 2, 0), 3 + shared);
    return (t[d * kLD + j] * c) * t[(tbl + idx) * kLD + j];
  }
  const int dl = pi[34 + j] - a;   // PhaseDurations::GetJacobianOfPos (phase_durations.cc:122-154): a = the column's phase
  return dl < 0 ? 0.0 : t[(dl > 0 ? d : d + v_off) * kLD + j];
}
// What an element is for the instances of this tile: out = (state[d] * c) * (state[w1] [+ state[w2]]) with rows that are the
// same for every instance (w1 = row 0, the constant 1, for an ordinary element; zero elements become row `zrow` times 0), or
// `slow`: the per-instance selection of PhaseVal.
struct ElemForm { int d, w1, w2; double c; bool slow; };
__device__ __forceinline__ ElemForm Classify(const double* t, unsigned x, int d, double c, int v_off, int dwin, int zrow) {
  ElemForm f{d, 0, -1, c, false};
  const unsigned kind = x & 3u;
  if (kind == kElemPlain) return f;
  const int a = (int)((x >> 8) & 0xFFu), info = (int)(x >> 16);
  const int* pi = reinterpret_cast<const int*>(t + info * kLD);
  if (kind == kElemNode) {
    const int2 mm = *reinterpret_cast<const int2*>(pi + 32);
    const int shared = (int)((x >> 3) & 1u);
    if (mm.y < a - 1 || mm.x > a + shared) { f.d = zrow; f.c = 0.0; return f; }   // no instance's polynomial touches the node(s)
    if (mm.y - mm.x > 2) { f.slow = true; return f; }
    const int s1 = a - mm.x, deriv = (int)((x >> 2) & 1u);
    const bool in1 = s1 >= 0 && s1 <= 3, in2 = shared && s1 + 1 >= 0 && s1 + 1 <= 3;
    if (in1) { f.w1 = info + 2 + 2 * s1 + deriv; if (in2) f.w2 = info + 2 + 2 * (s1 + 1); }
    else if (in2) f.w1 = info + 2 + 2 * (s1 + 1);
    else { f.d = zrow; f.c = 0.0; }
    return f;
  }
  const int2 mm = *reinterpret_cast<const int2*>(pi + 66);
  if (a > mm.y) { f.d = zrow; f.c = 0.0; }
  else if (a < mm.x) { }                                     // a column of an earlier phase for every instance: U
  else if (mm.y - mm.x < dwin) f.d = d + v_off * (1 + a - mm.x);   // finished column
  else f.slow = true;
  return f;
}
__device__ __forceinline__ double FormVal(const double* t, int j, const ElemForm& f, unsigned x, int d, double c, int v_off) {
  if (f.slow) return PhaseVal(t, j, x, d, c, v_off);
  const double w = f.w2 >= 0 ? t[f.w1 * kLD + j] + t[f.w2 * kLD + j] : t[f.w1 * kLD + j];
  return (t[f.d * kLD + j] * f.c) * w;
}
// the pair loop for sectors that hold phase elements: item = (pair, half of the tile's instances) as in StorePairs
__device__ __forceinline__ void StorePhasePairs(const double* t, const OutPair* __restrict__ pairs, const OutCoef* __restrict__ coefs,
                                                const PhaseExt* __restrict__ exts, int n_pairs, double* __restrict__ out, size_t stride,
                                                int n_inst, int v_off, int dwin, int zrow, int tid, int n_threads) {
  const int n_items = 2 * n_pairs;
  if (tid >= n_items) return;
  int noff = 0, nd0 = 0, nd1 = 0; double nc0 = 0.0, nc1 = 0.0; uint2 nx = make_uint2(0u, 0u);
  {
    const int k = tid < n_pairs ? tid : tid - n_pairs;
    LoadPair(pairs, coefs, k, n_pairs, &noff, &nd0, &nd1, &nc0, &nc1);
    nx = __ldg(reinterpret_cast<const uint2*>(exts) + k);
  }
  for (int i = tid; i < n_items; i += n_threads) {
    const int jb = i < n_pairs ? 0 : 16;
    const int off = noff, d0 = nd0, d1 = nd1; const double c0 = nc0, c1 = nc1; const uint2 x = nx;
    const int ni = i + n_threads;   // the next entry of this thread is fetched under the stores of the current one
    if (ni < n_items) {
      const int k = ni < n_pairs ? ni : ni - n_pairs;
      LoadPair(pairs, coefs, k, n_pairs, &noff, &nd0, &nd1, &nc0, &nc1);
      nx = __ldg(reinterpret_cast<const uint2*>(exts) + k);
    }
    double* o = out + off + (size_t)jb * stride;
    const ElemForm f0 = Classify(t, x.x, d0, c0, v_off, dwin, zrow), f1 = Classify(t, x.y, d1, c1, v_off, dwin, zrow);
    if (n_inst == 32 && !f0.slow && !f1.slow) {
      const double* r0 = t + f0.d * kLD + jb; const double* r1 = t + f1.d * kLD + jb;
      if ((f0.w1 | f1.w1) == 0 && f0.c == 0.0 && f1.c == 0.0) {   // zero for every instance of the tile (most phase elements)
#pragma unroll
        for (int j = 0; j < 16; ++j) { StoreOut2(o, 0.0, 0.0); o += stride; }
      } else if ((f0.w1 | f1.w1) == 0) {   // both elements are ordinary for this tile: the pair loop of StorePairs
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
          const double2 a = *reinterpret_cast<const double2*>(r0 + j), b = *reinterpret_cast<const double2*>(r1 + j);
          StoreOut2(o, a.x * f0.c, b.x * f1.c); o += stride;
          StoreOut2(o, a.y * f0.c, b.y * f1.c); o += stride;
        }
      } else if ((f0.w2 & f1.w2) < 0) {   // a weight row each (row 0 = 1 for an ordinary element)
        const double* w0 = t + f0.w1 * kLD + jb; const double* w1 = t + f1.w1 * kLD + jb;
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
          const double2 a = *reinterpret_cast<const double2*>(r0 + j), b = *reinterpret_cast<const double2*>(r1 + j);
          const double2 u = *reinterpret_cast<const double2*>(w0 + j), v = *reinterpret_cast<const double2*>(w1 + j);
          StoreOut2(o, (a.x * f0.c) * u.x, (b.x * f1.c) * v.x); o += stride;
          StoreOut2(o, (a.y * f0.c) * u.y, (b.y * f1.c) * v.y); o += stride;
        }
      } else {                            // shared stance positions: the sum of two weight rows (the zero row where there is none)
        const double* w0 = t + f0.w1 * kLD + jb; const double* w1 = t + f1.w1 * kLD + jb;
        const double* y0 = t + (f0.w2 >= 0 ? f0.w2 : zrow) * kLD + jb; const double* y1 = t + (f1.w2 >= 0 ? f1.w2 : zrow) * kLD + jb;
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
          const double2 a = *reinterpret_cast<const double2*>(r0 + j), b = *reinterpret_cast<const double2*>(r1 + j);
          const double2 u = *reinterpret_cast<const double2*>(w0 + j), v = *reinterpret_cast<const double2*>(w1 + j);
          const double2 p = *reinterpret_cast<const double2*>(y0 + j), r = *reinterpret_cast<const double2*>(y1 + j);
          StoreOut2(o, (a.x * f0.c) * (u.x + p.x), (b.x * f1.c) * (v.x + r.x)); o += stride;
          StoreOut2(o, (a.y * f0.c) * (u.y + p.y), (b.y * f1.c) * (v.y + r.y)); o += stride;
        }
      }
    } else if (n_inst == 32) {
#pragma unroll 4
      for (int j = jb; j < jb + 16; ++j) { StoreOut2(o, FormVal(t, j, f0, x.x, d0, c0, v_off), FormVal(t, j, f1, x.y, d1, c1, v_off)); o += stride; }
    } else {
      for (int j = jb; j < jb + 16; ++j) { if (j < n_inst) StoreOut2(o, FormVal(t, j, f0, x.x, d0, c0, v_off), FormVal(t, j, f1, x.y, d1, c1, v_off)); o += stride; }
    }
  }
}
// Entries handled with lane = instance: fetched with one coalesced load (lane = entry), broadcast with shuffles.
// fn(first, d0, coefficient) is called by every lane of the warp for every entry.
template <class F>
__device__ __forceinline__ void ForEachEntry(const OutPair* __restrict__ pairs, const OutCoef* __restrict__ coefs, int n, int lane, F&& fn) {
  for (int base = 0; base < n; base += 32) {
    uint2 raw = make_uint2(0u, 0u); double c = 0.0;
    if (base + lane < n) { raw = __ldg(reinterpret_cast<const uint2*>(pairs) + base + lane); c = __ldg(reinterpret_cast<const double*>(coefs + base + lane)); }
    const int cnt = min(32, n - base);
    for (int s = 0; s < cnt; ++s)
      fn(__shfl_sync(0xffffffffu, (int)raw.x, s), __shfl_sync(0xffffffffu, (int)(raw.y & 0xFFFFu), s), __shfl_sync(0xffffffffu, c, s));
  }
}
__device__ __forceinline__ OutRange LoadRange(const OutRange* r) {
  const int2 v = __ldg(reinterpret_cast<const int2*>(r)); return OutRange{v.x, v.y};
}
// constraint values of one unit: lane = instance writes GT[row][lane] (instance-tiled, 256 contiguous bytes per row and
// warp); TransposeOut turns the tiles into g[B][m] afterwards.  One unit owns only 3 - 10 constraint values per
// instance — written straight into g[B][m] they would be 8-byte pieces of sectors shared with other units.
__device__ __forceinline__ void StoreValuesTiled(const Plan& P, const double* t, const OutRange* values, double* __restrict__ gt_tile, int lane) {
  const OutRange r = LoadRange(values);
  ForEachEntry(P.pairs + r.first, P.coefs + r.first, r.count, lane,
               [&](int g_row, int d, double c) { gt_tile[(size_t)g_row * 32 + lane] = t[d * kLD + lane] * c; });
}
// Jacobian values of a whole CTA (after its barrier): every thread takes pairs of the CTA's list; warp 0 writes the
// single elements (sectors shared with a neighbouring CTA) with lane = instance.
template <bool kPhase = false>
__device__ __forceinline__ void StoreCta(const Plan& P, const double* cta_smem, const OutList* list, double* __restrict__ jac, int tile, int nb, const Stage st,
                                         int v_off = 0, int dwin = 0, int zrow = 0) {
#ifdef TWB_EXP_NOSTORE   // timing experiment: compute phase only
  return;
#endif
  const int nc = P.nc_jac, lane = threadIdx.x & 31;
  // all instances of the tile belong to alignment class q (interleaved tiles); consecutive lanes are nc rows apart
  const int q = tile % nc, n_inst = TileCount(nc, tile, nb);
  const size_t stride = (size_t)nc * P.nnz;
  double* __restrict__ jac_tile = jac + (size_t)TileInstance(nc, tile, 0) * P.nnz;
  {
    const OutRange rp = LoadRange(&list->pairs[q]);
    // warp 0 also owns the single elements: their range (and, below, their first 32 entries) is fetched BEFORE the pair
    // loop, so that the two dependent loads are in flight under the warp's pair stores instead of after them
    OutRange rs{0, 0};
    if (threadIdx.x < 32) rs = LoadRange(&list->singles[q]);
    uint2 raw = make_uint2(0u, 0u); double cs = 0.0; unsigned xs = 0u;
    if (lane < rs.count) {
      raw = __ldg(reinterpret_cast<const uint2*>(P.pairs + rs.first) + lane); cs = __ldg(reinterpret_cast<const double*>(P.coefs + rs.first + lane));
      if (kPhase) xs = __ldg(reinterpret_cast<const unsigned*>(P.exts + rs.first + lane));
    }
#if TWB_TMA
    const int run_off = __ldg(&list->run_off[q]);
    if (run_off >= 0 && 2 * rp.count <= st.cap && (32 % (blockDim.x >> 5)) == 0)
      StorePairsTma(cta_smem, P.pairs + rp.first, P.coefs + rp.first, rp.count, run_off, jac_tile, stride, 0, 1, n_inst, st);
    else
#endif
    StorePairs(cta_smem, P.pairs + rp.first, P.coefs + rp.first, rp.count, jac_tile, stride, n_inst, threadIdx.x, blockDim.x);
    if (kPhase) {
      const OutRange rq = LoadRange(&list->phase[q]);
      StorePhasePairs(cta_smem, P.pairs + rq.first, P.coefs + rq.first, P.exts + rq.first, rq.count, jac_tile, stride, n_inst, v_off, dwin, zrow,
                      threadIdx.x, blockDim.x);
    }
#ifndef TWB_EXP_NOSINGLES   // (timing experiment, profiles/README.md round 2: what the single-element stores cost)
    if (threadIdx.x < 32 && rs.count > 0) {
      const bool active = lane < n_inst;
      double* o = jac_tile + (size_t)lane * stride;
      const int cnt = min(32, rs.count);
      for (int sidx = 0; sidx < cnt; ++sidx) {
        const int off = __shfl_sync(0xffffffffu, (int)raw.x, sidx), d = __shfl_sync(0xffffffffu, (int)(raw.y & 0xFFFFu), sidx);
        const double c = __shfl_sync(0xffffffffu, cs, sidx);
        const unsigned x = kPhase ? __shfl_sync(0xffffffffu, xs, sidx) : 0u;
        if (active) StoreOut(o + off, kPhase ? FormVal(cta_smem, lane, Classify(cta_smem, x, d, c, v_off, dwin, zrow), x, d, c, v_off) : cta_smem[d * kLD + lane] * c);
      }
      for (int base = 32; base < rs.count; base += 32) {   // (rare) more than 32 single elements
        raw = make_uint2(0u, 0u); cs = 0.0; xs = 0u;
        if (base + lane < rs.count) {
          raw = __ldg(reinterpret_cast<const uint2*>(P.pairs + rs.first + base) + lane); cs = __ldg(reinterpret_cast<const double*>(P.coefs + rs.first + base + lane));
          if (kPhase) xs = __ldg(reinterpret_cast<const unsigned*>(P.exts + rs.first + base + lane));
        }
        const int more = min(32, rs.count - base);
        for (int sidx = 0; sidx < more; ++sidx) {
          const int off = __shfl_sync(0xffffffffu, (int)raw.x, sidx), d = __shfl_sync(0xffffffffu, (int)(raw.y & 0xFFFFu), sidx);
          const double c = __shfl_sync(0xffffffffu, cs, sidx);
          const unsigned x = kPhase ? __shfl_sync(0xffffffffu, xs, sidx) : 0u;
          if (active) StoreOut(o + off, kPhase ? FormVal(cta_smem, lane, Classify(cta_smem, x, d, c, v_off, dwin, zrow), x, d, c, v_off) : cta_smem[d * kLD + lane] * c);
        }
      }
    }
#endif
  }
}
// ---- constraint values straight into g[B][m] (TWB_GDIRECT) ----------------------------------------------------------------
#ifndef TWB_GDIRECT_PHASE
#define TWB_GDIRECT_PHASE 1   // 1: problems with optimised durations write g directly as well (their range-of-motion values lane = instance)
#endif
#ifndef TWB_G_ST
#define TWB_G_ST 1   // cache operator of the direct constraint-value stores: 0 .cs (evict-first), 1 default (ships: 132.0 vs 134.5 us per step on config 2 — rows shared by two CTAs merge in the L2)
#endif
__device__ __forceinline__ void StoreG(double* p, double v) {
#if TWB_G_ST == 1
  *p = v;
#else
  __stcs(p, v);
#endif
}
// The `n_units` consecutive units of a CTA own kPer consecutive constraint rows each, starting at row `row0`; unit w keeps its
// values in the state rows w * block_rows + d0 .. of the CTA's shared memory `t`.  All threads: consecutive threads write
// consecutive rows of one instance (kPer * n_units * 8 contiguous bytes per instance), after the CTA barrier.
template <int kPer>
__device__ __forceinline__ void StoreValuesDirect(const Plan& P, const double* t, double* __restrict__ g, int tile, int nb, int row0, int n_units,
                                                  int block_rows, int d0) {
  // thread = (row r of the CTA's run, instance j0), then every `per`-th instance: the index arithmetic happens once per thread
  const int nc = P.nc_jac, n_inst = TileCount(nc, tile, nb), N = kPer * n_units, per = (int)blockDim.x / N;
  const int j0 = (int)threadIdx.x / N, r = (int)threadIdx.x - j0 * N;
  if (j0 >= per) return;
  const int w = r / kPer, i = r - w * kPer;
  const double* src = t + (w * block_rows + d0 + i) * kLD;
  double* dst = g + (size_t)TileInstance(nc, tile, j0) * P.m + row0 + r;
  const size_t step = (size_t)per * nc * P.m;
  for (int j = j0; j < n_inst; j += per, dst += step) StoreG(dst, src[j]);
}
// non-finite check of this lane's own column (rows 1 .. n_rows-1); flags instance b
__device__ __forceinline__ void FlagNonFinite(const double* t, int n_rows, int lane, int* __restrict__ status, int b, int nb, int first_row = 1) {
  if (!status) return;
  double chk = 0.0;
  for (int r = first_row; r < n_rows; ++r) chk = fma(t[r * kLD + lane], 0.0, chk);
  if (chk != chk && b < nb) atomicOr(status + b, 1);
}

// DynamicConstraint: blockIdx.y = instance tile, warp = one of kDynWarps CONSECUTIVE samples, so a CTA writes
// several KB of contiguous CSR values per instance (the samples' rows are adjacent).
template <int kNEE, bool kPhase>
__device__ __forceinline__ void DynBody(const Plan& P, const double* __restrict__ XT, double* __restrict__ GT, double* __restrict__ jac,
                                        int* __restrict__ status, int nb, unsigned flags, double* out_smem, int cta, int tile, const Stage st,
                                        const double* __restrict__ FS = nullptr, double* __restrict__ g = nullptr) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = cta * kDynWarps + warp, b = TileInstance(P.nc_jac, tile, lane);
  // local rows: 1 | 3 | 36 | 6 per foot [| the 6 constraint values (TWB_GDIRECT); else they go straight into GT, coalesced]
  constexpr int n_rows = DynBlockRows(kNEE), g_d0 = n_rows - 6;
  const bool g_direct = TWB_GDIRECT && g != nullptr;
  double* t = out_smem + (size_t)warp * n_rows * kLD;
  if (k < P.n_dyn) {
    const DynUnit* u = P.dyn + k;
    t[lane] = 1.0;
#ifndef TWB_EXP_NOCOMPUTE   // (timing experiment: store phase only)
    DynamicUnit<kNEE, kPhase>(P, k, P.samples + __ldg(&u->sample0), TileCol(XT, tile, lane, P.n + 1), Col{t + kLD + lane, kLD},
                              g_direct ? Col{t + g_d0 * kLD + lane, kLD} : Col{GT + (((size_t)tile * P.m + (size_t)__ldg(&u->g_row0)) * 32) + lane, 32},
                              FS ? FS + (((size_t)tile * P.n_dyn + k) * (6 * kNEE)) * 32 + lane : nullptr);
    FlagNonFinite(t, n_rows, lane, status, b, nb);
#endif
  }
  __syncthreads();
  if (g_direct && (flags & 1u) && cta * kDynWarps < P.n_dyn)
    StoreValuesDirect<6>(P, out_smem, g, tile, nb, __ldg(&P.dyn[cta * kDynWarps].g_row0), min(kDynWarps, P.n_dyn - cta * kDynWarps), n_rows, g_d0);
  if (flags & 2u) StoreCta(P, out_smem, P.cta_lists + P.dyn_list0 + cta, jac, tile, nb, st);
}

// RangeOfMotionConstraint (range_of_motion_constraint.cc:58-109): g_e = R^T (p_e - c); Jacobian state R^T and
// D_e = d(R^T r_e)/d(theta) (EulerConverter::DerivOfRotVecMult(t, r_W, true)).  blockIdx.y = instance tile,
// warp = one of kRomWarps consecutive samples.  The rotation and its derivative are computed once per sample; the
// feet then take turns through two alternating buffers of 12 state rows (D_e, g_e): while the CTA writes the
// Jacobian values of foot e (one list per foot: the foot's rows of the CTA's samples are adjacent), every warp
// already evaluates foot e + 1 — one CTA barrier per foot.
template <int kNEE, bool kPhase>
__device__ __forceinline__ void RomBody(const Plan& P, const double* __restrict__ XT, double* __restrict__ GT, double* __restrict__ jac,
                                        int* __restrict__ status, int nb, unsigned flags, double* out_smem, int cta, int tile, const Stage st,
                                        double* __restrict__ g = nullptr) {
  const bool g_direct = TWB_GDIRECT && !kPhase && g != nullptr;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = cta * kRomWarps + warp, b = TileInstance(P.nc_jac, tile, lane);
  const bool valid = k < P.n_rom;
  constexpr int block_rows = RomBlockRowsP(kNEE, kPhase);
  double* t = out_smem + (size_t)warp * block_rows * kLD;
  const RomUnit* u = P.rom + (valid ? k : 0);
  const SplineSample* __restrict__ sp = P.samples + __ldg(&u->sample0);
  const ConstCol xs = TileCol(XT, tile, lane, P.n + 1);
  // local state rows 1..: R^T (0..8) | buffer 0: D_e (9..17), g_e (18..20) | buffer 1: (21..29), (30..32); with optimised durations a
  // buffer is D_e (9) | the PhaseSpline's info block (kInfoRows) | U (3) | X (3 kRomDurWin)   (g_e lives in registers only)
  const Col Sk{t + kLD + lane, kLD};
  t[lane] = 1.0;
#ifndef TWB_EXP_NOCOMPUTE
  double c[3], th[3], unused[3];
  EvalSpline<0>(P, sp + 0, xs, c, unused, unused);
  EvalSpline<0>(P, sp + 1, xs, th, unused, unused);
  const Trig tr = MakeTrig(th);
  double R[3][3]; RotationMatrix(tr, R);
  double dR[3][3][3]; RotationDerivative(tr, dR);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int d = 0; d < 3; ++d) Sk[i * 3 + d] = R[d][i];
#endif
#pragma unroll 1
  for (int e = 0; e < kNEE; ++e) {
    const int buf = RomBufferP(e, kPhase);
#ifndef TWB_EXP_NOCOMPUTE
    double pe[3];
    if (kPhase) {   // range_of_motion_constraint.cc:83-109 with the PhaseSpline of foot e: value, active polynomial, duration columns
      const PhaseFull mo = EvalPhaseFull(P, 2 * e, __ldg(&sp[2 + e].T), xs);
      pe[0] = mo.pos[0]; pe[1] = mo.pos[1]; pe[2] = mo.pos[2];
      StorePhaseInfo(mo, t, 19 + buf, lane);
      double U[3], V[3], RU[3], RV[3]; DurationVectors(mo, U, V);
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        RU[i] = (R[0][i] * U[0] + R[1][i] * U[1]) + R[2][i] * U[2];
        RV[i] = (R[0][i] * V[0] + R[1][i] * V[1]) + R[2][i] * V[2];
      }
      StorePhaseDurations<3, kRomDurWin>(mo.cur, RU, RV, t, 19 + buf, 19 + kInfoRows + buf, lane);
    } else {
      EvalSpline<0, false>(P, sp + 2 + e, xs, pe, unused, unused);
    }
    const double r[3] = {pe[0] - c[0], pe[1] - c[1], pe[2] - c[2]};
    double D[3][3]; RotVecDerivative<true>(dR, r, D);
    double ge[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) { ge[i] = R[0][i] * r[0] + R[1][i] * r[1] + R[2][i] * r[2]; if (!kPhase) Sk[18 + buf + i] = ge[i]; }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int d = 0; d < 3; ++d) Sk[9 + buf + i * 3 + d] = D[i][d];
    if (valid) {
      // non-finite check of this lane's R^T (first foot), D_e and g_e, from the registers
      double chk = 0.0;
      if (e == 0) {
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
          for (int d = 0; d < 3; ++d) chk = fma(R[i][d], 0.0, chk);
      }
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        chk = fma(ge[i], 0.0, chk);
#pragma unroll
        for (int d = 0; d < 3; ++d) chk = fma(D[i][d], 0.0, chk);
      }
      if (status && chk != chk && b < nb) atomicOr(status + b, 1);
    }
#endif
    if (kPhase && TWB_GDIRECT && g != nullptr) {   // optimised durations: g_e exists in registers only; lane = instance straight into g
#ifndef TWB_EXP_NOCOMPUTE
      if (valid && (flags & 1u) && b < nb) {
        double* gp = g + (size_t)b * P.m + P.rom_row0[e] + 3 * k;
#pragma unroll
        for (int i = 0; i < 3; ++i) StoreG(gp + i, ge[i]);
      }
#endif
    } else
    if (valid && (flags & 1u) && !g_direct) {   // rows rom_row0[e] + 3k .. + 2 (range_of_motion_constraint.cc:58-66), lane = instance into GT
      double* gt = GT + (((size_t)tile * P.m + (size_t)(P.rom_row0[e] + 3 * k)) * 32) + lane;
#ifndef TWB_EXP_NOCOMPUTE
#pragma unroll
      for (int i = 0; i < 3; ++i) gt[i * 32] = ge[i];
#else
      for (int i = 0; i < 3; ++i) gt[i * 32] = t[(19 + buf + i) * kLD + lane];
#endif
    }
#if !TWB_ROM_ALLFEET
    __syncthreads();   // foot e complete in every block; everybody is done reading buffer (e + 1) & 1 (the list of foot e - 1)
    if (g_direct && (flags & 1u))   // the foot's rows of the CTA's samples are adjacent: 3 kRomWarps consecutive values per instance
      StoreValuesDirect<3>(P, out_smem, g, tile, nb, P.rom_row0[e] + 3 * cta * kRomWarps, min(kRomWarps, P.n_rom - cta * kRomWarps), block_rows, 19 + buf);
    if (flags & 2u) StoreCta<kPhase>(P, out_smem, P.cta_lists + P.rom_list0 + cta * kNEE + e, jac, tile, nb, st, 3, kRomDurWin, 20 + buf);
#endif
  }
#if TWB_ROM_ALLFEET
  __syncthreads();
  if (flags & 2u) StoreCta<kPhase>(P, out_smem, P.cta_lists + P.rom_list0 + cta, jac, tile, nb, st, 3, kRomDurWin, 20);
#endif
}

// node groups: blockIdx.y = instance tile, warp = one of kNodeWarps consecutive groups
__device__ __forceinline__ void NodeBody(const Plan& P, const double* __restrict__ XT, double* __restrict__ GT, double* __restrict__ jac,
                                         int* __restrict__ status, const int* __restrict__ terrain_ids, int default_terrain, int nb,
                                         unsigned flags, double* node_smem, int cta, int tile, const Stage st, double* __restrict__ g = nullptr) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool g_direct = TWB_GDIRECT && g != nullptr;
  const int gi = cta * kNodeWarps + warp, b = TileInstance(P.nc_jac, tile, lane);
  double* t = node_smem + (size_t)warp * P.node_rows * kLD;
  if (gi < P.n_groups) {
    const ConstCol xs = TileCol(XT, tile, lane, P.n + 1);
    const NodeGroup* grp = P.groups + gi;
    const int kind = __ldg(&grp->kind), first = __ldg(&grp->first), count = __ldg(&grp->count);
    t[lane] = 1.0;
    int n_rows = 1;
#ifndef TWB_EXP_NOCOMPUTE
    if (kind == kGroupForce) {
      const int terrain = (terrain_ids && b < nb) ? __ldg(terrain_ids + b) : default_terrain;
      for (int q = 0; q < count; ++q)
        ForceUnitEval(P, P.force[first + q], terrain, xs, Col{t + (1 + 25 * q) * kLD + lane, kLD}, Col{t + (1 + 25 * count + 5 * q) * kLD + lane, kLD});
      n_rows = 1 + 30 * count;
    } else if (kind == kGroupTerrain) {
      const int terrain = (terrain_ids && b < nb) ? __ldg(terrain_ids + b) : default_terrain;
      for (int q = 0; q < count; ++q)
        TerrainUnitEval(P, P.terr[first + q], terrain, xs, Col{t + (1 + 2 * q) * kLD + lane, kLD}, Col{t + (1 + 2 * count + q) * kLD + lane, kLD});
      n_rows = 1 + 3 * count;
    } else if (kind == kGroupSwing) {
      if (flags & 1u) for (int q = 0; q < count; ++q) SwingUnitEval(P.swing[first + q], xs, Col{t + (1 + 4 * q) * kLD + lane, kLD});
      n_rows = (flags & 1u) ? 1 + 4 * count : 1;
    } else if (kind == kGroupAcc) {
      if (flags & 1u) for (int q = 0; q < count; ++q) AccUnitEval(P.acc[first + q], xs, Col{t + (1 + 3 * q) * kLD + lane, kLD});
      n_rows = (flags & 1u) ? 1 + 3 * count : 1;
    } else if (kind == kGroupBaseMotion) {
      if (flags & 1u) for (int q = 0; q < count; ++q) BaseMotionUnitEval(P, P.base_motion[first + q], xs, Col{t + (1 + 6 * q) * kLD + lane, kLD});
      n_rows = (flags & 1u) ? 1 + 6 * count : 1;
    }
    FlagNonFinite(t, n_rows, lane, status, b, nb);
#endif
    if ((flags & 1u) && g_direct) {   // the group's consecutive rows, this warp's own state: lanes = (instance, row) pairs
      const int g_row0 = __ldg(&grp->g_row0), nc = P.nc_jac, n_inst = TileCount(nc, tile, nb);
      __syncwarp();
      if (g_row0 >= 0) {
        const int d0 = __ldg(&grp->g_d0), gn = __ldg(&grp->g_n);
        if (gn <= 32) {   // lane = (row i, instance j0), then every `per`-th instance
          const int per = 32 / gn, j0 = lane / gn, i = lane - j0 * gn;
          if (j0 < per) {
            const double* src = t + (d0 + i) * kLD;
            double* dst = g + (size_t)TileInstance(nc, tile, j0) * P.m + g_row0 + i;
            const size_t step = (size_t)per * nc * P.m;
            for (int j = j0; j < n_inst; j += per, dst += step) StoreG(dst, src[j]);
          }
        } else {
          for (int j = 0; j < n_inst; ++j)
            for (int i = lane; i < gn; i += 32) StoreG(g + (size_t)TileInstance(nc, tile, j) * P.m + g_row0 + i, t[(d0 + i) * kLD + j]);
        }
      } else {
        const OutRange r = LoadRange(&grp->values);
        ForEachEntry(P.pairs + r.first, P.coefs + r.first, r.count, lane,
                     [&](int g_row, int d, double c) { if (b < nb) StoreG(g + (size_t)b * P.m + g_row, t[d * kLD + lane] * c); });
      }
    } else if (flags & 1u) {
      const int g_row0 = __ldg(&grp->g_row0);
      if (g_row0 >= 0) {
        const int d0 = __ldg(&grp->g_d0), gn = __ldg(&grp->g_n);
        double* gt = GT + (((size_t)tile * P.m + (size_t)g_row0) * 32) + lane;
        for (int i = 0; i < gn; ++i) gt[(size_t)i * 32] = t[(d0 + i) * kLD + lane];
      } else {
        StoreValuesTiled(P, t, &grp->values, GT + (size_t)tile * P.m * 32, lane);
      }
    }
  }
  __syncthreads();
  if (flags & 2u) StoreCta(P, node_smem, P.cta_lists + P.node_list0 + cta, jac, tile, nb, st);
}

// NodeCost::GetCost summed over terms (node_cost.cc:53-63; Composite::GetValues for costs) and the dense gradient row
// (node_cost.cc:65-76), both in the reference's order.  lane = instance (coalesced reads of XT); the gradient row is
// zeroed by a memset (coalesced) before this kernel, which then only touches the columns that carry a cost term.
__global__ void __launch_bounds__(128) CostKernel(const Plan P, const double* __restrict__ XT, double* __restrict__ cost,
                                                  double* __restrict__ grad, int nb) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  const ConstCol xs = TiledCol(XT, b, P.n + 1, P.nc_jac);
  double* gr = grad ? grad + (size_t)b * P.n : nullptr;
  double total_cost = 0.0, term = 0.0;
  for (int i = 0; i < P.n_cost; ++i) {
    const CostEntry ce = P.cost[i];
    if (ce.pad && i > 0) { total_cost += term; term = 0.0; }
    const double val = xs[ce.xi];
    term += ce.weight * (val * val);
    if (gr && ce.grad_col >= 0) gr[ce.grad_col] += ce.weight * 2.0 * val;
  }
  total_cost += term;
  if (cost) cost[b] = total_cost;
}

// ---- PhaseSpline columns of the dynamic constraint (optimised phase durations) --------------------------------
// dynamic_constraint.cc:91-113 with single_rigid_body_dynamics.cc:167-192: with PhaseSplines every dynamic row is
// structurally dense in all ee-motion / ee-force node variables and in the feet's duration variables (324 of the 348 entries
// of an angular row of config 4).  CTA = (dynamic sample, tile of 32 instances), warp = foot: lane = instance evaluates the
// foot's two PhaseSplines with everything their Jacobian needs (active polynomial, Hermite basis values, duration columns)
// into the foot's state block (device_tables.h: kTailRows); then all threads of the CTA walk the sample's list of phase
// elements — the same coalesced whole-sector pair loop as every other Jacobian value.  (Until round 2 these entries were
// scattered by lane = instance 8-byte stores over rows of zeros: 1.0 of config 4's 1.26 ms.)
#ifndef TWB_TAIL_CTAS
#define TWB_TAIL_CTAS 4   // resident CTAs per SM the DynTailOut kernel is compiled for (128 registers; 49 state rows per foot = 53 KB per CTA)
#endif
template <int kNEE>
__global__ void __launch_bounds__(kNEE * 32, TWB_TAIL_CTAS) DynTailOut(const Plan P, const double* __restrict__ XT, double* __restrict__ jac, int nb,
                                                        double* __restrict__ FS) {
  extern __shared__ __align__(16) double out_smem[];
  const int lane = threadIdx.x & 31, e = threadIdx.x >> 5, k = blockIdx.x;
  double* t = out_smem + (size_t)e * kTailRows * kLD;
  const SplineSample* __restrict__ sp = P.samples + __ldg(&P.dyn[k].sample0);
  const ConstCol xs = TileCol(XT, blockIdx.y, lane, P.n + 1);
#ifndef TWB_EXP_NOCOMPUTE
  double c[3], unused[3];
  EvalSpline<0>(P, sp, xs, c, unused, unused);
  const double tg = __ldg(&sp[2 + e].T);   // phase samples carry the global time
  const PhaseFull mo = EvalPhaseFull(P, 2 * e, tg, xs), fo = EvalPhaseFull(P, 2 * e + 1, tg, xs);
  const double r[3] = {c[0] - mo.pos[0], c[1] - mo.pos[1], c[2] - mo.pos[2]};
  t[lane] = 1.0;
#pragma unroll
  for (int d = 0; d < 3; ++d) { t[(1 + d) * kLD + lane] = fo.pos[d]; t[(4 + d) * kLD + lane] = r[d]; }
  if (FS) {   // p_e, f_e of this sample for the DynOut kernel that follows on the same stream
    double* fs = FS + (((size_t)blockIdx.y * P.n_dyn + k) * (6 * kNEE) + 6 * e) * 32 + lane;
#pragma unroll
    for (int d = 0; d < 3; ++d) { __stcg(fs + d * 32, mo.pos[d]); __stcg(fs + (3 + d) * 32, fo.pos[d]); }
  }
  StorePhaseInfo(mo, t, 7, lane);
  StorePhaseInfo(fo, t, 7 + kInfoRows, lane);
  double Cf[3][3], Cr[3][3];
  CrossMatrix(fo.pos, Cf); CrossMatrix(r, Cr);
  double jfU[3], jfV[3], jmU[3], jmV[3];
  DurationVectors(fo, jfU, jfV); DurationVectors(mo, jmU, jmV);
  double U[6], V[6];
#pragma unroll
  for (int i = 0; i < 3; ++i) {   // JacWrtForce + JacWrtEEPos of the duration columns (dynamic_constraint.cc:106-112)
    const int d1 = (i == 0) ? 1 : 0, d2 = (i == 2) ? 1 : 2;
    U[i] = (Cr[i][d1] * jfU[d1] + Cr[i][d2] * jfU[d2]) + (Cf[i][d1] * jmU[d1] + Cf[i][d2] * jmU[d2]);
    U[3 + i] = -jfU[i];
    V[i] = (Cr[i][d1] * jfV[d1] + Cr[i][d2] * jfV[d2]) + (Cf[i][d1] * jmV[d1] + Cf[i][d2] * jmV[d2]);
    V[3 + i] = -jfV[i];
  }
  StorePhaseDurations<6, kDynDurWin>(mo.cur, U, V, t, 7, 7 + 2 * kInfoRows, lane);
#endif
  __syncthreads();
  StoreCta<true>(P, out_smem, P.cta_lists + P.tail_list0 + k, jac, blockIdx.y, nb, Stage{nullptr, 0}, 6, kDynDurWin, 8);
}

// TotalDurationConstraint (total_duration_constraint.cc:36-72; the only rows no output kernel owns): value = sum of the foot's
// optimised durations, Jacobian = 1 in each of their columns, status bit 1 when the sum leaves nothing for the last phase
// (phase_durations.cc:92).  warp = tile of 32 instances, lane = instance; 8 entries per foot at the very end of the CSR row.
template <int kNEE>
__global__ void __launch_bounds__(32) PhaseJac(const Plan P, const double* __restrict__ XT, double* __restrict__ GT, double* __restrict__ g, double* __restrict__ jac,
                                               int* __restrict__ status, int nb, unsigned flags) {
  const int lane = threadIdx.x, b = TileInstance(P.nc_jac, blockIdx.x, lane);
  const bool live = b < nb;
  const ConstCol xs = TileCol(XT, blockIdx.x, lane, P.n + 1);
  for (int ui = 0; ui < P.n_phase_units; ++ui) {
    const PhaseUnit* u = P.phase_units + ui;
    for (int e = 0; e < kNEE; ++e) {
      const PhaseSplineDef def = P.phase_defs[2 * e];
      const int row = __ldg(&u->rows[e]), slot0 = __ldg(&u->slot0[e]);
      double sum = 0.0;
      for (int i = 0; i + 1 < def.n_phases; ++i) {
        sum += xs[def.sched0 + i];
        if (live && (flags & 2u)) StoreOut(jac + (size_t)b * P.nnz + slot0 + i, 1.0);
      }
      if (flags & 1u) {
        if (g) { if (live) StoreG(g + (size_t)b * P.m + row, sum); }
        else GT[((size_t)blockIdx.x * P.m + row) * 32 + lane] = sum;
      }
      if (live && status && !(def.t_total - sum > 0.0)) atomicOr(status + b, 2);
    }
  }
}

// The K values each lane holds for its instance -> out[instance][offset .. offset + K - 1] (row stride `stride` doubles), staged
// through the warp's shared-memory tile [K][33] so that consecutive lanes write consecutive addresses (a lane writing its own
// row would touch 32 different sectors per store instruction).
template <int K>
__device__ __forceinline__ void StoreRowsCoalesced(const double* o, double* stage, double* __restrict__ out, size_t stride, size_t offset,
                                                   int nc, int tile, int nb, int lane) {
#pragma unroll
  for (int i = 0; i < K; ++i) stage[i * 33 + lane] = o[i];
  __syncwarp();
  const int n_inst = TileCount(nc, tile, nb);
  for (int j = 0; j < n_inst; ++j) {
    double* dst = out + (size_t)TileInstance(nc, tile, j) * stride + offset;
    for (int i = lane; i < K; i += 32) dst[i] = stage[i * 33 + j];
  }
}

// ---- solution post-processing: fpowr::GetTrajectory (footstep_plan_extractor.h:19-53) --------------------------
// Eigen::Quaterniond(Matrix3d) (Eigen 3.3 Quaternion.h, quaternionbase_assign_impl<Other,3,3>); q = w, x, y, z
__device__ __forceinline__ void QuaternionFromMatrix(const double m[3][3], double q[4]) {
  double t = m[0][0] + m[1][1] + m[2][2];
  if (t > 0.0) {
    t = sqrt(t + 1.0); q[0] = 0.5 * t; t = 0.5 / t;
    q[1] = (m[2][1] - m[1][2]) * t; q[2] = (m[0][2] - m[2][0]) * t; q[3] = (m[1][0] - m[0][1]) * t;
  } else {
    int i = 0; if (m[1][1] > m[0][0]) i = 1; if (m[2][2] > m[i][i]) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    t = sqrt(m[i][i] - m[j][j] - m[k][k] + 1.0);
    double v[3];
    v[i] = 0.5 * t; t = 0.5 / t;
    q[0] = (m[k][j] - m[j][k]) * t; v[j] = (m[j][i] + m[i][j]) * t; v[k] = (m[k][i] + m[i][k]) * t;
    q[1] = v[0]; q[2] = v[1]; q[3] = v[2];
  }
}
// warp = (time step, tile of 32 instances), lane = instance; every lane writes its instance's 19 + 13 n_ee values
template <int kNEE, bool kPhase>
__global__ void __launch_bounds__(128) TrajectoryKernel(const Plan P, const double* __restrict__ XT, const SplineSample* __restrict__ samples,
                                                        const int* __restrict__ contact, int n_steps, double* __restrict__ out, int nb) {
  const int lane = threadIdx.x & 31, ti = blockIdx.x * 4 + (threadIdx.x >> 5), b = TileInstance(P.nc_jac, blockIdx.y, lane);
  if (ti >= n_steps) return;
  const ConstCol xs = TileCol(XT, blockIdx.y, lane, P.n + 1);
  const SplineSample* sp = samples + (size_t)ti * (2 + 2 * kNEE);
  constexpr int K = 19 + 13 * kNEE;
  double o[K];
  double th[3], thd[3], thdd[3], unused[3];
  EvalSpline<2>(P, sp + 0, xs, o, o + 3, o + 6);
  EvalSpline<2>(P, sp + 1, xs, th, thd, thdd);
  const Trig tr = MakeTrig(th);
  double R[3][3]; RotationMatrix(tr, R);
  QuaternionFromMatrix(R, o + 9);
  {  // EulerConverter::GetAngularVelocityInWorld / GetAngularAccelerationInWorld (euler_converter.cc:58-83), as in DynamicUnit
    const double sy = tr.sy, cy = tr.cy, sz = tr.sz, cz = tr.cz, yd = thd[1], zd = thd[2];
    const double M[3][3] = {{cy * cz, -sz, 0.0}, {cy * sz, cz, 0.0}, {-sy, 0.0, 1.0}};
    const double Md[3][3] = {{-cz * sy * yd - cy * sz * zd, -cz * zd, 0.0}, {cy * cz * zd - sy * sz * yd, -sz * zd, 0.0}, {-cy * yd, 0.0, 0.0}};
    o[13] = M[0][0] * thd[0] + M[0][1] * thd[1];
    o[14] = M[1][0] * thd[0] + M[1][1] * thd[1];
    o[15] = M[2][0] * thd[0] + thd[2];
    o[16] = (Md[0][0] * thd[0] + Md[0][1] * thd[1]) + (M[0][0] * thdd[0] + M[0][1] * thdd[1]);
    o[17] = (Md[1][0] * thd[0] + Md[1][1] * thd[1]) + (M[1][0] * thdd[0] + M[1][1] * thdd[1]);
    o[18] = (Md[2][0] * thd[0]) + (M[2][0] * thdd[0] + thdd[2]);
  }
#pragma unroll
  for (int e = 0; e < kNEE; ++e) {
    double* f = o + 19 + 13 * e;
    EvalSpline<2, kPhase>(P, sp + 2 + e, xs, f + 1, f + 4, f + 7);
    EvalSpline<0, kPhase>(P, sp + 2 + kNEE + e, xs, f + 10, unused, unused);
    if (kPhase) {   // PhaseDurations::IsContactPhase (phase_durations.cc:120-124) with this instance's durations
      const PhaseSplineDef def = P.phase_defs[2 * e];
      double sum = 0.0;
      for (int i = 0; i + 1 < def.n_phases; ++i) sum += xs[def.sched0 + i];
      const double last = def.t_total - sum, tg = __ldg(&sp[2 + e].T);
      double acc = 0.0; int phase = def.n_phases - 1; bool found = false;
      for (int ph = 0; ph < def.n_phases; ++ph) {
        acc += (ph == def.n_phases - 1) ? last : xs[def.sched0 + ph];
        if (!found && acc >= tg - 1e-10) { found = true; phase = ph; }
      }
      const bool first = __ldg(contact + e) != 0;   // contact: in_contact_at_start per foot
      f[0] = ((phase % 2 == 0) ? first : !first) ? 1.0 : 0.0;
    } else {
      f[0] = (double)__ldg(contact + (size_t)ti * kNEE + e);
    }
  }
  extern __shared__ __align__(16) double stage_smem[];
  StoreRowsCoalesced<K>(o, stage_smem + (size_t)(threadIdx.x >> 5) * K * 33, out, (size_t)n_steps * K, (size_t)ti * K, P.nc_jac, blockIdx.y, nb, lane);
}

// fpowr::ExtractInitialGuess (initial_guess_extractor.h:17-34) at caller-given times: per sample 49 doubles —
// time | state: base lin p, base ang p (Euler angles), base lin v, base ang v (12) | controls: ee-motion accelerations
// (12), joint torques = 0 (12), ee-forces (12); feet beyond n_ee stay 0.  warp = (time, tile), lane = instance.
template <int kNEE, bool kPhase>
__global__ void __launch_bounds__(128) InitialGuessKernel(const Plan P, const double* __restrict__ XT, const SplineSample* __restrict__ samples,
                                                          const double* __restrict__ times, int n_times, double* __restrict__ out, int nb) {
  const int lane = threadIdx.x & 31, ti = blockIdx.x * 4 + (threadIdx.x >> 5), b = TileInstance(P.nc_jac, blockIdx.y, lane);
  if (ti >= n_times) return;
  const ConstCol xs = TileCol(XT, blockIdx.y, lane, P.n + 1);
  const SplineSample* sp = samples + (size_t)ti * (2 + 2 * kNEE);
  double o[49];
#pragma unroll
  for (int i = 0; i < 49; ++i) o[i] = 0.0;
  o[0] = __ldg(times + ti);
  double unused[3];
  EvalSpline<2>(P, sp + 0, xs, o + 1, o + 7, unused);
  EvalSpline<2>(P, sp + 1, xs, o + 4, o + 10, unused);
#pragma unroll
  for (int e = 0; e < kNEE; ++e) {
    double pos[3];
    EvalSpline<1, kPhase>(P, sp + 2 + e, xs, pos, unused, o + 13 + 3 * e);
    EvalSpline<0, kPhase>(P, sp + 2 + kNEE + e, xs, o + 13 + 24 + 3 * e, unused, unused);
  }
  extern __shared__ __align__(16) double stage_smem[];
  StoreRowsCoalesced<49>(o, stage_smem + (size_t)(threadIdx.x >> 5) * 49 * 33, out, (size_t)n_times * 49, (size_t)ti * 49, P.nc_jac, blockIdx.y, nb, lane);
}

// fpowr::ExtractFootstepPlan (footstep_plan_extractor.h:68-133) without the nearest-plane lookup: the trajectory of
// fpowr::GetTrajectory(dt) is scanned for changes of the contact set (HasEndEffectorContactChanged, :55-66); every change
// (and the first state) is a footstep state.  Per footstep state V = 2 + 4 n_ee doubles: t_global | duration (time to the
// next footstep state, the last one up to time_horizon) | per foot: contact flag, ee position.
// Fused: the trajectory is never materialised.  Only the contact flags are walked, step by step, and the feet's ee-motion
// positions are evaluated at the change steps alone — from the same SplineSample entries, by the same EvalSpline position
// term (independent of kWant), at the same times (times[k] = the table's t += dt), so every value is bit-identical to
// sampling the trajectory and scanning it.  A change is coded (step << 4) | contact mask (bit e: foot e in contact).
// Fixed durations: the flags are structure-class data, and the host's table holds the change codes (`codes`, n_codes of
// them), the same for every instance.  Optimised durations: each lane walks the steps with its instance's durations and
// the phase search of TrajectoryKernel (acc >= t - 1e-10 over the phases, last phase = T - sum), resumed from the previous
// step's phase (the first phase that qualifies never moves back as t grows, so the result is the full search's), and
// keeps its codes in shared memory.  Warp = tile of 32 instances, lane = instance; each state row goes out through
// StoreRowsCoalesced; rows past the instance's count are written as 0.
template <int kNEE, bool kPhase>
__global__ void __launch_bounds__(128) FootstepPlanKernel(const Plan P, const double* __restrict__ XT, const SplineSample* __restrict__ samples,
                                                          const double* __restrict__ times, const int* __restrict__ contact, const int* __restrict__ codes,
                                                          int n_codes, int n_steps, double time_horizon, int max_states, int tiles, int* __restrict__ n_states,
                                                          double* __restrict__ out, int nb) {
  constexpr int V = 2 + 4 * kNEE;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, tile = blockIdx.x * 4 + warp, nc = P.nc_jac;
  if (tile >= tiles || TileCount(nc, tile, nb) == 0) return;   // whole warps
  const ConstCol xs = TileCol(XT, tile, lane, P.n + 1);
  extern __shared__ __align__(16) double fp_smem[];
  double* stage = fp_smem + (size_t)warp * V * 33;
  int* my_codes = reinterpret_cast<int*>(fp_smem + 4 * V * 33) + (size_t)warp * (max_states + 1) * 32 + lane;   // [max_states + 1][32]
  int count = n_codes;
  if (kPhase) {
    int ph[kNEE], n_ph[kNEE], s0[kNEE]; double acc[kNEE], last[kNEE]; bool first[kNEE];
#pragma unroll
    for (int e = 0; e < kNEE; ++e) {
      const PhaseSplineDef def = P.phase_defs[2 * e];
      n_ph[e] = def.n_phases; s0[e] = def.sched0;
      double sum = 0.0;
      for (int i = 0; i + 1 < def.n_phases; ++i) sum += xs[def.sched0 + i];
      last[e] = def.t_total - sum;
      ph[e] = 0; acc[e] = 0.0 + (def.n_phases == 1 ? last[e] : xs[def.sched0]);   // acc = 0, acc += first duration
      first[e] = __ldg(contact + e) != 0;
    }
    count = 0;
    unsigned prev = 0;
    for (int k = 0; k < n_steps; ++k) {
      const double thr = __ldg(times + k) - 1e-10;
      unsigned mask = 0;
#pragma unroll
      for (int e = 0; e < kNEE; ++e) {
        while (ph[e] < n_ph[e] - 1 && !(acc[e] >= thr)) { ++ph[e]; acc[e] += (ph[e] == n_ph[e] - 1) ? last[e] : xs[s0[e] + ph[e]]; }
        if ((ph[e] % 2 == 0) ? first[e] : !first[e]) mask |= 1u << e;
      }
      if (k == 0 || mask != prev) {
        if (count <= max_states) my_codes[(size_t)count * 32] = (k << 4) | (int)mask;
        ++count;
      }
      prev = mask;
    }
  }
  const int b = TileInstance(nc, tile, lane);
  if (b < nb) n_states[b] = count;
  for (int i = 0; i < max_states; ++i) {
    double o[V];
#pragma unroll
    for (int v = 0; v < V; ++v) o[v] = 0.0;
    if (i < count) {
      const int code = kPhase ? my_codes[(size_t)i * 32] : __ldg(codes + i), k = code >> 4;
      const double t = __ldg(times + k);
      o[0] = t;
      if (i + 1 < count) o[1] = __ldg(times + ((kPhase ? my_codes[(size_t)(i + 1) * 32] : __ldg(codes + i + 1)) >> 4)) - t;
      else o[1] = time_horizon - t;
      const SplineSample* sp = samples + (size_t)k * (2 + 2 * kNEE);
#pragma unroll
      for (int e = 0; e < kNEE; ++e) {
        double unused[3];
        o[2 + 4 * e] = ((code >> e) & 1) ? 1.0 : 0.0;
        EvalSpline<0, kPhase>(P, sp + 2 + e, xs, o + 3 + 4 * e, unused, unused);
      }
    }
    StoreRowsCoalesced<V>(o, stage, out, (size_t)max_states * V, (size_t)i * V, nc, tile, nb, lane);
    __syncwarp();   // the stage is rewritten by the next state
  }
}

// ---- fpowr::NearestPlaneLookup::GetNearestPlaneIndex (fpowr/include/fpowr/nearest_plane_lookup.h:62-84) ----------------
// boost::geometry::distance(point, polygon) with the default cartesian strategies, restated (boost is an un-vendored
// dependency): 0 when the point is inside or on the outer ring (winding number over the ring's segments), else the
// smallest distance to a segment of the ring, projected-point strategy (distance_projected_point.hpp: c1 = w.v <= 0 ->
// first end, c2 = v.v <= c1 -> second end, else the foot of the perpendicular), comparable (squared) distances, one sqrt.
// A ring is the vertex sequence AS GIVEN: bg::model::polygon is `closed` by default, i.e. the closing segment exists
// only if the caller repeats the first vertex (fpowr appends the message's boundary points as they are).
__device__ __forceinline__ double PolygonDistance(const double* __restrict__ v, int n, double px, double py) {
  if (n <= 0) return 1.7976931348623157e308;
  if (n == 1) { const double dx = px - v[0], dy = py - v[1]; return sqrt(dx * dx + dy * dy); }
  int winding = 0; bool touches = false;
  double best = 1.7976931348623157e308;
  for (int i = 0; i + 1 < n; ++i) {
    const double ax = __ldg(v + 2 * i), ay = __ldg(v + 2 * i + 1), bx = __ldg(v + 2 * i + 2), by = __ldg(v + 2 * i + 3);
    // winding: upward / downward crossings of the horizontal ray, side by the sign of the cross product
    const double side = (bx - ax) * (py - ay) - (px - ax) * (by - ay);
    if (ay <= py) { if (by > py && side > 0) ++winding; }
    else if (by <= py && side < 0) --winding;
    const double vx = bx - ax, vy = by - ay, wx = px - ax, wy = py - ay;
    const double c1 = wx * vx + wy * vy;
    double d2;
    if (c1 <= 0) d2 = wx * wx + wy * wy;
    else {
      const double c2 = vx * vx + vy * vy;
      if (c2 <= c1) { const double ex = px - bx, ey = py - by; d2 = ex * ex + ey * ey; }
      else { const double b = c1 / c2, qx = ax + b * vx, qy = ay + b * vy, ex = px - qx, ey = py - qy; d2 = ex * ex + ey * ey; }
    }
    if (d2 == 0.0) touches = true;
    if (d2 < best) best = d2;
  }
  if (touches || winding != 0) return 0.0;
  return sqrt(best);
}
// thread = (instance, footstep state, foot) of a footstep plan ([b][state][2 + 4 n_ee]): index of the nearest polygon for a
// foot in contact, -1 for a foot in the air (footstep_plan_extractor.h:106-116) and for unused states
__global__ void __launch_bounds__(128) NearestPlaneKernel(const double* __restrict__ plan, const int* __restrict__ n_states, int max_states, int n_ee,
                                                          const int* __restrict__ poly_offset, int n_polys, const double* __restrict__ verts,
                                                          int* __restrict__ out, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int e = (int)(i % n_ee); const long long bs = i / n_ee; const int st = (int)(bs % max_states); const long long b = bs / max_states;
  const int V = 2 + 4 * n_ee;
  const double* rec = plan + (size_t)bs * V + 2 + 4 * e;
  int idx = -1;
  if (st < n_states[b] && rec[0] != 0.0) {
    double min_distance = 1.7976931348623157e308;   // std::numeric_limits<double>::max(), :70
    for (int k = 0; k < n_polys; ++k) {
      const int o = __ldg(poly_offset + k), cnt = __ldg(poly_offset + k + 1) - o;
      const double d = PolygonDistance(verts + 2 * (size_t)o, cnt, rec[1], rec[2]);
      if (d < min_distance) { min_distance = d; idx = k; }
    }
  }
  out[i] = idx;
}

// ---- constant runs (device_tables.h: ConstRun): the TMA engine copies iterate-independent stretches of the CSR value rows ----
// CTA = (run, tile): one bulk copy global -> shared of the run's values (mbarrier, complete_tx), then one bulk copy
// shared -> global per instance of the tile.  No register or LSU traffic for these bytes (6 % of config 2's Jacobian).
__device__ __noinline__ void ConstRunBody(const ConstRun* __restrict__ runs, const double* __restrict__ vals, int nnz, double* __restrict__ jac, int nb, double* smem, int run, int tile) {
  __shared__ __align__(8) unsigned long long mbar;
  const ConstRun r = runs[run];
  const unsigned bytes = (unsigned)r.len * 8u;
  const int b0 = tile * 32;
  if (threadIdx.x == 0) {
    const unsigned mb = SmemAddr(&mbar);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mb) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(SmemAddr(smem)), "l"(vals + r.src), "r"(bytes), "r"(mb) : "memory");
    unsigned done = 0;
    while (!done)
      asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0, %2; selp.u32 %0, 1, 0, p; }" : "=r"(done) : "r"(mb), "r"(2000u) : "memory");   // (suspend-time hint: the thread sleeps in the wait instead of spinning)
  }
  __syncthreads();   // the values are in shared memory (written by the async proxy, observed through the mbarrier by thread 0)
  if (threadIdx.x < 32 && b0 + (int)threadIdx.x < nb) {
    // evict-first like the st.global.cs of the pair loop: the values are consumed by the host / a solver, they must not push
    // XT, GT and the lists out of the L2
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                 ::"l"(jac + (size_t)(b0 + threadIdx.x) * nnz + r.off), "r"(SmemAddr(smem)), "r"(bytes), "l"(pol) : "memory");
    BulkCommit();
#if TWB_CONST_WAIT_ALL
    BulkWaitAll();
#else
    BulkWaitRead<0>();   // the CTA may retire once the engine has read the staging row (the writes complete before the grid does)
#endif
  }
}

#if TWB_FUSED
// One kernel writes a whole tile of rows: blockIdx.y = instance tile, blockIdx.x walks the tile's CTAs in row
// order — dynamic samples, range-of-motion samples, node groups.
template <int kNEE, bool kPhase>
__global__ void __launch_bounds__(kWarps * 32, TWB_CTAS) EvalOut(const Plan P, const double* __restrict__ XT, double* __restrict__ GT,
                                                              double* __restrict__ jac, int* __restrict__ status,
                                                              const int* __restrict__ terrain_ids, int default_terrain, int nb, unsigned flags) {
  extern __shared__ __align__(16) double out_smem[];
  const int n_dyn_ctas = (P.n_dyn + kWarps - 1) / kWarps, n_rom_ctas = (P.n_rom + kWarps - 1) / kWarps;
  int cta = blockIdx.x;
  if (cta < n_dyn_ctas) { DynBody<kNEE, kPhase>(P, XT, GT, jac, status, nb, flags, out_smem, cta, blockIdx.y, Stage{nullptr, 0}); return; }
  cta -= n_dyn_ctas;
  if (cta < n_rom_ctas) { RomBody<kNEE, kPhase>(P, XT, GT, jac, status, nb, flags, out_smem, cta, blockIdx.y, Stage{nullptr, 0}); return; }
  cta -= n_rom_ctas;
  NodeBody(P, XT, GT, jac, status, terrain_ids, default_terrain, nb, flags, out_smem, cta, blockIdx.y, Stage{nullptr, 0});
}
#else
template <int kNEE, bool kPhase>
__global__ void __launch_bounds__(kDynWarps * 32, TWB_DYN_CTAS) DynOut(const Plan P, const double* __restrict__ XT, double* __restrict__ GT,
                                                           double* __restrict__ jac, int* __restrict__ status, int nb, unsigned flags,
                                                           int stage_off, int stage_cap, const double* __restrict__ FS, double* __restrict__ g,
                                                           int* __restrict__ tile_done, int done_total) {
  extern __shared__ __align__(16) double out_smem[];
  DynBody<kNEE, kPhase>(P, XT, GT, jac, status, nb, flags, out_smem, blockIdx.x, blockIdx.y, Stage{out_smem + stage_off, stage_cap}, FS, g);
  TileDone(tile_done, done_total, XT, P.n, P.nc_jac, blockIdx.y, nb);
#if TWB_TMA
  if ((threadIdx.x & 31) == 0) BulkWaitAll();   // the staging rows stay allocated until the last copy has left
#endif
}
template <int kNEE, bool kPhase>
__global__ void __launch_bounds__(kRomWarps * 32, TWB_ROM_CTAS) RomOut(const Plan P, const double* __restrict__ XT, double* __restrict__ GT,
                                                           double* __restrict__ jac, int* __restrict__ status, int nb, unsigned flags) {
  extern __shared__ __align__(16) double out_smem[];
  RomBody<kNEE, kPhase>(P, XT, GT, jac, status, nb, flags, out_smem, blockIdx.x, blockIdx.y, Stage{nullptr, 0});
}
__global__ void __launch_bounds__(kNodeWarps * 32, TWB_NODE_CTAS) NodeOut(const Plan P, const double* __restrict__ XT, double* __restrict__ GT,
                                                           double* __restrict__ jac, int* __restrict__ status,
                                                           const int* __restrict__ terrain_ids, int default_terrain, int nb, unsigned flags) {
  extern __shared__ __align__(16) double out_smem[];
  NodeBody(P, XT, GT, jac, status, terrain_ids, default_terrain, nb, flags, out_smem, blockIdx.x, blockIdx.y, Stage{nullptr, 0});
}
#if TWB_ROMNODE   // range-of-motion and node CTAs of a tile in one kernel (kRomWarps == kNodeWarps), in row order
template <int kNEE, bool kPhase>
__global__ void __launch_bounds__(kRomWarps * 32, TWB_ROM_CTAS) RomNodeOut(const Plan P, const double* __restrict__ XT, double* __restrict__ GT,
                                                               double* __restrict__ jac, int* __restrict__ status,
                                                               const int* __restrict__ terrain_ids, int default_terrain, int nb, unsigned flags,
                                                               int stage_off, int stage_cap, double* __restrict__ g,
                                                               int* __restrict__ tile_done, int done_total) {
  extern __shared__ __align__(16) double out_smem[];
  static_assert(kRomWarps == kNodeWarps, "TWB_ROMNODE needs equal CTA sizes");
  const Stage st{out_smem + stage_off, stage_cap};
#if TWB_PDL
  asm volatile("griddepcontrol.wait;" ::: "memory");   // XT complete and visible (programmatic dependency on TransposeIn)
#endif
  const int n_rom_ctas = (P.n_rom + kRomWarps - 1) / kRomWarps;
  const int n_node_ctas = (P.n_groups + kNodeWarps - 1) / kNodeWarps;
  if ((int)blockIdx.x >= n_rom_ctas + n_node_ctas) {   // constant runs: TMA only
    if (flags & 2u) ConstRunBody(P.const_runs, P.const_vals, P.nnz, jac, nb, out_smem, blockIdx.x - n_rom_ctas - n_node_ctas, blockIdx.y);
    TileDone(tile_done, done_total, XT, P.n, P.nc_jac, blockIdx.y, nb);
    return;
  }
  if ((int)blockIdx.x < n_rom_ctas) RomBody<kNEE, kPhase>(P, XT, GT, jac, status, nb, flags, out_smem, blockIdx.x, blockIdx.y, st, g);
#ifndef TWB_EXP_NONODE   // (timing experiment: node CTAs return at once)
  else NodeBody(P, XT, GT, jac, status, terrain_ids, default_terrain, nb, flags, out_smem, blockIdx.x - n_rom_ctas, blockIdx.y, st, g);
#endif
#if TWB_TMA
  if ((threadIdx.x & 31) == 0) BulkWaitAll();
#endif
  TileDone(tile_done, done_total, XT, P.n, P.nc_jac, blockIdx.y, nb);
}
#endif
#endif

// number of tiles that cover nb instances (whole groups of nc interleaved tiles)
inline int TileTotal(int nc, int nb) { return nc * ((nb + 32 * nc - 1) / (32 * nc)); }

// kernel launch with the optional attributes of this pipeline: programmatic dependent launch, L2 access-policy window
template <class... KArgs, class... Args>
cudaError_t LaunchK(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl, Args... args) {
  cudaLaunchConfig_t cfg{}; cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[2]; unsigned na = 0;
  if (pdl) { attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization; attr[na].val.programmaticStreamSerializationAllowed = 1; ++na; }
  if (t_l2_window) { attr[na].id = cudaLaunchAttributeAccessPolicyWindow; attr[na].val.accessPolicyWindow = *t_l2_window; ++na; }
  cfg.attrs = attr; cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// s: caller's stream (after TransposeIn); a0, a1: auxiliary streams already waiting on the transposition
template <int kNEE, bool kPhase>
cudaError_t LaunchOut(const Plan& P, const double* XT, double* GT, double* FS, double* g_direct, int* tile_done_in, double* jac, int* status, const int* terrain_ids, int default_terrain,
                      int nb, unsigned flags, int tiles, cudaStream_t s, cudaStream_t a0, cudaStream_t a1, int* count) {
  const size_t row_bytes = (size_t)kLD * sizeof(double);
  const int dyn_rows = DynBlockRows(kNEE), rom_rows = RomBlockRowsP(kNEE, kPhase), node_rows = P.node_rows;
  cudaError_t e = cudaSuccess;
  // CTAs per tile of the two output kernels (the count that completes a tile's counter, TileDone)
  const int done_total = (P.n_dyn > 0 ? (P.n_dyn + kDynWarps - 1) / kDynWarps : 0) +
                         (P.n_rom + kRomWarps - 1) / kRomWarps + (P.n_groups + kNodeWarps - 1) / kNodeWarps + P.n_const_runs;
  int* tile_done = (TWB_ROMNODE && !TWB_FUSED) ? tile_done_in : nullptr;
#if !TWB_FUSED
  // the dynamic rows on stream a0: with optimised durations and a Jacobian evaluation first DynTailOut (the PhaseSpline columns; it
  // leaves the feet's positions and forces in FS), then DynOut (base columns and the constraint values)
  auto launch_dyn = [&]() -> cudaError_t {
    if (P.n_dyn <= 0) return cudaSuccess;
    cudaError_t err;
    const bool tail = kPhase && (flags & 2u);
    if (tail) {
      const size_t tail_smem = (size_t)kNEE * kTailRows * row_bytes;
      if ((err = cudaFuncSetAttribute(DynTailOut<kNEE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tail_smem)) != cudaSuccess) return err;
      DynTailOut<kNEE><<<dim3(P.n_dyn, tiles), kNEE * 32, tail_smem, a0>>>(P, XT, jac, nb, FS);
      ++*count; TWB_MARK("DynTailOut", a0);
    }
    const size_t state_bytes = (size_t)kDynWarps * dyn_rows * row_bytes;
    const int stage_off = (int)(state_bytes / sizeof(double));
    int stage_cap = TWB_TMA_DYN ? P.stage_dyn : 0;
    if (state_bytes + (size_t)kDynWarps * (TWB_TMA_BUF * TWB_TMA_G) * stage_cap * sizeof(double) > 200 * 1024) stage_cap = 0;
    const size_t smem = state_bytes + (size_t)kDynWarps * (TWB_TMA_BUF * TWB_TMA_G) * stage_cap * sizeof(double);
    if ((err = cudaFuncSetAttribute(DynOut<kNEE, kPhase>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return err;
    if ((err = LaunchK(DynOut<kNEE, kPhase>, dim3((P.n_dyn + kDynWarps - 1) / kDynWarps, tiles), dim3(kDynWarps * 32), smem, a0, false, P, XT, GT, jac, status, nb, flags,
                       stage_off, stage_cap, (const double*)(tail ? FS : nullptr), g_direct, tile_done, done_total)) != cudaSuccess) return err;
    ++*count; TWB_MARK("DynOut", a0);
    return cudaSuccess;
  };
#endif
#if TWB_FUSED
  const int n_ctas = (P.n_dyn + kWarps - 1) / kWarps + (P.n_rom + kWarps - 1) / kWarps + (P.n_groups + kWarps - 1) / kWarps;
  if (n_ctas == 0) return cudaSuccess;
  if (kPhase) return cudaErrorNotSupported;   // the fused experiment does not carry the PhaseSpline columns
  const int rows = std::max(std::max(P.n_dyn > 0 ? dyn_rows : 0, P.n_rom > 0 ? rom_rows : 0), P.n_groups > 0 ? node_rows : 0);
  const size_t smem = (size_t)kWarps * rows * row_bytes;
  if ((e = cudaFuncSetAttribute(EvalOut<kNEE, kPhase>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
  EvalOut<kNEE, kPhase><<<dim3(n_ctas, tiles), kWarps * 32, smem, s>>>(P, XT, GT, jac, status, terrain_ids, default_terrain, nb, flags);
  ++*count; TWB_MARK("EvalOut", s);
#else
#if TWB_ROMNODE
  {
    const size_t state_bytes = (size_t)kRomWarps * std::max(rom_rows, node_rows) * row_bytes;
    const int stage_off = (int)(state_bytes / sizeof(double));
    int stage_cap = TWB_TMA_ROM ? std::max(P.stage_rom, P.stage_node) : 0;
    if (state_bytes + (size_t)kRomWarps * (TWB_TMA_BUF * TWB_TMA_G) * stage_cap * sizeof(double) > 100 * 1024) stage_cap = 0;   // dense rows (optimised durations): st.global path
    const size_t smem = std::max(state_bytes + (size_t)kRomWarps * (TWB_TMA_BUF * TWB_TMA_G) * stage_cap * sizeof(double),
                                 P.n_const_runs > 0 ? (size_t)kConstRunMax * sizeof(double) : (size_t)0);
    if ((e = cudaFuncSetAttribute(RomNodeOut<kNEE, kPhase>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    const int n_ctas = (P.n_rom + kRomWarps - 1) / kRomWarps + (P.n_groups + kNodeWarps - 1) / kNodeWarps + P.n_const_runs;
    if (n_ctas > 0) {
      if ((e = LaunchK(RomNodeOut<kNEE, kPhase>, dim3(n_ctas, tiles), dim3(kRomWarps * 32), smem, s, TWB_PDL != 0, P, XT, GT, jac, status, terrain_ids,
                       default_terrain, nb, flags, stage_off, stage_cap, g_direct, tile_done, done_total)) != cudaSuccess) return e;
      ++*count; TWB_MARK("RomNodeOut", s);
    }
  }
  if ((e = launch_dyn()) != cudaSuccess) return e;
  return cudaSuccess;
#endif
  if (P.n_rom > 0) {
    const size_t smem = (size_t)kRomWarps * rom_rows * row_bytes;
    if ((e = cudaFuncSetAttribute(RomOut<kNEE, kPhase>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    RomOut<kNEE, kPhase><<<dim3((P.n_rom + kRomWarps - 1) / kRomWarps, tiles), kRomWarps * 32, smem, s>>>(P, XT, GT, jac, status, nb, flags);
    ++*count; TWB_MARK("RomOut", s);
  }
  if ((e = launch_dyn()) != cudaSuccess) return e;
  if (P.n_groups > 0) {
    const size_t smem = (size_t)kNodeWarps * node_rows * row_bytes;
    if ((e = cudaFuncSetAttribute(NodeOut, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    NodeOut<<<dim3((P.n_groups + kNodeWarps - 1) / kNodeWarps, tiles), kNodeWarps * 32, smem, a1>>>(P, XT, GT, jac, status, terrain_ids, default_terrain, nb, flags);
    ++*count; TWB_MARK("NodeOut", a1);
  }
#endif
  return cudaSuccess;
}

}  // namespace

// ---- host launchers ------------------------------------------------------------------

int LaunchTrajectory(const Plan& P, const double* x, double* XT, const SplineSample* samples, const int* contact, int n_steps,
                     double* out, int nb, cudaStream_t s) {
  if (nb <= 0 || n_steps <= 0) return 0;
  const int tiles = TileTotal(P.nc_jac, nb);
  TransposeIn<<<dim3((P.n + 32 * kTinTiles - 1) / (32 * kTinTiles), tiles), dim3(32, 8), 0, s>>>(x, XT, nullptr, P.n, nb, P.nc_jac);
  const dim3 grid((n_steps + 3) / 4, tiles);
  const bool phase = P.n_phase_defs > 0;
  // dynamic shared memory: the four warps' staging tiles [19 + 13 n_ee][33] of the coalesced stores
#define TWB_TRAJ(NEE) { const size_t sm = 4 * (size_t)(19 + 13 * NEE) * 33 * sizeof(double);                                                     \
    if (phase) { cudaFuncSetAttribute(TrajectoryKernel<NEE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);                       \
                 TrajectoryKernel<NEE, true><<<grid, 128, sm, s>>>(P, XT, samples, contact, n_steps, out, nb); }                                 \
    else { cudaFuncSetAttribute(TrajectoryKernel<NEE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);                            \
           TrajectoryKernel<NEE, false><<<grid, 128, sm, s>>>(P, XT, samples, contact, n_steps, out, nb); } }
  switch (P.n_ee) {
    case 1: TWB_TRAJ(1); break;
    case 2: TWB_TRAJ(2); break;
    case 4: TWB_TRAJ(4); break;
    default: return (int)cudaErrorInvalidValue;
  }
#undef TWB_TRAJ
  return (int)cudaGetLastError();
}

int LaunchInitialGuess(const Plan& P, const double* x, double* XT, const SplineSample* samples, const double* times, int n_times,
                       double* out, int nb, cudaStream_t s) {
  if (nb <= 0 || n_times <= 0) return 0;
  const int tiles = TileTotal(P.nc_jac, nb);
  TransposeIn<<<dim3((P.n + 32 * kTinTiles - 1) / (32 * kTinTiles), tiles), dim3(32, 8), 0, s>>>(x, XT, nullptr, P.n, nb, P.nc_jac);
  const dim3 grid((n_times + 3) / 4, tiles);
  const bool phase = P.n_phase_defs > 0;
#define TWB_IG(NEE) { const size_t sm = 4 * (size_t)49 * 33 * sizeof(double);                                                                    \
    if (phase) { cudaFuncSetAttribute(InitialGuessKernel<NEE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);                     \
                 InitialGuessKernel<NEE, true><<<grid, 128, sm, s>>>(P, XT, samples, times, n_times, out, nb); }                                 \
    else { cudaFuncSetAttribute(InitialGuessKernel<NEE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);                          \
           InitialGuessKernel<NEE, false><<<grid, 128, sm, s>>>(P, XT, samples, times, n_times, out, nb); } }
  switch (P.n_ee) {
    case 1: TWB_IG(1); break;
    case 2: TWB_IG(2); break;
    case 4: TWB_IG(4); break;
    default: return (int)cudaErrorInvalidValue;
  }
#undef TWB_IG
  return (int)cudaGetLastError();
}

int LaunchFootstepPlan(const Plan& P, const double* x, double* XT, const SplineSample* samples, const double* times, const int* contact,
                       const int* codes, int n_codes, int n_steps, double time_horizon, int max_states, int* n_states, double* out, int nb,
                       cudaStream_t s) {
  if (nb <= 0 || max_states <= 0) return 0;
  const int tiles = TileTotal(P.nc_jac, nb);
  TransposeIn<<<dim3((P.n + 32 * kTinTiles - 1) / (32 * kTinTiles), tiles), dim3(32, 8), 0, s>>>(x, XT, nullptr, P.n, nb, P.nc_jac);
  const bool phase = P.n_phase_defs > 0;
  // dynamic shared memory per warp: the staging tile [V][33] of the coalesced stores; optimised durations: the change codes [max_states + 1][32]
#define TWB_FSP(NEE) { const size_t sm = 4 * ((size_t)(2 + 4 * NEE) * 33 * sizeof(double) + (phase ? (size_t)(max_states + 1) * 32 * sizeof(int) : 0)); \
    if (phase) { cudaFuncSetAttribute(FootstepPlanKernel<NEE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);                           \
                 FootstepPlanKernel<NEE, true><<<(tiles + 3) / 4, 128, sm, s>>>(P, XT, samples, times, contact, codes, n_codes, n_steps,            \
                                                                                 time_horizon, max_states, tiles, n_states, out, nb); }             \
    else { cudaFuncSetAttribute(FootstepPlanKernel<NEE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);                                \
           FootstepPlanKernel<NEE, false><<<(tiles + 3) / 4, 128, sm, s>>>(P, XT, samples, times, contact, codes, n_codes, n_steps,                  \
                                                                            time_horizon, max_states, tiles, n_states, out, nb); } }
  switch (P.n_ee) {
    case 1: TWB_FSP(1); break;
    case 2: TWB_FSP(2); break;
    case 4: TWB_FSP(4); break;
    default: return (int)cudaErrorInvalidValue;
  }
#undef TWB_FSP
  return (int)cudaGetLastError();
}

int LaunchNearestPlanes(const double* plan, const int* n_states, int max_states, int n_ee, const int* poly_offset, int n_polys,
                        const double* verts, int* out, int nb, cudaStream_t s) {
  const long long total = (long long)nb * max_states * n_ee;
  if (total <= 0) return 0;
  NearestPlaneKernel<<<(unsigned)((total + 127) / 128), 128, 0, s>>>(plan, n_states, max_states, n_ee, poly_offset, n_polys, verts, out, total);
  return (int)cudaGetLastError();
}

// ---- the two components outside Parameters::ConstraintName: LinearEqualityConstraint and SoftConstraint -----------------
// towr::LinearEqualityConstraint::GetValues (linear_constraint.cc:46-51): g = M x_set, thread = (row, instance), lane = instance
__global__ void __launch_bounds__(128) LinearEqualityKernel(const double* __restrict__ XT, int n, int col0, int n_cols, const double* __restrict__ M,
                                                            int rows, double* __restrict__ g, int nb, int nc) {
  const int b = TileInstance(nc, blockIdx.y, threadIdx.x & 31), r = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const ConstCol xs = TileCol(XT, blockIdx.y, threadIdx.x & 31, n + 1);
  double acc = 0.0;
  for (int c = 0; c < n_cols; ++c) acc += __ldg(M + (size_t)r * n_cols + c) * xs[col0 + c];   // Eigen's dense row-times-vector order
  if (b < nb) g[(size_t)b * rows + r] = acc;
}
// towr::SoftConstraint (soft_constraint.cc:53-72): cost = 0.5 (g - b)^T W (g - b), gradient = J^T W (g - b) of one constraint
// set (rows row0 .. row0 + n_rows - 1 of g / the CSR); block = instance, the gradient is accumulated in shared memory
__global__ void __launch_bounds__(128) SoftConstraintKernel(const double* __restrict__ g, const double* __restrict__ jac, const int* __restrict__ row_ptr,
                                                            const int* __restrict__ col_idx, int n, int m, int nnz, int row0, int n_rows,
                                                            const double* __restrict__ b_avg, const double* __restrict__ w,
                                                            double* __restrict__ cost, double* __restrict__ grad, int nb) {
  extern __shared__ double acc[];   // [n] gradient | [128] partial costs
  const int b = blockIdx.x;
  if (b >= nb) return;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc[i] = 0.0;
  __syncthreads();
  double part = 0.0;
  for (int r = threadIdx.x; r < n_rows; r += blockDim.x) {
    const double d = g[(size_t)b * m + row0 + r] - b_avg[r], wd = w[r] * d;
    part += d * wd;
    for (int k = __ldg(row_ptr + row0 + r); k < __ldg(row_ptr + row0 + r + 1); ++k) atomicAdd(acc + __ldg(col_idx + k), jac[(size_t)b * nnz + k] * wd);
  }
  acc[n + threadIdx.x] = part;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) grad[(size_t)b * n + i] = acc[i];
  if (threadIdx.x == 0) { double c = 0.0; for (int i = 0; i < (int)blockDim.x; ++i) c += acc[n + i]; cost[b] = 0.5 * c; }
}
int LaunchLinearEquality(const Plan& P, const double* x, double* XT, int col0, int n_cols, const double* M, int rows, double* g, int nb, cudaStream_t s) {
  if (nb <= 0 || rows <= 0) return 0;
  const int tiles = TileTotal(P.nc_jac, nb);
  TransposeIn<<<dim3((P.n + 32 * kTinTiles - 1) / (32 * kTinTiles), tiles), dim3(32, 8), 0, s>>>(x, XT, nullptr, P.n, nb, P.nc_jac);
  LinearEqualityKernel<<<dim3((rows + 3) / 4, tiles), 128, 0, s>>>(XT, P.n, col0, n_cols, M, rows, g, nb, P.nc_jac);
  return (int)cudaGetLastError();
}
int LaunchSoftConstraint(const Plan& P, const double* g, const double* jac, const int* row_ptr, const int* col_idx, int row0, int n_rows,
                         const double* b_avg, const double* w, double* cost, double* grad, int nb, cudaStream_t s) {
  if (nb <= 0) return 0;
  SoftConstraintKernel<<<nb, 128, (P.n + 128) * sizeof(double), s>>>(g, jac, row_ptr, col_idx, P.n, P.m, P.nnz, row0, n_rows, b_avg, w, cost, grad, nb);
  return (int)cudaGetLastError();
}

// ---- batched setup (SURVEY 8f-3): x0 and variable bounds of goal-randomised instances, block = instance ------------------
// NlpFormulation::GetVariableSets (nlp_formulation.cc:95-181) through the per-variable recipe Plan::goal_vars; the terrain
// under the goal is the instance's own (per-instance id, height grids included — which the host path cannot serve).
__global__ void __launch_bounds__(128) GoalInstanceKernel(const Plan P, const GoalSetup S, const double* __restrict__ goals, const int* __restrict__ terrain_ids,
                                                          int default_terrain, double* __restrict__ x0, double* __restrict__ lo, double* __restrict__ up, int nb) {
  __shared__ double a_[2 + 2 * kMaxEE][3], b_[2 + 2 * kMaxEE][3];   // (initial, final) per set: lin, ang, motion_e.., force_e..
  const int b = blockIdx.x;
  if (b >= nb) return;
  const double* gp = goals + 6 * (size_t)b;
  const int terrain = terrain_ids ? __ldg(terrain_ids + b) : default_terrain;
  if (threadIdx.x == 0) {
    const double fx = gp[0], fy = gp[1];
    const double fz = EvalTerrain(P, terrain, fx, fy).h - S.nominal[0][2];
    const double fin[3] = {fx, fy, fz};
    for (int d = 0; d < 3; ++d) { a_[0][d] = S.initial_lin[d]; b_[0][d] = fin[d]; a_[1][d] = S.initial_ang[d]; b_[1][d] = gp[3 + d]; }
  } else if ((int)threadIdx.x <= P.n_ee) {
    const int e = threadIdx.x - 1;
    double sz, cz; sincos(gp[5], &sz, &cz);   // yaw-only rotation of the nominal stance (EulerConverter::GetRotationMatrixBaseToWorld with x = y = 0)
    const double* nom = S.nominal[e];
    const double R[3][3] = {{cz, -sz, 0.0}, {sz, cz, 0.0}, {-0.0, 0.0, 1.0}};
    double w[3];
    for (int i = 0; i < 3; ++i) w[i] = gp[i] + (R[i][0] * nom[0] + R[i][1] * nom[1] + R[i][2] * nom[2]);
    const double goal[3] = {w[0], w[1], EvalTerrain(P, terrain, w[0], w[1]).h};
    for (int d = 0; d < 3; ++d) {
      a_[2 + e][d] = S.initial_ee[e][d]; b_[2 + e][d] = goal[d];
      a_[2 + kMaxEE + e][d] = b_[2 + kMaxEE + e][d] = (d == 2) ? S.f_stance_z : 0.0;
    }
  }
  __syncthreads();
  const double inf = 1e20;
  for (int i = threadIdx.x; i < P.n; i += blockDim.x) {
    const GoalVar v = P.goal_vars[i];
    double x, l = -inf, u = inf;
    if (v.kind == kGoalConst) x = v.frac;
    else {
      const int set = v.kind == kGoalLin ? 0 : v.kind == kGoalAng ? 1 : v.kind == kGoalMotion ? 2 + v.ee : 2 + kMaxEE + v.ee;
      const double a = a_[set][v.dim], dp = b_[set][v.dim] - a;
      x = v.deriv == 0 ? a + v.frac * dp : dp / S.t_total;
    }
    if (v.bound == kBoundConst) l = u = v.c0;
    else if (v.bound == kBoundGoalLin) l = u = gp[v.dim];
    else if (v.bound == kBoundGoalAng) l = u = gp[3 + v.dim];
    else if (v.bound == kBoundPair) { l = v.c0; u = v.c1; }
    const size_t o = (size_t)b * P.n + i;
    if (x0) x0[o] = x;
    if (lo) lo[o] = l;
    if (up) up[o] = u;
  }
}
int LaunchGoalInstances(const Plan& P, const GoalSetup& S, const double* goals, const int* terrain_ids, int default_terrain, double* x0, double* lo,
                        double* up, int nb, cudaStream_t s) {
  if (nb <= 0) return 0;
  GoalInstanceKernel<<<nb, 128, 0, s>>>(P, S, goals, terrain_ids, default_terrain, x0, lo, up, nb);
  return (int)cudaGetLastError();
}

// 1 when the constraint values go through GT and the TransposeOut kernel (optimised durations, experimental variants), else 0
int TransposeOutPerEval(const Plan& P) { return (TWB_GDIRECT && TWB_ROMNODE && !TWB_FUSED && (TWB_GDIRECT_PHASE || P.n_phase_defs == 0)) ? 0 : 1; }
int OutKernelsPerEval(const Plan& P, unsigned flags) {
  const int dyn = (P.n_dyn > 0) * ((P.n_phase_defs > 0 && (flags & 2u)) ? 2 : 1);   // DynOut [+ DynTailOut]
#if TWB_FUSED
  (void)dyn; return (P.n_dyn + P.n_rom + P.n_groups) > 0;
#elif TWB_ROMNODE
  return dyn + ((P.n_rom + P.n_groups) > 0);
#else
  return dyn + (P.n_rom > 0) + (P.n_groups > 0);
#endif
}

// XT / GT are the instance-tiled iterate and constraint-value matrices of the whole batch (first tile = first
// instance of x / g / jac).  Streams: `s` carries TransposeIn -> [out kernels] -> TransposeOut; with separate
// out kernels DynOut / NodeOut (and the CostKernel) run beside RomOut on aux0 / aux1 after the transposition
// (ev[0]) and are joined back into `s` (ev[1], ev[2]) before TransposeOut.
int LaunchEval(const Plan& P, const double* x, double* XT, double* GT, double* FS, int* TD, double* g, double* jac, double* cost, double* grad,
               int* status, const int* terrain_ids, int default_terrain, int nb, unsigned flags, cudaStream_t s,
               cudaStream_t aux0, cudaStream_t aux1, cudaEvent_t* ev, int* launches) {
  if (nb <= 0) return 0;
  int count = 0;
  const bool serial = (g_after_launch != nullptr);
  if (serial) aux0 = aux1 = s;
  const int tiles = TileTotal(P.nc_jac, nb);
  const unsigned out_flags = flags & 3u;
  const bool want_cost = (flags & 4u) && P.n_cost > 0;
  TWB_MARK("begin", s);
#if TWB_TIN_PERSIST
  {
    const int n_ctiles = (P.n + 31) / 32, total = n_ctiles * tiles;
    LaunchK(TransposeInP, dim3(std::min(total, 148 * TWB_TIN_PERSIST)), dim3(32, 8), 0, s, false, x, XT, status, P.n, nb, P.nc_jac, n_ctiles, total); ++count; TWB_MARK("TransposeIn", s);
  }
#else
  LaunchK(TransposeIn, dim3((P.n + 32 * kTinTiles - 1) / (32 * kTinTiles), tiles), dim3(32, 8), 0, s, false, x, XT, status, P.n, nb, P.nc_jac); ++count; TWB_MARK("TransposeIn", s);
#endif
  const bool fork = !serial && (want_cost || (!TWB_FUSED && out_flags));
  if (fork) { cudaEventRecord(ev[0], s); cudaStreamWaitEvent(aux0, ev[0], 0); cudaStreamWaitEvent(aux1, ev[0], 0); }
  cudaError_t e = cudaSuccess;
  // fixed durations: the output kernels write the constraint values straight into g (no GT, no TransposeOut)
  const bool direct = TWB_GDIRECT && TWB_ROMNODE && !TWB_FUSED && (TWB_GDIRECT_PHASE || P.n_phase_defs == 0);
  double* g_direct = (direct && (out_flags & 1u)) ? g : nullptr;
  if (out_flags) {
    const bool phase = P.n_phase_defs > 0;
    switch (P.n_ee) {
      case 1: e = phase ? LaunchOut<1, true>(P, XT, GT, FS, g_direct, direct ? TD : nullptr, jac, status, terrain_ids, default_terrain, nb, out_flags, tiles, s, aux0, aux1, &count)
                       : LaunchOut<1, false>(P, XT, GT, FS, g_direct, direct ? TD : nullptr, jac, status, terrain_ids, default_terrain, nb, out_flags, tiles, s, aux0, aux1, &count); break;
      case 2: e = phase ? LaunchOut<2, true>(P, XT, GT, FS, g_direct, direct ? TD : nullptr, jac, status, terrain_ids, default_terrain, nb, out_flags, tiles, s, aux0, aux1, &count)
                       : LaunchOut<2, false>(P, XT, GT, FS, g_direct, direct ? TD : nullptr, jac, status, terrain_ids, default_terrain, nb, out_flags, tiles, s, aux0, aux1, &count); break;
      case 4: e = phase ? LaunchOut<4, true>(P, XT, GT, FS, g_direct, direct ? TD : nullptr, jac, status, terrain_ids, default_terrain, nb, out_flags, tiles, s, aux0, aux1, &count)
                       : LaunchOut<4, false>(P, XT, GT, FS, g_direct, direct ? TD : nullptr, jac, status, terrain_ids, default_terrain, nb, out_flags, tiles, s, aux0, aux1, &count); break;
      default: return (int)cudaErrorInvalidValue;
    }
    if (e != cudaSuccess) return (int)e;
  }
  if (out_flags && P.n_phase_units > 0) {   // TotalDurationConstraint rows: needs XT only, beside the output kernels on the third stream
    switch (P.n_ee) {
      case 1: PhaseJac<1><<<tiles, 32, 0, aux1>>>(P, XT, GT, g_direct, jac, status, nb, out_flags); break;
      case 2: PhaseJac<2><<<tiles, 32, 0, aux1>>>(P, XT, GT, g_direct, jac, status, nb, out_flags); break;
      default: PhaseJac<4><<<tiles, 32, 0, aux1>>>(P, XT, GT, g_direct, jac, status, nb, out_flags); break;
    }
    ++count; TWB_MARK("PhaseJac", aux1);
  }
  if (want_cost) {
    if (grad) cudaMemsetAsync(grad, 0, sizeof(double) * (size_t)nb * P.n, aux1);
    CostKernel<<<(nb + 127) / 128, 128, 0, aux1>>>(P, XT, cost, grad, nb); ++count; TWB_MARK("CostKernel", aux1);
  }
  if (fork) {
    cudaEventRecord(ev[1], aux0); cudaEventRecord(ev[2], aux1);
    cudaStreamWaitEvent(s, ev[1], 0); cudaStreamWaitEvent(s, ev[2], 0);
  }
  if ((out_flags & 1u) && !direct) { LaunchK(TransposeOut, dim3((P.m + 31) / 32, tiles), dim3(32, 8), 0, s, false, (const double*)GT, g, P.m, nb, XT, P.n, P.nc_jac); ++count; TWB_MARK("TransposeOut", s); }
  if (launches) *launches += count;
  return (int)cudaGetLastError();
}

}  // namespace twb
