// grf_math.cuh -- the per-robot arithmetic of Dynamiccclass (GO1/src/whole_body_dynamics/dynmics_compute.cpp), shared by
// every kernel that runs it:
//   force_distribution, force_opt + solve_grf_opt, compute_joint_torques   grf_qp.cu (the single-stage entries)
//   all three, K servo ticks per robot                                      servo_torque.cu (servo_torque_kernel)
// grf_qp.cu is built with FMA contraction, servo_torque.cu with -fmad=false (it runs servo_math.cuh).  So that both compute
// the same bits, every multiply-add here is written out: fma(a, b, c) where the contracting build fuses it, __dmul_rn /
// __dadd_rn where the reference's order is kept unfused; no a*b+c is left for the compiler to decide.
#pragma once
#include <cuda_runtime.h>
#define GO1_GI_FMA      // gi_warp.cuh's multiply-adds as fma(), as grf_qp.cu has always compiled them
#include "gi_warp.cuh"
#include "kernels.h"

namespace go1 {

constexpr int GN = 12, GP = 12, GM = 24;   // force QP: 12 variables, 12 equality columns, 24 inequalities

// Legs that carry no force (:315-350), bit l = FR, FL, RR, RL: the force QP's equality rows, and the swing legs of the
// torque map in servo_torque_kernel.
__device__ __forceinline__ unsigned grf_zero_legs(int mode, int right_support) {
  unsigned zero_legs = 0u;
  if (mode == 102) zero_legs = (right_support == 0) ? 0x6u : ((right_support == 1) ? 0x9u : 0u);
  else if (mode == 101) zero_legs = (right_support == 0) ? 0x5u : ((right_support == 1) ? 0xAu : 0u);
  return zero_legs;
}

// dense policy of gi_loop over shared-memory matrices (column-major, one constraint per column)
struct GrfSmemPolicy {
  const double *CI, *ci0, *CE, *ce0v;
  int n, m;
  __device__ __forceinline__ void eval_s(const GiWs& w, int lane, double& psi) const {
    for (int c = lane; c < m; c += 32) {
      const double* col = CI + c * n;
      double acc = 0.0;
      for (int j = 0; j < n; j++) acc = fma(col[j], w.x[j], acc);
      const double sv = acc + ci0[c];
      w.s[c] = sv;
      psi += fmin(0.0, sv);
    }
  }
  __device__ __forceinline__ void load_np(const GiWs& w, int ip, int lane, int& klo, int& khi) const {
    for (int j = lane; j < n; j += 32) w.np[j] = CI[ip * n + j];
    klo = 0; khi = n;
    __syncwarp();
  }
  __device__ __forceinline__ double eval_one(const GiWs& w, int ip, int lane) const {
    double acc = 0.0;
    for (int j = lane; j < n; j += 32) acc = fma(CI[ip * n + j], w.x[j], acc);
    return warp_sum(acc) + ci0[ip];
  }
  __device__ __forceinline__ void load_eq(const GiWs& w, int i, int lane, bool& allzero) const {
    bool z = true;
    for (int j = lane; j < n; j += 32) { const double v = CE[i * n + j]; w.np[j] = v; z = z && (fabs(v) <= 1e-12); }
    allzero = __all_sync(FULL_MASK, z);
    __syncwarp();
  }
  __device__ __forceinline__ double ce0(int i) const { return ce0v[i]; }
};

// CTA-shared inequality data of the force QP in smem: CI = -qp_H' (12 x 24), then ci0 = qp_h (24).  Every thread of the CTA
// calls it.
__device__ __forceinline__ void grf_ci_build(double* CI, double fz_max, double mu) {
  double* ci0 = CI + GN * GM;
  for (int t = threadIdx.x; t < GN * GM + GM; t += blockDim.x) CI[t] = 0.0;
  __syncthreads();
  if (threadIdx.x < 4) {
    const int i = threadIdx.x;
    // rows 2i, 2i+1: -fz <= 0, fz <= fz_max; rows 8+2i(+1): -+fx - mu fz <= 0; rows 16+2i(+1): -+fy - mu fz <= 0
    CI[(2 * i) * GN + 3 * i + 2] = 1.0;           CI[(2 * i + 1) * GN + 3 * i + 2] = -1.0;  ci0[2 * i + 1] = fz_max;
    CI[(8 + 2 * i) * GN + 3 * i] = 1.0;           CI[(8 + 2 * i) * GN + 3 * i + 2] = mu;
    CI[(8 + 2 * i + 1) * GN + 3 * i] = -1.0;      CI[(8 + 2 * i + 1) * GN + 3 * i + 2] = mu;
    CI[(16 + 2 * i) * GN + 3 * i + 1] = 1.0;      CI[(16 + 2 * i) * GN + 3 * i + 2] = mu;
    CI[(16 + 2 * i + 1) * GN + 3 * i + 1] = -1.0; CI[(16 + 2 * i + 1) * GN + 3 * i + 2] = mu;
  }
  __syncthreads();
}

// What one force QP ended with, in registers on every lane: its status (diag word 0) and whether x held a NaN, so that the
// closed-form guess was returned (diag word 6 = 0)
struct GrfQpOutcome { int status; bool nan; };

// force_opt (:265-373) + solve_grf_opt (:387-427) for one robot, one warp.  recs: the robot's 48-double record in the layout of
// GrfKParams::in (shared memory); A (6 x 12), g0, CE, ce0: the warp's scratch; w: its QP workspace.  Writes out[0..16) in
// GrfKParams::out's layout and, when dg is non-null, the 32 diagnostic ints; returns the outcome.
__device__ __forceinline__ GrfQpOutcome grf_force_opt_warp(const GrfKParams& P, const double* CI, const GiWs& w, double* A, double* g0,
                                                   double* CE, double* ce0, const double* recs, double* out, int* dg, int lane) {
  const double* ci0 = CI + GN * GM;
  auto field = [&](int k) -> double { return recs[k]; };
  const double base_x = field(0);
  const int mode = (int)field(45), right_support = (int)field(46);
  // A = [I I I I; W_FR W_FL W_RR W_RL], W from skew_hat with its comma-operator reading of vec_w[0]
  for (int t = lane; t < 72; t += 32) {
    const int col = t / 6, r = t - 6 * col, l = col / 3, k = col - 3 * l;
    double v;
    if (r < 3) v = (r == k) ? 1.0 : 0.0;
    else {
      const double w0 = base_x - field(3 + 3 * l);
      const int rr = r - 3;
      v = (rr == k) ? 0.0 : (((k - rr + 3) % 3 == 1) ? -w0 : w0);    // [0 -w w; w 0 -w; -w w 0]
    }
    A[t] = v;
  }
  for (int t = lane; t < GN * GP; t += 32) CE[t] = 0.0;
  if (lane < GP) ce0[lane] = 0.0;
  __syncwarp();
  const unsigned zero_legs = grf_zero_legs(mode, right_support);
  if (lane < GN && ((zero_legs >> (lane / 3)) & 1u)) CE[lane * GN + lane] = 1.0;
  // G = sym(2 (alpha A'A + (beta + gama) I)) into w.R (lower triangle is what the factorisation reads)
  double tr = 0.0;
  for (int t = lane; t < GN * GN; t += 32) {
    const int j = t / GN, i = t - GN * j;
    double a1 = 0.0, a2 = 0.0;
    for (int r = 0; r < 6; r++) { a1 = fma(P.qp_alpha * A[i * 6 + r], A[j * 6 + r], a1); a2 = fma(P.qp_alpha * A[j * 6 + r], A[i * 6 + r], a2); }
    const double unit = (i == j) ? 1.0 : 0.0;
    const double hij = fma(P.qp_beta + P.qp_gama, unit, a1), hji = fma(P.qp_beta + P.qp_gama, unit, a2);
    const double g = fma(2.0, hij, 2 * hji) / 2.0;    // (qji + qij) / 2 with q = 2 h, qij's product fused into the sum
    w.R[j * w.ld + i] = g;
    if (i == j) tr += g;
  }
  const double c1 = warp_sum(tr);
  if (lane < GN) {
    double acc = 0.0;
    for (int r = 0; r < 6; r++) acc = fma(P.qp_alpha * A[lane * 6 + r], field(15 + r), acc);
    g0[lane] = -2 * fma(P.qp_gama, field(33 + lane), fma(P.qp_beta, field(21 + lane), acc));
  }
  for (int t = lane; t < GN * w.ld; t += 32) w.J[t] = 0.0;
  if (lane < GN) w.x[lane] = field(33 + lane);
  __syncwarp();
  GiResult res; res.f = 0.0; res.iq = 0; res.status = ST_OK;
  res.it_outer = res.it_add = res.it_drop = res.it_degen = res.it_l2a = 0; res.flops = gi_flops_setup(GN, GP);
  const bool pd = gi_llt(w, GN, lane);
  if (!pd) { res.status = ST_NOT_PD; res.f = CUDART_INF; }
  else {
    gi_inv_lt(w, GN, 0, lane);
    double c2 = (lane < GN) ? w.J[lane * w.ld + lane] : 0.0;
    c2 = warp_sum(c2);
    for (int t = lane; t < GN * w.ld; t += 32) w.R[t] = 0.0;
    if (lane < GN) w.np[lane] = g0[lane];
    __syncwarp();
    gi_compute_d(w, 0, GN, lane);
    gi_update_z(w, 0, lane);
    double f = 0.0;
    if (lane < GN) { const double xv = -w.z[lane]; w.x[lane] = xv; f = g0[lane] * xv; }
    res.f = 0.5 * warp_sum(f);
    __syncwarp();
    GrfSmemPolicy pol{CI, ci0, CE, ce0, GN, GM};
    gi_loop(w, pol, c1, c2, P.cap, res, lane);
  }
  // qp_solution = "no NaN in X"; on failure the reference falls back to the closed-form guess (:364-367)
  bool nan = (lane < GN) && (w.x[lane] != w.x[lane]);
  nan = __any_sync(FULL_MASK, nan);
  if (nan && (res.status == ST_OK || res.status == ST_EQ_DEP)) res.status = ST_NAN;
  const double guess = field(21 + (lane % GN));
  if (lane < GN) out[lane] = nan ? guess : w.x[lane];
  if (lane == 0) { out[12] = res.f; out[13] = nan ? 0.0 : 1.0; out[14] = 0.0; out[15] = 0.0; }
  if (dg) {
    if (lane == 0) { dg[0] = res.status; dg[1] = pd ? res.iq : 0; dg[2] = res.it_outer; dg[3] = res.it_add; dg[4] = res.it_drop; dg[5] = res.it_degen; dg[6] = nan ? 0 : 1; dg[7] = 0; }
    if (lane < 24) dg[8 + lane] = (pd && lane < res.iq) ? w.A[lane] : -99;
  }
  return GrfQpOutcome{res.status, nan};
}

// force_distribution (:141-261) for one robot: com [3], leg [12] (FR, FL, RR, RL xyz), F [6] (L xyz, R xyz), rf / lf [3]
// -> out [12] (FR, FL, RR, RL xyz), every entry written for gait modes 101 / 102; other modes leave out as it is.
__device__ __forceinline__ void grf_distribute(int mode, double yc, const double com[3], const double leg[12], const double F[6],
                                               const double rf[3], const double lf[3], double out[12]) {
#define FR_(r, c) out[(c) * 3 + (r)]
  if (mode == 101) {
    double dis[4];
    for (int l = 0; l < 4; l++) {
      const double a = com[0] - leg[3 * l], bb = com[1] - leg[3 * l + 1], cc = com[2] - leg[3 * l + 2];
      dis[l] = sqrt(fma(cc, cc, fma(a, a, bb * bb)));
    }
    const double FRd = dis[0], FLd = dis[1], RRd = dis[2], RLd = dis[3];
    double f;
    f = F[0] * FLd / (FLd + RLd);       FR_(0, 3) = f; FR_(0, 1) = F[0] - f;
    f = F[1] * FLd / (FLd + RLd) * yc;  FR_(1, 3) = f; FR_(1, 1) = fma(F[1], yc, -f);
    f = F[2] * FLd / (FLd + RLd);       FR_(2, 3) = f; FR_(2, 1) = F[2] - f;
    f = F[3] * FRd / (FRd + RRd);       FR_(0, 2) = f; FR_(0, 0) = F[3] - f;
    f = F[4] * FRd / (FRd + RRd) * yc;  FR_(1, 2) = f; FR_(1, 0) = fma(F[4], yc, -f);
    f = F[5] * FRd / (FRd + RRd);       FR_(2, 2) = f; FR_(2, 0) = F[5] - f;
  } else if (mode == 102) {
    double v[3], w[3], f;
    for (int k = 0; k < 3; k++) { v[k] = leg[9 + k] - leg[k]; w[k] = lf[k] - leg[k]; }
    double len = sqrt(fma(v[2], v[2], fma(v[0], v[0], v[1] * v[1])));
    double prj = fma(v[2], w[2], fma(v[0], w[0], v[1] * w[1]));
    double r = fmax(fmin(prj / len, 1.0), 0.0);
    f = F[0] * r;       FR_(0, 3) = f; FR_(0, 0) = F[0] - f;
    f = F[1] * r * yc;  FR_(1, 3) = f; FR_(1, 0) = fma(F[1], yc, -f);
    f = F[2] * r;       FR_(2, 3) = f; FR_(2, 0) = F[2] - f;
    for (int k = 0; k < 3; k++) { v[k] = leg[6 + k] - leg[3 + k]; w[k] = rf[k] - leg[3 + k]; }
    len = sqrt(fma(v[2], v[2], fma(v[0], v[0], v[1] * v[1])));
    prj = fma(v[2], w[2], fma(v[0], w[0], v[1] * w[1]));
    r = fmax(fmin(prj / len, 1.0), 0.0);
    f = F[3] * r;       FR_(0, 2) = f; FR_(0, 1) = F[3] - f;
    f = F[4] * r * yc;  FR_(1, 2) = f; FR_(1, 1) = fma(F[4], yc, -f);
    f = F[5] * r;       FR_(2, 2) = f; FR_(2, 1) = F[5] - f;
  }
#undef FR_
}

// compute_joint_torques (:109-138), the reference's operation order without FMA.  Swing leg: w = swing_kp (p_des - p_est) +
// swing_kd (pv_des - pv_est), one component; a stance leg's w is its force.
__device__ __forceinline__ double grf_swing_w(double kp, double kd, double p_des, double p_est, double pv_des, double pv_est) {
  return __dadd_rn(__dmul_rn(kp, __dsub_rn(p_des, p_est)), __dmul_rn(kd, __dsub_rn(pv_des, pv_est)));
}
// tau_i of leg `leg` = -(column i of Jaco)' w + gravity_compensate(i, leg); j[r] = Jaco(r, i)
__device__ __forceinline__ double grf_tau(int leg, int i, const double j[3], const double w[3]) {
  double acc = 0.0;
  for (int r = 0; r < 3; r++) acc = __dadd_rn(acc, __dmul_rn(-j[r], w[r]));
  const double grav = (i == 0) ? ((leg & 1) ? 0.80 : -0.80) : 0.0;    // gravity_compensate, dynmics_compute.cpp:39-41
  return __dadd_rn(acc, grav);
}

}  // namespace go1
