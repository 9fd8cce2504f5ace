// grf_qp.cu -- ground-reaction-force distribution of go1_servo's 1 kHz loop, batched.
//
// Replaces Dynamiccclass (GO1 = unitree_ros/go1_rt_control):
//   force_distribution     GO1/src/whole_body_dynamics/dynmics_compute.cpp:141-261  (thread per robot)
//   force_opt              :265-373   (warp per robot: condensation of the 12-variable QP in shared
//   solve_grf_opt          :387-427    memory + the warp-cooperative Goldfarb-Idnani core; 12 equality
//                                      columns -- the stance legs' are all-zero and skipped while
//                                      me = p = 12 stays, EiQuadProg.cpp:238-241,288,370 -- and 24
//                                      inequalities: unilateral + friction pyramid per leg)
//   skew_hat               :375-385   (frozen bug: vec_w[2,0] is the comma operator -> every entry is vec_w[0])
//   compute_joint_torques  :109-138   (thread per leg)
// Records are instance-major (a warp reads its robot's 48-double record with coalesced loads).  The per-robot arithmetic is
// grf_math.cuh's, which servo_torque_kernel also runs.
#include <cuda_runtime.h>
#include "grf_math.cuh"
#include "kernels.h"

namespace go1 {

int grf_warp_doubles() { return gi_ws_doubles(GN, GM) + 72 + GN + GN * GP + GP + GRF_IN_DOUBLES; }   // ws | A(6x12) | g0 | CE | ce0 | record

template <int WPC>
__global__ void __launch_bounds__(WPC * 32) grf_force_opt_kernel(GrfKParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* smem = reinterpret_cast<double*>(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* CI = smem;                             // CTA-shared inequality data: CI = -qp_H' (12 x 24), ci0 = qp_h
  grf_ci_build(CI, P.fz_max, P.mu);
  double* wbase = smem + GN * GM + GM + (size_t)warp * P.warp_doubles;
  GiWs w;
  gi_ws_carve(w, wbase, GN, GP, GM);
  double* A = wbase + gi_ws_doubles(GN, GM);     // 6 x 12 column-major
  double* g0 = A + 72;
  double* CE = g0 + GN;
  double* ce0 = CE + GN * GP;
  double* recs = ce0 + GP;                       // the robot's input record

  for (int b = blockIdx.x * WPC + warp; b < P.B; b += gridDim.x * WPC) {
    const double* rec = P.in + (size_t)b * GRF_IN_DOUBLES;
    // record: base_p 3 | leg_p 12 | FT 6 | F_leg_guess 12 | grf_prev 12 | mode | right_support | pad
    recs[lane] = rec[lane];
    if (lane < GRF_IN_DOUBLES - 32) recs[32 + lane] = rec[32 + lane];
    __syncwarp();
    grf_force_opt_warp(P, CI, w, A, g0, CE, ce0, recs, P.out + (size_t)b * GRF_OUT_DOUBLES,
                       P.diag ? P.diag + (size_t)b * GRF_DIAG_INTS : nullptr, lane);
    __syncwarp();
  }
}

// force_distribution (:141-261), one thread per robot; SoA in/out
__global__ void __launch_bounds__(256) grf_force_distribution_kernel(GrfDistParams P) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= P.B) return;
  const size_t B = (size_t)P.B;
  double com[3], leg[12], F[6], rf[3], lf[3], out[12];
  for (int k = 0; k < 3; k++) { com[k] = P.com[k * B + b]; rf[k] = P.rfoot[k * B + b]; lf[k] = P.lfoot[k * B + b]; }
  for (int k = 0; k < 12; k++) { leg[k] = P.leg[k * B + b]; out[k] = 0.0; }
  for (int k = 0; k < 6; k++) F[k] = P.F[k * B + b];
  grf_distribute(P.mode, P.y_coefficient, com, leg, F, rf, lf, out);
  for (int k = 0; k < 12; k++) P.F_leg_ref[k * B + b] = out[k];
}

// compute_joint_torques (:109-138), one thread per leg; SoA in/out.  tau = -Jaco' * w + gravity_compensate(:, leg) with
// w = swing_kp (p_des - p_est) + swing_kd (pv_des - pv_est) for a swing leg, the leg's column of F_leg_ref for a stance
// leg.  The reference's operation order, no contraction into FMA (bit-identical to the oracle).
__global__ void __launch_bounds__(256) grf_joint_torques_kernel(GrfTauParams P) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 4 * P.B) return;
  const size_t B = (size_t)P.B;
  const int leg = t / P.B;                 // leg-major over the grid: consecutive threads = consecutive robots
  const size_t b = (size_t)(t - leg * P.B);
  double w[3];
  if (P.swing[leg * B + b]) {
    for (int k = 0; k < 3; k++) {
      const size_t i = (size_t)(3 * leg + k) * B + b;
      w[k] = grf_swing_w(P.swing_kp, P.swing_kd, P.p_des[i], P.p_est[i], P.pv_des[i], P.pv_est[i]);
    }
  } else {
    for (int k = 0; k < 3; k++) w[k] = P.F_leg_ref[(long long)(3 * leg + k) * P.f_ks + (long long)b * P.f_bs];
  }
  for (int i = 0; i < 3; i++) {
    double j[3];
    for (int r = 0; r < 3; r++) j[r] = P.jac[(size_t)(9 * leg + 3 * r + i) * B + b];
    P.tau[(size_t)(3 * leg + i) * B + b] = grf_tau(leg, i, j, w);
  }
}

template <int WPC>
static cudaError_t launch_opt(const GrfKParams& P0, int sms, cudaStream_t st) {
  GrfKParams P = P0;
  P.warp_doubles = grf_warp_doubles();
  const size_t smem = (size_t)(GN * GM + GM + WPC * P.warp_doubles) * sizeof(double);
  cudaError_t e = cudaFuncSetAttribute(grf_force_opt_kernel<WPC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  int grid = (P.B + WPC - 1) / WPC;
  if (grid > sms * 6) grid = sms * 6;
  grf_force_opt_kernel<WPC><<<grid, WPC * 32, smem, st>>>(P);
  return cudaGetLastError();
}
cudaError_t grf_force_opt_launch(GrfKParams P, int sms, cudaStream_t st) { return launch_opt<4>(P, sms, st); }
cudaError_t grf_force_distribution_launch(GrfDistParams P, cudaStream_t st) {
  grf_force_distribution_kernel<<<(P.B + 255) / 256, 256, 0, st>>>(P);
  return cudaGetLastError();
}

cudaError_t grf_joint_torques_launch(GrfTauParams P, cudaStream_t st) {
  grf_joint_torques_kernel<<<(4 * P.B + 255) / 256, 256, 0, st>>>(P);
  return cudaGetLastError();
}

}  // namespace go1
