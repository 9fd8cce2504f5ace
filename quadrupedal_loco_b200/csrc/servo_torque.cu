// servo_torque.cu -- the force stage of go1_servo's 1 kHz tick after the servo stack (go1mpc_servo_torque_tick_async):
// force_distribution -> the 12-variable force QP -> 4 x compute_joint_torques, K ticks per robot in order (the QP's gama term
// chains grf_opt from tick to tick).  One warp per robot, grf_force_opt_kernel's layout: CI / ci0 shared by the CTA, the QP
// workspace and the tick's record in the warp's slice.  Per tick, lanes 0-3 (one leg each) rebuild the IK's body pose and foot
// target from the filtered channels servo_stack_kernel<true> stored, the IK Jacobian at the tick's joint angles (fk_any: the
// IK's J bit for bit) and the FK of the measured joints; lane 0 runs the distribution; the warp solves the QP; lanes 0-11 map
// one joint torque each.  grf_opt and F_leg_ref stay in shared memory over the K ticks and are stored once.
// Built with -fmad=false (servo_math.cuh); grf_math.cuh writes its multiply-adds out, so the force stage equals grf_qp.cu's.
#include <cuda_runtime.h>
#include "grf_math.cuh"      // first: it selects gi_warp.cuh's fma() form
#include "servo_math.cuh"
#include "kernels.h"

namespace go1 {

namespace {
// out record | IK J | p_est | pv_est | pv_des | F_leg_ref | per-call leg data: homing, measured q, dq [4][9] | R [9] | F_force_des [6]
constexpr int TQ_EXTRA = GRF_OUT_DOUBLES + 36 + 12 + 12 + 12 + 12 + 36 + 9 + 6 + 1;
}

// The per-call leg data lives in shared memory, not in registers across the QP, so that 4 CTAs (16 warps) fit an SM without
// spills: the QP is latency-bound and wants as many warps per SM as the registers allow.
// H: also count, per tick, the force QP's outcome (FH_GRF_OK / FH_GRF_FAILED, FH_GRF_FALLBACK on a NaN solution) and a non-finite
// q or tau of the robot (FH_NONFINITE) in registers of lane 0, which adds them to the health rows and ORs FH_EVENTS once per robot.
template <int WPC, bool H = false>
__global__ void __launch_bounds__(WPC * 32, 4) servo_torque_kernel(ServoTorqueKParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* smem = reinterpret_cast<double*>(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* CI = smem;
  grf_ci_build(CI, P.g.fz_max, P.g.mu);
  double* wbase = smem + GN * GM + GM + (size_t)warp * P.g.warp_doubles;
  GiWs w;
  gi_ws_carve(w, wbase, GN, GP, GM);
  double* A = wbase + gi_ws_doubles(GN, GM);
  double* g0 = A + 72;
  double* CE = g0 + GN;
  double* ce0 = CE + GN * GP;
  double* recs = ce0 + GP;                 // the tick's force-QP record (GrfKParams::in layout)
  double* out = recs + GRF_IN_DOUBLES;     // its out record
  double* Jq = out + GRF_OUT_DOUBLES;      // [4][9] IK Jacobians
  double* pest = Jq + 36;                  // [12] measured foot positions
  double* pvest = pest + 12;               // [12] measured foot velocities
  double* pvdes = pvest + 12;              // [12] desired foot velocities
  double* fref = pvdes + 12;               // [12] F_leg_ref (FR, FL, RR, RL xyz)
  double* legd = fref + 12;                // [4][9] per leg: homing | measured q | measured dq
  double* Rs = legd + 36;                  // [9] body rotation (roll, pitch of /rtMPC/traj 72 / 73, yaw 0)
  double* Fd = Rs + 9;                     // [6] F_force_des: /MPC/Gait 15-20 (F_L xyz, F_R xyz)

  const size_t B = (size_t)P.B;
  const int K = P.K, mode = P.gait_mode;
  const int leg = lane & 3;                // lanes 0..3
  const bool right = servo_follows_right(mode, leg);
  const LegC lc = leg_consts(leg);
  for (int bi = blockIdx.x * WPC + warp; bi < P.B; bi += gridDim.x * WPC) {
    const size_t b = (size_t)bi;
    const double* G = P.gait + b;          // /MPC/Gait slot s at G[s * B]
    const bool rst = P.reset && P.reset[b];
    if (lane < 12) {
      recs[33 + lane] = rst ? 0.0 : P.force[(size_t)lane * B + b];
      fref[lane] = rst ? 0.0 : P.force[(size_t)(12 + lane) * B + b];
    }
    // FT_total_des = (F_L + F_R, M_L + M_R): slots 15-17 + 18-20, 21-23 + 24-26
    if (lane < 6) recs[15 + lane] = G[(size_t)(lane < 3 ? 15 + lane : 18 + lane) * B] + G[(size_t)(lane < 3 ? 18 + lane : 21 + lane) * B];
    const double rs = G[(size_t)99 * B];
    if (lane == 0) { recs[45] = (double)mode; recs[46] = rs; recs[47] = 0.0; }
    const unsigned swing = grf_zero_legs(mode, (int)rs);
    if (lane < 4) {
      for (int k = 0; k < 3; k++) {
        legd[9 * leg + k] = P.homing[(size_t)(3 * leg + k) * B + b];
        legd[9 * leg + 3 + k] = P.meas[(size_t)(3 * leg + k) * B + b];
        legd[9 * leg + 6 + k] = P.meas[(size_t)(12 + 3 * leg + k) * B + b];
        pvdes[3 * leg + k] = G[(size_t)((right ? 46 : 49) + k) * B];
      }
    }
    if (lane == 0) {
      double R[9];
      body_rotation(P.traj[72 * B + b], P.traj[73 * B + b], 0.0, R);
      for (int k = 0; k < 9; k++) Rs[k] = R[k];
    }
    if (lane < 6) Fd[lane] = G[(size_t)(15 + lane) * B];
    __syncwarp();
    int n_ok = 0, n_fail = 0, n_fallback = 0, n_nonfinite = 0;   // H only
    for (int k = 0; k < K; k++) {
      bool nonfinite = false;                                   // H only: this tick's q or tau of the robot
      double ch[SERVO_LPF_CHANNELS];
      if (lane < 4) {
#pragma unroll
        for (int c = 0; c < SERVO_LPF_CHANNELS; c++) ch[c] = P.ch[((size_t)k * SERVO_LPF_CHANNELS + c) * B + b];
        Body bd;
        bd.on = true;
        bd.p[0] = ch[0]; bd.p[1] = ch[1] * P.y_offset; bd.p[2] = ch[2];
        for (int j = 0; j < 9; j++) bd.R[j] = Rs[j];
        const double* ld = legd + 9 * leg;
        const double hom[3] = {ld[0], ld[1], ld[2]}, qm[3] = {ld[3], ld[4], ld[5]}, dqm[3] = {ld[6], ld[7], ld[8]};
        const double vf[3] = {right ? ch[6] : ch[3], right ? ch[7] : ch[4], right ? ch[8] : ch[5]};
        double pdes[3], pos[3], J[9];
        servo_leg_target(hom, vf, right, P.half_hip_width, pdes);
        const double* qk = P.q + b * (size_t)(12 * K) + 12 * k + 3 * leg;
        const double qq[3] = {qk[0], qk[1], qk[2]};
        if constexpr (H) nonfinite = !isfinite(qq[0]) || !isfinite(qq[1]) || !isfinite(qq[2]);
        fk_any(qq, lc, bd, pos, J);
        for (int j = 0; j < 9; j++) Jq[9 * leg + j] = J[j];
        fk_any(qm, lc, bd, pos, J);
        for (int i = 0; i < 3; i++) {
          pest[3 * leg + i] = pos[i];
          pvest[3 * leg + i] = __dadd_rn(__dadd_rn(__dmul_rn(J[3 * i], dqm[0]), __dmul_rn(J[3 * i + 1], dqm[1])), __dmul_rn(J[3 * i + 2], dqm[2]));
          recs[3 + 3 * leg + i] = pdes[i];
        }
        if (lane == 0) for (int i = 0; i < 3; i++) recs[i] = bd.p[i];
      }
      __syncwarp();
      if (lane == 0 && (mode == 101 || mode == 102)) {       // other gait modes hold F_leg_ref
        const double rf[3] = {ch[6], ch[7], ch[8]}, lf[3] = {ch[3], ch[4], ch[5]};
        double o[12];
        grf_distribute(mode, P.y_coefficient, recs, recs + 3, Fd, rf, lf, o);
        for (int j = 0; j < 12; j++) fref[j] = o[j];
      }
      __syncwarp();
      if (lane < 12) recs[21 + lane] = fref[lane];            // F_leg_guess
      __syncwarp();
      const GrfQpOutcome qo = grf_force_opt_warp(P.g, CI, w, A, g0, CE, ce0, recs, out,
                                                 (k == K - 1 && P.grf_diag) ? P.grf_diag + b * GRF_DIAG_INTS : nullptr, lane);
      if constexpr (H) {
        n_ok += qo.status == ST_OK;
        n_fail += qo.status != ST_OK;
        n_fallback += qo.nan;
      }
      __syncwarp();
      if (lane < 12) {
        const int l = lane / 3, i = lane - 3 * l;
        const bool sw = (swing >> l) & 1u;
        double wv[3], jc[3];
        for (int r = 0; r < 3; r++) {
          const int e = 3 * l + r;
          wv[r] = sw ? grf_swing_w(P.swing_kp, P.swing_kd, recs[3 + e], pest[e], pvdes[e], pvest[e]) : out[e];
          jc[r] = Jq[9 * l + 3 * r + i];
        }
        const double tq = grf_tau(l, i, jc, wv);
        P.tau[b * (size_t)(12 * K) + 12 * k + lane] = tq;
        if constexpr (H) nonfinite = nonfinite || !isfinite(tq);
        recs[33 + lane] = out[lane];                          // grf_opt -> the next tick's previous solution
      }
      if constexpr (H) n_nonfinite += __any_sync(FULL_MASK, nonfinite) ? 1 : 0;
      __syncwarp();
    }
    if constexpr (H) {
      if (lane == 0) {
        const int add[4] = {n_ok, n_fail, n_fallback, n_nonfinite};
        const int row[4] = {FH_GRF_OK, FH_GRF_FAIL, FH_GRF_FALLBACK, FH_NONFINITE};
        int ev = 0;
#pragma unroll
        for (int j = 0; j < 4; j++)
          if (add[j]) { P.health[(size_t)row[j] * B + b] += add[j]; ev |= 1 << row[j]; }
        if (ev) P.health[(size_t)FH_EVENTS * B + b] |= ev;
      }
    }
    if (lane < 12) {
      P.force[(size_t)lane * B + b] = recs[33 + lane];
      P.force[(size_t)(12 + lane) * B + b] = fref[lane];
    }
    if (P.grf && lane < GRF_OUT_DOUBLES) P.grf[b * GRF_OUT_DOUBLES + lane] = out[lane];
    __syncwarp();
  }
}

cudaError_t servo_torque_launch(ServoTorqueKParams P, int sms, cudaStream_t st) {
  constexpr int WPC = 4;
  P.g.warp_doubles = grf_warp_doubles() + TQ_EXTRA;
  const size_t smem = (size_t)(GN * GM + GM + WPC * P.g.warp_doubles) * sizeof(double);
  auto kern = P.health ? servo_torque_kernel<WPC, true> : servo_torque_kernel<WPC>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  int per_sm = 0;
  if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WPC * 32, smem)) != cudaSuccess) return e;
  int grid = (P.B + WPC - 1) / WPC;                 // one wave of resident CTAs, grid-stride over the robots
  if (grid > sms * per_sm) grid = sms * per_sm;
  kern<<<grid, WPC * 32, smem, st>>>(P);
  return cudaGetLastError();
}

}  // namespace go1
