// nlp_chain.cu -- the 40 Hz planner node of mosek_nlp_kmp around the step-timing SQP, batched: one tick of B robots.
//
// Replaces, for B independent robots (NLP = unitree_ros/mosek_nlp_kmp):
//   NLPRTControlClass::WalkingReactStepping   NLP/src/NLPRTControl/NLPRTControlClass.cpp:191-396 (squat / walk / over / idle
//                                             branches :196-283, the 100-slot /MPC/Gait message :288-392)
//   StartWalking / StopWalking                :400-432 (per-robot command word)
//   rt_nlp_gait                               :436-596
//   NLPClass::X_CoM_position_squat            NLP/src/NLP/NLPClass_sqp.cpp:2958-3015 (instance independent: a host table)
//   NLPClass::Zmp_distributor                 :3650-3831, zmp_interpolation :3834-3869, Force_torque_calculate :3872-3897
// around the existing planner kernels (step_sqp.cu: step_timing_opti_loop + CoM_height_solve; foot_traj.cu:
// Foot_trajectory_solve_mod2 with its stop-walking branch).  Six launches per tick:
//   nlp_pre_kernel    thread per robot: commands, branch, the planner's tick index (0 = no planner tick) and inputs
//   step_sqp / step_height / step_finish / foot_traj   (skip robots whose tick index is 0)
//   nlp_post_kernel   thread per robot: ZMP samples i+3 .. i+_nTdx-1 of the LIPM roll-out (:938-955, only Zmp_distributor
//                     reads them) into the robot's ZMP ring, force / moment distribution, the outgoing message
// With an active mask (per-robot clocks of the gait stack) a robot whose entry is 0 leaves the node untouched: nlp_pre_kernel gives it
// tick index 0, which the four planner kernels skip, and both node kernels return before touching its rows or its message.
// Node state: ONE SoA buffer [NLP_NODE_DOUBLES][B] -- rows [0,202) planner state, [202,234) swing-foot window, then the ZMP
// ring (the reference's whole-walk _zmpx_real / _zmpy_real as 2 x 64 entries, index & 63, with the highest index written)
// and the members of NLPRTControlClass that persist (layout of oracle/nlp_node.c).  Checkpoint = memcpy.
// Frozen quirks (oracle/nlp_node.c): the planner gets the all-zero member _estimated_state, Force_torque_calculate gets zero
// foot positions and angular acceleration, 0 / 0 weights propagate as NaN.  Compiled with -fmad=false, reference operation
// order; integer powers correctly rounded (reference: libm pow): parity 1e-9, integer slots exact.
#include <cuda_runtime.h>
#include <math_constants.h>
#include "kernels.h"
#include "powi.cuh"

namespace go1 {

namespace {
constexpr int NS = 27;
// planner state rows
constexpr int S_TS = 0, S_TX = 27, S_FX = 54, S_FY = 81, S_BJX1 = 201;
// node rows (oracle/nlp_node.c) + device-only hand-over rows
constexpr int N_RING = 234, N_ZHI = 362, N_LIFT0 = 363, N_RESTART = 364, N_STOP = 365, N_AGAIN = 366, N_TINT = 367,
              N_MPCSTOP = 368, N_RSUP = 369, N_BJX1 = 370, N_PEL = 371, N_LF = 380, N_RF = 383, N_ZMPREF = 386, N_DCMREF = 389,
              N_FL = 392, N_FR = 395, N_ML = 398, N_MR = 401, N_BODY = 404, N_RL = 442, N_COL = 460, N_COR = 463, N_COMX = 466,
              N_COMA = 469, N_TS1OLD = 472, N_MODE = 473, N_W1 = 474;
static_assert(N_W1 < NLP_NODE_DOUBLES, "node layout");
constexpr int MODE_NONE = 0, MODE_SQUAT = 1, MODE_GAIT = 2, MODE_OVER = 3, MODE_IDLE = 4;
}  // namespace

// ------------------------------------------------------------------------------------------------------------ pre
__global__ void __launch_bounds__(128) nlp_pre_kernel(NlpKParams P) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= P.B) return;
  if (P.active && !P.active[b]) { P.tick[b] = 0; return; }     // robot skips the node this call: its rows stay as they are
  const size_t B = (size_t)P.B;
  double* Nn = P.node + b;
#define N(f) Nn[(size_t)(f) * B]
  // StopWalking / StartWalking (:400-432) arrive as a command word and act before the tick
  const int cmd = P.cmd ? P.cmd[b] : 0;
  if (cmd == 1) { if (!(N(N_TINT) < 10)) N(N_STOP) = 1.0; }
  if (cmd == 2) { if (N(N_STOP) != 0.0) N(N_AGAIN) = 1.0; N(N_STOP) = 0.0; }
  const int walkdtime = P.walkdtime[b];
  int w1 = walkdtime - (int)N(N_RESTART);
  const bool start = P.start ? (P.start[b] != 0) : true;
  int mode = MODE_NONE, tick = 0;
  if (start) {
    if (N(N_AGAIN) == 0.0) {
      if (w1 * P.dtx <= P.height_offset_time) {
        mode = MODE_SQUAT;
      } else {
        w1 = (int)(w1 - (int)P.height_offset_time / P.dtx);      // :246, int -= double
        if (w1 < P.walkdtime_max) {
          N(N_TINT) = (double)w1;
          mode = MODE_GAIT;
          tick = w1 >= 1 ? w1 : 0;
        } else {
          mode = MODE_OVER;
        }
      }
    }
  } else {
    mode = MODE_IDLE;
  }
  N(N_MODE) = (double)mode; N(N_W1) = (double)w1;
  N(N_TS1OLD) = N(S_TS + 1);        // _td(1) = 0.2 _ts(1) as the previous tick left it: _nTdx of this tick (:933)
  P.tick[b] = tick;
  // planner inputs: _estimated_state (zero, see the header), the foot-location feedback, flat ground
  double* IN = P.in + b;
#pragma unroll
  for (int k = 0; k < 20; k++) IN[(size_t)k * B] = 0.0;
  if (P.rfoot_fb) { IN[(size_t)6 * B] = P.rfoot_fb[b]; IN[(size_t)7 * B] = P.rfoot_fb[B + b]; }
  if (P.lfoot_fb) { IN[(size_t)8 * B] = P.lfoot_fb[b]; IN[(size_t)9 * B] = P.lfoot_fb[B + b]; }
#undef N
}

// ------------------------------------------------------------------------------------------------------------ post
namespace {
struct Ring {
  double* base;      // row N_RING of this robot
  size_t B;
  int hi;
  __device__ __forceinline__ double get(int row, int idx) const {
    if (idx < 0 || idx > hi) return 0.0;                         // never written: the arrays' initial zero
    return base[(size_t)(64 * row + (idx & 63)) * B];
  }
  __device__ __forceinline__ void put(int row, int idx, double v) { base[(size_t)(64 * row + (idx & 63)) * B] = v; }
};

// the weights of a double-support phase (:3695-3711 and its three siblings)
__device__ __forceinline__ void dsp_weights(double* co_a, double* co_b, const double zi[2], const double ze[2], const double zr[2]) {
  const double d1 = ze[1] - zi[1], d0 = ze[0] - zi[0];
  double a = fabs((d1 * (zr[1] - zi[1]) + d0 * (zr[0] - zi[0])) / (d1 * d1 + d0 * d0));
  double a1 = a;
  if (a > 1) a = 1;
  if (a1 > 1) a1 = 1;
  co_a[0] = a; co_a[1] = a1;
  co_a[2] = sqrt((co_a[0] * co_a[0] + co_a[0] * co_a[0]) / 2);
#pragma unroll
  for (int k = 0; k < 3; k++) co_b[k] = 1.0 - co_a[k];
}
}  // namespace

__global__ void __launch_bounds__(128) nlp_post_kernel(NlpKParams P) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= P.B) return;
  if (P.active && !P.active[b]) return;
  const size_t B = (size_t)P.B;
  double* Nn = P.node + b;
#define N(f) Nn[(size_t)(f) * B]
  const int mode = (int)N(N_MODE);
  const int w1 = (int)N(N_W1);
  const double hw = P.half_hip_width, dt = P.dt;
  if (mode == MODE_SQUAT) {
    // :207-244; X_CoM_position_squat from the host table (column = walktime)
    const int col = w1 < 0 ? 0 : (w1 >= P.squat_n ? P.squat_n - 1 : w1);
#pragma unroll
    for (int k = 0; k < 9; k++) N(N_PEL + k) = 0.0;
    N(N_PEL + 2) = P.squat[col]; N(N_PEL + 5) = P.squat[P.squat_n + col]; N(N_PEL + 8) = P.squat[2 * P.squat_n + col];
#pragma unroll
    for (int k = 0; k < 3; k++) { N(N_FR + k) = 0.0; N(N_FL + k) = 0.0; N(N_MR + k) = 0.0; N(N_ML + k) = 0.0; }
    N(N_FR + 2) = 9.8 / 2 * P.mass; N(N_FL + 2) = 9.8 / 2 * P.mass;
    N(N_LF) = 0.0; N(N_LF + 1) = hw; N(N_LF + 2) = 0.0; N(N_RF) = 0.0; N(N_RF + 1) = -hw; N(N_RF + 2) = 0.0;
    const double z3[3] = {(0.0 + 0.0) / 2, (hw + -hw) / 2, (0.0 + 0.0) / 2};
#pragma unroll
    for (int k = 0; k < 3; k++) { N(N_ZMPREF + k) = z3[k]; N(N_DCMREF + k) = z3[k]; }
    N(N_BODY + 13) = z3[0]; N(N_BODY + 14) = z3[1]; N(N_BODY + 15) = z3[0]; N(N_BODY + 16) = z3[1];
    N(N_BJX1) = 1.0;
  } else if (mode == MODE_GAIT) {
    // ---- rt_nlp_gait :436-596 ----
    const int t_int = (int)N(N_TINT);
    Ring ring{Nn + (size_t)N_RING * B, B, (int)N(N_ZHI)};
    if (t_int >= 1) {
      const double* O = P.out38 + b;
      double body[38];
#pragma unroll
      for (int k = 0; k < 38; k++) { body[k] = O[(size_t)k * B]; N(N_BODY + k) = body[k]; }
      // ZMP samples of the roll-out: i, i+1, i+2 are outputs; i+3 .. i+_nTdx-1 are rebuilt from the tick's LIPM state and
      // CoM-height polynomial exactly as :938-955 / CoM_height_solve :2438-2457 evaluate them
      int ntdx = (int)round(0.2 * N(N_TS1OLD) / dt) + 1;
      if (ntdx > NLP_NTD_MAX) ntdx = NLP_NTD_MAX;
      if (ntdx < 3) ntdx = 3;
      // entries between the old top and t_int that no tick wrote (a jump ahead) are stale ring slots: zero them
      {
        int k0 = ring.hi + 1;
        if (t_int - k0 > 64) k0 = t_int - 64;
        for (int k = k0; k < t_int; k++) { ring.put(0, k, 0.0); ring.put(1, k, 0.0); }
      }
      ring.put(0, t_int, body[9]); ring.put(1, t_int, body[10]);
      ring.put(0, t_int + 1, body[13]); ring.put(1, t_int + 1, body[14]);
      ring.put(0, t_int + 2, body[17]); ring.put(1, t_int + 2, body[18]);
      if (ntdx > 3) {
        const double* LP = P.lipm + b;
        const double isx = LP[0], visx = LP[B], isy = LP[2 * B], visy = LP[3 * B], px = LP[4 * B], py = LP[5 * B];
        const double* HC = P.hz_co + b;
        double co[7];
#pragma unroll
        for (int r = 0; r < 7; r++) co[r] = HC[(size_t)r * B];
        const double base = HC[(size_t)7 * B];
        const double Wn = P.Wn;
        for (int q = 3; q < ntdx; q++) {
          const int jxx = q + 1;
          const double ch = P.ch_w[q], sh = P.sh_w[q];
          const double cx = isx * ch + visx * 1 / Wn * sh + px;
          const double cy = isy * ch + visy * 1 / Wn * sh + py;
          const double ax = (Wn * Wn) * isx * ch + visx * Wn * sh;
          const double ay = (Wn * Wn) * isy * ch + visy * Wn * sh;
          const double t = (t_int + jxx - base) * dt;
          double pw[7];
          powi_all(t, pw);
          const double pp[7] = {pw[6], pw[5], pw[4], pw[3], pw[2], pw[1], 1};
          const double aa[7] = {30 * pw[4], 20 * pw[3], 12 * pw[2], 6 * pw[1], 2, 0, 0};
          double z = 0.0, az = 0.0;
#pragma unroll
          for (int k = 0; k < 7; k++) { z = z + pp[k] * co[k]; az = az + aa[k] * co[k]; }
          const double hz = (z - 0.0) / (az + P.ggg);            // _Zsc = 0: flat ground
          ring.put(0, t_int + q, cx - hz * ax);
          ring.put(1, t_int + q, cy - hz * ay);
        }
      }
      if (t_int + ntdx - 1 > ring.hi) { ring.hi = t_int + ntdx - 1; N(N_ZHI) = (double)ring.hi; }
#pragma unroll
      for (int k = 0; k < 9; k++) N(N_PEL + k) = body[k];
      N(N_COMX) = body[0]; N(N_COMX + 1) = body[1]; N(N_COMX + 2) = body[2];      // :1093-1099
      N(N_COMA) = body[6]; N(N_COMA + 1) = body[7]; N(N_COMA + 2) = body[8];
      const double* F18 = P.out18 + b;
#pragma unroll
      for (int k = 0; k < 18; k++) N(N_RL + k) = F18[(size_t)k * B];
#pragma unroll
      for (int k = 0; k < 3; k++) { N(N_RF + k) = F18[(size_t)k * B]; N(N_LF + k) = F18[(size_t)(3 + k) * B]; }
      N(N_RSUP) = (double)P.right_support[b];
    }
    // ---- NLPClass::Zmp_distributor :3650-3831 (walktime = _walkdtime1, dt_sample = _dtx) ----
    const int bjx1 = (int)N(S_BJX1);
    const int j_index = (int)floor(w1 / (dt / P.dtx));
    double t_des = w1 * P.dtx - j_index * dt;
    if (t_des <= 0) t_des = 0.0001;
    double zr[2];
    if (j_index >= 1) {
      zr[0] = (ring.get(0, j_index) - ring.get(0, j_index - 1)) / dt * t_des + ring.get(0, j_index - 1);
      zr[1] = (ring.get(1, j_index) - ring.get(1, j_index - 1)) / dt * t_des + ring.get(1, j_index - 1);
    } else {
      zr[0] = ring.get(0, j_index) / dt * t_des + 0;
      zr[1] = ring.get(1, j_index) / dt * t_des + 0;
    }
    double col[3], cor[3];
#pragma unroll
    for (int k = 0; k < 3; k++) { col[k] = N(N_COL + k); cor[k] = N(N_COR + k); }
    if (bjx1 >= 2 && bjx1 <= NS) {
      const double tx1 = N(S_TX + bjx1 - 1), td1 = 0.2 * N(S_TS + bjx1 - 1);
      const bool dsp = (j_index + 1 - round(tx1 / dt)) * dt < td1;
      double* mine = (bjx1 % 2 == 0) ? col : cor;
      double* other = (bjx1 % 2 == 0) ? cor : col;
      if (dsp) {
        const int nTx_n = (int)round(tx1 / dt), nTx_n_dsp = (int)round((tx1 + td1) / dt);
        const double zi[2] = {ring.get(0, nTx_n - 2), ring.get(1, nTx_n - 2)};
        const double ze[2] = {ring.get(0, nTx_n_dsp - 1), ring.get(1, nTx_n_dsp - 1)};
        dsp_weights(mine, other, zi, ze, zr);
      } else {
#pragma unroll
        for (int k = 0; k < 3; k++) { mine[k] = 1.0; other[k] = 0.0; }
      }
    } else if (bjx1 == 0) {
#pragma unroll
      for (int k = 0; k < 3; k++) { col[k] = 0.5; cor[k] = 0.5; }
    } else if (bjx1 == 1) {
      const double zi[2] = {N(S_FX + 0), -P.stepwidth0};         // _footxyz_real(1, 0) = -_stepwidth(0)
      const double ze[2] = {N(S_FX + 1), N(S_FY + 1)};
      dsp_weights(cor, col, zi, ze, zr);
    }
    // ---- Force_torque_calculate :3872-3897 ----
    {
      const double com[3] = {N(N_COMX), N(N_COMX + 1), N(N_COMX + 2)}, coma[3] = {N(N_COMA), N(N_COMA + 1), N(N_COMA + 2)};
      const double gra[3] = {0, 0, -P.ggg};
      const double j_ini = P.mass * (P.rad * P.rad);
      double Ft[3], FR[3], FL[3], rd[3], ld[3];
      const double Lt[3] = {j_ini * 0.0, j_ini * 0.0, j_ini * 0.0};
#pragma unroll
      for (int k = 0; k < 3; k++) {
        Ft[k] = P.mass * (coma[k] - gra[k]);
        FR[k] = cor[k] * Ft[k]; FL[k] = col[k] * Ft[k];
        rd[k] = 0.0 - com[k]; ld[k] = 0.0 - com[k];
      }
      const double crR[3] = {FR[1] * rd[2] - FR[2] * rd[1], FR[2] * rd[0] - FR[0] * rd[2], FR[0] * rd[1] - FR[1] * rd[0]};
      const double crL[3] = {FL[1] * ld[2] - FL[2] * ld[1], FL[2] * ld[0] - FL[0] * ld[2], FL[0] * ld[1] - FL[1] * ld[0]};
#pragma unroll
      for (int k = 0; k < 3; k++) {
        const double Mt = Lt[k] - crR[k] - crL[k];
        N(N_FR + k) = FR[k]; N(N_FL + k) = FL[k];
        N(N_MR + k) = cor[k] * Mt; N(N_ML + k) = col[k] * Mt;
        N(N_COL + k) = col[k]; N(N_COR + k) = cor[k];
      }
    }
    N(N_ZMPREF) = N(N_BODY + 9); N(N_ZMPREF + 1) = N(N_BODY + 10); N(N_ZMPREF + 2) = 0.0;
    N(N_DCMREF) = N(N_BODY + 11); N(N_DCMREF + 1) = N(N_BODY + 12);
    N(N_BJX1) = N(S_BJX1);
  } else if (mode == MODE_OVER) {
    N(N_RSUP) = 2.0;
    N(N_RESTART) = (double)P.walkdtime[b];
    N(N_MPCSTOP) = 2.0;
  } else if (mode == MODE_IDLE) {
#pragma unroll
    for (int k = 0; k < 3; k++) {
      N(N_ZMPREF + k) = (N(N_LF + k) + N(N_RF + k)) / 2;
      N(N_FR + k) = 0.0; N(N_FL + k) = 0.0; N(N_MR + k) = 0.0; N(N_ML + k) = 0.0;
    }
    N(N_FR + 2) = 9.8 / 2 * P.mass; N(N_FL + 2) = 9.8 / 2 * P.mass;
    N(N_BJX1) = 1.0;
  }
  // ---- /MPC/Gait :288-392 ----
  double* M = P.msg + b;
#define MSG(k) M[(size_t)(k) * B]
#pragma unroll
  for (int k = 0; k < 3; k++) {
    MSG(k) = N(N_PEL + k); MSG(3 + k) = 0.0; MSG(6 + k) = N(N_LF + k); MSG(9 + k) = N(N_RF + k); MSG(12 + k) = N(N_ZMPREF + k);
    MSG(15 + k) = N(N_FL + k); MSG(18 + k) = N(N_FR + k); MSG(21 + k) = N(N_ML + k); MSG(24 + k) = N(N_MR + k);
    MSG(28 + k) = 0.0; MSG(31 + k) = 0.0;
    MSG(36 + k) = N(N_PEL + 3 + k); MSG(39 + k) = N(N_PEL + 6 + k);
  }
  MSG(27) = N(N_BJX1);
  MSG(34) = N(N_DCMREF); MSG(35) = N(N_DCMREF + 1);
#pragma unroll
  for (int k = 0; k < 4; k++) MSG(42 + k) = N(N_BODY + 13 + k);
#pragma unroll
  for (int k = 0; k < 12; k++) MSG(46 + k) = N(N_RL + 6 + k);
#pragma unroll
  for (int k = 58; k < 76; k++) MSG(k) = 0.0;
#pragma unroll
  for (int k = 0; k < 21; k++) MSG(76 + k) = N(N_BODY + 17 + k);
  MSG(97) = N(N_MPCSTOP);
  MSG(98) = 0.0;
  MSG(99) = N(N_RSUP);
#undef MSG
#undef N
}

cudaError_t nlp_pre_launch(NlpKParams P, cudaStream_t st) {
  nlp_pre_kernel<<<(P.B + 127) / 128, 128, 0, st>>>(P);
  return cudaGetLastError();
}
cudaError_t nlp_post_launch(NlpKParams P, cudaStream_t st) {
  nlp_post_kernel<<<(P.B + 127) / 128, 128, 0, st>>>(P);
  return cudaGetLastError();
}

}  // namespace go1
