// rt_chain.cu -- the 100 Hz node of rt_mpc_qp around the body-inclination MPC, batched: message in, message out.
//
// Replaces, for B independent robots, one tick of the main loop of RT/src/gait_fast.cpp:505-746 (RT = unitree_ros/rt_mpc_qp):
//   xget_position_interpolation()            gait_fast.cpp:113-372   40 Hz -> 100 Hz sample bookkeeping
//   PRMPCClass::XGetSolution_position_mod3   RT/src/FastMPC/PRMPCClass.cpp:1170-1261 (CoM, CoM acceleration, ZMP, DCM)
//   PRMPCClass::Foot_trajectory_solve_mod2   :1756-2195, solve_AAA_inv2 :2224-2236   swing-foot positions over the horizon
//   PRMPCClass::XGetSolution_Foot_rotation   :2255-2380                               swing-foot roll / pitch reference
//   the 2 x nh reference windows             gait_fast.cpp:568-616 (row 0 of rfoot written twice, row 1 never -- mirrored)
//   PRMPCClass::body_theta_mpc               the existing body tick kernels, fed with the record rt_pre_kernel assembles
//   the 100-slot /rtMPC/traj                 gait_fast.cpp:633-729
// Three launches per tick: rt_pre_kernel (thread per robot: everything up to the body-MPC input record), the body tick,
// rt_post_kernel (thread per robot: the outgoing message).  All per-robot state is one SoA buffer [field][B]: the node's
// members (layout of oracle/rt_glue.c), the swing-foot members (oracle/rt_foot.c) and the foot-rotation members; the body
// MPC's state is its output record.  Compiled with -fmad=false, the reference's operation order; integer powers are
// correctly rounded (the reference: libm pow), cos is CUDA's: parity 1e-9, integer slots exact.
#include <cuda_runtime.h>
#include <math_constants.h>
#include "kernels.h"
#include "powi.cuh"

namespace go1 {

namespace {
constexpr int NS = 27;
// node layout (oracle/rt_glue.c)
constexpr int N_LOOP = 0, N_MPC = 1, N_CNT = 2, N_TINT = 3, N_FLAGOLD = 4, N_COM = 5, N_COMV = 17, N_ACC = 20, N_ZMP = 32, N_DCM = 44, N_INTER = 56;
// swing-foot layout (oracle/rt_foot.c), relative to its base
constexpr int F_TS = 0, F_FX = 27, F_LIFT = 108, F_RY = 135, F_BJXX = 136, F_BJX1 = 137, F_ARR = 138;
constexpr int NH_MAX = 40, W_MAX = NH_MAX + 2;   // GO1MPC_BODY_NH_MAX; window width nh + 2

__device__ __forceinline__ int ni_of(int nh) { return 9 + 3 * (nh - 1); }

// inverse by Gauss-Jordan with partial (row) pivoting, first maximal |pivot| wins (the reference's 4x4 .inverse() through
// oracle/eigen_shim); row-major
__device__ void gj4(double* a, double* r) {
  constexpr int n = 4;
  for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) r[i * n + j] = (i == j) ? 1.0 : 0.0;
  for (int k = 0; k < n; k++) {
    int piv = k;
    double best = fabs(a[k * n + k]);
    for (int i = k + 1; i < n; i++) if (fabs(a[i * n + k]) > best) { best = fabs(a[i * n + k]); piv = i; }
    if (piv != k)
      for (int j = 0; j < n; j++) {
        double t = a[k * n + j]; a[k * n + j] = a[piv * n + j]; a[piv * n + j] = t;
        t = r[k * n + j]; r[k * n + j] = r[piv * n + j]; r[piv * n + j] = t;
      }
    const double d = a[k * n + k];
    for (int j = 0; j < n; j++) { a[k * n + j] = a[k * n + j] / d; r[k * n + j] = r[k * n + j] / d; }
    for (int i = 0; i < n; i++) {
      if (i == k) continue;
      const double f = a[i * n + k];
      for (int j = 0; j < n; j++) { a[i * n + j] -= f * a[k * n + j]; r[i * n + j] -= f * r[k * n + j]; }
    }
  }
}
__device__ __forceinline__ double row_inv_temp(const double row[4], const double* inv, const double temp[4]) {
  double v[4];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < 4; k++) acc += row[k] * inv[4 * k + j];
    v[j] = acc;
  }
  double acc = 0.0;
#pragma unroll
  for (int k = 0; k < 4; k++) acc += v[k] * temp[k];
  return acc;
}
}  // namespace

__global__ void __launch_bounds__(128) rt_pre_kernel(RtKParams P) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= P.B) return;
  const size_t B = (size_t)P.B;
  const int nh = P.nh, NI = ni_of(nh), W = nh + 2;
  double* st = P.state + b;
  const double* M = P.msg + b;
#define N_(f) st[(size_t)(f) * B]
#define MSG(k) M[(size_t)(k) * B]
  const int o_foot = N_INTER + 4 * NI, o_rot = o_foot + 6 * (nh + 1), o_thx = o_rot + 6 * nh;
  const int node_d = o_thx + 3 + 14;
  const int fs = node_d;                                   // swing-foot members
  const int rs = fs + F_ARR + 6 * W;                       // foot-rotation members: bjxx | bjx1 | Rr[3][nh] | Lr[3][nh]
#define FS_(f) st[(size_t)(fs + (f)) * B]
#define RS_(f) st[(size_t)(rs + (f)) * B]
  const double dt_fast = P.dt_mpc, dt_slow = P.dt_slow;
  const int n_t_int = (int)floor(dt_slow / dt_fast);
  const double flag = MSG(99);
  const bool ctrl = P.ctl_msg ? (P.ctl_msg[b] > 0) : (P.ctrl ? (P.ctrl[b] > 0) : true);
  bool active = false;
  double cmpc = 0.0;
  // the step table _ts: read once, written back once (the message may re-time one step)
  double ts[NS];
#pragma unroll
  for (int i = 0; i < NS; i++) ts[i] = FS_(F_TS + i);
  double* rec = P.body_in + (size_t)b * P.in_stride;
  const double* bout = P.body_out + (size_t)b * P.out_stride;
  if (ctrl) {
    const double loop = N_(N_LOOP) + 1;
    N_(N_LOOP) = loop;
    const double tint = N_(N_TINT) + (int)floor(loop / n_t_int);
    N_(N_TINT) = tint;
    if (flag > 0) {
      active = true;
      cmpc = N_(N_MPC) + 1;
      N_(N_MPC) = cmpc;
      // ---- xget_position_interpolation (:113-372) ----
      const double cnt = N_(N_CNT) + 1;
      N_(N_CNT) = cnt;
      if (tint > 2) {
        const int walktime = (int)cnt;
#pragma unroll 1
        for (int qn = 0; qn < 4; qn++) {
          const int src = (qn == 0) ? N_COM : (qn == 1 ? N_ACC : (qn == 2 ? N_ZMP : N_DCM));
          const int dst = N_INTER + qn * NI;
          double s[12];
#pragma unroll
          for (int k = 0; k < 12; k++) s[k] = N_(src + k);
          for (int jx = 0; jx < nh; jx++) {
            const double t = walktime * dt_fast + jx * dt_fast;
            const double t2 = powi(t, 2), t3 = powi(t, 3);
            const double p[4] = {t3, t2, t, 1.0};
            const double v[4] = {3 * t2, 2 * t, 1.0, 0.0};
            const double a[4] = {6 * t, 2.0, 0.0, 0.0};
#pragma unroll
            for (int c = 0; c < 3; c++) {
              const double temp[4] = {s[c], s[3 + c], s[6 + c], s[9 + c]};
              if (jx == 0) {
                N_(dst + c) = row_inv_temp(p, P.inv, temp);
                N_(dst + 3 + c) = row_inv_temp(v, P.inv, temp);
                N_(dst + 6 + c) = row_inv_temp(a, P.inv, temp);
              } else {
                N_(dst + 8 + 3 * jx - 2 + c) = row_inv_temp(p, P.inv, temp);
              }
            }
          }
        }
      }
      if (((int)cnt) % n_t_int == 0) {
#pragma unroll 1
        for (int qn = 0; qn < 4; qn++) {
          const int src = (qn == 0) ? N_COM : (qn == 1 ? N_ACC : (qn == 2 ? N_ZMP : N_DCM));
          for (int k = 0; k < 3; k++) { N_(src + k) = N_(src + 3 + k); N_(src + 3 + k) = N_(src + 6 + k); }
        }
        if (flag > N_(N_FLAGOLD)) {
          for (int k = 0; k < 3; k++) {
            const double c0 = MSG(k), cv = MSG(36 + k);
            N_(N_COM + 6 + k) = c0; N_(N_COMV + k) = cv;
            N_(N_COM + 9 + k) = c0 + cv * dt_slow;
            N_(N_ACC + 6 + k) = MSG(39 + k); N_(N_ACC + 9 + k) = MSG(80 + k);
          }
          N_(N_ZMP + 6) = MSG(12); N_(N_ZMP + 7) = MSG(13); N_(N_ZMP + 9) = MSG(42); N_(N_ZMP + 10) = MSG(43);
          N_(N_DCM + 6) = MSG(34); N_(N_DCM + 7) = MSG(35); N_(N_DCM + 9) = MSG(44); N_(N_DCM + 10) = MSG(45);
        } else {
          for (int k = 0; k < 3; k++) {
            double c0 = MSG(k), cv = MSG(36 + k);
            c0 += cv * dt_slow;
            cv += MSG(39 + k) * dt_slow;
            N_(N_COM + 6 + k) = c0; N_(N_COMV + k) = cv;
            N_(N_COM + 9 + k) = c0 + cv * dt_slow;
            N_(N_ACC + 6 + k) = MSG(80 + k); N_(N_ACC + 9 + k) = MSG(83 + k);
          }
          N_(N_ZMP + 6) = MSG(42); N_(N_ZMP + 7) = MSG(43); N_(N_ZMP + 9) = MSG(76); N_(N_ZMP + 10) = MSG(77);
          N_(N_DCM + 6) = MSG(44); N_(N_DCM + 7) = MSG(45); N_(N_DCM + 9) = MSG(78); N_(N_DCM + 10) = MSG(79);
        }
        N_(N_CNT) = 0;
        N_(N_FLAGOLD) = flag;
      }
      // ---- swing foot + foot rotation (:534-555) ----
      if (cmpc * dt_fast > 1) {
        const int jf = (int)(cmpc - (int)1 / dt_fast);
        // Foot_trajectory_solve_mod2 (:1756-2195); members as oracle/rt_foot.c lays them out
        const int bjxx_nrt = (int)MSG(86);
        if (bjxx_nrt >= 0 && bjxx_nrt + 1 < NS) {
          FS_(F_FX + bjxx_nrt) = MSG(87); FS_(F_FX + bjxx_nrt + 1) = MSG(88);
          FS_(F_FX + 27 + bjxx_nrt) = MSG(89); FS_(F_FX + 27 + bjxx_nrt + 1) = MSG(90);
          FS_(F_FX + 54 + bjxx_nrt) = MSG(91); FS_(F_FX + 54 + bjxx_nrt + 1) = MSG(92);
        }
        const int bjxp = (int)MSG(93);
        if (MSG(94) > 0 && bjxp >= 0 && bjxp < NS) { ts[bjxp] = MSG(94); FS_(F_TS + bjxp) = ts[bjxp]; }
      }
    }
  }
  // step tables rebuilt from _ts (:1774-1784); _t_end_footstep with 2 tstep (the swing-foot call's)
  double tx[NS];
  tx[0] = 0.0;
  for (int i = 1; i < NS; i++) { double v = tx[i - 1] + ts[i - 1]; tx[i] = round(v / dt_slow) * dt_slow - 0.00001; }
  const double t_end = round((tx[NS - 1] - 2 * P.tstep) / dt_fast);
  // The swing-foot window, the lift heights and the foot-rotation horizons live in local arrays for the whole horizon loop:
  // loaded once, stored once.  Same operations in the same order as the reference, so the results are bit-identical.
  const bool swung = active && cmpc * dt_fast > 1;
  double arr[6 * W_MAX], rot[6 * NH_MAX];
  if (swung) {
    const int j_indexx = (int)(cmpc - (int)1 / dt_fast);
    int bjxx = (int)FS_(F_BJXX), bjx1 = (int)FS_(F_BJX1);
    double ry = FS_(F_RY);
    for (int i = 0; i < 6 * W; i++) arr[i] = FS_(F_ARR + i);
    double lift[NS];
#pragma unroll
    for (int i = 0; i < NS; i++) lift[i] = FS_(F_LIFT + i);
    // the reference zeroes lift heights 24..26 on every horizon step; nothing in the loop sets them, so once is the same
#pragma unroll
    for (int it = 24; it < NS; it++) lift[it] = 0.0;
#define ARR(foot, k, idx) arr[((foot) * 3 + (k)) * W + (idx)]      /* foot 0 = right, 1 = left */
#define FXYZ(k, idx) FS_(F_FX + 27 * (k) + (idx))
    FXYZ(1, 0) = -P.stepwidth0;
    int fx_key = -1000;            // bjxx the footstep cache below belongs to
    double fq[3], fq2[3];          // FXYZ(k, bq), FXYZ(k, bq2)
    for (int j_index = j_indexx; j_index < j_indexx + nh; j_index++) {
      const int q = j_index - j_indexx;
      if (j_index <= t_end) {
        int jp = 0;
        while (jp < NS && j_index * dt_fast >= tx[jp]) jp++;
        bjxx = (jp - 1) + 1;
        jp = 0;
        while (jp < NS && (j_index + 1) * dt_fast >= tx[jp]) jp++;
        bjx1 = (jp - 1) + 1;
      }
      if (j_index > t_end) for (int it = bjx1 + 1; it < NS; it++) lift[it] = 0.0;       // (stop-walking flag: not raised by the node)
      if (bjx1 >= 2 && j_index <= t_end) {
        const int sup = (bjx1 % 2 == 0) ? 1 : 0, swg = 1 - sup;       // even: left support, right swing
        for (int k = 0; k < 3; k++) { const double v = ARR(sup, k, q); ARR(sup, k, q + 1) = v; ARR(sup, k, q + 2) = v; }
        const double ts1 = ts[bjx1 - 1], td1 = P.tdsp_ratio * ts1;
        const double s0 = round(tx[bjx1 - 1] / dt_fast);
        if ((j_index + 1 - s0) * dt_fast < td1) {
          for (int k = 0; k < 3; k++) { const double v = ARR(swg, k, q); ARR(swg, k, q + 1) = v; ARR(swg, k, q + 2) = v; }
        } else {
          const double t_des = (j_index + 1 - s0 + 1) * dt_fast;
          const double tp[3] = {t_des - dt_fast, (td1 + ts1) / 2 + 0.0001, ts1 - (2 * dt_fast + 0.001)};
          if (bjxx != fx_key) {
            const int bq = bjxx < NS ? bjxx : NS - 1, bq2 = bjxx - 2 >= 0 ? (bjxx - 2 < NS ? bjxx - 2 : NS - 1) : 0;
#pragma unroll
            for (int k = 0; k < 3; k++) { fq[k] = FXYZ(k, bq); fq2[k] = FXYZ(k, bq2); }
            fx_key = bjxx;
          }
          if (fabs(t_des - ts1) <= (dt_fast)) {
#pragma unroll
            for (int k = 0; k < 3; k++) { const double v = fq[k]; ARR(swg, k, q + 1) = v; ARR(swg, k, q + 2) = v; }
          } else {
            double A[16], Ai[16];
            for (int r = 0; r < 3; r++) { A[4 * r] = powi(tp[r], 3); A[4 * r + 1] = powi(tp[r], 2); A[4 * r + 2] = powi(tp[r], 1); A[4 * r + 3] = 1; }
            A[12] = 3 * powi(tp[2], 2); A[13] = 2 * powi(tp[2], 1); A[14] = powi(tp[2], 0); A[15] = 0;
            gj4(A, Ai);
            const double tap[4] = {powi(t_des, 3), powi(t_des, 2), powi(t_des, 1), 1};
            const double tav[4] = {3 * powi(t_des, 2), 2 * powi(t_des, 1), 1, 0};
            if ((j_index + 1 - s0) * dt_fast < td1 + dt_fast) ry = (fq[1] + fq2[1]) / 2;
#pragma unroll
            for (int k = 0; k < 3; k++) {
              double plan[4];
              plan[0] = ARR(swg, k, q);
              if (k == 0) plan[1] = (fq2[0] + fq[0]) / 2;
              else if (k == 1) plan[1] = ry;
              else plan[1] = fmax(fq2[2], fq[2]) + lift[bjx1 - 1];
              plan[2] = fq[k];
              plan[3] = 0;
              double co[4];
              for (int r = 0; r < 4; r++) { double a_ = 0.0; for (int m = 0; m < 4; m++) a_ += Ai[4 * r + m] * plan[m]; co[r] = a_; }
              double p_ = 0.0, v_ = 0.0;
              for (int m = 0; m < 4; m++) { p_ += tap[m] * co[m]; v_ += tav[m] * co[m]; }
              ARR(swg, k, q + 1) = p_;
              ARR(swg, k, q + 2) = p_ + dt_fast * v_;
            }
          }
        }
      } else {
        if (j_index > t_end) {
          for (int k = 0; k < 3; k++) { ARR(0, k, q + 1) = ARR(0, k, q); ARR(1, k, q + 1) = ARR(1, k, q); }
        } else {
          ARR(0, 1, q + 1) = -P.stepwidth0;
          ARR(1, 1, q + 1) = P.stepwidth0;
        }
      }
    }
    for (int jjj = 0; jjj < nh + 1; jjj++)
      for (int k = 0; k < 3; k++) { N_(o_foot + 6 * jjj + k) = ARR(0, k, jjj + 1); N_(o_foot + 6 * jjj + 3 + k) = ARR(1, k, jjj + 1); }
    // column 0 of the stored window takes column 1 (the reference's shift after the horizon); the local copy stays unshifted:
    // the record below reads columns 1..nh only
    for (int i = 0; i < 6 * W; i++) FS_(F_ARR + i) = (i % W == 0) ? arr[i + 1] : arr[i];
#pragma unroll
    for (int i = 0; i < NS; i++) FS_(F_LIFT + i) = lift[i];
    FS_(F_BJXX) = bjxx; FS_(F_BJX1) = bjx1; FS_(F_RY) = ry;
    // XGetSolution_Foot_rotation (:2255-2380) with the members Foot_trajectory_solve_mod2 just updated; rot = Rr[3][nh] | Lr[3][nh]
    for (int i = 0; i < 6 * nh; i++) rot[i] = RS_(2 + i);
    int rbjxx = (int)RS_(0), rbjx1 = (int)RS_(1);
    for (int walktime = j_indexx; walktime < j_indexx + nh; walktime++) {
      const int col = walktime - j_indexx;
      if (walktime <= t_end) {
        int jp = 0;
        while (jp < NS && walktime * dt_fast >= tx[jp]) jp++;
        rbjxx = (jp - 1) + 1;
        jp = 0;
        while (jp < NS && (walktime + 1) * dt_fast >= tx[jp]) jp++;
        rbjx1 = (jp - 1) + 1;
      }
      const int k = rbjx1 - 1;
      if (rbjx1 >= 2 && walktime <= t_end) {
        const double tsk = ts[k], tdk = P.tdsp_ratio * tsk;
        const double t_des = (walktime + 1) * dt_fast - (tx[k] + 2 * tdk / 4);
        const double sarg = t_des + 2 * tdk / 4;
        const int i1 = rbjx1 < NS ? rbjx1 : NS - 1;
        const double dfx = FXYZ(0, i1) - FXYZ(0, rbjx1 - 1);
        const int base = (rbjx1 % 2 == 0) ? 0 : 3 * nh;          // even: the right foot swings
        const double amp = (rbjx1 % 2 == 0) ? -0.065 : 0.075;
        rot[base + 0 * nh + col] = amp * (1 - cos(2 * CUDART_PI / tsk * sarg));
        if (sarg >= tsk / 2) {
          if (dfx > 0) rot[base + 1 * nh + col] = 0.075 * dfx / P.footx_max * (cos(4 * CUDART_PI / tsk * sarg) - 1);
        } else {
          rot[base + 1 * nh + col] = 0;
        }
      }
      N_(o_rot + 6 * col + 0) = rot[0 * nh + col]; N_(o_rot + 6 * col + 1) = rot[1 * nh + col]; N_(o_rot + 6 * col + 2) = rot[2 * nh + 0];
      N_(o_rot + 6 * col + 3) = rot[3 * nh + col]; N_(o_rot + 6 * col + 4) = rot[4 * nh + col]; N_(o_rot + 6 * col + 5) = rot[5 * nh + 0];
    }
    // rows 0, 1 of each foot are the ones the loop writes
    for (int i = 0; i < 2 * nh; i++) { RS_(2 + i) = rot[i]; RS_(2 + 3 * nh + i) = rot[3 * nh + i]; }
    RS_(0) = rbjxx; RS_(1) = rbjx1;
#undef FXYZ
  }
  if (active) N_(N_ZMP + 8) = 0.0;          // zmpxyz_ref(2) = _Zsc = 0
  // ---- body-MPC input record (:568-620); an inactive robot gets a gated tick (0): its body state stays as it is ----
  for (int k = 0; k < NS; k++) rec[k] = tx[k];
  rec[27] = active ? cmpc : 0.0;
  for (int k = 0; k < 4; k++) { rec[28 + k] = bout[14 + k]; rec[32 + k] = P.ctl_msg ? P.ctl_msg[(size_t)(k < 2 ? 10 + k : 11 + k) * B + b]       // state_feedback(10, 11, 13, 14), :105-108
                             : (P.bodyangle_state ? P.bodyangle_state[(size_t)k * B + b] : 0.0); }
  for (int k = 0; k < 2 * nh; k++) rec[36 + k] = bout[18 + k];
  double* rows = rec + 36 + 2 * nh;
  if (active) {
    const int zi = N_INTER + 2 * NI, ai = N_INTER + NI;
    for (int jxx = 0; jxx < nh; jxx++) {
      rows[0 * nh + jxx] = (jxx == 0) ? N_(zi + 0) : N_(zi + 8 + 3 * jxx - 2);
      rows[1 * nh + jxx] = (jxx == 0) ? N_(zi + 1) : N_(zi + 8 + 3 * jxx - 1);
      // the horizons of this tick when the swing section ran, else the stale ones the state holds
      const double r0 = swung ? rot[jxx] : N_(o_rot + jxx * 6), l0 = swung ? rot[3 * nh + jxx] : N_(o_rot + jxx * 6 + 3);
      const double r1 = swung ? rot[nh + jxx] : N_(o_rot + jxx * 6 + 1), l1 = swung ? rot[4 * nh + jxx] : N_(o_rot + jxx * 6 + 4);
      const double a0 = (r0 + l0) / 5, a1 = (r1 + l1) / 5;
      rows[2 * nh + jxx] = a0; rows[3 * nh + jxx] = a1;
      rows[4 * nh + jxx] = swung ? ARR(0, 1, jxx + 1) : N_(o_foot + jxx * 6 + 1);        // row 0 written twice (x, then y), row 1 never
      rows[5 * nh + jxx] = 0.0;
      rows[6 * nh + jxx] = swung ? ARR(1, 0, jxx + 1) : N_(o_foot + jxx * 6 + 3);
      rows[7 * nh + jxx] = swung ? ARR(1, 1, jxx + 1) : N_(o_foot + jxx * 6 + 4);
      rows[8 * nh + jxx] = (jxx == 0) ? N_(ai + 2) : N_(ai + 8 + 3 * jxx);
      if (jxx == 0) { N_(o_thx + 0) = a0; N_(o_thx + 1) = a1; }
    }
  } else {
    for (int k = 0; k < 9 * nh; k++) rows[k] = 0.0;
  }
  if (P.in_stride > 36 + 11 * nh) rec[36 + 11 * nh] = 0.0;
  if (P.active) P.active[b] = active ? 1 : 0;
#undef ARR
#undef N_
#undef MSG
#undef FS_
#undef RS_
}

__global__ void __launch_bounds__(128) rt_post_kernel(RtKParams P) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= P.B) return;
  const size_t B = (size_t)P.B;
  const int nh = P.nh, NI = ni_of(nh);
  double* st = P.state + b;
  const double* M = P.msg + b;
  double* O = P.out + b;
#define N_(f) st[(size_t)(f) * B]
  const int o_foot = N_INTER + 4 * NI, o_rot = o_foot + 6 * (nh + 1), o_thx = o_rot + 6 * nh, o_bm = o_thx + 3;
  const bool ctrl = P.ctl_msg ? (P.ctl_msg[b] > 0) : (P.ctrl ? (P.ctrl[b] > 0) : true);
  const bool active = ctrl && M[(size_t)99 * B] > 0;
  if (active) {
    const double* bout = P.body_out + (size_t)b * P.out_stride;
    for (int k = 0; k < 14; k++) N_(o_bm + k) = bout[k];
  }
  for (int k = 0; k < 36; k++) O[(size_t)k * B] = M[(size_t)k * B];
  double inte[51];
  for (int k = 0; k < 51; k++) inte[k] = 0.0;
  for (int k = 0; k < 3; k++) { inte[k] = N_(N_INTER + k); inte[3 + k] = N_(o_thx + k); inte[6 + k] = N_(o_foot + 3 + k); inte[9 + k] = N_(o_foot + k); }
  inte[12] = N_(N_INTER + 2 * NI); inte[13] = N_(N_INTER + 2 * NI + 1); inte[14] = N_(N_ZMP + 8);
  inte[27] = M[(size_t)27 * B];
  for (int k = 0; k < 3; k++) { inte[28 + k] = N_(o_rot + 3 + k); inte[31 + k] = N_(o_rot + k); }
  inte[34] = N_(N_INTER + 3 * NI); inte[35] = N_(N_INTER + 3 * NI + 1);
  for (int k = 0; k < 14; k++) inte[36 + k] = N_(o_bm + k);
  for (int k = 36; k <= 86; k++) O[(size_t)k * B] = inte[k - 36];
  for (int k = 87; k < 98; k++) O[(size_t)k * B] = 0.0;
  // _tx_total = _tx(26) of the rebuilt table; (int) binds to it (:727)
  {
    const int fs = o_bm + 14;
    double txv = 0.0;
    for (int i = 1; i < NS; i++) { const double v = txv + st[(size_t)(fs + F_TS + i - 1) * B]; txv = round(v / P.dt_slow) * P.dt_slow - 0.00001; }
    O[(size_t)98 * B] = (double)(int)txv / 0.001;
  }
  O[(size_t)99 * B] = N_(N_LOOP);
  if (P.rt2nrt) {
    // /rt2nrt/state (:519-527): state_feedback = the control message with slot 0 replaced by t_int
    double* R = P.rt2nrt + b;
    R[0] = N_(N_TINT);
    for (int k = 1; k < 25; k++) R[(size_t)k * B] = P.ctl_msg ? P.ctl_msg[(size_t)k * B + b] : 0.0;
  }
#undef N_
}

cudaError_t rt_pre_launch(RtKParams P, cudaStream_t st) {
  rt_pre_kernel<<<(P.B + 127) / 128, 128, 0, st>>>(P);
  return cudaGetLastError();
}
cudaError_t rt_post_launch(RtKParams P, cudaStream_t st) {
  rt_post_kernel<<<(P.B + 127) / 128, 128, 0, st>>>(P);
  return cudaGetLastError();
}

}  // namespace go1
