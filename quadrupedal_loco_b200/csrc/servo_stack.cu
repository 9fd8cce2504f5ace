// servo_stack.cu -- K consecutive ticks of go1_servo's 1 kHz loop for B robots, fed from the messages the gait stack keeps
// resident (go1mpc_servo_stack_tick_async).  Per robot and tick:
//   9 butterworthLPF objects (3 Hz) on the held /MPC/Gait slots 0 1 2 (CoM) | 6 7 8 (left foot) | 9 10 11 (right foot)
//   -> the gait_mode leg mapping and 4 x Inverse_kinematics_g (servo.cpp:935-1051) with the body pose (filtered CoM,
//      /rtMPC/traj slots 72 / 73 = roll / pitch, yaw 0), from the previous tick's joint angles.
// One thread per (robot, leg), a robot's four legs on adjacent lanes (the servo_kin_kernel mapping).  Filter channel c is
// stepped by lane c % 4 of the group (lane 0 also takes channel 8) and the group shares the outputs by shuffle.  The message
// slots, the filter state, the joint angles and the homing positions are loaded once per call and carried in registers over
// the K ticks; q is stored per tick, the state once at the end.  The arithmetic is servo_math.cuh's, which lpf_kernel and
// servo_kin_kernel also run: the call equals K x (go1mpc_lpf_batch + go1mpc_servo_kin_tick_batch) bit for bit.
#include <cuda_runtime.h>
#include "kernels.h"
#include "servo_math.cuh"

namespace go1 {

namespace {
// /MPC/Gait slot filtered by channel c (0 1 2 | 6 7 8 | 9 10 11)
__device__ __forceinline__ constexpr int lpf_slot(int c) { return c < 3 ? c : c + 3; }
}  // namespace

// CH: also store each tick's nine filtered channels to P.ch [K][9][B] (the servo torque tick's second kernel reads them).
// H: also count the leg-ticks whose IK applied all 15 updates into the robot's health row FH_IK_CAP (the group's four legs summed
// by shuffle, lane 0 of the group writes) and mark the row in FH_EVENTS.
template <bool CH, bool H = false>
__global__ void __launch_bounds__(256) servo_stack_kernel(ServoStackKParams P) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t B = (size_t)P.B;
  // 4B threads and 256-thread blocks: a robot's group is either wholly live or wholly out of range
  const unsigned live = __ballot_sync(0xffffffffu, idx < 4 * B);
  if (idx >= 4 * B) return;
  const size_t b = idx >> 2;
  const int leg = (int)(idx & 3);
  const int nch = leg == 0 ? 3 : 2;             // this lane's channels: leg, leg + 4 (, 8)

  LpfState fs[3];
  double y[3];
#pragma unroll
  for (int j = 0; j < 3; j++) {
    const int c = leg + 4 * j;
    if (j < nch) {
      const double* S = P.state + (size_t)(SERVO_ROW_LPF + c) * B + b;
      const size_t CB = (size_t)SERVO_LPF_CHANNELS * B;
      fs[j] = LpfState{S[0], S[CB], S[2 * CB], S[3 * CB], S[4 * CB]};
      y[j] = P.gait[(size_t)lpf_slot(c) * B + b];
    } else {
      fs[j] = LpfState{0.0, 0.0, 0.0, 0.0, 0.0};
      y[j] = 0.0;
    }
  }
  const bool right = servo_follows_right(P.gait_mode, leg);
  const LegC lc = leg_consts(leg);
  double hom[3], q[3];
#pragma unroll
  for (int k = 0; k < 3; k++) {
    hom[k] = P.state[(size_t)(SERVO_ROW_HOMING + 3 * leg + k) * B + b];
    q[k] = P.state[(size_t)(SERVO_ROW_Q + 3 * leg + k) * B + b];
  }
  Body bd;
  bd.on = true;
  body_rotation(P.traj[72 * B + b], P.traj[73 * B + b], 0.0, bd.R);

  double* qo = P.q_out + b * (size_t)(12 * P.K) + 3 * leg;
  double pdes[3], J[9];
  int it = 0, capped = 0;
  for (int k = 0; k < P.K; k++) {
    double f[3];
#pragma unroll
    for (int j = 0; j < 3; j++) f[j] = (j < nch) ? lpf_step(P.coef, fs[j], y[j]) : 0.0;
    if constexpr (CH) {
#pragma unroll
      for (int j = 0; j < 3; j++)
        if (j < nch) P.ch[((size_t)k * SERVO_LPF_CHANNELS + leg + 4 * j) * B + b] = f[j];
    }
    double ch[SERVO_LPF_CHANNELS];                // channel c: lane c % 4 of the group, its f[c / 4]
#pragma unroll
    for (int c = 0; c < SERVO_LPF_CHANNELS; c++) ch[c] = __shfl_sync(live, f[c >> 2], c & 3, 4);
    bd.p[0] = ch[0]; bd.p[1] = ch[1] * P.y_offset; bd.p[2] = ch[2];
    const double vf[3] = {right ? ch[6] : ch[3], right ? ch[7] : ch[4], right ? ch[8] : ch[5]};
    servo_leg_target(hom, vf, right, P.half_hip_width, pdes);
    it = servo_leg_ik(lc, bd, pdes, q, J);
    if constexpr (H) capped += (it == 15);
    qo[12 * k] = q[0]; qo[12 * k + 1] = q[1]; qo[12 * k + 2] = q[2];
  }

#pragma unroll
  for (int k = 0; k < 3; k++) P.state[(size_t)(SERVO_ROW_Q + 3 * leg + k) * B + b] = q[k];
#pragma unroll
  for (int j = 0; j < 3; j++) {
    if (j < nch) {
      double* S = P.state + (size_t)(SERVO_ROW_LPF + leg + 4 * j) * B + b;
      const size_t CB = (size_t)SERVO_LPF_CHANNELS * B;
      S[0] = fs[j].i; S[CB] = fs[j].y_p; S[2 * CB] = fs[j].y_pp; S[3 * CB] = fs[j].x_p; S[4 * CB] = fs[j].x_pp;
    }
  }
  if (P.jac) for (int k = 0; k < 9; k++) P.jac[(size_t)(9 * leg + k) * B + b] = J[k];
  if (P.foot_des) for (int k = 0; k < 3; k++) P.foot_des[(size_t)(3 * leg + k) * B + b] = pdes[k];
  if (P.iters) P.iters[(size_t)leg * B + b] = it;
  if constexpr (H) {
    capped += __shfl_xor_sync(live, capped, 1, 4);
    capped += __shfl_xor_sync(live, capped, 2, 4);
    if (leg == 0 && capped) {
      P.health[(size_t)FH_IK_CAP * B + b] += capped;
      P.health[(size_t)FH_EVENTS * B + b] |= 1 << FH_IK_CAP;
    }
  }
}

cudaError_t servo_stack_launch(const ServoStackKParams& P, cudaStream_t st) {
  const size_t threads = 4 * (size_t)P.B;
  if (P.health) servo_stack_kernel<true, true><<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(P);
  else if (P.ch) servo_stack_kernel<true><<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(P);
  else servo_stack_kernel<false><<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(P);
  return cudaGetLastError();
}

}  // namespace go1
