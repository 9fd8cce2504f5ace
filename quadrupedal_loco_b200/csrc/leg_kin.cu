// leg_kin.cu -- Go1 leg forward kinematics, analytic Jacobian and damped-Newton IK, one thread per leg.
//
// Replaces Kinematicclass (GO1 = unitree_ros/go1_rt_control):
//   Forward_kinematics    GO1/src/kinematics/Kinematics.cpp:63-142   (hip frame)
//   Forward_kinematics_g  :145-229  (world frame: body position + roll/pitch/yaw)
//   Inverse_kinematics    :233-267  (lamda 0.5, <= 10 updates, stop: max(dq) < 1e-4, no abs)
//   Inverse_kinematics_g  :270-304  (lamda 0.5, <= 15 updates, stop: |dp|^2 <= 1e-6)
// and its Jacobian_kin side channel (Kinematics.h:60), returned as an output array.
// The reference's expanded trigonometric polynomials are evaluated in factored form:
//   p = body_P + Rz Ry Rx p_hip(q),  J = R J_hip(q),  K = lc sin(q2+q3) + lt sin q2,
//   L = lc cos(q2+q3) + lt cos q2  -- 6 sincos (+3 for the body) instead of ~600 flops of
// repeated products.  Layout: structure of arrays, element-major / batch-minor ([f*B + b]):
// every access of a warp is one coalesced 256-byte segment.  HBM-bound in principle
// (FK: 4 + 8*(3+6) B in, 8*12 B out per leg), sincos-bound in practice.
#include <cuda_runtime.h>
#include "kernels.h"
#include "servo_math.cuh"   // fk / Jacobian / Newton step, the servo leg stage

namespace go1 {

namespace {
__device__ __forceinline__ Body load_body(const double* bp, const double* br, size_t B, int b) {
  Body bd;
  bd.on = (bp != nullptr);
  if (bd.on) {
    for (int k = 0; k < 3; k++) bd.p[k] = bp[k * B + b];
    body_rotation(br[b], br[B + b], br[2 * B + b], bd.R);
  }
  return bd;
}
}  // namespace

__global__ void __launch_bounds__(256) leg_fk_kernel(LegKParams P) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= P.B) return;
  const size_t B = (size_t)P.B;
  const double q[3] = {P.q_in[b], P.q_in[B + b], P.q_in[2 * B + b]};
  const LegC c = leg_consts(P.leg[b]);
  const Body bd = load_body(P.body_p, P.body_r, B, b);
  double pos[3], J[9];
  fk_any(q, c, bd, pos, J);
  for (int k = 0; k < 3; k++) P.pos_out[k * B + b] = pos[k];
  if (P.jac_out) for (int k = 0; k < 9; k++) P.jac_out[k * B + b] = J[k];
}

__global__ void __launch_bounds__(256) leg_ik_kernel(LegKParams P) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= P.B) return;
  const size_t B = (size_t)P.B;
  const double pdes[3] = {P.pdes[b], P.pdes[B + b], P.pdes[2 * B + b]};
  double q[3] = {P.q_in[b], P.q_in[B + b], P.q_in[2 * B + b]};
  const LegC c = leg_consts(P.leg[b]);
  const Body bd = load_body(P.body_p, P.body_r, B, b);
  const int maxit = bd.on ? 15 : 10;
  double pc[3], J[9], dp[3], dq[3];
  fk_any(q, c, bd, pc, J);
  int it = 0;
  for (int j = 0; j < maxit; j++) {
    for (int k = 0; k < 3; k++) dp[k] = pdes[k] - pc[k];
    newton_step(J, dp, 0.5, dq);
    bool stop;
    if (bd.on) stop = fabs(dp[0] * dp[0] + dp[1] * dp[1] + dp[2] * dp[2]) <= 0.000001;
    else stop = fmax(dq[0], fmax(dq[1], dq[2])) < 0.0001;       // no abs: the reference's test, Kinematics.cpp:249
    if (stop) break;
    q[0] += dq[0]; q[1] += dq[1]; q[2] += dq[2];
    fk_any(q, c, bd, pc, J);
    it++;
  }
  for (int k = 0; k < 3; k++) P.q_out[k * B + b] = q[k];
  if (P.jac_out) for (int k = 0; k < 9; k++) P.jac_out[k * B + b] = J[k];
  if (P.iters) P.iters[b] = it;
}

// ---------------------------------------------------------------------------------------------
// Servo kinematics tick (GO1/src/servo_control/servo.cpp:935-1051): the planner's virtual right /
// left foot is mapped onto the four legs by gait_mode (101 pace: FR,RR <- right, FL,RL <- left;
// 102 trot: FR,RL <- right, FL,RR <- left; 103 gallop: FR,FL <- right, RR,RL <- left), each foot
// target = homing position + virtual foot displacement -+ half hip width, then
// Inverse_kinematics_g per leg from the previous joint angles, Jacobian side channel included.
// One thread per (robot, leg): 4 B threads, the body pose is shared by a robot's four threads.
__global__ void __launch_bounds__(256) servo_kin_kernel(ServoKParams P) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 4 * P.B) return;
  const int b = idx >> 2, leg = idx & 3;
  const size_t B = (size_t)P.B;
  const bool right = servo_follows_right(P.gait_mode, leg);
  const double* vf = right ? P.rfoot : P.lfoot;
  const double hom[3] = {P.homing[(size_t)(3 * leg) * B + b], P.homing[(size_t)(3 * leg + 1) * B + b], P.homing[(size_t)(3 * leg + 2) * B + b]};
  const double v[3] = {vf[b], vf[B + b], vf[2 * B + b]};
  double pdes[3];
  servo_leg_target(hom, v, right, P.half_hip_width, pdes);
  const LegC c = leg_consts(leg);
  Body bd;
  bd.on = true;
  bd.p[0] = P.com[b]; bd.p[1] = P.com[B + b] * P.y_offset; bd.p[2] = P.com[2 * B + b];
  body_rotation(P.theta[b], P.theta[B + b], P.theta[2 * B + b], bd.R);
  double q[3] = {P.q[(size_t)(3 * leg) * B + b], P.q[(size_t)(3 * leg + 1) * B + b], P.q[(size_t)(3 * leg + 2) * B + b]};
  double J[9];
  const int it = servo_leg_ik(c, bd, pdes, q, J);
  for (int k = 0; k < 3; k++) P.q[(size_t)(3 * leg + k) * B + b] = q[k];
  if (P.jac) for (int k = 0; k < 9; k++) P.jac[(size_t)(9 * leg + k) * B + b] = J[k];
  if (P.foot_des) for (int k = 0; k < 3; k++) P.foot_des[(size_t)(3 * leg + k) * B + b] = pdes[k];
  if (P.iters) P.iters[(size_t)leg * B + b] = it;
}

cudaError_t servo_kin_launch(ServoKParams P, cudaStream_t st) {
  servo_kin_kernel<<<(4 * P.B + 255) / 256, 256, 0, st>>>(P);
  return cudaGetLastError();
}

cudaError_t leg_fk_launch(LegKParams P, cudaStream_t st) {
  leg_fk_kernel<<<(P.B + 255) / 256, 256, 0, st>>>(P);
  return cudaGetLastError();
}
cudaError_t leg_ik_launch(LegKParams P, cudaStream_t st) {
  leg_ik_kernel<<<(P.B + 255) / 256, 256, 0, st>>>(P);
  return cudaGetLastError();
}

// Fused tick glue: body orientation for the servo stage from the body-MPC output records (AoS, stride doubles):
// roll = out[0], pitch = out[1] (the Vec14's next-step angles, PRMPCClass.cpp:696-712), yaw = 0.  -> theta [3][B] SoA.
__global__ void __launch_bounds__(256) body_theta_gather_kernel(int B, const double* body_out, int stride, double* theta) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const double* o = body_out + (size_t)b * stride;
  theta[b] = o[0];
  theta[(size_t)B + b] = o[1];
  theta[2 * (size_t)B + b] = 0.0;
}
cudaError_t body_theta_gather_launch(int B, const double* body_out, int stride, double* theta, cudaStream_t st) {
  body_theta_gather_kernel<<<(B + 255) / 256, 256, 0, st>>>(B, body_out, stride, theta);
  return cudaGetLastError();
}

}  // namespace go1
