// servo_math.cuh -- the per-sample arithmetic of go1_servo's 1 kHz loop, shared by every kernel that runs it:
//   leg kinematics + the servo's leg mapping and Inverse_kinematics_g   leg_kin.cu (leg_fk / leg_ik / servo_kin_kernel)
//   the butterworthLPF step                                            filters.cu (lpf_kernel)
//   both, K ticks in registers                                         servo_stack.cu (servo_stack_kernel)
// One copy of the arithmetic: the fused servo stack tick and the single-stage entries compute the same bits by
// construction.  Every file that includes this header is compiled with -fmad=false (the reference's operation order).
#pragma once
#include <cuda_runtime.h>
#include "kernels.h"

namespace go1 {

// ---------------------------------------------------------------------------------------------- leg kinematics
// Kinematicclass (GO1/src/kinematics/Kinematics.cpp:63-304) in factored form, see leg_kin.cu
constexpr double L_THIGH = -0.213, L_CALF = -0.213;

struct LegC { double ox, oy, ty; };
__device__ __forceinline__ LegC leg_consts(int leg) {
  LegC c;
  c.ox = (leg == 0 || leg == 1) ? 0.1881 : -0.1881;
  c.oy = (leg == 0 || leg == 2) ? -0.04675 : 0.04675;
  c.ty = (leg == 0 || leg == 2) ? -0.08 : 0.08;
  return c;
}
__device__ __forceinline__ void fk_hip(const double q[3], const LegC& c, double pos[3], double J[9]) {
  double s1, c1, s2, c2, s3, c3;
  sincos(q[0], &s1, &c1); sincos(q[1], &s2, &c2); sincos(q[2], &s3, &c3);
  const double s23 = c3 * s2 + c2 * s3, c23 = c3 * c2 - s3 * s2;
  const double K = L_CALF * s23 + L_THIGH * s2;
  const double L = L_CALF * c23 + L_THIGH * c2;
  pos[0] = c.ox + K;
  pos[1] = c.oy + c.ty * c1 - s1 * L;
  pos[2] = c.ty * s1 + c1 * L;
  J[0] = 0.0;                     J[1] = L;        J[2] = L_CALF * c23;
  J[3] = -(c.ty * s1 + c1 * L);   J[4] = s1 * K;   J[5] = s1 * (L_CALF * s23);
  J[6] = c.ty * c1 - s1 * L;      J[7] = -c1 * K;  J[8] = -c1 * (L_CALF * s23);
}
struct Body { bool on; double p[3], R[9]; };
__device__ __forceinline__ void fk_any(const double q[3], const LegC& c, const Body& bd, double pos[3], double J[9]) {
  if (!bd.on) { fk_hip(q, c, pos, J); return; }
  double pl[3], Jl[9];
  fk_hip(q, c, pl, Jl);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    pos[i] = bd.p[i] + (bd.R[3 * i] * pl[0] + bd.R[3 * i + 1] * pl[1] + bd.R[3 * i + 2] * pl[2]);
#pragma unroll
    for (int j = 0; j < 3; j++) J[3 * i + j] = bd.R[3 * i] * Jl[j] + bd.R[3 * i + 1] * Jl[3 + j] + bd.R[3 * i + 2] * Jl[6 + j];
  }
}
// body rotation Rz(yaw) Ry(pitch) Rx(roll), row-major
__device__ __forceinline__ void body_rotation(double roll, double pitch, double yaw, double R[9]) {
  double sr, cr, sp, cp, sy, cy;
  sincos(roll, &sr, &cr); sincos(pitch, &sp, &cp); sincos(yaw, &sy, &cy);
  R[0] = cp * cy; R[1] = cy * sp * sr - cr * sy; R[2] = sr * sy + cr * cy * sp;
  R[3] = cp * sy; R[4] = cr * cy + sp * sr * sy; R[5] = cr * sp * sy - cy * sr;
  R[6] = -sp;     R[7] = cp * sr;                R[8] = cp * cr;
}
// dq = lamda J^-1 dp by cofactors
__device__ __forceinline__ void newton_step(const double J[9], const double dp[3], double lamda, double dq[3]) {
  const double c00 = J[4] * J[8] - J[5] * J[7], c01 = J[5] * J[6] - J[3] * J[8], c02 = J[3] * J[7] - J[4] * J[6];
  const double det = J[0] * c00 + J[1] * c01 + J[2] * c02;
  const double id = 1.0 / det;
  const double i00 = c00 * id, i01 = (J[2] * J[7] - J[1] * J[8]) * id, i02 = (J[1] * J[5] - J[2] * J[4]) * id;
  const double i10 = c01 * id, i11 = (J[0] * J[8] - J[2] * J[6]) * id, i12 = (J[2] * J[3] - J[0] * J[5]) * id;
  const double i20 = c02 * id, i21 = (J[1] * J[6] - J[0] * J[7]) * id, i22 = (J[0] * J[4] - J[1] * J[3]) * id;
  dq[0] = (lamda * i00) * dp[0] + (lamda * i01) * dp[1] + (lamda * i02) * dp[2];
  dq[1] = (lamda * i10) * dp[0] + (lamda * i11) * dp[1] + (lamda * i12) * dp[2];
  dq[2] = (lamda * i20) * dp[0] + (lamda * i21) * dp[1] + (lamda * i22) * dp[2];
}

// ---------------------------------------------------------------------------------------------- servo leg stage
// GO1/src/servo_control/servo.cpp:935-1051.  Does leg `leg` (FR=0, FL=1, RR=2, RL=3) follow the planner's virtual right foot?
// 101 pace: FR, RR <- right, FL, RL <- left; 102 trot: FR, RL <- right; 103 gallop: FR, FL <- right.
__device__ __forceinline__ bool servo_follows_right(int gait_mode, int leg) {
  const unsigned right_mask = (gait_mode == 101) ? 0x5u : ((gait_mode == 102) ? 0x9u : 0x3u);
  return (right_mask >> leg) & 1u;
}
// foot target = homing position + virtual foot displacement -+ half hip width (y)
__device__ __forceinline__ void servo_leg_target(const double hom[3], const double vf[3], bool right, double half_hip_width,
                                                 double pdes[3]) {
  for (int k = 0; k < 3; k++) pdes[k] = hom[k] + vf[k];
  pdes[1] = hom[1] + vf[1] + (right ? half_hip_width : -half_hip_width);
}
// Inverse_kinematics_g (Kinematics.cpp:270-304: lamda 0.5, <= 15 updates, stop |dp|^2 <= 1e-6) from the joint angles q
// (in/out); J = the Jacobian at the returned q.  Returns the number of updates applied.
__device__ __forceinline__ int servo_leg_ik(const LegC& c, const Body& bd, const double pdes[3], double q[3], double J[9]) {
  double pc[3], dp[3], dq[3];
  fk_any(q, c, bd, pc, J);
  int it = 0;
  for (int j = 0; j < 15; j++) {
    for (int k = 0; k < 3; k++) dp[k] = pdes[k] - pc[k];
    newton_step(J, dp, 0.5, dq);
    if (fabs(dp[0] * dp[0] + dp[1] * dp[1] + dp[2] * dp[2]) <= 0.000001) break;
    q[0] += dq[0]; q[1] += dq[1]; q[2] += dq[2];
    fk_any(q, c, bd, pc, J);
    it++;
  }
  return it;
}

// ---------------------------------------------------------------------------------------------- signal filter
// butterworthLPF::filter (GO1/src/Filter/butterworthLPF.cpp:104-121) on one sample y: the first three calls run the
// first-order start-up filter and count, later calls the second-order section.  State = one object's members.
struct LpfState { double i, y_p, y_pp, x_p, x_pp; };
__device__ __forceinline__ double lpf_step(const LpfCoef& k, LpfState& s, double y) {
  double out;
  if (s.i > 2) {
    out = k.b0 * y + k.b1 * s.y_p + k.b2 * s.y_pp + k.a1 * s.x_p + k.a2 * s.x_pp;
  } else {
    out = s.x_p + k.a * (y - s.x_p);
    s.i = s.i + 1;
  }
  s.y_pp = s.y_p; s.y_p = y; s.x_pp = s.x_p; s.x_p = out;
  return out;
}

}  // namespace go1
