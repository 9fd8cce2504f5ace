// gait_stack.cu -- the two copy kernels of the gait stack tick (go1mpc_gait_stack_tick_host_async): both MPC nodes of the
// reference behind one host call, everything the nodes keep as members resident in one SoA state [row][B].
//
//   gait_stack_pre_kernel  : when the planner ticks, walkdtime += 1 in the state (kept as an exact integer double) and as the
//                            int the planner node reads; the 11 uploaded sensor rows -> their slots of /control2rtmpc/state
//   gait_stack_pack_kernel : the selected slots of /MPC/Gait and /rtMPC/traj -> one row of n_slots doubles per robot
// Thread per robot (pre) / per output double (pack): every warp access is coalesced over B.
#include "kernels.h"

namespace go1 {

namespace {
// /control2rtmpc/state slot of uploaded sensor row k: 0 | 10 11 13 14 | 19 20 21 | 22 23 24 (flag | body angles / rates |
// left foot xyz | right foot xyz)
__device__ __forceinline__ constexpr int sensor_slot(int k) { return k == 0 ? 0 : (k < 3 ? 9 + k : (k < 5 ? 10 + k : 14 + k)); }
}  // namespace

__global__ void __launch_bounds__(256) gait_stack_pre_kernel(int B, int planner, double* __restrict__ walkdtime_row,
                                                             int* __restrict__ walkdtime_i, const double* __restrict__ sensor,
                                                             double* __restrict__ ctl) {
  const size_t Bs = (size_t)B;
  for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < Bs; b += (size_t)gridDim.x * blockDim.x) {
    if (planner) {
      const double w = walkdtime_row[b] + 1.0;
      walkdtime_row[b] = w;
      walkdtime_i[b] = (int)w;
    }
#pragma unroll
    for (int k = 0; k < GAIT_STACK_SENSOR_ROWS; k++) ctl[(size_t)sensor_slot(k) * Bs + b] = sensor[(size_t)k * Bs + b];
  }
}

__global__ void __launch_bounds__(256) gait_stack_pack_kernel(GaitStackSlots S, int B, const double* __restrict__ gait,
                                                              const double* __restrict__ traj, double* __restrict__ rows) {
  const size_t Bs = (size_t)B, total = Bs * S.n;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t b = idx / S.n;
    const int s = S.slot[idx - b * S.n];
    rows[idx] = s < 100 ? gait[(size_t)s * Bs + b] : traj[(size_t)(s - 100) * Bs + b];
  }
}

static int stack_grid(size_t total, int sms) {
  size_t g = (total + 255) / 256;
  const size_t cap = (size_t)sms * 8;
  return (int)(g < cap ? (g ? g : 1) : cap);
}

cudaError_t gait_stack_pre_launch(int B, int planner, double* walkdtime_row, int* walkdtime_i, const double* sensor, double* ctl,
                                  int sms, cudaStream_t st) {
  gait_stack_pre_kernel<<<stack_grid((size_t)B, sms), 256, 0, st>>>(B, planner, walkdtime_row, walkdtime_i, sensor, ctl);
  return cudaGetLastError();
}
cudaError_t gait_stack_pack_launch(const GaitStackSlots& S, int B, const double* gait, const double* traj, double* rows, int sms,
                                   cudaStream_t st) {
  gait_stack_pack_kernel<<<stack_grid((size_t)B * S.n, sms), 256, 0, st>>>(S, B, gait, traj, rows);
  return cudaGetLastError();
}

}  // namespace go1
