// farm_health.cu -- the health counters of a controller farm after a clocked gait stack tick
// (go1mpc_gait_stack_tick_clocked_health_async).  Thread per robot, after the pack kernel: the robot's counters restart when its
// clock was 0 at the start of the call, then the statuses the planner and body MPC wrote into the call's diag workspaces and a
// non-finite value in the robot's rows_d row are counted, and FH_EVENTS is overwritten with the rows that grew.  The torque tick's
// kernels add their rows and OR their bits afterwards (servo_stack.cu, servo_torque.cu).
#include "kernels.h"

namespace go1 {

namespace {
// solver status -> OK / INFEASIBLE / FAILED row offset, or -1 for "no solve" (status < 0)
__device__ __forceinline__ int status_row(int s) { return s < 0 ? -1 : (s == 0 ? 0 : (s == 2 ? 1 : 2)); }
}  // namespace

__global__ void __launch_bounds__(256) farm_health_stack_kernel(FarmHealthStackParams P) {
  const size_t Bs = (size_t)P.B;
  for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < Bs; b += (size_t)gridDim.x * blockDim.x) {
    int h[FARM_HEALTH_ROWS - 1];
    const bool restart = P.clock[b] == 1;      // the clock was 0 when the call started: a fresh episode
#pragma unroll
    for (int r = 0; r < FARM_HEALTH_ROWS - 1; r++) h[r] = restart ? 0 : P.health[(size_t)r * Bs + b];
    int add[FARM_HEALTH_ROWS - 1];
#pragma unroll
    for (int r = 0; r < FARM_HEALTH_ROWS - 1; r++) add[r] = 0;
    // the SQP kernels write nothing for a robot without a planner tick: its diag column is stale.  Within a tick, unsolved
    // iterations read status -1.
    if (P.node_tick[b] >= 1) {
#pragma unroll
      for (int q = 0; q < STEP_MAX_SQP; q++) {
        const int o = status_row(P.step_diag[(size_t)(STEP_DIAG_HEAD + q * STEP_DIAG_PER) * Bs + b]);
        if (o >= 0) add[FH_PLAN_OK + o]++;
      }
    }
    const int ob = status_row(P.body_diag[b * (size_t)P.body_diag_stride]);   // -1: gated tick
    if (ob >= 0) add[FH_BODY_OK + ob]++;
    bool bad = false;
    const double* row = P.rows + b * (size_t)P.n_slots;
    for (int k = 0; k < P.n_slots; k++) bad = bad || !isfinite(row[k]);
    add[FH_NONFINITE] = bad ? 1 : 0;
    int ev = 0;
#pragma unroll
    for (int r = 0; r < FARM_HEALTH_ROWS - 1; r++) {
      if (restart || add[r]) P.health[(size_t)r * Bs + b] = h[r] + add[r];
      if (add[r]) ev |= 1 << r;
    }
    P.health[(size_t)FH_EVENTS * Bs + b] = ev;
  }
}

cudaError_t farm_health_stack_launch(const FarmHealthStackParams& P, int sms, cudaStream_t st) {
  size_t g = ((size_t)P.B + 255) / 256;
  const size_t cap = (size_t)sms * 8;
  farm_health_stack_kernel<<<(unsigned)(g < cap ? g : cap), 256, 0, st>>>(P);
  return cudaGetLastError();
}

}  // namespace go1
