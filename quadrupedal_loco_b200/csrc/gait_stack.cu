// gait_stack.cu -- the copy kernels of the gait stack ticks (go1mpc_gait_stack_tick_host_async, go1mpc_gait_stack_tick_clocked_async)
// and the robot reset (go1mpc_gait_stack_reset_async): both MPC nodes of the reference behind one host call, everything the nodes
// keep as members resident in one SoA state [row][B].
//
//   gait_stack_pre_kernel  : when the planner ticks, walkdtime += 1 in the state (kept as an exact integer double) and as the
//                            int the planner node reads; the 11 uploaded sensor rows -> their slots of /control2rtmpc/state
//   gait_stack_pack_kernel : the selected slots of /MPC/Gait and /rtMPC/traj -> one row of n_slots doubles per robot
//   gait_stack_clocked_pre_kernel : per-robot clocks (periods since the robot's reset): whether each robot's planner ticks this
//                            call, into a mask the planner node reads; walkdtime += 1 for those robots; clock += 1; the sensor scatter
//   gait_stack_reset_mark_kernel / gait_stack_reset_column_kernel : robot resets, see below
//   farm_copy_list_kernel / farm_copy_column_kernel : whole robot columns copied between two farms (go1mpc_farm_copy_async)
//                            (the health rows of farm_health.cu travel with the clock, in the list kernel)
// Thread per robot (pre) / per output double (pack): every warp access is coalesced over B.
#include "kernels.h"

namespace go1 {

namespace {
// /control2rtmpc/state slot of uploaded sensor row k: 0 | 10 11 13 14 | 19 20 21 | 22 23 24 (flag | body angles / rates |
// left foot xyz | right foot xyz)
__device__ __forceinline__ constexpr int sensor_slot(int k) { return k == 0 ? 0 : (k < 3 ? 9 + k : (k < 5 ? 10 + k : 14 + k)); }

__device__ __forceinline__ void scatter_sensors(size_t b, size_t Bs, const double* __restrict__ sensor, double* __restrict__ ctl) {
#pragma unroll
  for (int k = 0; k < GAIT_STACK_SENSOR_ROWS; k++) ctl[(size_t)sensor_slot(k) * Bs + b] = sensor[(size_t)k * Bs + b];
}
__device__ __forceinline__ void bump_walkdtime(size_t b, double* __restrict__ walkdtime_row, int* __restrict__ walkdtime_i) {
  const double w = walkdtime_row[b] + 1.0;
  walkdtime_row[b] = w;
  walkdtime_i[b] = (int)w;
}
// Reserves a slot of a device list for every flagged lane of the warp with one atomicAdd on *count per warp, and returns whether
// this lane is flagged, its slot in *slot.  Every lane of the warp must arrive.  Slots of one warp are consecutive and in lane order.
__device__ __forceinline__ bool warp_list_slot(bool flag, int* count, int* slot) {
  const unsigned m = __ballot_sync(0xffffffffu, flag);
  if (!m) return false;
  const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
  int base = 0;
  if (lane == leader) base = atomicAdd(count, __popc(m));
  base = __shfl_sync(0xffffffffu, base, leader);
  if (!flag) return false;
  *slot = base + __popc(m & ((1u << lane) - 1));
  return true;
}
}  // namespace

__global__ void __launch_bounds__(256) gait_stack_pre_kernel(int B, int planner, double* __restrict__ walkdtime_row,
                                                             int* __restrict__ walkdtime_i, const double* __restrict__ sensor,
                                                             double* __restrict__ ctl) {
  const size_t Bs = (size_t)B;
  for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < Bs; b += (size_t)gridDim.x * blockDim.x) {
    if (planner) bump_walkdtime(b, walkdtime_row, walkdtime_i);
    scatter_sensors(b, Bs, sensor, ctl);
  }
}

// The reference's clock, per robot: the fast tick at 10c ms after the robot's reset runs the planner first when a multiple of 25
// lies in (10(c-1), 10c], i.e. c = 0, 3, 5, 8, 10, ... (c mod 5 in {0, 3}).  64-bit products: no overflow at any int clock.
__global__ void __launch_bounds__(256) gait_stack_clocked_pre_kernel(int B, int* __restrict__ clock, int* __restrict__ plan,
                                                                     double* __restrict__ walkdtime_row, int* __restrict__ walkdtime_i,
                                                                     const double* __restrict__ sensor, double* __restrict__ ctl) {
  const size_t Bs = (size_t)B;
  for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < Bs; b += (size_t)gridDim.x * blockDim.x) {
    const long long c = clock[b];
    const int p = (c == 0 || (10 * c) / 25 > (10 * (c - 1)) / 25) ? 1 : 0;
    plan[b] = p;
    if (p) bump_walkdtime(b, walkdtime_row, walkdtime_i);
    clock[b] = (int)(c + 1);
    scatter_sensors(b, Bs, sensor, ctl);
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

// ---- robot resets.  Thread per robot: the flagged robots are appended to a list with one atomic per warp, and get their small
// writes here -- clock 0, the body-MPC record zeroed with 16-byte stores (records are 16-byte aligned, an even number of doubles),
// the servo joint angles q0 and zero filter rows (the homing rows are the caller's input and stay).  Every lane reaches the ballot:
// the grid covers B exactly, lanes past B vote 0.
__global__ void __launch_bounds__(256) gait_stack_reset_mark_kernel(StackResetParams P) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const bool flag = b < P.B && P.reset[b] != 0;
  int slot;
  if (!warp_list_slot(flag, P.count, &slot)) return;
  P.list[slot] = b;
  P.clock[b] = 0;
  double2* rec = reinterpret_cast<double2*>(P.body_out + (size_t)b * P.out_stride);
  const double2 z = make_double2(0.0, 0.0);
  for (int k = 0; k < P.out_stride / 2; k++) rec[k] = z;
  if (P.servo) {
    const size_t Bs = (size_t)P.B;
    double* S = P.servo + b;
#pragma unroll
    for (int k = 0; k < 12; k++) S[(size_t)(SERVO_ROW_Q + k) * Bs] = P.q0[k];
#pragma unroll 5
    for (int k = SERVO_ROW_LPF; k < SERVO_STATE_ROWS; k++) S[(size_t)k * Bs] = 0.0;
  }
}

// Grid-stride over (row, listed robot), robot-minor: the count is read on the device, so the launch does not depend on how many
// robots reset, and a call with no reset costs one read of the count per thread.
__global__ void __launch_bounds__(256) gait_stack_reset_column_kernel(StackResetParams P) {
  const size_t n = (size_t)*P.count, total = n * (size_t)P.rows, Bs = (size_t)P.B;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t r = idx / n;
    P.state[r * Bs + P.list[idx - r * n]] = P.column[r];
  }
}

// ---- farm column copy.  Thread per destination column: the columns with a valid source are listed with one atomic per warp, with
// their source beside them, and get their clock and health counters here.  Entries outside -1..src_B-1 are counted (one atomic per warp) and never read
// through.  Every lane reaches the ballots: lanes past dst_B hold -1.
__global__ void __launch_bounds__(256) farm_copy_list_kernel(FarmCopyParams P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int s = i < P.dst_B ? P.index[i] : -1;
  if (P.bad) {
    const unsigned mb = __ballot_sync(0xffffffffu, s < -1 || s >= P.src_B);
    if (mb && (threadIdx.x & 31) == __ffs(mb) - 1) atomicAdd(P.bad, __popc(mb));
  }
  const bool take = s >= 0 && s < P.src_B;
  int slot;
  if (!warp_list_slot(take, P.count, &slot)) return;
  P.dlist[slot] = i;
  P.slist[slot] = s;
  if (P.dst_clock) P.dst_clock[i] = P.src_clock[s];
  if (P.dst_health) {
#pragma unroll
    for (int r = 0; r < FARM_HEALTH_ROWS; r++) P.dst_health[(size_t)r * P.dst_B + i] = P.src_health[(size_t)r * P.src_B + s];
  }
}

constexpr int FARM_TASK_ROWS = 32;   // SoA rows per warp task
constexpr int FARM_UNROLL = 8;       // loads in flight per lane

__device__ __forceinline__ void farm_soa_row(const FarmCopyParams& P, int r, const double*& s, double*& d) {
  if (r < P.rows) {
    s = P.src_state + (size_t)r * P.src_B; d = P.dst_state + (size_t)r * P.dst_B;
  } else if (r < P.servo_end) {
    s = P.src_servo + (size_t)(r - P.rows) * P.src_B; d = P.dst_servo + (size_t)(r - P.rows) * P.dst_B;
  } else {
    s = P.src_force + (size_t)(r - P.servo_end) * P.src_B; d = P.dst_force + (size_t)(r - P.servo_end) * P.dst_B;
  }
}

// The listed columns, count read on the device.  SoA rows: a warp task is 32 consecutive list entries (one per lane, loaded once)
// x FARM_TASK_ROWS rows, so every row is one warp-wide access -- the stores coalesced over the listed destinations, the loads
// coalesced where the index is monotone and L2 hits where many destinations share few sources.  The row is uniform over the warp,
// so picking the state / servo / force block does not diverge.  Body records: grid-stride over (listed column, double2), the
// double2 fastest; the (column, double2) pair advances by the stride's quotient and remainder, with no division in the loop.
__global__ void __launch_bounds__(256) farm_copy_column_kernel(FarmCopyParams P) {
  const int n = *P.count;
  if (!n) return;
  const int lane = threadIdx.x & 31;
  const int ngroups = (n + 31) >> 5, nchunks = (P.soa_rows + FARM_TASK_ROWS - 1) / FARM_TASK_ROWS;
  const long long tasks = (long long)ngroups * nchunks, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long t = (((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5); t < tasks; t += nwarps) {
    const int g = (int)(t % ngroups), r0 = (int)(t / ngroups) * FARM_TASK_ROWS;
    const int j = (g << 5) + lane;
    if (j >= n) continue;
    const int dc = P.dlist[j], sc = P.slist[j];
    const int r1 = min(r0 + FARM_TASK_ROWS, P.soa_rows);
    for (int r = r0; r < r1; r += FARM_UNROLL) {
      double v[FARM_UNROLL];
      double* d[FARM_UNROLL];
#pragma unroll
      for (int u = 0; u < FARM_UNROLL; u++) {
        d[u] = nullptr;
        if (r + u < r1) {
          const double* s;
          farm_soa_row(P, r + u, s, d[u]);
          v[u] = s[sc];
          d[u] += dc;
        }
      }
#pragma unroll
      for (int u = 0; u < FARM_UNROLL; u++)
        if (d[u]) *d[u] = v[u];
    }
  }
  const size_t h = (size_t)P.rec2, stride = (size_t)gridDim.x * blockDim.x, t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t dj = stride / h, dk = stride - dj * h;
  for (size_t j = t0 / h, k = t0 - j * h; j < (size_t)n;) {
    P.dst_body[(size_t)P.dlist[j] * h + k] = P.src_body[(size_t)P.slist[j] * h + k];
    j += dj; k += dk;
    if (k >= h) { k -= h; j++; }
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
cudaError_t gait_stack_clocked_pre_launch(int B, int* clock, int* plan, double* walkdtime_row, int* walkdtime_i, const double* sensor,
                                          double* ctl, int sms, cudaStream_t st) {
  gait_stack_clocked_pre_kernel<<<stack_grid((size_t)B, sms), 256, 0, st>>>(B, clock, plan, walkdtime_row, walkdtime_i, sensor, ctl);
  return cudaGetLastError();
}
cudaError_t gait_stack_reset_launch(const StackResetParams& P, int sms, cudaStream_t st) {
  gait_stack_reset_mark_kernel<<<(P.B + 255) / 256, 256, 0, st>>>(P);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  gait_stack_reset_column_kernel<<<stack_grid((size_t)P.B * P.rows, sms), 256, 0, st>>>(P);
  return cudaGetLastError();
}
cudaError_t farm_copy_launch(const FarmCopyParams& P, int sms, cudaStream_t st) {
  farm_copy_list_kernel<<<(P.dst_B + 255) / 256, 256, 0, st>>>(P);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  // sized for every column copied; the shape depends on dst_B only
  const size_t tasks = (size_t)((P.dst_B + 31) / 32) * ((P.soa_rows + FARM_TASK_ROWS - 1) / FARM_TASK_ROWS);
  farm_copy_column_kernel<<<stack_grid(tasks * 32, sms), 256, 0, st>>>(P);
  return cudaGetLastError();
}
cudaError_t gait_stack_pack_launch(const GaitStackSlots& S, int B, const double* gait, const double* traj, double* rows, int sms,
                                   cudaStream_t st) {
  gait_stack_pack_kernel<<<stack_grid((size_t)B * S.n, sms), 256, 0, st>>>(S, B, gait, traj, rows);
  return cudaGetLastError();
}

}  // namespace go1
