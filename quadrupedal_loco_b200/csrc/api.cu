// api.cu -- C ABI of libgo1mpc.so (include/go1mpc.h): handle, model tables, launches.
//
// Host side of the boundary.  No CPU compute path exists here: every entry point
// either launches the sm_100a kernels or fails with an error code.
#include <cuda_runtime.h>
#include <assert.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <initializer_list>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include "../../include/go1mpc.h"
#include "kernels.h"

using namespace go1;

namespace {

struct BodyModel {
  int nh = 0, tab_doubles = 0;
  std::vector<double> pps, pvs, ppu, pvu, ppu2, pvu2;   // host copies (column-major)
  double* tab_d = nullptr;
  std::vector<double> tab_h;       // host copy of the device table (kernels that take it as a launch parameter)
  int nstepx = 0, nsum_mpc = 0, gate = 0;
  double tx0[GO1MPC_FOOTSTEPS];
};

// device buffer grown on demand by grow(); freed with its owner
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { reset(); }
  void reset() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// Workspace of one caller stream.  Keyed by stream because launches on one stream are ordered: a buffer is free again when
// the next call on that stream starts, and calls on different streams never share one.
struct StreamWs {
  // {next, done} scheduler counters of the persistent body kernels and the hand-over list {count, total, ids[kFlistCap]}
  DevBuf ctl;
  // body_tri workspace, laid out for capB instances: J | half state | half result | queue | meta | hand-over at off[], then the
  // 16-byte queue control block at qctl_off
  struct { DevBuf buf; int capB = 0; size_t off[6] = {0, 0, 0, 0, 0, 0}; size_t qctl_off = 0; } tri;
  // go1mpc_control_tick_host_async; zero_B: batch size for which rows 10..19 of the planner inputs are known zero
  struct { DevBuf tick, step_in, body_tick_in, body_in, out38, step_diag, body_diag; int zero_B = -1; } control;
  // go1mpc_nlp_node_tick_batch
  struct { DevBuf tick, in, out38, out18, right_support, hz_co, lipm; } nlp;
  // gait stack ticks: sensor | /control2rtmpc/state | walkdtime ints | cmd | start | body-MPC input records | planner mask of
  // the clocked tick; zero_B: batch size for which the control message's other slots are zero
  struct { DevBuf sensor, ctl_msg, walkdtime, cmd, start, body_in, plan; int zero_B = -1; } stack;
  DevBuf reset_list;   // go1mpc_gait_stack_reset_async: {count, 3 pad, flags[B], robot list[B]}
  DevBuf copy_list;    // go1mpc_farm_copy_async: {count, 3 pad, destination list[dst.B], source list[dst.B]}
  DevBuf servo_ch, servo_reset;   // go1mpc_servo_torque_tick_async: filtered channels [SERVO_TICKS_MAX][9][B], reset flags [B]
  // go1mpc_gait_stack_tick_clocked_health_async: the planner's step diag [STEP_DIAG_INTS][B] and the body MPC's diag records
  struct { DevBuf step_diag, body_diag; } health;
};

}  // namespace

struct go1mpc {
  int device = 0;
  int sms = 0;
  size_t smem_optin = 0;
  cudaStream_t stream = nullptr;
  Go1MpcConfig cfg;
  std::string err;
  long long launches = 0;
  std::map<int, BodyModel> body_models;
  DevBuf stage[16];   // device staging for the synchronous *_host entry points
  // lanes of the asynchronous *_host_async entry points (8: a lane is busy for H2D + kernel + D2H, a few
  // hundred microseconds at batch 4096, while the PCIe link needs a new batch every ~100 us): consecutive calls go to consecutive lanes
  // (own stream, own staging), so the H2D copy of one batch overlaps the kernel of the previous
  // one and the D2H copy of the one before that.  Each entry stages into its own slots.
  struct Lane { cudaStream_t stream = nullptr; DevBuf body[3], resident[4], step[4]; };
  static const int kLanes = 8;
  Lane lanes[8];
  unsigned lane_next = 0;
  // device-resident buffers the pipelined calls read AND write (planner state): the last
  // enqueued writer per buffer, so that a later call on another lane is ordered after it
  std::map<const void*, cudaEvent_t> last_writer;
  std::map<cudaStream_t, StreamWs> ws;   // per caller stream, at most 256 (stream_ws)
  cudaStream_t side = nullptr;     // side stream of the planner tick's out-of-place state copy
  bool phase_timing = false;       // go1mpc_body_phase_timing: events around the three launches of the body tick
  cudaEvent_t phase_ev[4] = {nullptr, nullptr, nullptr, nullptr};
  double* squat_d = nullptr;       // X_CoM_position_squat table of the planner node (host libm), built on first use
  std::map<int, double*> stack_col_d;   // go1mpc_gait_stack_default_state(nh) on the device, per nh, built on first use
  double* trtab_d = nullptr;       // remaining-time bound table of the planner tick (host libm), built on first use
  std::vector<cudaEvent_t> ev_pool;   // go1mpc_stream_wait: events, reused round-robin
  unsigned ev_next = 0;
  std::recursive_mutex mu;         // guards the handle's host-side bookkeeping (maps, lane cursor, launch counter)
  int body_mode = 3;               // GO1MPC_BODY_MODE: 0 "fast" combined kernel only, 1 "split" halves side by side in
                                   // one warp, 2 "tri" setup / 4-lanes-per-half solve / merge launches, 3 "auto" (default):
                                   // tri from body_tri_min instances per call on (throughput: 2.6x the combined kernel at
                                   // 65536, 2.6x at 4096 with calls in flight on several streams), the combined kernel below
                                   // (latency of a lone small batch: 64 vs 95 us at 256)
  int body_tri_min = 2048;         // GO1MPC_BODY_TRI_MIN
  bool force_generic = false;      // GO1MPC_FORCE_GENERIC=1: always use the run-time-sized kernel
  int step_mode = 0;               // 0 auto, 1 thread per planner, 2 warp per planner (GO1MPC_STEP_MODE)
  int step_warp_below = 1024;      // auto: warp per planner below this batch size (measured: 82 vs 124 us at B = 256,
                                   // 107 vs 137 us at 1024, but 404 vs 190 us at 4096 -- the scalar front-end is
                                   // replicated per warp, so it only pays while the GPU is mostly empty)
};
static const int kFlistCap = 8190;   // ints per hand-over list; beyond it the combined kernel redoes the whole batch

namespace {

int fail(go1mpc* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  return code;
}
int cuda_fail(go1mpc* h, cudaError_t e, const char* what) {
  return fail(h, GO1MPC_E_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(h, call)                                        \
  do {                                                     \
    cudaError_t e_ = (call);                               \
    if (e_ != cudaSuccess) return cuda_fail(h, e_, #call); \
  } while (0)

// C = A(m x k) * B(k x n), column-major, ascending inner index
void mm(const double* A, const double* B, double* C, int m, int k, int n) {
  for (int j = 0; j < n; j++)
    for (int i = 0; i < m; i++) {
      double acc = 0.0;
      for (int t = 0; t < k; t++) acc += A[t * m + i] * B[j * k + t];
      C[j * m + i] = acc;
    }
}

// Horizon model of the double-integrator body-angle dynamics.
// Replaces PRMPCClass::Initialize (model part, RT/src/FastMPC/PRMPCClass.cpp:168-220)
// and Matrix_ps / Matrix_pu (:741-796): the same power recurrences, so the tables are
// what the reference would hold for this nh.
int build_body_model(go1mpc* h, int nh, BodyModel& M) {
  const Go1BodyMpcConfig& c = h->cfg.body;
  M.nh = nh;
  M.pps.assign(nh * 2, 0.0); M.pvs.assign(nh * 2, 0.0);
  M.ppu.assign(nh * nh, 0.0); M.pvu.assign(nh * nh, 0.0);
  M.ppu2.assign(nh * nh, 0.0); M.pvu2.assign(nh * nh, 0.0);
  const double a[4] = {1, 0, c.dt_mpc, 1};
  const double b[2] = {pow(c.dt_mpc, 2) / 2, c.dt_mpc};
  const double cp[2] = {1, 0}, cv[2] = {0, 1};
  for (int sel = 0; sel < 2; sel++) {
    const double* cx = sel ? cv : cp;
    std::vector<double>& ps = sel ? M.pvs : M.pps;
    std::vector<double>& pu = sel ? M.pvu : M.ppu;
    for (int i = 0; i < nh; i++) {           // row i of Pps: cx * a^(i+1)
      double A[4] = {1, 0, 0, 1}, T[4], r[2];
      for (int j = 1; j < i + 2; j++) { mm(A, a, T, 2, 2, 2); memcpy(A, T, sizeof A); }
      mm(cx, A, r, 1, 2, 2);
      ps[i] = r[0]; ps[nh + i] = r[1];
    }
    for (int i = 1; i <= nh; i++)            // Ppu(i,j) = cx * a^(i-j) * b, lower triangular
      for (int j = 1; j <= i; j++) {
        double A[4] = {1, 0, 0, 1}, T[4], r[2], v[1];
        for (int k = 1; k < i - j + 1; k++) { mm(A, a, T, 2, 2, 2); memcpy(A, T, sizeof A); }
        mm(cx, A, r, 1, 2, 2);
        mm(r, b, v, 1, 2, 1);
        pu[(j - 1) * nh + (i - 1)] = v[0];
      }
  }
  std::vector<double> T(nh * nh);
  for (int j = 0; j < nh; j++) for (int i = 0; i < nh; i++) T[j * nh + i] = M.pvu[i * nh + j];
  mm(T.data(), M.pvu.data(), M.pvu2.data(), nh, nh, nh);
  for (int j = 0; j < nh; j++) for (int i = 0; i < nh; i++) T[j * nh + i] = M.ppu[i * nh + j];
  mm(T.data(), M.ppu.data(), M.ppu2.data(), nh, nh, nh);

  // step tables (PRMPCClass.cpp:168-185)
  M.nstepx = (int)round(c.tstep / c.dt_mpc);
  M.tx0[0] = 0.0;
  for (int i = 1; i < GO1MPC_FOOTSTEPS; i++) {
    M.tx0[i] = M.tx0[i - 1] + c.tstep;
    M.tx0[i] = round(M.tx0[i] / c.dt_slow) * c.dt_slow - 0.00001;
  }
  M.nsum_mpc = (int)floor(M.tx0[GO1MPC_FOOTSTEPS - 1] / c.dt_mpc);
  M.gate = (int)round(c.height_offset_time / c.dt_mpc);

  // device table: ppu | gc0 | s2 | m1 | m2 | pps   (see body_mpc.cu)
  int td = 3 * nh * nh + 6 * nh;
  td = (td + 1) & ~1;
  M.tab_doubles = td;
  std::vector<double> tab(td, 0.0);
  double* ppu = tab.data();
  double* gc0 = ppu + nh * nh;
  double* s2 = gc0 + nh * nh;
  double* m1 = s2 + nh * nh;
  double* m2 = m1 + 2 * nh;
  double* pps = m2 + 2 * nh;
  std::vector<double> s1(nh * nh);
  for (int j = 0; j < nh; j++)
    for (int i = 0; i < nh; i++) {
      ppu[j * nh + i] = M.ppu[j * nh + i];
      double unit = (i == j) ? 1.0 : 0.0;
      // PRMPCClass.cpp:511: the three tick-independent terms of _WthetaX, in the reference's order
      gc0[j * nh + i] = c.Rtheta / 2 * unit + c.alphatheta / 2 * M.pvu2[j * nh + i] + c.beltatheta / 2 * M.ppu2[j * nh + i];
      s1[j * nh + i] = c.alphatheta * M.pvu[i * nh + j];   // alpha * Pvu'
      s2[j * nh + i] = c.beltatheta * M.ppu[i * nh + j];   // beta  * Ppu'
    }
  mm(s1.data(), M.pvs.data(), m1, nh, nh, 2);   // (alpha Pvu') Pvs   (cpp:523)
  mm(s2, M.pps.data(), m2, nh, nh, 2);          // (beta  Ppu') Pps
  memcpy(pps, M.pps.data(), sizeof(double) * 2 * nh);

  M.tab_h = tab;
  CU(h, cudaMalloc(&M.tab_d, sizeof(double) * td));
  CU(h, cudaMemcpyAsync(M.tab_d, tab.data(), sizeof(double) * td, cudaMemcpyHostToDevice, h->stream));
  CU(h, cudaStreamSynchronize(h->stream));
  return GO1MPC_OK;
}

int get_body_model(go1mpc* h, int nh, BodyModel** out) {
  auto it = h->body_models.find(nh);
  if (it == h->body_models.end()) {
    BodyModel M;
    int rc = build_body_model(h, nh, M);
    if (rc) return rc;
    it = h->body_models.emplace(nh, std::move(M)).first;
  }
  *out = &it->second;
  return GO1MPC_OK;
}

// The workspace record of stream `st`, created on first use.  One handle serves at most 256 distinct streams.
int stream_ws(go1mpc* h, cudaStream_t st, StreamWs** out) {
  auto it = h->ws.find(st);
  if (it == h->ws.end()) {
    if (h->ws.size() >= 256) return fail(h, GO1MPC_E_UNSUPPORTED, "more than 256 distinct streams used with one handle");
    it = h->ws.try_emplace(st).first;
  }
  *out = &it->second;
  return GO1MPC_OK;
}

// Makes `b` hold at least `bytes`.  A buffer that is too small is replaced: `st`, the stream that used it, is synchronised
// first (its earlier work may still read the old buffer), and the new one has headroom so that slowly rising sizes do not
// reallocate on every call.  *grew (optional) tells the caller that the contents are gone.
int grow(go1mpc* h, DevBuf& b, size_t bytes, cudaStream_t st, bool* grew = nullptr) {
  if (grew) *grew = false;
  if (bytes <= b.cap) return GO1MPC_OK;
  if (b.p) {
    CU(h, cudaStreamSynchronize(st));
    b.reset();
  }
  const size_t cap = bytes + bytes / 4 + 256;
  CU(h, cudaMalloc(&b.p, cap));
  b.cap = cap;
  if (grew) *grew = true;
  return GO1MPC_OK;
}

// The workspace record of `st` with its scheduler counters and hand-over list (allocated and zeroed on first use)
int stream_ctl(go1mpc* h, cudaStream_t st, StreamWs** out) {
  int rc = stream_ws(h, st, out);
  if (rc) return rc;
  DevBuf& c = (*out)->ctl;
  if (!c.p) {
    const size_t bytes = sizeof(int) * (size_t)(kFlistCap + 4);
    if ((rc = grow(h, c, bytes, st))) return rc;
    cudaError_t e = cudaMemset(c.p, 0, bytes);
    if (e != cudaSuccess) { c.reset(); return cuda_fail(h, e, "cudaMemset(stream control block)"); }
  }
  return GO1MPC_OK;
}

// Device staging of one host-buffer call in a set of slots, on one stream.  Each up / inout / out takes the next slot, also
// for a null host pointer, so that a buffer keeps its slot from call to call.  H2D copies are enqueued at once, D2H copies by
// finish() in staging order.  The first failure is kept in rc; later staging then does nothing.
struct Staging {
  go1mpc* h;
  DevBuf* slot;
  int nslots;
  cudaStream_t st;
  int rc = GO1MPC_OK, next = 0, ndown = 0;
  struct Down { void* host; const void* dev; size_t bytes; } down[16];   // at most one per slot

  template <int N>
  Staging(go1mpc* h_, DevBuf (&s)[N], cudaStream_t st_) : h(h_), slot(s), nslots(N), st(st_) {
    static_assert(N <= 16, "one D2H copy per slot at most");
    cudaError_t e = cudaSetDevice(h->device);   // a host thread other than the creating one starts on device 0
    if (e != cudaSuccess) rc = cuda_fail(h, e, "cudaSetDevice");
  }

  void* stage(size_t bytes) {
    assert(next < nslots);
    DevBuf& b = slot[next++];
    if (!rc) rc = grow(h, b, bytes, st);
    return rc ? nullptr : b.p;
  }
  // copied up; a null host pointer gives a null device pointer
  template <class T> T* up(const T* host, size_t bytes) {
    if (!host) { next++; return nullptr; }
    void* d = stage(bytes);
    cudaError_t e = rc ? cudaSuccess : cudaMemcpyAsync(d, host, bytes, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) rc = cuda_fail(h, e, "cudaMemcpyAsync(H2D staging)");
    return (T*)d;
  }
  // copied up, and down again by finish(); null gives null
  template <class T> T* inout(T* host, size_t bytes) {
    T* d = (T*)up(host, bytes);
    if (host) down[ndown++] = Down{host, d, bytes};
    return d;
  }
  // copied down by finish(); null gives null
  template <class T> T* out(T* host, size_t bytes) {
    if (!host) { next++; return nullptr; }
    return out_always(host, bytes, bytes);
  }
  // staged even for a null host pointer (the kernel writes it either way); down_bytes are copied down when host is given
  template <class T> T* out_always(T* host, size_t bytes, size_t down_bytes) {
    void* d = stage(bytes);
    if (host) down[ndown++] = Down{host, d, down_bytes};
    return (T*)d;
  }
  // enqueues the D2H copies; with sync, waits for them
  int finish(bool sync) {
    for (int k = 0; k < ndown; k++) CU(h, cudaMemcpyAsync(down[k].host, down[k].dev, down[k].bytes, cudaMemcpyDeviceToHost, st));
    if (sync) CU(h, cudaStreamSynchronize(st));
    return GO1MPC_OK;
  }
  // the device entry, when staging succeeded, then finish()
  template <class F> int run(bool sync, F launch) {
    if (rc) return rc;
    if (int r = launch()) return r;
    return finish(sync);
  }
};

// Launch parameters of the body-MPC kernels common to every path; a path adds its scheduler, hand-over list and workspace
BodyKParams body_params(const go1mpc* h, const BodyModel& M, int nh, int B, const double* in_d, double* out_d, int* diag_d) {
  const Go1BodyMpcConfig& c = h->cfg.body;
  BodyKParams P{};
  P.nh = nh; P.B = B; P.in_stride = go1mpc_body_in_stride(nh); P.out_stride = go1mpc_body_out_stride(nh);
  P.diag_stride = go1mpc_body_diag_stride(nh);
  P.tab_doubles = M.tab_doubles; P.warp_doubles = 0;
  P.cap_scale = h->cfg.qp_iter_cap_scale; P.gate = M.gate; P.nstepx = M.nstepx; P.nsum_mpc = M.nsum_mpc;
  P.in = in_d; P.out = out_d; P.diag = diag_d; P.tab = M.tab_d; P.sched = nullptr;
  P.flist = nullptr; P.flist_count = nullptr; P.flist_cap = 0;
  P.dt_mpc = c.dt_mpc; P.j_ini = c.j_ini; P.mass = c.mass; P.g = c.g; P.gama = c.gama_zmp;
  P.theta_lim = c.theta_lim; P.torque_lim = c.torque_lim;
  for (int k = 0; k < 4; k++) P.lamda[k] = c.lamda[k];
  return P;
}

// The 12-variable force QP of Dynamiccclass::force_opt: weights, friction and force bound of dynmics_compute.cpp:59-63
GrfKParams grf_params(const go1mpc* h, int B, const double* in_d, double* out_d, int* diag_d) {
  GrfKParams P;
  P.B = B; P.cap = h->cfg.qp_iter_cap_scale * (12 + 12 + 24) + 50; P.warp_doubles = 0;
  P.qp_alpha = 10000; P.qp_beta = 1000; P.qp_gama = 10; P.fz_max = 160; P.mu = 0.25;
  P.in = in_d; P.out = out_d; P.diag = diag_d;
  return P;
}
constexpr double kSwingKp = 1, kSwingKd = 0.01;   // swing-leg gains of compute_joint_torques (dynmics_compute.cpp:37-38)

// The servo stack kernel's parameters from a Go1ServoStackTick or a Go1ServoTorqueTick (the same leading fields); ch: null or
// where the kernel stores each tick's filtered channels
template <class Tick>
ServoStackKParams servo_stack_params(const go1mpc* h, int B, const Tick* t, double* ch) {
  const size_t b = (size_t)B;
  ServoStackKParams P;
  P.B = B; P.K = t->K; P.gait_mode = t->gait_mode;
  P.half_hip_width = h->cfg.step.half_hip_width; P.y_offset = t->y_offset;
  double k6[6];
  go1mpc_lpf_coefficients(1000.0, 3.0, k6);                     // the servo loop's 3 Hz filters at 1 kHz
  P.coef = LpfCoef{k6[0], k6[1], k6[2], k6[3], k6[4], k6[5]};
  P.gait = t->stack_state_d + GO1MPC_STACK_ROW_GAIT * b;
  P.traj = t->stack_state_d + GO1MPC_STACK_ROW_TRAJ * b;
  P.state = t->servo_state_d; P.q_out = t->q_d;
  P.jac = t->jac_d; P.foot_des = t->foot_des_d; P.iters = t->iters_d; P.ch = ch; P.health = nullptr;
  return P;
}

}  // namespace

extern "C" {

const char* go1mpc_version(void) { return GO1MPC_VERSION_STRING " (sm_100a, fp64)"; }

int go1mpc_config_default(Go1MpcConfig* cfg) {
  if (!cfg) return GO1MPC_E_INVALID;
  memset(cfg, 0, sizeof *cfg);
  Go1BodyMpcConfig& b = cfg->body;
  b.dt_mpc = 0.01; b.dt_slow = 0.025; b.tstep = 0.7; b.height_offset_time = 1.0;
  b.g = 9.8; b.mass = 12.0; b.j_ini = 12 * 0.1 * 0.1;
  b.foot_length = 0.02; b.foot_width = 0.02;
  b.theta_lim = 10 * M_PI / 180; b.torque_lim = 20.0;
  b.Rtheta = 100.0; b.alphatheta = 10.0; b.beltatheta = 5000000000.0; b.gama_zmp = 5000.0;
  Go1StepMpcConfig& s = cfg->step;
  s.dt = 0.025; s.ggg = 9.8; s.Wn = sqrt(9.8 / (0.309458 - 0.000));
  s.t_min = 0.5; s.t_max = 1;
  s.footx_max = 0.15; s.footx_min = -0.05;
  s.footx_vmax = 3; s.footx_vmin = -2.875; s.footy_vmax = 2; s.footy_vmin = -1;
  s.comax_max = 5; s.comax_min = -5; s.comay_max = 6; s.comay_min = -6;
  s.aax = 50000; s.aay = 50000; s.aaxv = 1000; s.aayv = 500;
  s.bbx = 2000000; s.bby = 10000000; s.rr1 = 1000000; s.rr2 = 1000000;
  s.half_hip_width = 0.12675; s.foot_width = 0.03;
  s.hcom = 0.309458 - 0.000; s.ext_height = 0;
  s.stepwidth0 = 0.12675; s.lift_height = 0.03;
  cfg->qp_iter_cap_scale = 20;
  return GO1MPC_OK;
}

int go1mpc_create(const Go1MpcConfig* cfg, int device, go1mpc_t** out) {
  if (!out) return GO1MPC_E_INVALID;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return GO1MPC_E_NO_DEVICE;
  go1mpc* h = new go1mpc();
  if (cfg) h->cfg = *cfg; else go1mpc_config_default(&h->cfg);
  if (h->cfg.qp_iter_cap_scale <= 0) h->cfg.qp_iter_cap_scale = 20;
  if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) { delete h; return GO1MPC_E_NO_DEVICE; } }
  if (device >= ndev) { delete h; return GO1MPC_E_INVALID; }
  h->device = device;
  cudaDeviceProp prop;
  if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&prop, device) != cudaSuccess ||
      cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete h;
    return GO1MPC_E_CUDA;
  }
  h->sms = prop.multiProcessorCount;
  h->smem_optin = prop.sharedMemPerBlockOptin;
  for (auto& L : h->lanes)
    if (cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking) != cudaSuccess) { go1mpc_destroy(h); return GO1MPC_E_CUDA; }
  if (cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking) != cudaSuccess) { go1mpc_destroy(h); return GO1MPC_E_CUDA; }
  for (int k = 0; k < 64; k++) {        // events of go1mpc_stream_wait, created up front (none is created during a graph capture)
    cudaEvent_t e;
    if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) { go1mpc_destroy(h); return GO1MPC_E_CUDA; }
    h->ev_pool.push_back(e);
  }
  const char* bm = getenv("GO1MPC_BODY_MODE");
  if (bm && !strcmp(bm, "fast")) h->body_mode = 0;
#ifdef GO1MPC_AB_VARIANTS
  else if (bm && !strcmp(bm, "split")) h->body_mode = 1;
#endif
  else if (bm && !strcmp(bm, "tri")) h->body_mode = 2;
  else if (bm && !strcmp(bm, "duo")) h->body_mode = 4;      // the any-horizon interleaved-halves kernel also at nh = 4 / 10 (A/B)
  const char* btm = getenv("GO1MPC_BODY_TRI_MIN");
  if (btm && atoi(btm) > 0) h->body_tri_min = atoi(btm);
  const char* fg = getenv("GO1MPC_FORCE_GENERIC");
  h->force_generic = fg && fg[0] == '1';
  const char* sm = getenv("GO1MPC_STEP_MODE");
  if (sm && !strcmp(sm, "thread")) h->step_mode = 1;
  if (sm && !strcmp(sm, "warp")) h->step_mode = 2;
  *out = h;
  return GO1MPC_OK;
}

void go1mpc_destroy(go1mpc_t* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  for (auto& kv : h->body_models) if (kv.second.tab_d) cudaFree(kv.second.tab_d);
  for (auto& kv : h->last_writer) cudaEventDestroy(kv.second);
  for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
  if (h->trtab_d) cudaFree(h->trtab_d);
  if (h->squat_d) cudaFree(h->squat_d);
  for (cudaEvent_t e : h->phase_ev) if (e) cudaEventDestroy(e);
  for (auto& kv : h->stack_col_d) cudaFree(kv.second);
  for (auto& L : h->lanes) if (L.stream) cudaStreamDestroy(L.stream);
  if (h->side) cudaStreamDestroy(h->side);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;   // frees the staging and every stream's workspace (DevBuf)
}

const char* go1mpc_last_error(const go1mpc_t* h) { return h ? h->err.c_str() : "null handle"; }
int go1mpc_device(const go1mpc_t* h) { return h ? h->device : -1; }
long long go1mpc_launch_count(const go1mpc_t* h) { return h ? h->launches : 0; }
void* go1mpc_stream(const go1mpc_t* h) { return h ? (void*)h->stream : nullptr; }
int go1mpc_sm_count(const go1mpc_t* h) { return h ? h->sms : 0; }
// device-to-device copy on a stream of the caller's choice: planner / MPC state is plain SoA memory,
// so checkpointing or restoring a batch is a memcpy
int go1mpc_copy_device_async(go1mpc_t* h, void* dst_d, const void* src_d, size_t bytes, void* stream) {
  if (!h || !dst_d || !src_d) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  CU(h, cudaSetDevice(h->device));     // a host thread other than the creating one starts on device 0
  CU(h, cudaMemcpyAsync(dst_d, src_d, bytes, cudaMemcpyDeviceToDevice, stream ? (cudaStream_t)stream : h->stream));
  return GO1MPC_OK;
}
int go1mpc_synchronize(go1mpc_t* h) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  CU(h, cudaSetDevice(h->device));
  CU(h, cudaStreamSynchronize(h->stream));
  for (auto& L : h->lanes) CU(h, cudaStreamSynchronize(L.stream));
  return GO1MPC_OK;
}

// ------------------------------------------------------------------ dense QP
int go1mpc_qp_solve_batch(go1mpc_t* h, int n, int p, int m, int B, const double* G_d, const double* g0_d,
                          const double* CE_d, const double* ce0_d, const double* CI_d, const double* ci0_d,
                          double* x_d, double* cost_d, int* active_d, int* nactive_d, int* iters_d,
                          int* status_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (n < 1 || p < 0 || m < 0 || B < 0 || !G_d || !g0_d || !x_d || (m && (!CI_d || !ci0_d)) || (p && (!CE_d || !ce0_d)))
    return fail(h, GO1MPC_E_INVALID, "qp_solve_batch: bad argument");
  if (n > 96 || m + p > 1024 || p > n) return fail(h, GO1MPC_E_UNSUPPORTED, "qp_solve_batch: n <= 96, m + p <= 1024, p <= n");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  int wpc = 4;
  size_t smem = dense_smem_bytes(n, m, wpc);
  while (wpc > 1 && smem > h->smem_optin / 2) { wpc >>= 1; smem = dense_smem_bytes(n, m, wpc); }
  if (smem > h->smem_optin) return fail(h, GO1MPC_E_UNSUPPORTED, "qp_solve_batch: workspace exceeds shared memory");
  int occ = 0;
  CU(h, dense_qp_occupancy(wpc, smem, &occ));
  if (occ < 1) return fail(h, GO1MPC_E_UNSUPPORTED, "qp_solve_batch: kernel does not fit on an SM");
  int grid = (B + wpc - 1) / wpc;
  if (grid > h->sms * occ) grid = h->sms * occ;
  DenseKParams P;
  P.n = n; P.p = p; P.m = m; P.B = B; P.cap = h->cfg.qp_iter_cap_scale * (m + p + n) + 50;
  P.G = G_d; P.g0 = g0_d; P.CE = CE_d; P.ce0 = ce0_d; P.CI = CI_d; P.ci0 = ci0_d;
  P.x = x_d; P.cost = cost_d; P.active = active_d; P.nactive = nactive_d; P.iters = iters_d; P.status = status_d;
  CU(h, dense_qp_launch(P, wpc, grid, smem, st));
  h->launches++;
  return GO1MPC_OK;
}

int go1mpc_qp_solve_batch_host(go1mpc_t* h, int n, int p, int m, int B, const double* G, const double* g0,
                               const double* CE, const double* ce0, const double* CI, const double* ci0,
                               double* x, double* cost, int* active, int* nactive, int* iters, int* status) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  const size_t szd = sizeof(double), szi = sizeof(int), b = (size_t)B;
  Staging S(h, h->stage, h->stream);
  const double* dG = S.up(G, b * n * n * szd);
  const double* dg0 = S.up(g0, b * n * szd);
  const double* dCE = S.up(p ? CE : nullptr, b * n * p * szd);
  const double* dce0 = S.up(p ? ce0 : nullptr, b * p * szd);
  const double* dCI = S.up(m ? CI : nullptr, b * n * m * szd);
  const double* dci0 = S.up(m ? ci0 : nullptr, b * m * szd);
  double* dx = S.inout(x, b * n * szd);
  double* dcost = S.out_always(cost, b * szd, b * szd);
  int* dact = S.out_always(active, b * (m + p + 1) * szi, b * (m + p) * szi);
  int* dna = S.out_always(nactive, b * szi, b * szi);
  int* dit = S.out_always(iters, b * 6 * szi, b * 6 * szi);
  int* dst = S.out_always(status, b * szi, b * szi);
  return S.run(true, [&] {
    return go1mpc_qp_solve_batch(h, n, p, m, B, dG, dg0, dCE, dce0, dCI, dci0, dx, dcost, dact, dna, dit, dst, S.st);
  });
}

// ------------------------------------------------------------------ body MPC
int go1mpc_body_in_stride(int nh) { int s = 36 + 11 * nh; return (s + 1) & ~1; }
int go1mpc_body_out_stride(int nh) { int s = 18 + 2 * nh + 1; return (s + 1) & ~1; }
int go1mpc_body_diag_stride(int nh) { return 10 + 2 * nh; }

int go1mpc_body_mpc_step_batch(go1mpc_t* h, int nh, int B, const double* in_d, double* out_d, int* diag_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !in_d || !out_d) return fail(h, GO1MPC_E_INVALID, "body_mpc_step_batch: bad argument");
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "body_mpc_step_batch: 3 <= nh <= 40");
  if (((uintptr_t)in_d & 15) || ((uintptr_t)out_d & 15)) return fail(h, GO1MPC_E_INVALID, "body_mpc_step_batch: in/out must be 16-byte aligned");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  BodyModel* M;
  int rc = get_body_model(h, nh, &M);
  if (rc) return rc;
  BodyKParams P = body_params(h, *M, nh, B, in_d, out_d, diag_d);
  if (body_fast_supported(nh) && !h->force_generic && h->body_mode != 4) {
    StreamWs* W;
    if ((rc = stream_ctl(h, st, &W))) return rc;
    int* ctl = (int*)W->ctl.p;
    P.sched = ctl;
    if (body_tri_supported(nh) && (h->body_mode == 2 || (h->body_mode == 3 && B >= h->body_tri_min))) {
      if (!W->tri.buf.p) {
        // a caller that keeps creating streams: past 64 streams with a workspace, drop them all (their work is done after
        // the sync)
        int held = 0;
        for (auto& kv : h->ws) held += kv.second.tri.buf.p != nullptr;
        if (held >= 64) {
          CU(h, cudaDeviceSynchronize());
          for (auto& kv : h->ws) { kv.second.tri.buf.reset(); kv.second.tri.capB = 0; }
        }
      }
      auto& T = W->tri;
      if (T.capB < B) {
        // laid out anew for B instances, with the queue control block cleared
        const size_t bytes = body_tri_workspace_bytes(nh, B, T.off);
        T.qctl_off = bytes;
        if ((rc = grow(h, T.buf, bytes + 16, st))) return rc;
        CU(h, cudaMemsetAsync((char*)T.buf.p + T.qctl_off, 0, 16, st));
        T.capB = B;
      }
      char* p = (char*)T.buf.p;
      P.tri_jb = (double*)(p + T.off[0]); P.tri_hs = (double*)(p + T.off[1]); P.tri_res = (double*)(p + T.off[2]);
      P.tri_queue = (int*)(p + T.off[3]); P.tri_qctl = (int*)(p + T.qctl_off); P.tri_meta = (int*)(p + T.off[4]); P.tri_fr = (double*)(p + T.off[5]);
      int* fl = ctl + 2;
      P.flist_count = fl; P.flist = fl + 2; P.flist_cap = kFlistCap;
      CU(h, body_tri_launch(P, M->tab_h.data(), h->sms, st, h->phase_timing ? h->phase_ev : nullptr));
      CU(h, body_fast_launch(P, h->sms, st));   // list mode: what the merge kernel handed over (normally nothing)
      h->launches += 4;
      return GO1MPC_OK;
    }
#ifdef GO1MPC_AB_VARIANTS
    if (body_split_supported(nh) && h->body_mode == 1) {
      // A/B variant (GO1MPC_BUILD_AB=1 builds): halves side by side; what it cannot reproduce goes through the
      // combined kernel right behind it
      int* fl = ctl + 2;
      P.flist_count = fl; P.flist = fl + 2; P.flist_cap = kFlistCap;
      CU(h, body_split_launch(P, h->sms, st));
      CU(h, body_fast_launch(P, h->sms, st));
      h->launches += 2;
      return GO1MPC_OK;
    }
#endif
    CU(h, body_fast_launch(P, h->sms, st));
    h->launches++;
    return GO1MPC_OK;
  }
  // every other horizon: the interleaved-halves kernel (body_duo.cu) with the dense kernel in list mode right behind it for
  // the instances it hands over (normally none); GO1MPC_FORCE_GENERIC=1 keeps the dense kernel alone
  const bool duo = !h->force_generic;
  int wpc = 4, wd = 0;
  size_t smem = body_smem_bytes(nh, wpc, P.in_stride, P.out_stride, M->tab_doubles, &wd);
  while (wpc > 1 && smem > h->smem_optin / 2) { wpc >>= 1; smem = body_smem_bytes(nh, wpc, P.in_stride, P.out_stride, M->tab_doubles, &wd); }
  if (smem > h->smem_optin) return fail(h, GO1MPC_E_UNSUPPORTED, "body_mpc_step_batch: workspace exceeds shared memory");
  int occ = 0;
  CU(h, body_mpc_occupancy(wpc, smem, &occ));
  if (occ < 1) return fail(h, GO1MPC_E_UNSUPPORTED, "body_mpc_step_batch: kernel does not fit on an SM");
  int grid = (B + wpc - 1) / wpc;
  if (grid > h->sms * occ) grid = h->sms * occ;
  P.warp_doubles = wd;
  if (duo) {
    StreamWs* W;
    if ((rc = stream_ctl(h, st, &W))) return rc;
    int* fl = (int*)W->ctl.p + 2;
    P.flist_count = fl; P.flist = fl + 2; P.flist_cap = kFlistCap;
    CU(h, body_duo_launch(P, h->sms, h->smem_optin, st));
    CU(h, body_mpc_launch(P, wpc, grid, smem, st));           // list mode
    CU(h, cudaMemsetAsync(fl, 0, sizeof(int), st));
    h->launches += 2;
    return GO1MPC_OK;
  }
  CU(h, body_mpc_launch(P, wpc, grid, smem, st));
  h->launches++;
  return GO1MPC_OK;
}

// Per-kernel timing of the three-launch body tick (measurement aid): while enabled, every go1mpc_body_mpc_step_batch call that
// takes the three-launch path records CUDA events around its setup / solve / merge launches; go1mpc_body_phase_ms waits for the
// last call and returns the three durations.  Not for use inside a graph capture.
int go1mpc_body_phase_timing(go1mpc_t* h, int enable) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  CU(h, cudaSetDevice(h->device));
  if (enable) for (cudaEvent_t& e : h->phase_ev) if (!e) CU(h, cudaEventCreate(&e));
  h->phase_timing = enable != 0;
  return GO1MPC_OK;
}
int go1mpc_body_phase_ms(go1mpc_t* h, float* ms3) {
  if (!h || !ms3) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (!h->phase_ev[3]) return fail(h, GO1MPC_E_INVALID, "body_phase_ms: phase timing was never enabled");
  CU(h, cudaEventSynchronize(h->phase_ev[3]));
  for (int k = 0; k < 3; k++) CU(h, cudaEventElapsedTime(ms3 + k, h->phase_ev[k], h->phase_ev[k + 1]));
  return GO1MPC_OK;
}

// instances the split kernel handed to the combined kernel since the handle was created (synchronises)
int go1mpc_body_handover_total(go1mpc_t* h, long long* total) {
  if (!h || !total) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  CU(h, cudaSetDevice(h->device));
  CU(h, cudaDeviceSynchronize());
  long long t = 0;
  for (auto& kv : h->ws) {
    if (!kv.second.ctl.p) continue;
    int v = 0;
    CU(h, cudaMemcpy(&v, (int*)kv.second.ctl.p + 3, sizeof(int), cudaMemcpyDeviceToHost));
    t += v;
  }
  *total = t;
  return GO1MPC_OK;
}

// health counter of the three-launch body path: warps of the solve kernel that left through the defensive
// iteration guard (always 0 unless there is a bug); synchronises
int go1mpc_body_guard_trips(go1mpc_t* h, long long* total) {
  if (!h || !total) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  CU(h, cudaSetDevice(h->device));
  CU(h, cudaDeviceSynchronize());
  long long t = 0;
  for (auto& kv : h->ws) {
    const auto& T = kv.second.tri;
    if (!T.buf.p) continue;
    int v = 0;
    CU(h, cudaMemcpy(&v, (char*)T.buf.p + T.qctl_off + 8, sizeof(int), cudaMemcpyDeviceToHost));
    t += v;
  }
  *total = t;
  return GO1MPC_OK;
}

int go1mpc_body_mpc_step_batch_host(go1mpc_t* h, int nh, int B, const double* in, double* out, int* diag) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!in || !out) return fail(h, GO1MPC_E_INVALID, "body_mpc_step_batch_host: bad argument");
  const size_t b = (size_t)B;
  Staging S(h, h->stage, h->stream);
  const double* din = S.up(in, b * go1mpc_body_in_stride(nh) * sizeof(double));
  double* dout = S.inout(out, b * go1mpc_body_out_stride(nh) * sizeof(double));   // out14 is in/out (gated ticks)
  int* ddiag = S.out(diag, b * go1mpc_body_diag_stride(nh) * sizeof(int));
  return S.run(true, [&] { return go1mpc_body_mpc_step_batch(h, nh, B, din, dout, ddiag, S.st); });
}

int go1mpc_body_model(go1mpc_t* h, int nh, double* pps, double* pvs, double* ppu, double* pvu, double* ppu_2, double* pvu_2) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (nh < 1 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "body_model: 1 <= nh <= 40");
  CU(h, cudaSetDevice(h->device));
  BodyModel* M;
  int rc = get_body_model(h, nh, &M);
  if (rc) return rc;
  if (pps) memcpy(pps, M->pps.data(), sizeof(double) * 2 * nh);
  if (pvs) memcpy(pvs, M->pvs.data(), sizeof(double) * 2 * nh);
  if (ppu) memcpy(ppu, M->ppu.data(), sizeof(double) * nh * nh);
  if (pvu) memcpy(pvu, M->pvu.data(), sizeof(double) * nh * nh);
  if (ppu_2) memcpy(ppu_2, M->ppu2.data(), sizeof(double) * nh * nh);
  if (pvu_2) memcpy(pvu_2, M->pvu2.data(), sizeof(double) * nh * nh);
  return GO1MPC_OK;
}

int go1mpc_body_default_tx(go1mpc_t* h, double* tx27) {
  if (!h || !tx27) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  CU(h, cudaSetDevice(h->device));
  BodyModel* M;
  int rc = get_body_model(h, 4, &M);
  if (rc) return rc;
  memcpy(tx27, M->tx0, sizeof M->tx0);
  return GO1MPC_OK;
}

// ------------------------------------------------------------------ step timing
namespace {
int step_tick_enqueue(go1mpc_t* h, int n_sqp, int B, const int* tick_d, const double* state_d, double* state_out_d,
                      const double* in_d, double* out_d, int* diag_d, void* stream, double* hz_co_d, double* lipm_d);
}
int go1mpc_step_timing_step_batch(go1mpc_t* h, int n_sqp, int B, const int* tick_d, const double* state_d, double* state_out_d,
                                  const double* in_d, double* out_d, int* diag_d, void* stream) {
  return step_tick_enqueue(h, n_sqp, B, tick_d, state_d, state_out_d, in_d, out_d, diag_d, stream, nullptr, nullptr);
}
namespace {
// hz_co_d / lipm_d: optional hand-over rows for the planner node (nlp_chain.cu); they force the three-launch mapping
int step_tick_enqueue(go1mpc_t* h, int n_sqp, int B, const int* tick_d, const double* state_d, double* state_out_d,
                      const double* in_d, double* out_d, int* diag_d, void* stream, double* hz_co_d, double* lipm_d) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !tick_d || !state_d || !state_out_d || !in_d || !out_d) return fail(h, GO1MPC_E_INVALID, "step_timing_step_batch: bad argument");
  if (n_sqp < 1 || n_sqp > STEP_MAX_SQP) return fail(h, GO1MPC_E_UNSUPPORTED, "step_timing_step_batch: 1 <= n_sqp <= 5");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  const Go1StepMpcConfig& c = h->cfg.step;
  StepKParams P;
  P.B = B; P.n_sqp = n_sqp; P.cap = h->cfg.qp_iter_cap_scale * (4 + 24 + 1) + 50;
  P.tick = tick_d; P.state = state_d; P.state_out = state_out_d; P.in = in_d; P.out = out_d; P.diag = diag_d;
  P.hz_co = hz_co_d; P.lipm = lipm_d;
  StepCfgDev& d = P.cfg;
  d.dt = c.dt; d.Wn = c.Wn; d.ggg = c.ggg; d.t_min = c.t_min; d.t_max = c.t_max;
  d.footx_max = c.footx_max; d.footx_min = c.footx_min;
  d.footx_vmax = c.footx_vmax; d.footx_vmin = c.footx_vmin; d.footy_vmax = c.footy_vmax; d.footy_vmin = c.footy_vmin;
  d.comax_max = c.comax_max; d.comax_min = c.comax_min; d.comay_max = c.comay_max; d.comay_min = c.comay_min;
  d.aax = c.aax; d.aay = c.aay; d.aaxv = c.aaxv; d.aayv = c.aayv; d.bbx = c.bbx; d.bby = c.bby; d.rr1 = c.rr1; d.rr2 = c.rr2;
  d.half_hip_width = c.half_hip_width; d.foot_width = c.foot_width;
  for (int k = 0; k < 4; k++) d.lamda[k] = c.lamda[k];
  d.hcom = c.hcom; d.ext_height = c.ext_height;
  // instance-independent transcendentals, evaluated once per launch by the host libm (the values the CPU reference uses)
  d.sh_dt = sinh(c.Wn * c.dt); d.ch_dt = cosh(c.Wn * c.dt);
  for (int jxx = 1; jxx <= 3; jxx++) { const double w = c.Wn * c.dt * jxx; d.sh_w[jxx - 1] = sinh(w); d.ch_w[jxx - 1] = cosh(w); }
  // one thread per planner is the throughput mapping; below a few waves of threads the latency of the
  // thread-serial tick dominates and one warp per planner is faster (GO1MPC_STEP_MODE=thread|warp forces one)
  bool warp_mode = B < h->step_warp_below;
  if (h->step_mode == 1) warp_mode = false;
  if (h->step_mode == 2) warp_mode = true;
  if (hz_co_d || lipm_d) warp_mode = false;
  if (!h->trtab_d) {
    // tr1_min, tr2_min, tr1_max, tr2_max of NLPClass_sqp.cpp:745-757 as functions of k_yu (the samples elapsed in the step)
    double tab[STEP_TRTAB_ROWS * 4];
    for (int k = 0; k < STEP_TRTAB_ROWS; k++) {
      const double tmin = ((c.t_min - k * c.dt) >= 0.001) ? (c.t_min - k * c.dt) : 0.001;
      tab[4 * k + 0] = cosh(c.Wn * tmin); tab[4 * k + 1] = sinh(c.Wn * tmin);
      tab[4 * k + 2] = cosh(c.Wn * (c.t_max - k * c.dt)); tab[4 * k + 3] = sinh(c.Wn * (c.t_max - k * c.dt));
    }
    CU(h, cudaMalloc((void**)&h->trtab_d, sizeof tab));
    CU(h, cudaMemcpy(h->trtab_d, tab, sizeof tab, cudaMemcpyHostToDevice));
  }
  P.trtab = h->trtab_d;
  if (warp_mode) {
    CU(h, step_timing_launch(P, st));                 // one launch, warp per planner
    h->launches++;
  } else {
    // SQP kernel, CoM-height kernel, back-end kernel.  Out of place, the new state starts as a copy of the old one (the back-end
    // updates the changed fields): that copy runs on the handle's side stream beside the compute-bound SQP kernel.
    const bool oop = (state_out_d != state_d);
    if (oop) {
      int rc = go1mpc_stream_wait(h, h->side, st);
      if (rc) return rc;
      CU(h, cudaMemcpyAsync(state_out_d, state_d, (size_t)B * STEP_STATE_DOUBLES * sizeof(double), cudaMemcpyDeviceToDevice, h->side));
    }
    CU(h, step_sqp_launch(P, st));
    CU(h, step_height_launch(P, st));
    if (oop) {
      int rc = go1mpc_stream_wait(h, st, h->side);
      if (rc) return rc;
    }
    CU(h, step_post_launch(P, st));
    h->launches += 3;
  }
  return GO1MPC_OK;
}
}  // namespace

int go1mpc_step_timing_step_batch_host(go1mpc_t* h, int n_sqp, int B, const int* tick, double* state, const double* in,
                                       double* out, int* diag) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!tick || !state || !in || !out) return fail(h, GO1MPC_E_INVALID, "step_timing_step_batch_host: bad argument");
  const size_t b = (size_t)B;
  Staging S(h, h->stage, h->stream);
  const int* dt_ = S.up(tick, b * sizeof(int));
  double* ds = S.inout(state, b * STEP_STATE_DOUBLES * sizeof(double));
  const double* di = S.up(in, b * STEP_IN_DOUBLES * sizeof(double));
  double* do_ = S.out(out, b * STEP_OUT_DOUBLES * sizeof(double));
  int* dd = S.out(diag, b * STEP_DIAG_INTS * sizeof(int));
  return S.run(true, [&] { return go1mpc_step_timing_step_batch(h, n_sqp, B, dt_, ds, ds, di, do_, dd, S.st); });
}

// NLPClass::FootStepInputs (NLP/NLP/NLPClass_sqp.cpp:51-75) + Initialize (:131-206) step tables
int go1mpc_step_default_state(go1mpc_t* h, double steplength, double stepwidth, double stepheight, double tstep, double* s) {
  if (!h || !s) return GO1MPC_E_INVALID;
  const int NS = GO1MPC_FOOTSTEPS;
  const double dt = h->cfg.step.dt;
  double sl[GO1MPC_FOOTSTEPS], sw[GO1MPC_FOOTSTEPS], sh[GO1MPC_FOOTSTEPS];
  memset(s, 0, sizeof(double) * STEP_STATE_DOUBLES);
  double *ts = s, *tx = s + 27, *fx = s + 54, *fy = s + 81, *fz = s + 108, *Lxx = s + 135, *Lyy = s + 162;
  for (int j = 0; j < NS; j++) { sl[j] = steplength; sw[j] = stepwidth; sh[j] = stepheight; }
  sl[NS - 1] = sl[NS - 2] = sl[NS - 3] = sl[NS - 4] = sl[NS - 5] = 0;
  sl[0] = sl[1] = sl[2] = 0; sl[3] = steplength / 2;
  sw[0] = sw[0] / 2;
  sl[14] = 0;
  for (int j = 15; j <= 21; j++) sl[j] *= -1;
  for (int j = 0; j < NS; j++) { Lxx[j] = sl[j]; Lyy[j] = (int)pow(-1, j) * sw[j]; }
  for (int j = 1; j < NS; j++) {
    fx[j] = fx[j - 1] + sl[j - 1];
    fy[j] = fy[j - 1] + (int)pow(-1, j - 1) * sw[j - 1];
    fz[j] = fz[j - 1] + sh[j - 1];
  }
  for (int j = 0; j < NS; j++) ts[j] = tstep;
  for (int j = 1; j < NS; j++) { tx[j] = tx[j - 1] + ts[j - 1]; tx[j] = round(tx[j] / dt) * dt - 0.000001; }
  return GO1MPC_OK;
}

// ------------------------------------------------------------------ swing-foot trajectory
namespace {
int foot_enqueue(go1mpc_t* h, int B, const int* tick_d, const double* state_d, const double* out38_d, double* foot_d, double* out18_d,
                 int* right_support_d, void* stream, double* lift0_d, const double* stop_d, int t_end);
}
int go1mpc_foot_trajectory_batch(go1mpc_t* h, int B, const int* tick_d, const double* state_d, const double* out38_d,
                                 double* foot_d, double* out18_d, int* right_support_d, void* stream) {
  return foot_enqueue(h, B, tick_d, state_d, out38_d, foot_d, out18_d, right_support_d, stream, nullptr, nullptr, 0);
}
int go1mpc_foot_trajectory_stop_batch(go1mpc_t* h, int B, const int* tick_d, const double* state_d, const double* out38_d,
                                      double* foot_d, double* out18_d, int* right_support_d, double* lift0_d,
                                      const double* stop_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  if (!lift0_d) return fail(h, GO1MPC_E_INVALID, "foot_trajectory_stop_batch: bad argument");
  return foot_enqueue(h, B, tick_d, state_d, out38_d, foot_d, out18_d, right_support_d, stream, lift0_d, stop_d, go1mpc_nlp_t_end_footstep(h));
}
namespace {
int foot_enqueue(go1mpc_t* h, int B, const int* tick_d, const double* state_d, const double* out38_d, double* foot_d, double* out18_d,
                 int* right_support_d, void* stream, double* lift0_d, const double* stop_d, int t_end) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !tick_d || !state_d || !out38_d || !foot_d || !out18_d) return fail(h, GO1MPC_E_INVALID, "foot_trajectory_batch: bad argument");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  FootKParams P;
  P.B = B; P.tick = tick_d; P.state = state_d; P.out38 = out38_d; P.foot = foot_d; P.out18 = out18_d; P.right_support = right_support_d;
  P.dt = h->cfg.step.dt; P.stepwidth0 = h->cfg.step.stepwidth0; P.lift_height = h->cfg.step.lift_height;
  P.lift0 = lift0_d; P.stop = stop_d; P.t_end = t_end;
  CU(h, foot_traj_launch(P, stream ? (cudaStream_t)stream : h->stream));
  h->launches++;
  return GO1MPC_OK;
}
}  // namespace
int go1mpc_foot_trajectory_batch_host(go1mpc_t* h, int B, const int* tick, const double* state, const double* out38,
                                      double* foot, double* out18, int* right_support) {
  return go1mpc_foot_trajectory_stop_batch_host(h, B, tick, state, out38, foot, out18, right_support, nullptr, nullptr);
}
int go1mpc_foot_trajectory_stop_batch_host(go1mpc_t* h, int B, const int* tick, const double* state, const double* out38,
                                           double* foot, double* out18, int* right_support, double* lift0, const double* stop) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!tick || !state || !out38 || !foot || !out18) return fail(h, GO1MPC_E_INVALID, "foot_trajectory_batch_host: bad argument");
  const size_t b = (size_t)B;
  Staging S(h, h->stage, h->stream);
  const int* dt_ = S.up(tick, b * sizeof(int));
  const double* ds = S.up(state, b * STEP_STATE_DOUBLES * sizeof(double));
  const double* do_ = S.up(out38, b * STEP_OUT_DOUBLES * sizeof(double));
  double* df = S.inout(foot, b * FOOT_STATE_DOUBLES * sizeof(double));
  double* d18 = S.out(out18, b * FOOT_OUT_DOUBLES * sizeof(double));
  int* drs = S.out(right_support, b * sizeof(int));
  double* dl0 = S.inout(lift0, b * sizeof(double));
  const double* dstop = S.up(lift0 ? stop : nullptr, b * sizeof(double));
  return S.run(true, [&] {
    return foot_enqueue(h, B, dt_, ds, do_, df, d18, drs, S.st, dl0, dstop, lift0 ? go1mpc_nlp_t_end_footstep(h) : 0);
  });
}
// initial foot window: _Rfooty = -stepwidth(0), _Lfooty = +stepwidth(0), rest 0 (NLPClass_sqp.cpp:496-500)
int go1mpc_foot_default_state(go1mpc_t* h, double* fs) {
  if (!h || !fs) return GO1MPC_E_INVALID;
  const double sw0 = h->cfg.step.stepwidth0;
  for (int k = 0; k < 4; k++) { double* p = fs + 6 * k; p[0] = 0; p[1] = -sw0; p[2] = 0; p[3] = 0; p[4] = sw0; p[5] = 0; }
  for (int k = 24; k < 30; k++) fs[k] = 0.0;
  fs[30] = -1.0; fs[31] = 0.0;
  return GO1MPC_OK;
}

// ------------------------------------------------------------------ GRF distribution
int go1mpc_grf_force_opt_batch(go1mpc_t* h, int B, const double* in_d, double* out_d, int* diag_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !in_d || !out_d) return fail(h, GO1MPC_E_INVALID, "grf_force_opt_batch: bad argument");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  CU(h, grf_force_opt_launch(grf_params(h, B, in_d, out_d, diag_d), h->sms, stream ? (cudaStream_t)stream : h->stream));
  h->launches++;
  return GO1MPC_OK;
}
int go1mpc_grf_force_distribution_batch(go1mpc_t* h, int B, int gait_mode, double y_coefficient, const double* com_des_d,
                                        const double* leg_des_d, const double* F_force_des_d, const double* rfoot_des_d,
                                        const double* lfoot_des_d, double* F_leg_ref_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !com_des_d || !leg_des_d || !F_force_des_d || !rfoot_des_d || !lfoot_des_d || !F_leg_ref_d)
    return fail(h, GO1MPC_E_INVALID, "grf_force_distribution_batch: bad argument");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  GrfDistParams P;
  P.B = B; P.mode = gait_mode; P.y_coefficient = y_coefficient;
  P.com = com_des_d; P.leg = leg_des_d; P.F = F_force_des_d; P.rfoot = rfoot_des_d; P.lfoot = lfoot_des_d; P.F_leg_ref = F_leg_ref_d;
  CU(h, grf_force_distribution_launch(P, stream ? (cudaStream_t)stream : h->stream));
  h->launches++;
  return GO1MPC_OK;
}

int go1mpc_grf_joint_torques_batch(go1mpc_t* h, int B, const double* jac_d, const int* swing_d, const double* p_des_d,
                                   const double* p_est_d, const double* pv_des_d, const double* pv_est_d,
                                   const double* F_leg_ref_d, long long F_elem_stride, long long F_robot_stride, double* tau_d,
                                   void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !jac_d || !swing_d || !p_des_d || !p_est_d || !pv_des_d || !pv_est_d || !F_leg_ref_d || !tau_d)
    return fail(h, GO1MPC_E_INVALID, "grf_joint_torques_batch: bad argument");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  GrfTauParams P;
  P.B = B; P.swing_kp = kSwingKp; P.swing_kd = kSwingKd;
  P.jac = jac_d; P.swing = swing_d; P.p_des = p_des_d; P.p_est = p_est_d; P.pv_des = pv_des_d; P.pv_est = pv_est_d;
  P.F_leg_ref = F_leg_ref_d; P.f_ks = F_elem_stride; P.f_bs = F_robot_stride; P.tau = tau_d;
  CU(h, grf_joint_torques_launch(P, stream ? (cudaStream_t)stream : h->stream));
  h->launches++;
  return GO1MPC_OK;
}

// synchronous host-buffer forms of the three GRF entries (staging on the handle's stream)
int go1mpc_grf_force_opt_batch_host(go1mpc_t* h, int B, const double* in, double* out, int* diag) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!in || !out) return fail(h, GO1MPC_E_INVALID, "grf_force_opt_batch_host: bad argument");
  const size_t b = (size_t)B;
  Staging S(h, h->stage, h->stream);
  const double* di = S.up(in, b * GRF_IN_DOUBLES * sizeof(double));
  double* do_ = S.out(out, b * GRF_OUT_DOUBLES * sizeof(double));
  int* dd = S.out(diag, b * GRF_DIAG_INTS * sizeof(int));
  return S.run(true, [&] { return go1mpc_grf_force_opt_batch(h, B, di, do_, dd, S.st); });
}
int go1mpc_grf_force_distribution_batch_host(go1mpc_t* h, int B, int gait_mode, double y_coefficient, const double* com_des,
                                             const double* leg_des, const double* F_force_des, const double* rfoot_des,
                                             const double* lfoot_des, double* F_leg_ref) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!com_des || !leg_des || !F_force_des || !rfoot_des || !lfoot_des || !F_leg_ref)
    return fail(h, GO1MPC_E_INVALID, "grf_force_distribution_batch_host: bad argument");
  const size_t d = (size_t)B * sizeof(double);
  Staging S(h, h->stage, h->stream);
  const double* dcom = S.up(com_des, 3 * d);
  const double* dleg = S.up(leg_des, 12 * d);
  const double* dF = S.up(F_force_des, 6 * d);
  const double* drf = S.up(rfoot_des, 3 * d);
  const double* dlf = S.up(lfoot_des, 3 * d);
  double* dref = S.out(F_leg_ref, 12 * d);
  return S.run(true, [&] {
    return go1mpc_grf_force_distribution_batch(h, B, gait_mode, y_coefficient, dcom, dleg, dF, drf, dlf, dref, S.st);
  });
}
int go1mpc_grf_joint_torques_batch_host(go1mpc_t* h, int B, const double* jac, const int* swing, const double* p_des,
                                        const double* p_est, const double* pv_des, const double* pv_est,
                                        const double* F_leg_ref, long long F_elem_stride, long long F_robot_stride, double* tau) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!jac || !swing || !p_des || !p_est || !pv_des || !pv_est || !F_leg_ref || !tau || F_elem_stride < 0 || F_robot_stride < 0)
    return fail(h, GO1MPC_E_INVALID, "grf_joint_torques_batch_host: bad argument");
  const size_t d = (size_t)B * sizeof(double);
  const size_t fdoubles = (size_t)(11 * F_elem_stride + (B - 1) * F_robot_stride + 1);   // extent the strides address
  Staging S(h, h->stage, h->stream);
  const double* djac = S.up(jac, 36 * d);
  const int* dsw = S.up(swing, 4 * (size_t)B * sizeof(int));
  const double* dpd = S.up(p_des, 12 * d);
  const double* dpe = S.up(p_est, 12 * d);
  const double* dvd = S.up(pv_des, 12 * d);
  const double* dve = S.up(pv_est, 12 * d);
  const double* dF = S.up(F_leg_ref, fdoubles * sizeof(double));
  double* dtau = S.out(tau, 12 * d);
  return S.run(true, [&] {
    return go1mpc_grf_joint_torques_batch(h, B, djac, dsw, dpd, dpe, dvd, dve, dF, F_elem_stride, F_robot_stride, dtau, S.st);
  });
}

// ------------------------------------------------------------------ 40 Hz -> 100 Hz reference interpolation
namespace {
// _AAA_inv_mod of PRMPCClass::solve_AAA_inv_mod1 (PRMPCClass.cpp:1344-1361): inverse of the rows (t^3, t^2, t, 1) at
// t = -dt, 0, dt, 2 dt by row-pivoted Gauss-Jordan (first maximal pivot wins), row-major.
void build_aaa_inv_mod(double dt, double inv[16]) {
  const double t[4] = {-dt, 0.0, dt, 2 * dt};
  double a[4][4], r[4][4];
  for (int i = 0; i < 4; i++) {
    a[i][0] = pow(t[i], 3); a[i][1] = pow(t[i], 2); a[i][2] = pow(t[i], 1); a[i][3] = 1.0;
    for (int j = 0; j < 4; j++) r[i][j] = (i == j) ? 1.0 : 0.0;
  }
  for (int k = 0; k < 4; k++) {
    int piv = k;
    double best = fabs(a[k][k]);
    for (int i = k + 1; i < 4; i++) if (fabs(a[i][k]) > best) { best = fabs(a[i][k]); piv = i; }
    if (piv != k) for (int j = 0; j < 4; j++) { std::swap(a[k][j], a[piv][j]); std::swap(r[k][j], r[piv][j]); }
    const double d = a[k][k];
    for (int j = 0; j < 4; j++) { a[k][j] = a[k][j] / d; r[k][j] = r[k][j] / d; }
    for (int i = 0; i < 4; i++) {
      if (i == k) continue;
      const double f = a[i][k];
      for (int j = 0; j < 4; j++) {
        const double pa = f * a[k][j], pr = f * r[k][j];     // separate statements: no contraction into FMA
        a[i][j] = a[i][j] - pa; r[i][j] = r[i][j] - pr;
      }
    }
  }
  memcpy(inv, r, sizeof r);
}
}  // namespace

// host part of the interpolation (no device needed): _AAA_inv_mod (row-major) and _t_end_footstep for a configuration
int go1mpc_ref_interp_model(const Go1MpcConfig* cfg, double* inv16, int* t_end_footstep) {
  if (!inv16 && !t_end_footstep) return GO1MPC_E_INVALID;
  Go1MpcConfig def;
  if (!cfg) { go1mpc_config_default(&def); cfg = &def; }
  const Go1BodyMpcConfig& c = cfg->body;
  if (inv16) build_aaa_inv_mod(c.dt_slow, inv16);
  if (t_end_footstep) {
    // _tx and _t_end_footstep of PRMPCClass::Initialize (:174-179)
    double tx = 0.0;
    for (int i = 1; i < GO1MPC_FOOTSTEPS; i++) { tx = tx + c.tstep; tx = round(tx / c.dt_slow) * c.dt_slow - 0.00001; }
    *t_end_footstep = (int)round((tx - 3 * c.tstep) / c.dt_mpc);
  }
  return GO1MPC_OK;
}

int go1mpc_ref_interp_batch(go1mpc_t* h, int B, int nh, const int* walktime_d, double dt_sample, const double* samples_d,
                            double* out_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !walktime_d || !samples_d || !out_d) return fail(h, GO1MPC_E_INVALID, "ref_interp_batch: bad argument");
  if (nh < 1 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "ref_interp_batch: 1 <= nh <= 40");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  RefInterpParams P;
  P.B = B; P.nh = nh; P.dt_sample = dt_sample;
  go1mpc_ref_interp_model(&h->cfg, P.inv, &P.t_end_footstep);
  P.walktime = walktime_d; P.samples = samples_d; P.out = out_d;
  CU(h, ref_interp_launch(P, stream ? (cudaStream_t)stream : h->stream));
  h->launches++;
  return GO1MPC_OK;
}

// ------------------------------------------------------------------ signal filters of the servo loop
// coefficients of butterworthLPF::init (GO1/src/Filter/butterworthLPF.cpp:82-100), host libm; CPU-callable
int go1mpc_lpf_coefficients(double fsampling, double fcutoff, double* coef6) {
  if (!coef6 || !(fsampling > 0)) return GO1MPC_E_INVALID;
  const double ff = fcutoff / fsampling;
  const double ita = 1.0 / tan(3.14159265359 * ff);
  const double q = sqrt(2.0);
  const double qi = q * ita, ii = ita * ita;
  const double b0 = 1.0 / (1.0 + qi + ii);
  coef6[0] = b0; coef6[1] = 2 * b0; coef6[2] = b0;
  const double t1 = 2.0 * (ii - 1.0);
  coef6[3] = t1 * b0;
  const double t2 = -(1.0 - qi + ii);
  coef6[4] = t2 * b0;
  const double w = 2.0 * 3.14159265359 * ff;
  coef6[5] = w / (w + 1.0);
  return GO1MPC_OK;
}
int go1mpc_lpf_batch(go1mpc_t* h, int B, int C, const double* coef, const double* in_d, const int* in_rows_d, double* state_d,
                     double* out_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || C < 0 || !coef || !in_d || !state_d || !out_d) return fail(h, GO1MPC_E_INVALID, "lpf_batch: bad argument");
  if (C > LPF_MAX_CHANNELS) return fail(h, GO1MPC_E_UNSUPPORTED, "lpf_batch: at most 32 channels per call");
  if (B == 0 || C == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  LpfKParams P;
  P.B = B; P.C = C;
  for (int c = 0; c < C; c++) { const double* k = coef + 6 * c; P.coef[c] = LpfCoef{k[0], k[1], k[2], k[3], k[4], k[5]}; }
  P.in = in_d; P.in_rows = in_rows_d; P.state = state_d; P.out = out_d;
  CU(h, lpf_launch(P, h->sms, stream ? (cudaStream_t)stream : h->stream));
  h->launches++;
  return GO1MPC_OK;
}
int go1mpc_force_filter_batch(go1mpc_t* h, int B, int C, const double* in_d, double* state_d, double* out_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || C < 0 || !in_d || !state_d || !out_d) return fail(h, GO1MPC_E_INVALID, "force_filter_batch: bad argument");
  if (B == 0 || C == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  CU(h, force_filter_launch(B, C, in_d, state_d, out_d, h->sms, stream ? (cudaStream_t)stream : h->stream));
  h->launches++;
  return GO1MPC_OK;
}

// ------------------------------------------------------------------ the 40 Hz planner node (message out)
namespace {
// reference constants of NLPRTControlClass / NLPClass (NLPRTControlClass.h:16-18, NLPClass.h:35-38, NLPClass_sqp.cpp:262)
constexpr double kNlpDtx = 0.025, kNlpHeightOffsetTime = 1.0, kNlpSquatTime = 1.0, kNlpHeightOffset = 0.0, kNlpMass = 12.0, kNlpRad = 0.1;
constexpr double kNlpStepLength = 0.075, kNlpStepHeight = 0.0, kNlpTstep = 0.7;
constexpr int kNlpRing = 234, kNlpZhi = 362, kNlpLift0 = 363, kNlpStop = 365, kNlpRsup = 369, kNlpPel = 371, kNlpLf = 380, kNlpRf = 383, kNlpComx = 466;

// the default step table's last entry (_tx(last) of Initialize): _t_end_footstep and _walkdtime_max derive from it
void nlp_limits(const go1mpc* h, int* t_end, int* walkdtime_max) {
  const double dt = h->cfg.step.dt;
  double tx = 0.0;
  for (int j = 1; j < GO1MPC_FOOTSTEPS; j++) { tx = tx + kNlpTstep; tx = round(tx / dt) * dt - 0.000001; }
  if (t_end) *t_end = (int)round((tx - 2 * kNlpTstep) / dt);                                  // NLPClass_sqp.cpp:593
  const int nsum = (GO1MPC_FOOTSTEPS - 1) * (int)round(kNlpTstep / dt);                        // NLPClass.h:35-36
  const int omit = 2 * (int)round(kNlpTstep / dt);                                             // :311
  if (walkdtime_max) *walkdtime_max = (int)((nsum - omit - 1) * floor(dt / kNlpDtx)) + 1;      // :3026-3032, NLPRTControlClass.cpp:93
}

// NLPClass::X_CoM_position_squat (NLPClass_sqp.cpp:2958-3015, solve_AAA_inv_x :3585-3628) for walktime = 0 .. n-1: the squat
// does not depend on the robot, so the node reads a table built once by the host libm (the reference's own pow / divisions)
void build_squat_table(double z_c, int n, double* tab /* [3][n] */) {
  const double tp[3] = {0.00001, kNlpSquatTime / 2 + 0.0001, kNlpSquatTime + 0.0001};
  double A[49], R[49];
  const int rowt[7] = {0, 0, 0, 1, 2, 2, 2}, kind[7] = {1, 2, 0, 0, 0, 1, 2};
  for (int r = 0; r < 7; r++) {
    const double t = tp[rowt[r]];
    double* a = A + 7 * r;
    if (kind[r] == 0) { a[0] = pow(t, 6); a[1] = pow(t, 5); a[2] = pow(t, 4); a[3] = pow(t, 3); a[4] = pow(t, 2); a[5] = pow(t, 1); a[6] = 1; }
    else if (kind[r] == 1) { a[0] = 6 * pow(t, 5); a[1] = 5 * pow(t, 4); a[2] = 4 * pow(t, 3); a[3] = 3 * pow(t, 2); a[4] = 2 * pow(t, 1); a[5] = 1; a[6] = 0; }
    else { a[0] = 30 * pow(t, 4); a[1] = 20 * pow(t, 3); a[2] = 12 * pow(t, 2); a[3] = 6 * pow(t, 1); a[4] = 2; a[5] = 0; a[6] = 0; }
  }
  for (int i = 0; i < 7; i++) for (int j = 0; j < 7; j++) R[i * 7 + j] = (i == j) ? 1.0 : 0.0;
  for (int k = 0; k < 7; k++) {       // row-pivoted Gauss-Jordan, first maximal pivot wins
    int piv = k;
    double best = fabs(A[k * 7 + k]);
    for (int i = k + 1; i < 7; i++) if (fabs(A[i * 7 + k]) > best) { best = fabs(A[i * 7 + k]); piv = i; }
    if (piv != k) for (int j = 0; j < 7; j++) { std::swap(A[k * 7 + j], A[piv * 7 + j]); std::swap(R[k * 7 + j], R[piv * 7 + j]); }
    const double d = A[k * 7 + k];
    for (int j = 0; j < 7; j++) { A[k * 7 + j] = A[k * 7 + j] / d; R[k * 7 + j] = R[k * 7 + j] / d; }
    for (int i = 0; i < 7; i++) {
      if (i == k) continue;
      const double f = A[i * 7 + k];
      for (int j = 0; j < 7; j++) {
        const double pa = f * A[k * 7 + j], pr = f * R[k * 7 + j];
        A[i * 7 + j] = A[i * 7 + j] - pa; R[i * 7 + j] = R[i * 7 + j] - pr;
      }
    }
  }
  const double plan[7] = {0, 0, z_c, z_c - kNlpHeightOffset / 2, z_c - kNlpHeightOffset, 0, 0};
  double co[7];
  for (int r = 0; r < 7; r++) { double acc = 0.0; for (int k = 0; k < 7; k++) { const double pr = R[7 * r + k] * plan[k]; acc = acc + pr; } co[r] = acc; }
  for (int w = 0; w < n; w++) {
    const double t = w * kNlpDtx;
    double z = 0.0, vz = 0.0, az = 0.0;
    if (t <= kNlpSquatTime) {
      const double p[7] = {pow(t, 6), pow(t, 5), pow(t, 4), pow(t, 3), pow(t, 2), pow(t, 1), 1};
      const double v[7] = {6 * pow(t, 5), 5 * pow(t, 4), 4 * pow(t, 3), 3 * pow(t, 2), 2 * pow(t, 1), 1, 0};
      const double a[7] = {30 * pow(t, 4), 20 * pow(t, 3), 12 * pow(t, 2), 6 * pow(t, 1), 2, 0, 0};
      for (int k = 0; k < 7; k++) {
        const double a1 = p[k] * co[k], a2 = v[k] * co[k], a3 = a[k] * co[k];
        z = z + a1; vz = vz + a2; az = az + a3;
      }
    } else {
      z = z_c - kNlpHeightOffset;
    }
    tab[w] = z; tab[n + w] = vz; tab[2 * n + w] = az;
  }
}
constexpr int kSquatN = 48;
}  // namespace

int go1mpc_nlp_node_state_doubles(void) { return NLP_NODE_DOUBLES; }
int go1mpc_nlp_t_end_footstep(const go1mpc_t* h) { int t = 0; if (h) nlp_limits(h, &t, nullptr); return t; }
int go1mpc_nlp_walkdtime_max(const go1mpc_t* h) { int w = 0; if (h) nlp_limits(h, nullptr, &w); return w; }
// members as NLPRTControlClass() (NLPRTControlClass.cpp:25-189) and NLPClass::Initialize leave them
int go1mpc_nlp_node_default_state(go1mpc_t* h, double* s) {
  if (!h || !s) return GO1MPC_E_INVALID;
  memset(s, 0, sizeof(double) * NLP_NODE_DOUBLES);
  const double hw = h->cfg.step.half_hip_width, z_c = h->cfg.step.hcom + kNlpHeightOffset;
  int rc = go1mpc_step_default_state(h, kNlpStepLength, 2 * hw, kNlpStepHeight, kNlpTstep, s);
  if (rc) return rc;
  if ((rc = go1mpc_foot_default_state(h, s + STEP_STATE_DOUBLES))) return rc;
  s[kNlpZhi] = -1.0; s[kNlpLift0] = GO1MPC_FOOTSTEPS; s[kNlpRsup] = 2.0;
  s[kNlpPel + 2] = z_c; s[kNlpLf + 1] = hw; s[kNlpRf + 1] = -hw;
  s[kNlpComx + 2] = z_c - kNlpHeightOffset;
  return GO1MPC_OK;
}

namespace {
int nlp_node_enqueue(go1mpc_t* h, int B, double* state_d, const int* walkdtime_d, const int* start_d, const int* cmd_d,
                     const double* rfoot_fb_d, const double* lfoot_fb_d, double* msg_d, const int* active_d, int* step_diag_d,
                     void* stream);
}
int go1mpc_nlp_node_tick_batch(go1mpc_t* h, int B, double* state_d, const int* walkdtime_d, const int* start_d, const int* cmd_d,
                               const double* rfoot_fb_d, const double* lfoot_fb_d, double* msg_d, void* stream) {
  return nlp_node_enqueue(h, B, state_d, walkdtime_d, start_d, cmd_d, rfoot_fb_d, lfoot_fb_d, msg_d, nullptr, nullptr, stream);
}
namespace {
// active_d: [B] ints or null (= all); robots with 0 leave the node untouched (per-robot clocks of the gait stack).
// step_diag_d: [STEP_DIAG_INTS][B] or null, the planner tick's diag (written only for robots whose node tick is >= 1)
int nlp_node_enqueue(go1mpc_t* h, int B, double* state_d, const int* walkdtime_d, const int* start_d, const int* cmd_d,
                     const double* rfoot_fb_d, const double* lfoot_fb_d, double* msg_d, const int* active_d, int* step_diag_d,
                     void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !state_d || !walkdtime_d || !msg_d) return fail(h, GO1MPC_E_INVALID, "nlp_node_tick_batch: bad argument");
  if (h->cfg.step.ext_height) return fail(h, GO1MPC_E_UNSUPPORTED, "nlp_node_tick_batch: cfg.step.ext_height must be 0 (the node owns CoM_height_solve)");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  const Go1StepMpcConfig& c = h->cfg.step;
  if (!h->squat_d) {
    double tab[3 * kSquatN];
    build_squat_table(c.hcom + kNlpHeightOffset, kSquatN, tab);
    CU(h, cudaMalloc((void**)&h->squat_d, sizeof tab));
    CU(h, cudaMemcpy(h->squat_d, tab, sizeof tab, cudaMemcpyHostToDevice));
  }
  StreamWs* W;
  int rc = stream_ws(h, st, &W);
  if (rc) return rc;
  auto& ws = W->nlp;
  const size_t b = (size_t)B, d = b * sizeof(double);
  if ((rc = grow(h, ws.tick, b * sizeof(int), st)) || (rc = grow(h, ws.in, STEP_IN_DOUBLES * d, st)) ||
      (rc = grow(h, ws.out38, STEP_OUT_DOUBLES * d, st)) || (rc = grow(h, ws.out18, FOOT_OUT_DOUBLES * d, st)) ||
      (rc = grow(h, ws.right_support, b * sizeof(int), st)) || (rc = grow(h, ws.hz_co, 8 * d, st)) || (rc = grow(h, ws.lipm, 6 * d, st)))
    return rc;
  NlpKParams P;
  P.B = B;
  nlp_limits(h, &P.t_end, &P.walkdtime_max);
  P.dt = c.dt; P.dtx = kNlpDtx; P.height_offset_time = kNlpHeightOffsetTime; P.half_hip_width = c.half_hip_width;
  P.stepwidth0 = c.stepwidth0; P.mass = kNlpMass; P.rad = kNlpRad; P.ggg = c.ggg; P.z_c = c.hcom + kNlpHeightOffset;
  P.height_offset = kNlpHeightOffset; P.Wn = c.Wn;
  for (int q = 0; q < NLP_NTD_MAX; q++) { const double w = c.Wn * c.dt * (q + 1); P.sh_w[q] = sinh(w); P.ch_w[q] = cosh(w); }
  P.squat = h->squat_d; P.squat_n = kSquatN;
  P.node = state_d; P.walkdtime = walkdtime_d; P.start = start_d; P.cmd = cmd_d; P.rfoot_fb = rfoot_fb_d; P.lfoot_fb = lfoot_fb_d;
  P.tick = (int*)ws.tick.p; P.in = (double*)ws.in.p; P.out38 = (double*)ws.out38.p; P.out18 = (double*)ws.out18.p;
  P.right_support = (int*)ws.right_support.p; P.hz_co = (double*)ws.hz_co.p; P.lipm = (double*)ws.lipm.p; P.msg = msg_d;
  P.active = active_d;
  CU(h, nlp_pre_launch(P, st));
  h->launches++;
  // the planner state is rows [0, 202) of the node, the swing-foot window rows [202, 234): same SoA stride B
  rc = step_tick_enqueue(h, 3, B, P.tick, state_d, state_d, P.in, P.out38, step_diag_d, st, P.hz_co, P.lipm);
  if (rc) return rc;
  rc = foot_enqueue(h, B, P.tick, state_d, P.out38, state_d + (size_t)STEP_STATE_DOUBLES * B, P.out18, P.right_support, st,
                    state_d + (size_t)kNlpLift0 * B, state_d + (size_t)kNlpStop * B, P.t_end);
  if (rc) return rc;
  CU(h, nlp_post_launch(P, st));
  h->launches++;
  return GO1MPC_OK;
}
}  // namespace

// host form: SoA host buffers of the same shapes; state and msg are copied up, the tick runs, state and msg come down
int go1mpc_nlp_node_tick_batch_host(go1mpc_t* h, int B, double* state, const int* walkdtime, const int* start, const int* cmd,
                                    const double* rfoot_fb, const double* lfoot_fb, double* msg) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!state || !walkdtime || !msg) return fail(h, GO1MPC_E_INVALID, "nlp_node_tick_batch_host: bad argument");
  const size_t b = (size_t)B, ib = b * sizeof(int), fb = b * 3 * sizeof(double);
  Staging S(h, h->stage, h->stream);
  double* ds = S.inout(state, b * NLP_NODE_DOUBLES * sizeof(double));
  const int* dw = S.up(walkdtime, ib);
  const int* dst_ = S.up(start, ib);
  const int* dc = S.up(cmd, ib);
  const double* drf = S.up(rfoot_fb, fb);
  const double* dlf = S.up(lfoot_fb, fb);
  double* dm = S.out(msg, b * 100 * sizeof(double));
  return S.run(true, [&] { return go1mpc_nlp_node_tick_batch(h, B, ds, dw, dst_, dc, drf, dlf, dm, S.st); });
}

// ------------------------------------------------------------------ the 100 Hz node (message in, message out)
int go1mpc_rt_node_state_doubles(int nh) {
  const int ni = 9 + 3 * (nh - 1);
  return (56 + 4 * ni + 6 * (nh + 1) + 6 * nh + 3 + 14) + (138 + 6 * (nh + 2)) + (2 + 6 * nh);
}
// members as the node's main() (RT/gait_fast.cpp:383-447) and PRMPCClass::Initialize / FootStepInputs (:46-55,105-139,2198-2221) leave them
int go1mpc_rt_node_default_state(go1mpc_t* h, int nh, double* s) {
  if (!h || !s) return GO1MPC_E_INVALID;
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "rt_node_default_state: 3 <= nh <= 40");
  const Go1BodyMpcConfig& c = h->cfg.body;
  const int S = go1mpc_rt_node_state_doubles(nh), ni = 9 + 3 * (nh - 1), W = nh + 2;
  memset(s, 0, sizeof(double) * S);
  const double zc = h->cfg.step.hcom, hw = h->cfg.step.half_hip_width;
  for (int q = 0; q < 4; q++) s[5 + 3 * q + 2] = zc;            // COM_in1, COM_in2, COMxyz_ref, COM_ref2: z = Z_C
  s[56 + 2] = zc;                                              // rpy_mpc_body(2)
  double* foot = s + 56 + 4 * ni;
  for (int j = 0; j < nh + 1; j++) { foot[6 * j + 1] = -hw; foot[6 * j + 4] = hw; }
  double* fs = s + 56 + 4 * ni + 6 * (nh + 1) + 6 * nh + 3 + 14;
  double sw[GO1MPC_FOOTSTEPS];
  const double lift = 0.015;                                   // PRMPCClass::Initialize :51
  for (int i = 0; i < GO1MPC_FOOTSTEPS; i++) { sw[i] = 2 * hw; fs[i] = c.tstep; fs[108 + i] = lift; }
  sw[0] = sw[0] / 2;
  fs[108 + 26] = 0; fs[108 + 25] = 0; fs[108 + 24] = lift / 2; fs[108 + 23] = lift;
  for (int i = 1; i < GO1MPC_FOOTSTEPS; i++) fs[54 + i] = fs[54 + i - 1] + (int)pow(-1, i - 1) * sw[i - 1];
  for (int k = 0; k < W; k++) { fs[138 + 1 * W + k] = -sw[0]; fs[138 + 4 * W + k] = sw[0]; }
  return GO1MPC_OK;
}
namespace {
int rt_node_enqueue(go1mpc_t* h, int nh, int B, double* state_d, const double* msg_d, const int* ctrl_d, const double* bodyangle_state_d,
                    const double* ctl_msg_d, double* body_in_d, double* body_out_d, int* body_diag_d, double* out100_d,
                    double* rt2nrt_d, int* active_d, void* stream);
}
int go1mpc_rt_node_tick_batch(go1mpc_t* h, int nh, int B, double* state_d, const double* msg_d, const int* ctrl_d,
                              const double* bodyangle_state_d, double* body_in_d, double* body_out_d, int* body_diag_d,
                              double* out100_d, int* active_d, void* stream) {
  return rt_node_enqueue(h, nh, B, state_d, msg_d, ctrl_d, bodyangle_state_d, nullptr, body_in_d, body_out_d, body_diag_d, out100_d,
                         nullptr, active_d, stream);
}
int go1mpc_rt_node_tick_msgs_batch(go1mpc_t* h, int nh, int B, double* state_d, const double* gait_msg_d, const double* ctl_msg_d,
                                   double* body_in_d, double* body_out_d, int* body_diag_d, double* traj_msg_d, double* rt2nrt_msg_d,
                                   void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  if (!ctl_msg_d) return fail(h, GO1MPC_E_INVALID, "rt_node_tick_msgs_batch: bad argument");
  return rt_node_enqueue(h, nh, B, state_d, gait_msg_d, nullptr, nullptr, ctl_msg_d, body_in_d, body_out_d, body_diag_d, traj_msg_d,
                         rt2nrt_msg_d, nullptr, stream);
}
namespace {
int rt_node_enqueue(go1mpc_t* h, int nh, int B, double* state_d, const double* msg_d, const int* ctrl_d, const double* bodyangle_state_d,
                    const double* ctl_msg_d, double* body_in_d, double* body_out_d, int* body_diag_d, double* out100_d,
                    double* rt2nrt_d, int* active_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !state_d || !msg_d || !body_in_d || !body_out_d || !out100_d) return fail(h, GO1MPC_E_INVALID, "rt_node_tick_batch: bad argument");
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "rt_node_tick_batch: 3 <= nh <= 40");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  const Go1BodyMpcConfig& c = h->cfg.body;
  RtKParams P;
  P.B = B; P.nh = nh; P.in_stride = go1mpc_body_in_stride(nh); P.out_stride = go1mpc_body_out_stride(nh);
  P.dt_mpc = c.dt_mpc; P.dt_slow = c.dt_slow; P.tstep = c.tstep; P.tdsp_ratio = 0.1;      // PRMPCClass::Initialize :169
  P.stepwidth0 = h->cfg.step.half_hip_width; P.footx_max = 0.15;                              // :52,149
  build_aaa_inv_mod(c.dt_slow, P.inv);
  P.state = state_d; P.msg = msg_d; P.ctrl = ctrl_d; P.bodyangle_state = bodyangle_state_d;
  P.body_in = body_in_d; P.body_out = body_out_d; P.out = out100_d; P.active = active_d;
  P.ctl_msg = ctl_msg_d; P.rt2nrt = rt2nrt_d;
  CU(h, rt_pre_launch(P, st));
  h->launches++;
  int rc = go1mpc_body_mpc_step_batch(h, nh, B, body_in_d, body_out_d, body_diag_d, st);
  if (rc) return rc;
  CU(h, rt_post_launch(P, st));
  h->launches++;
  return GO1MPC_OK;
}
}  // namespace

// host form of the 100 Hz node: state / msg / body_out (the body MPC's state) are host SoA / record buffers
int go1mpc_rt_node_tick_batch_host(go1mpc_t* h, int nh, int B, double* state, const double* msg, const int* ctrl,
                                   const double* bodyangle_state, double* body_out, double* out100) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!state || !msg || !body_out || !out100) return fail(h, GO1MPC_E_INVALID, "rt_node_tick_batch_host: bad argument");
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "rt_node_tick_batch_host: 3 <= nh <= 40");
  const size_t b = (size_t)B, mb = b * 100 * sizeof(double);
  Staging S(h, h->stage, h->stream);
  double* ds = S.inout(state, b * go1mpc_rt_node_state_doubles(nh) * sizeof(double));
  const double* dm = S.up(msg, mb);
  const int* dc = S.up(ctrl, b * sizeof(int));
  const double* da = S.up(bodyangle_state, b * 4 * sizeof(double));
  double* dbi = S.out_always((double*)nullptr, b * go1mpc_body_in_stride(nh) * sizeof(double), 0);   // the node writes the records
  double* dbo = S.inout(body_out, b * go1mpc_body_out_stride(nh) * sizeof(double));
  double* dout = S.out(out100, mb);
  return S.run(true, [&] { return go1mpc_rt_node_tick_batch(h, nh, B, ds, dm, dc, da, dbi, dbo, nullptr, dout, nullptr, S.st); });
}

// ------------------------------------------------------------------ gait stack tick: both nodes behind one host call
static_assert(GO1MPC_STACK_ROW_GAIT == GO1MPC_STACK_ROW_NLP + NLP_NODE_DOUBLES && GO1MPC_STACK_ROW_RT2NRT == GO1MPC_STACK_ROW_GAIT + 100 &&
              GO1MPC_STACK_ROW_WALKDTIME == GO1MPC_STACK_ROW_RT2NRT + 25 && GO1MPC_STACK_ROW_TRAJ == GO1MPC_STACK_ROW_WALKDTIME + 1 &&
              GO1MPC_STACK_ROW_RT == GO1MPC_STACK_ROW_TRAJ + 100, "gait stack state layout");
static_assert(GO1MPC_STACK_SENSOR_ROWS == GAIT_STACK_SENSOR_ROWS && GO1MPC_STACK_SLOTS_MAX == GAIT_STACK_SLOTS_MAX, "gait stack sizes");
int go1mpc_gait_stack_state_doubles(int nh) { return GO1MPC_STACK_ROW_RT + go1mpc_rt_node_state_doubles(nh); }
int go1mpc_gait_stack_default_state(go1mpc_t* h, int nh, double* s) {
  if (!h || !s) return GO1MPC_E_INVALID;
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "gait_stack_default_state: 3 <= nh <= 40");
  memset(s, 0, sizeof(double) * GO1MPC_STACK_ROW_RT);
  int rc = go1mpc_nlp_node_default_state(h, s + GO1MPC_STACK_ROW_NLP);
  if (rc) return rc;
  return go1mpc_rt_node_default_state(h, nh, s + GO1MPC_STACK_ROW_RT);
}

namespace {
struct Block { const void* p; size_t bytes; };
// Whether the device input [in, in + bytes) shares a byte with one of the blocks a call writes (null blocks are skipped).  The
// kernels that read the inputs declare their pointers __restrict__, so a caller's input must not alias what the call writes.
bool overlaps_written(const void* in, size_t bytes, std::initializer_list<Block> written) {
  if (!in) return false;
  const uintptr_t lo = (uintptr_t)in, hi = lo + bytes;
  for (const Block& w : written)
    if (w.p && (uintptr_t)w.p < hi && lo < (uintptr_t)w.p + w.bytes) return true;
  return false;
}

// The node sequence of both gait stack ticks.  clock_d == null: every robot gets t.planner (go1mpc_gait_stack_tick_host_async);
// otherwise each robot's planner flag comes from its clock (go1mpc_gait_stack_tick_clocked_async), and the planner node is always
// enqueued, with the robots that do not plan masked out -- the same launches every period, so one captured graph fits all.
// health_d (clocked only, else null): the planner and body MPC write their diag into the stream's workspace, and one more kernel
// after the pack updates the farm's health counters from it.
int gait_stack_enqueue(go1mpc_t* h, int B, const Go1GaitStackTick* t, int* clock_d, int* health_d, void* stream, const char* name) {
  const std::string nm(name);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!t || !t->sensor == !t->sensor_d || !t->state_d || !t->body_out_d || !t->rows_d) return fail(h, GO1MPC_E_INVALID, nm + ": bad argument");
  if ((t->cmd && t->cmd_d) || (t->start && t->start_d))
    return fail(h, GO1MPC_E_INVALID, nm + ": at most one of cmd / cmd_d and one of start / start_d");
  const int nh = t->nh, n = t->n_slots;
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, nm + ": 3 <= nh <= 40");
  if (h->cfg.step.ext_height)
    return fail(h, GO1MPC_E_UNSUPPORTED, nm + ": cfg.step.ext_height must be 0 (the planner node owns CoM_height_solve)");
  if (n < 1 || n > GO1MPC_STACK_SLOTS_MAX) return fail(h, GO1MPC_E_INVALID, nm + ": 1 <= n_slots <= 64");
  GaitStackSlots S;
  S.n = n;
  for (int k = 0; k < GO1MPC_STACK_SLOTS_MAX; k++) {
    S.slot[k] = k < n ? t->slots[k] : 0;
    if (S.slot[k] < 0 || S.slot[k] >= 200) return fail(h, GO1MPC_E_INVALID, nm + ": slots must lie in 0..199");
  }
  // the body kernels read and write body_out_d with 16-byte loads / TMA; the pack kernel stores doubles into rows_d
  if (((uintptr_t)t->body_out_d & 15) || ((uintptr_t)t->rows_d & 7))
    return fail(h, GO1MPC_E_INVALID, nm + ": body_out_d must be 16-byte and rows_d 8-byte aligned");
  if (((uintptr_t)t->sensor_d & 7) || (((uintptr_t)t->cmd_d | (uintptr_t)t->start_d) & 3))
    return fail(h, GO1MPC_E_INVALID, nm + ": sensor_d must be 8-byte and cmd_d / start_d 4-byte aligned");
  {
    const size_t b = (size_t)B;
    const std::initializer_list<Block> written = {{t->state_d, b * go1mpc_gait_stack_state_doubles(nh) * sizeof(double)},
                                                  {t->body_out_d, b * go1mpc_body_out_stride(nh) * sizeof(double)},
                                                  {t->rows_d, b * n * sizeof(double)}, {clock_d, b * sizeof(int)}};
    if (overlaps_written(t->sensor_d, b * GO1MPC_STACK_SENSOR_ROWS * sizeof(double), written) ||
        overlaps_written(t->cmd_d, b * sizeof(int), written) || overlaps_written(t->start_d, b * sizeof(int), written))
      return fail(h, GO1MPC_E_INVALID, nm + ": sensor_d / cmd_d / start_d overlap state_d, body_out_d, rows_d or clock_d");
    if (health_d) {
      if ((uintptr_t)health_d & 3) return fail(h, GO1MPC_E_INVALID, nm + ": health_d must be 4-byte aligned");
      if (overlaps_written(health_d, b * GO1MPC_HEALTH_ROWS * sizeof(int),
                           {{t->state_d, b * go1mpc_gait_stack_state_doubles(nh) * sizeof(double)},
                            {t->body_out_d, b * go1mpc_body_out_stride(nh) * sizeof(double)}, {t->rows_d, b * n * sizeof(double)},
                            {clock_d, b * sizeof(int)}, {t->sensor_d, b * GO1MPC_STACK_SENSOR_ROWS * sizeof(double)},
                            {t->cmd_d, b * sizeof(int)}, {t->start_d, b * sizeof(int)}}))
        return fail(h, GO1MPC_E_INVALID, nm + ": health_d overlaps state_d, body_out_d, rows_d, clock_d, sensor_d, cmd_d or start_d");
    }
  }
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  StreamWs* W;
  int rc = stream_ws(h, st, &W);
  if (rc) return rc;
  auto& ws = W->stack;
  const size_t b = (size_t)B, sb = b * GO1MPC_STACK_SENSOR_ROWS * sizeof(double), cb = b * 25 * sizeof(double), ib = b * sizeof(int);
  bool fresh = false;   // the control message buffer was (re)allocated
  if ((rc = grow(h, ws.sensor, sb, st)) || (rc = grow(h, ws.ctl_msg, cb, st, &fresh)) || (rc = grow(h, ws.walkdtime, ib, st)) ||
      (rc = grow(h, ws.cmd, ib, st)) || (rc = grow(h, ws.start, ib, st)) ||
      (rc = grow(h, ws.body_in, b * go1mpc_body_in_stride(nh) * sizeof(double), st)) || (clock_d && (rc = grow(h, ws.plan, ib, st))))
    return rc;
  int *step_diag = nullptr, *body_diag = nullptr;
  if (health_d) {
    if ((rc = grow(h, W->health.step_diag, STEP_DIAG_INTS * ib, st)) ||
        (rc = grow(h, W->health.body_diag, b * go1mpc_body_diag_stride(nh) * sizeof(int), st)))
      return rc;
    step_diag = (int*)W->health.step_diag.p;
    body_diag = (int*)W->health.body_diag.p;
  }
  if (fresh) ws.zero_B = -1;
  double* ctl = (double*)ws.ctl_msg.p;
  int* walkdtime = (int*)ws.walkdtime.p;
  if (ws.zero_B != B) {
    // the 14 slots of /control2rtmpc/state the stack does not upload read as zero: cleared once per batch size
    CU(h, cudaMemsetAsync(ctl, 0, cb, st));
    ws.zero_B = B;
  }
  double* state = t->state_d;
  // device inputs are read in place; host inputs go up into the stream's staging buffers
  const double* sensor = t->sensor_d;
  if (!sensor) { CU(h, cudaMemcpyAsync(ws.sensor.p, t->sensor, sb, cudaMemcpyHostToDevice, st)); sensor = (const double*)ws.sensor.p; }
  // with per-robot clocks some robot may plan in any call, so cmd / start go up whenever they are given
  const bool planner = clock_d || t->planner;
  const int* cmd_d = t->cmd_d;
  const int* start_d = t->start_d;
  if (planner && t->cmd) { CU(h, cudaMemcpyAsync(ws.cmd.p, t->cmd, ib, cudaMemcpyHostToDevice, st)); cmd_d = (const int*)ws.cmd.p; }
  if (planner && t->start) { CU(h, cudaMemcpyAsync(ws.start.p, t->start, ib, cudaMemcpyHostToDevice, st)); start_d = (const int*)ws.start.p; }
  int* plan_d = (int*)ws.plan.p;
  if (clock_d)
    CU(h, gait_stack_clocked_pre_launch(B, clock_d, plan_d, state + GO1MPC_STACK_ROW_WALKDTIME * b, walkdtime, sensor, ctl, h->sms, st));
  else
    CU(h, gait_stack_pre_launch(B, t->planner ? 1 : 0, state + GO1MPC_STACK_ROW_WALKDTIME * b, walkdtime, sensor, ctl, h->sms, st));
  h->launches++;
  double* gait = state + GO1MPC_STACK_ROW_GAIT * b;
  double* rt2nrt = state + GO1MPC_STACK_ROW_RT2NRT * b;
  double* traj = state + GO1MPC_STACK_ROW_TRAJ * b;
  if (planner &&
      (rc = nlp_node_enqueue(h, B, state + GO1MPC_STACK_ROW_NLP * b, walkdtime, start_d, cmd_d, rt2nrt + 22 * b, rt2nrt + 19 * b,
                             gait, clock_d ? plan_d : nullptr, step_diag, st)))
    return rc;
  if ((rc = rt_node_enqueue(h, nh, B, state + GO1MPC_STACK_ROW_RT * b, gait, nullptr, nullptr, ctl, (double*)ws.body_in.p, t->body_out_d,
                            body_diag, traj, rt2nrt, nullptr, st)))
    return rc;
  CU(h, gait_stack_pack_launch(S, B, gait, traj, t->rows_d, h->sms, st));
  h->launches++;
  if (health_d) {
    FarmHealthStackParams H;
    H.B = B; H.n_slots = n; H.body_diag_stride = go1mpc_body_diag_stride(nh);
    H.clock = clock_d; H.node_tick = (const int*)W->nlp.tick.p; H.step_diag = step_diag; H.body_diag = body_diag; H.rows = t->rows_d;
    H.health = health_d;
    CU(h, farm_health_stack_launch(H, h->sms, st));
    h->launches++;
  }
  if (t->rows) CU(h, cudaMemcpyAsync(t->rows, t->rows_d, b * n * sizeof(double), cudaMemcpyDeviceToHost, st));
  return GO1MPC_OK;
}
}  // namespace

int go1mpc_gait_stack_tick_host_async(go1mpc_t* h, int B, const Go1GaitStackTick* t, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  return gait_stack_enqueue(h, B, t, nullptr, nullptr, stream, "gait_stack_tick_host_async");
}

namespace {
int gait_stack_clocked_enqueue(go1mpc_t* h, int B, const Go1GaitStackClockedTick* t, int* health_d, void* stream, const char* name) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!t || !t->clock_d) return fail(h, GO1MPC_E_INVALID, std::string(name) + ": bad argument");
  Go1GaitStackTick u;
  u.nh = t->nh; u.planner = 0; u.sensor = t->sensor; u.cmd = t->cmd; u.start = t->start; u.state_d = t->state_d;
  u.body_out_d = t->body_out_d; u.n_slots = t->n_slots; u.rows_d = t->rows_d; u.rows = t->rows;
  u.sensor_d = t->sensor_d; u.cmd_d = t->cmd_d; u.start_d = t->start_d;
  memcpy(u.slots, t->slots, sizeof u.slots);
  return gait_stack_enqueue(h, B, &u, t->clock_d, health_d, stream, name);
}
}  // namespace

int go1mpc_gait_stack_tick_clocked_async(go1mpc_t* h, int B, const Go1GaitStackClockedTick* t, void* stream) {
  return gait_stack_clocked_enqueue(h, B, t, nullptr, stream, "gait_stack_tick_clocked_async");
}

int go1mpc_gait_stack_tick_clocked_health_async(go1mpc_t* h, int B, const Go1GaitStackClockedTick* t, int* health_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (!health_d) return fail(h, GO1MPC_E_INVALID, "gait_stack_tick_clocked_health_async: health_d must be given");
  return gait_stack_clocked_enqueue(h, B, t, health_d, stream, "gait_stack_tick_clocked_health_async");
}

int go1mpc_gait_stack_reset_async(go1mpc_t* h, int B, const Go1GaitStackReset* r, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!r || !r->reset == !r->reset_d || !r->clock_d || !r->state_d || !r->body_out_d)
    return fail(h, GO1MPC_E_INVALID, "gait_stack_reset_async: bad argument");
  const int nh = r->nh;
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "gait_stack_reset_async: 3 <= nh <= 40");
  if ((uintptr_t)r->body_out_d & 15) return fail(h, GO1MPC_E_INVALID, "gait_stack_reset_async: body_out_d must be 16-byte aligned");
  if ((uintptr_t)r->reset_d & 3) return fail(h, GO1MPC_E_INVALID, "gait_stack_reset_async: reset_d must be 4-byte aligned");
  if (overlaps_written(r->reset_d, (size_t)B * sizeof(int),
                       {{r->state_d, (size_t)B * go1mpc_gait_stack_state_doubles(nh) * sizeof(double)},
                        {r->body_out_d, (size_t)B * go1mpc_body_out_stride(nh) * sizeof(double)},
                        {r->clock_d, (size_t)B * sizeof(int)}, {r->servo_state_d, (size_t)B * SERVO_STATE_ROWS * sizeof(double)}}))
    return fail(h, GO1MPC_E_INVALID, "gait_stack_reset_async: reset_d overlaps state_d, body_out_d, clock_d or servo_state_d");
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  const int rows = go1mpc_gait_stack_state_doubles(nh);
  auto it = h->stack_col_d.find(nh);
  if (it == h->stack_col_d.end()) {
    std::vector<double> col(rows);
    int rc = go1mpc_gait_stack_default_state(h, nh, col.data());
    if (rc) return rc;
    double* p = nullptr;
    CU(h, cudaMalloc((void**)&p, sizeof(double) * rows));
    cudaError_t e = cudaMemcpy(p, col.data(), sizeof(double) * rows, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(p); return cuda_fail(h, e, "cudaMemcpy(default gait stack column)"); }
    it = h->stack_col_d.emplace(nh, p).first;
  }
  StreamWs* W;
  int rc = stream_ws(h, st, &W);
  if (rc) return rc;
  const size_t b = (size_t)B;
  if ((rc = grow(h, W->reset_list, (4 + 2 * b) * sizeof(int), st))) return rc;
  StackResetParams P;
  P.B = B; P.rows = rows; P.out_stride = go1mpc_body_out_stride(nh);
  P.count = (int*)W->reset_list.p; P.reset = r->reset_d ? r->reset_d : P.count + 4; P.list = P.count + 4 + B;
  P.clock = r->clock_d; P.state = r->state_d; P.column = it->second; P.body_out = r->body_out_d; P.servo = r->servo_state_d;
  memcpy(P.q0, r->servo_q0, sizeof P.q0);
  if (r->reset) CU(h, cudaMemcpyAsync((void*)P.reset, r->reset, b * sizeof(int), cudaMemcpyHostToDevice, st));
  CU(h, cudaMemsetAsync(P.count, 0, sizeof(int), st));
  CU(h, gait_stack_reset_launch(P, h->sms, st));
  h->launches += 2;
  return GO1MPC_OK;
}

int go1mpc_farm_copy_async(go1mpc_t* h, const Go1FarmCopy* c, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (!c) return fail(h, GO1MPC_E_INVALID, "farm_copy_async: bad argument");
  const Go1FarmColumns &D = c->dst, &S = c->src;
  if (D.B < 0 || S.B < 0) return fail(h, GO1MPC_E_INVALID, "farm_copy_async: negative B");
  if (D.B == 0) return GO1MPC_OK;
  if (S.B < 1) return fail(h, GO1MPC_E_INVALID, "farm_copy_async: src.B must be at least 1");
  if (!D.state_d || !D.body_out_d || !S.state_d || !S.body_out_d || !c->index_d)
    return fail(h, GO1MPC_E_INVALID, "farm_copy_async: bad argument");
  if (!D.clock_d != !S.clock_d || !D.servo_state_d != !S.servo_state_d || !D.force_state_d != !S.force_state_d ||
      !D.health_d != !S.health_d)
    return fail(h, GO1MPC_E_INVALID,
                "farm_copy_async: clock_d, servo_state_d, force_state_d and health_d must be given on both sides or neither");
  if (((uintptr_t)D.health_d | (uintptr_t)S.health_d) & 3) return fail(h, GO1MPC_E_INVALID, "farm_copy_async: health_d must be 4-byte aligned");
  if (((uintptr_t)D.body_out_d | (uintptr_t)S.body_out_d) & 15)
    return fail(h, GO1MPC_E_INVALID, "farm_copy_async: body_out_d must be 16-byte aligned");
  const int nh = c->nh;
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "farm_copy_async: 3 <= nh <= 40");
  const int rows = go1mpc_gait_stack_state_doubles(nh), out_stride = go1mpc_body_out_stride(nh);
  // the kernels read the source while they write the destination: no destination block may share a byte with a source block
  auto blocks = [&](const Go1FarmColumns& F, uintptr_t* lo, uintptr_t* hi) {
    const size_t b = (size_t)F.B;
    const void* p[6] = {F.state_d, F.body_out_d, F.clock_d, F.servo_state_d, F.force_state_d, F.health_d};
    const size_t n[6] = {b * rows * sizeof(double), b * out_stride * sizeof(double), b * sizeof(int), b * SERVO_STATE_ROWS * sizeof(double),
                         b * SERVO_FORCE_ROWS * sizeof(double), b * GO1MPC_HEALTH_ROWS * sizeof(int)};
    for (int k = 0; k < 6; k++) { lo[k] = (uintptr_t)p[k]; hi[k] = p[k] ? lo[k] + n[k] : lo[k]; }
  };
  uintptr_t dlo[6], dhi[6], slo[6], shi[6];
  blocks(D, dlo, dhi);
  blocks(S, slo, shi);
  for (int i = 0; i < 6; i++)
    for (int k = 0; k < 6; k++)
      if (dlo[i] < shi[k] && slo[k] < dhi[i])
        return fail(h, GO1MPC_E_INVALID, "farm_copy_async: a destination block overlaps a source block");
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  StreamWs* W;
  int rc = stream_ws(h, st, &W);
  if (rc) return rc;
  if ((rc = grow(h, W->copy_list, (4 + 2 * (size_t)D.B) * sizeof(int), st))) return rc;
  FarmCopyParams P;
  P.dst_B = D.B; P.src_B = S.B;
  P.rows = rows;
  P.servo_end = rows + (D.servo_state_d ? SERVO_STATE_ROWS : 0);
  P.soa_rows = P.servo_end + (D.force_state_d ? SERVO_FORCE_ROWS : 0);
  P.rec2 = out_stride / 2;
  P.index = c->index_d; P.bad = c->bad_d;
  P.dst_state = D.state_d; P.dst_servo = D.servo_state_d; P.dst_force = D.force_state_d;
  P.src_state = S.state_d; P.src_servo = S.servo_state_d; P.src_force = S.force_state_d;
  P.dst_body = reinterpret_cast<double2*>(D.body_out_d); P.src_body = reinterpret_cast<const double2*>(S.body_out_d);
  P.dst_clock = D.clock_d; P.src_clock = S.clock_d;
  P.dst_health = D.health_d; P.src_health = S.health_d;
  P.count = (int*)W->copy_list.p; P.dlist = P.count + 4; P.slist = P.count + 4 + D.B;
  CU(h, cudaMemsetAsync(P.count, 0, sizeof(int), st));
  CU(h, farm_copy_launch(P, h->sms, st));
  h->launches += 2;
  return GO1MPC_OK;
}

// ------------------------------------------------------------------ servo stack tick: K 1 kHz servo ticks from the resident messages
static_assert(GO1MPC_SERVO_TICKS_MAX == SERVO_TICKS_MAX && GO1MPC_SERVO_STATE_ROWS == SERVO_STATE_ROWS &&
              GO1MPC_SERVO_ROW_Q == SERVO_ROW_Q && GO1MPC_SERVO_ROW_HOMING == SERVO_ROW_HOMING && GO1MPC_SERVO_ROW_LPF == SERVO_ROW_LPF,
              "servo stack state layout");
int go1mpc_servo_stack_tick_async(go1mpc_t* h, int B, const Go1ServoStackTick* t, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!t || !t->stack_state_d || !t->servo_state_d || !t->q_d) return fail(h, GO1MPC_E_INVALID, "servo_stack_tick_async: bad argument");
  if (t->K < 1 || t->K > GO1MPC_SERVO_TICKS_MAX) return fail(h, GO1MPC_E_INVALID, "servo_stack_tick_async: 1 <= K <= 10");
  if ((uintptr_t)t->q_d & 7) return fail(h, GO1MPC_E_INVALID, "servo_stack_tick_async: q_d must be 8-byte aligned");
  if (t->gait_mode < 101 || t->gait_mode > 103) return fail(h, GO1MPC_E_UNSUPPORTED, "servo_stack_tick_async: gait_mode 101, 102 or 103");
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  CU(h, servo_stack_launch(servo_stack_params(h, B, t, nullptr), st));
  h->launches++;
  if (t->q) CU(h, cudaMemcpyAsync(t->q, t->q_d, (size_t)B * 12 * t->K * sizeof(double), cudaMemcpyDeviceToHost, st));
  return GO1MPC_OK;
}

// ------------------------------------------------------------------ servo torque tick: the servo stack + force QP + torque map
static_assert(GO1MPC_SERVO_FORCE_ROWS == SERVO_FORCE_ROWS, "servo force state layout");
static_assert(GO1MPC_HEALTH_ROWS == FARM_HEALTH_ROWS && GO1MPC_HEALTH_PLAN_OK == FH_PLAN_OK && GO1MPC_HEALTH_PLAN_INFEASIBLE == FH_PLAN_INF &&
              GO1MPC_HEALTH_PLAN_FAILED == FH_PLAN_FAIL && GO1MPC_HEALTH_BODY_OK == FH_BODY_OK && GO1MPC_HEALTH_BODY_INFEASIBLE == FH_BODY_INF &&
              GO1MPC_HEALTH_BODY_FAILED == FH_BODY_FAIL && GO1MPC_HEALTH_GRF_OK == FH_GRF_OK && GO1MPC_HEALTH_GRF_FAILED == FH_GRF_FAIL &&
              GO1MPC_HEALTH_GRF_FALLBACK == FH_GRF_FALLBACK && GO1MPC_HEALTH_IK_CAP == FH_IK_CAP && GO1MPC_HEALTH_NONFINITE == FH_NONFINITE &&
              GO1MPC_HEALTH_EVENTS == FH_EVENTS && GO1MPC_QP_OK == 0 && GO1MPC_QP_INFEASIBLE == 2, "farm health rows");
namespace {
// health_d: null, or the farm's health counters, which the health instantiations of both kernels update
int servo_torque_enqueue(go1mpc_t* h, int B, const Go1ServoTorqueTick* t, int* health_d, void* stream, const char* name) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  const std::string nm(name);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!t || !t->stack_state_d || !t->servo_state_d || !t->q_d || !t->force_state_d || !t->meas_d || !t->tau_d)
    return fail(h, GO1MPC_E_INVALID, nm + ": bad argument");
  if (t->K < 1 || t->K > GO1MPC_SERVO_TICKS_MAX) return fail(h, GO1MPC_E_INVALID, nm + ": 1 <= K <= 10");
  if (((uintptr_t)t->q_d | (uintptr_t)t->tau_d) & 7)
    return fail(h, GO1MPC_E_INVALID, nm + ": q_d and tau_d must be 8-byte aligned");
  if (t->gait_mode < 101 || t->gait_mode > 103) return fail(h, GO1MPC_E_UNSUPPORTED, nm + ": gait_mode 101, 102 or 103");
  if (t->reset && t->reset_d) return fail(h, GO1MPC_E_INVALID, nm + ": at most one of reset / reset_d");
  if ((uintptr_t)t->reset_d & 3) return fail(h, GO1MPC_E_INVALID, nm + ": reset_d must be 4-byte aligned");
  {
    const size_t b = (size_t)B, kb = b * 12 * t->K * sizeof(double);
    if (overlaps_written(t->reset_d, b * sizeof(int),
                         {{t->force_state_d, b * SERVO_FORCE_ROWS * sizeof(double)}, {t->servo_state_d, b * SERVO_STATE_ROWS * sizeof(double)},
                          {t->q_d, kb}, {t->tau_d, kb}}))
      return fail(h, GO1MPC_E_INVALID, nm + ": reset_d overlaps force_state_d, servo_state_d, q_d or tau_d");
    if (health_d) {
      if ((uintptr_t)health_d & 3) return fail(h, GO1MPC_E_INVALID, nm + ": health_d must be 4-byte aligned");
      // the stack state's size depends on nh, which this call does not take: its rows before the 100 Hz node's are checked
      if (overlaps_written(health_d, b * GO1MPC_HEALTH_ROWS * sizeof(int),
                           {{t->stack_state_d, b * GO1MPC_STACK_ROW_RT * sizeof(double)},
                            {t->servo_state_d, b * SERVO_STATE_ROWS * sizeof(double)},
                            {t->force_state_d, b * SERVO_FORCE_ROWS * sizeof(double)}, {t->meas_d, b * SERVO_MEAS_ROWS * sizeof(double)},
                            {t->q_d, kb}, {t->tau_d, kb}, {t->reset_d, b * sizeof(int)},
                            {t->grf_d, b * GRF_OUT_DOUBLES * sizeof(double)}, {t->grf_diag_d, b * GRF_DIAG_INTS * sizeof(int)},
                            {t->jac_d, b * 36 * sizeof(double)}, {t->foot_des_d, b * 12 * sizeof(double)}, {t->iters_d, b * 4 * sizeof(int)}}))
        return fail(h, GO1MPC_E_INVALID, nm + ": health_d overlaps a block the call reads or writes");
    }
  }
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  StreamWs* W;
  int rc = stream_ws(h, st, &W);
  if (rc) return rc;
  const size_t b = (size_t)B, rb = b * sizeof(int);
  // sized for K = GO1MPC_SERVO_TICKS_MAX, so that K changes do not reallocate
  if ((rc = grow(h, W->servo_ch, b * SERVO_TICKS_MAX * SERVO_LPF_CHANNELS * sizeof(double), st)) ||
      (t->reset && (rc = grow(h, W->servo_reset, rb, st))))
    return rc;
  void* rst = t->reset ? W->servo_reset.p : nullptr;
  ServoStackKParams S = servo_stack_params(h, B, t, (double*)W->servo_ch.p);
  S.health = health_d;
  ServoTorqueKParams P;
  P.g = grf_params(h, B, nullptr, nullptr, nullptr);
  P.B = B; P.K = t->K; P.gait_mode = t->gait_mode;
  P.half_hip_width = S.half_hip_width; P.y_offset = t->y_offset; P.y_coefficient = t->y_coefficient;
  P.swing_kp = kSwingKp; P.swing_kd = kSwingKd;
  P.gait = S.gait; P.traj = S.traj; P.homing = t->servo_state_d + SERVO_ROW_HOMING * b; P.ch = S.ch; P.q = t->q_d;
  P.meas = t->meas_d; P.reset = t->reset_d ? t->reset_d : (const int*)rst; P.force = t->force_state_d; P.tau = t->tau_d;
  P.grf = t->grf_d; P.grf_diag = t->grf_diag_d; P.health = health_d;
  if (rst) CU(h, cudaMemcpyAsync(rst, t->reset, rb, cudaMemcpyHostToDevice, st));
  CU(h, servo_stack_launch(S, st));
  h->launches++;
  CU(h, servo_torque_launch(P, h->sms, st));
  h->launches++;
  const size_t kb = b * 12 * t->K * sizeof(double);
  if (t->q) CU(h, cudaMemcpyAsync(t->q, t->q_d, kb, cudaMemcpyDeviceToHost, st));
  if (t->tau) CU(h, cudaMemcpyAsync(t->tau, t->tau_d, kb, cudaMemcpyDeviceToHost, st));
  return GO1MPC_OK;
}
}  // namespace

int go1mpc_servo_torque_tick_async(go1mpc_t* h, int B, const Go1ServoTorqueTick* t, void* stream) {
  return servo_torque_enqueue(h, B, t, nullptr, stream, "servo_torque_tick_async");
}

int go1mpc_servo_torque_tick_health_async(go1mpc_t* h, int B, const Go1ServoTorqueTick* t, int* health_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (!health_d) return fail(h, GO1MPC_E_INVALID, "servo_torque_tick_health_async: health_d must be given");
  return servo_torque_enqueue(h, B, t, health_d, stream, "servo_torque_tick_health_async");
}

// ------------------------------------------------------------------ pipelined host entries
int go1mpc_body_mpc_step_batch_host_async(go1mpc_t* h, int nh, int B, const double* in, double* out, int* diag) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!in || !out) return fail(h, GO1MPC_E_INVALID, "body_mpc_step_batch_host_async: bad argument");
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "body_mpc_step_batch_host_async: 3 <= nh <= 40");
  CU(h, cudaSetDevice(h->device));
  BodyModel* M;
  int rc = get_body_model(h, nh, &M);
  if (rc) return rc;
  const int is = go1mpc_body_in_stride(nh);
  const size_t b = (size_t)B, ob = b * go1mpc_body_out_stride(nh) * sizeof(double);
  // the previous outputs are only read by gated ticks (the reference returns its stale members):
  // upload them only when the batch has one
  bool gated = false;
  for (int k = 0; k < B && !gated; k++) {
    const int t = (int)in[(size_t)k * is + 27];
    gated = (t < M->gate) || !(t - M->gate < M->nsum_mpc - nh);
  }
  go1mpc::Lane& L = h->lanes[h->lane_next++ % go1mpc::kLanes];
  Staging S(h, L.body, L.stream);
  const double* din = S.up(in, b * is * sizeof(double));
  double* dout = gated ? S.inout(out, ob) : S.out(out, ob);
  int* ddiag = S.out(diag, b * go1mpc_body_diag_stride(nh) * sizeof(int));
  return S.run(false, [&] { return go1mpc_body_mpc_step_batch(h, nh, B, din, dout, ddiag, S.st); });
}

// Same tick with tx and the previous output record resident on the device (body_resident.cu): per instance
// 9+9nh doubles go up and 20 doubles (+ diagnostics) come down.
int go1mpc_body_tick_in_stride(int nh) { return (9 + 9 * nh + 1) & ~1; }
int go1mpc_body_mpc_step_batch_resident_host_async(go1mpc_t* h, int nh, int B, const double* tx_d, double* out_d,
                                                   const double* tick_in, double* tick_out, int* diag) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!tx_d || !out_d || !tick_in || !tick_out) return fail(h, GO1MPC_E_INVALID, "body_mpc_step_batch_resident_host_async: bad argument");
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "body_mpc_step_batch_resident_host_async: 3 <= nh <= 40");
  const int is = go1mpc_body_in_stride(nh), os = go1mpc_body_out_stride(nh), ts = go1mpc_body_tick_in_stride(nh);
  const size_t b = (size_t)B;
  go1mpc::Lane& L = h->lanes[h->lane_next++ % go1mpc::kLanes];
  Staging S(h, L.resident, L.stream);
  double* drec = S.out_always((double*)nullptr, b * is * sizeof(double), 0);   // the expand kernel writes the records
  const double* dtick = S.up(tick_in, b * ts * sizeof(double));
  double* dto = S.out(tick_out, b * GO1MPC_BODY_TICK_OUT * sizeof(double));
  int* ddiag = S.out(diag, b * go1mpc_body_diag_stride(nh) * sizeof(int));
  if (S.rc) return S.rc;
  // consecutive ticks of the same instances sit on different lanes: order them through the resident records
  {
    auto it = h->last_writer.find((const void*)out_d);
    if (it != h->last_writer.end()) CU(h, cudaStreamWaitEvent(L.stream, it->second, 0));
  }
  CU(h, body_record_expand_launch(B, nh, is, ts, os, tx_d, dtick, out_d, drec, h->sms, L.stream));
  h->launches++;
  int rc = go1mpc_body_mpc_step_batch(h, nh, B, drec, out_d, ddiag, L.stream);
  if (rc) return rc;
  CU(h, body_record_pack_launch(B, nh, os, out_d, dto, h->sms, L.stream));
  h->launches++;
  {
    cudaEvent_t& ev = h->last_writer[(const void*)out_d];
    if (!ev) CU(h, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CU(h, cudaEventRecord(ev, L.stream));
  }
  return S.finish(false);
}

int go1mpc_step_timing_step_batch_host_async(go1mpc_t* h, int n_sqp, int B, const int* tick, const double* state_d,
                                             double* state_out_d, const double* in, double* out, int* diag) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!tick || !state_d || !state_out_d || !in || !out) return fail(h, GO1MPC_E_INVALID, "step_timing_step_batch_host_async: bad argument");
  CU(h, cudaSetDevice(h->device));
  const size_t b = (size_t)B;
  go1mpc::Lane& L = h->lanes[h->lane_next++ % go1mpc::kLanes];
  // consecutive ticks of the same planners sit on different lanes: order them through the state buffers
  for (const void* key : {(const void*)state_d, (const void*)state_out_d}) {
    auto it = h->last_writer.find(key);
    if (it != h->last_writer.end()) CU(h, cudaStreamWaitEvent(L.stream, it->second, 0));
  }
  Staging S(h, L.step, L.stream);
  const int* dt_ = S.up(tick, b * sizeof(int));
  const double* di = S.up(in, b * STEP_IN_DOUBLES * sizeof(double));
  double* do_ = S.out(out, b * STEP_OUT_DOUBLES * sizeof(double));
  int* dd = S.out(diag, b * STEP_DIAG_INTS * sizeof(int));
  if (S.rc) return S.rc;
  int rc = go1mpc_step_timing_step_batch(h, n_sqp, B, dt_, state_d, state_out_d, di, do_, dd, L.stream);
  if (rc) return rc;
  // the buffer read and the buffer written: a later call on another lane that WRITES the state this call read must come after
  // it too (write-after-read when state_out_d != state_d)
  for (const void* key : {(const void*)state_out_d, (const void*)state_d}) {
    cudaEvent_t& ev = h->last_writer[key];
    if (!ev) CU(h, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CU(h, cudaEventRecord(ev, L.stream));
    if (state_out_d == state_d) break;
  }
  return S.finish(false);
}

// The pipelined entries order calls that share a device-resident buffer through an event kept per buffer address; a caller that
// frees such a buffer tells the handle, so that the entry does not outlive the allocation (and a new allocation at the same
// address does not inherit it)
int go1mpc_forget_buffer(go1mpc_t* h, const void* buf_d) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  auto it = h->last_writer.find(buf_d);
  if (it != h->last_writer.end()) {
    if (it->second) { cudaEventSynchronize(it->second); cudaEventDestroy(it->second); }
    h->last_writer.erase(it);
  }
  return GO1MPC_OK;
}

// ------------------------------------------------------------------ leg kinematics
int go1mpc_leg_fk_batch(go1mpc_t* h, int B, const double* q_d, const int* leg_d, const double* body_p_d, const double* body_r_d,
                        double* pos_d, double* jac_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !q_d || !leg_d || !pos_d || ((body_p_d == nullptr) != (body_r_d == nullptr)))
    return fail(h, GO1MPC_E_INVALID, "leg_fk_batch: bad argument");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  LegKParams P{};
  P.B = B; P.q_in = q_d; P.leg = leg_d; P.body_p = body_p_d; P.body_r = body_r_d; P.pos_out = pos_d; P.jac_out = jac_d;
  CU(h, leg_fk_launch(P, stream ? (cudaStream_t)stream : h->stream));
  h->launches++;
  return GO1MPC_OK;
}
int go1mpc_leg_ik_batch(go1mpc_t* h, int B, const double* pdes_d, const double* qini_d, const int* leg_d, const double* body_p_d,
                        const double* body_r_d, double* q_d, double* jac_d, int* iters_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !pdes_d || !qini_d || !leg_d || !q_d || ((body_p_d == nullptr) != (body_r_d == nullptr)))
    return fail(h, GO1MPC_E_INVALID, "leg_ik_batch: bad argument");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  LegKParams P{};
  P.B = B; P.q_in = qini_d; P.leg = leg_d; P.body_p = body_p_d; P.body_r = body_r_d; P.pdes = pdes_d;
  P.q_out = q_d; P.jac_out = jac_d; P.iters = iters_d;
  CU(h, leg_ik_launch(P, stream ? (cudaStream_t)stream : h->stream));
  h->launches++;
  return GO1MPC_OK;
}
int go1mpc_servo_kin_tick_batch(go1mpc_t* h, int B, int gait_mode, double y_offset, const double* com_d, const double* theta_d,
                                const double* rfoot_d, const double* lfoot_d, const double* homing_d, double* q_d, double* jac_d,
                                double* foot_des_d, int* iters_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !com_d || !theta_d || !rfoot_d || !lfoot_d || !homing_d || !q_d) return fail(h, GO1MPC_E_INVALID, "servo_kin_tick_batch: bad argument");
  if (gait_mode < 101 || gait_mode > 103) return fail(h, GO1MPC_E_UNSUPPORTED, "servo_kin_tick_batch: gait_mode 101, 102 or 103");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  ServoKParams P;
  P.B = B; P.gait_mode = gait_mode; P.half_hip_width = h->cfg.step.half_hip_width; P.y_offset = y_offset;
  P.com = com_d; P.theta = theta_d; P.rfoot = rfoot_d; P.lfoot = lfoot_d; P.homing = homing_d;
  P.q = q_d; P.jac = jac_d; P.foot_des = foot_des_d; P.iters = iters_d;
  CU(h, servo_kin_launch(P, stream ? (cudaStream_t)stream : h->stream));
  h->launches++;
  return GO1MPC_OK;
}
// ------------------------------------------------------------------ fused tick (planner -> swing foot -> body MPC -> servo IK)
int go1mpc_fused_tick_batch(go1mpc_t* h, int B, const Go1FusedTick* t, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (!t || B < 0) return fail(h, GO1MPC_E_INVALID, "fused_tick_batch: bad argument");
  if (!t->servo_theta_d || !t->out38_d || !t->out18_d || !t->body_out_d) return fail(h, GO1MPC_E_INVALID, "fused_tick_batch: bad argument");
  if (B == 0) return GO1MPC_OK;
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  int rc;
  if ((rc = go1mpc_step_timing_step_batch(h, t->n_sqp, B, t->tick_d, t->step_state_d, t->step_state_d, t->step_in_d, t->out38_d,
                                          t->step_diag_d, st))) return rc;
  if ((rc = go1mpc_foot_trajectory_batch(h, B, t->tick_d, t->step_state_d, t->out38_d, t->foot_d, t->out18_d, t->right_support_d, st))) return rc;
  if ((rc = go1mpc_body_mpc_step_batch(h, t->nh, B, t->body_in_d, t->body_out_d, t->body_diag_d, st))) return rc;
  CU(h, cudaSetDevice(h->device));
  CU(h, body_theta_gather_launch(B, t->body_out_d, go1mpc_body_out_stride(t->nh), t->servo_theta_d, st));
  h->launches++;
  // SoA: the CoM position is rows 0..2 of out38, the right / left foot positions rows 0..2 / 3..5 of out18
  if ((rc = go1mpc_servo_kin_tick_batch(h, B, t->gait_mode, t->y_offset, t->out38_d, t->servo_theta_d, t->out18_d,
                                        t->out18_d + (size_t)3 * B, t->homing_d, t->q_d, t->jac_d, t->foot_des_d, t->ik_iters_d, st))) return rc;
  // 5 (optional): force QP and torque map on the Jacobians stage 4 just wrote
  if (!t->grf_in_d) return GO1MPC_OK;
  if (!t->grf_out_d) return fail(h, GO1MPC_E_INVALID, "fused_tick_batch: grf_in_d without grf_out_d");
  if ((rc = go1mpc_grf_force_opt_batch(h, B, t->grf_in_d, t->grf_out_d, t->grf_diag_d, st))) return rc;
  if (!t->tau_d) return GO1MPC_OK;
  if (!t->jac_d) return fail(h, GO1MPC_E_INVALID, "fused_tick_batch: tau_d needs jac_d");
  return go1mpc_grf_joint_torques_batch(h, B, t->jac_d, t->swing_d, t->p_des_d, t->p_est_d, t->pv_des_d, t->pv_est_d, t->grf_out_d, 1,
                                        GRF_OUT_DOUBLES, t->tau_d, st);
}

int go1mpc_leg_fk_batch_host(go1mpc_t* h, int B, const double* q, const int* leg, const double* body_p, const double* body_r,
                             double* pos, double* jac) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!q || !leg || !pos || ((body_p == nullptr) != (body_r == nullptr))) return fail(h, GO1MPC_E_INVALID, "leg_fk_batch_host: bad argument");
  const size_t v3 = (size_t)B * 3 * sizeof(double);
  Staging S(h, h->stage, h->stream);
  const double* dq = S.up(q, v3);
  const int* dl = S.up(leg, (size_t)B * sizeof(int));
  const double* dbp = S.up(body_p, v3);
  const double* dbr = S.up(body_r, v3);
  double* dpos = S.out(pos, v3);
  double* dj = S.out(jac, 3 * v3);
  return S.run(true, [&] { return go1mpc_leg_fk_batch(h, B, dq, dl, dbp, dbr, dpos, dj, S.st); });
}
int go1mpc_leg_ik_batch_host(go1mpc_t* h, int B, const double* pdes, const double* qini, const int* leg, const double* body_p,
                             const double* body_r, double* q, double* jac, int* iters) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!pdes || !qini || !leg || !q || ((body_p == nullptr) != (body_r == nullptr))) return fail(h, GO1MPC_E_INVALID, "leg_ik_batch_host: bad argument");
  const size_t v3 = (size_t)B * 3 * sizeof(double), vi = (size_t)B * sizeof(int);
  Staging S(h, h->stage, h->stream);
  const double* dpdes = S.up(pdes, v3);
  const double* dqini = S.up(qini, v3);
  const int* dl = S.up(leg, vi);
  const double* dbp = S.up(body_p, v3);
  const double* dbr = S.up(body_r, v3);
  double* dq = S.out(q, v3);
  double* dj = S.out(jac, 3 * v3);
  int* dit = S.out(iters, vi);
  return S.run(true, [&] { return go1mpc_leg_ik_batch(h, B, dpdes, dqini, dl, dbp, dbr, dq, dj, dit, S.st); });
}

// ------------------------------------------------------------------ control tick with host inputs and compact results
int go1mpc_pack_compact_batch(go1mpc_t* h, int B, int nh, const double* out38_d, const int* step_diag_d, const double* body_out_d,
                              const int* body_diag_d, double* compact_d, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B < 0 || !out38_d || !body_out_d || !compact_d) return fail(h, GO1MPC_E_INVALID, "pack_compact_batch: bad argument");
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "pack_compact_batch: 3 <= nh <= 40");
  if (((uintptr_t)body_out_d & 15) || ((uintptr_t)compact_d & 15)) return fail(h, GO1MPC_E_INVALID, "pack_compact_batch: 16-byte alignment");
  if (B == 0) return GO1MPC_OK;
  CU(h, cudaSetDevice(h->device));
  CU(h, compact_pack_launch(B, nh, go1mpc_body_out_stride(nh), go1mpc_body_diag_stride(nh), out38_d, step_diag_d, body_out_d, body_diag_d,
                            compact_d, h->sms, stream ? (cudaStream_t)stream : h->stream));
  h->launches++;
  return GO1MPC_OK;
}

int go1mpc_control_tick_host_async(go1mpc_t* h, int B, const Go1ControlTick* t, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!t || !t->tick || !t->step_in || !t->body_tick_in || !t->step_state_d || !t->tx_d || !t->body_out_d || !t->compact_d)
    return fail(h, GO1MPC_E_INVALID, "control_tick_host_async: bad argument");
  const int nh = t->nh;
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "control_tick_host_async: 3 <= nh <= 40");
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  StreamWs* W;
  int rc = stream_ws(h, st, &W);
  if (rc) return rc;
  auto& ws = W->control;
  const size_t b = (size_t)B;
  const int is = go1mpc_body_in_stride(nh), os = go1mpc_body_out_stride(nh), ts = go1mpc_body_tick_in_stride(nh), ds = go1mpc_body_diag_stride(nh);
  const size_t tb = b * sizeof(int), tib = b * ts * sizeof(double), ob = b * STEP_OUT_DOUBLES * sizeof(double);
  const size_t sdb = b * STEP_DIAG_INTS * sizeof(int), bdb = b * ds * sizeof(int);
  const int in_rows = (t->step_in_rows > 0 && t->step_in_rows < STEP_IN_DOUBLES) ? t->step_in_rows : STEP_IN_DOUBLES;
  if (in_rows < STEP_IN_DOUBLES && (in_rows < 10 || h->cfg.step.ext_height))
    return fail(h, GO1MPC_E_INVALID, "control_tick_host_async: step_in_rows must cover the 10 sensor rows, and all 20 with cfg.step.ext_height");
  bool fresh = false;   // the planner input buffer was (re)allocated
  if ((rc = grow(h, ws.tick, tb, st)) || (rc = grow(h, ws.step_in, b * STEP_IN_DOUBLES * sizeof(double), st, &fresh)) ||
      (rc = grow(h, ws.body_tick_in, tib, st)) || (rc = grow(h, ws.body_in, b * is * sizeof(double), st)) ||
      (rc = grow(h, ws.out38, ob, st)) || (rc = grow(h, ws.step_diag, sdb, st)) || (rc = grow(h, ws.body_diag, bdb, st)))
    return rc;
  if (fresh) ws.zero_B = -1;
  int* tick = (int*)ws.tick.p;
  double* step_in = (double*)ws.step_in.p;
  double* body_tick_in = (double*)ws.body_tick_in.p;
  double* body_in = (double*)ws.body_in.p;
  double* out38 = (double*)ws.out38.p;
  int* step_diag = (int*)ws.step_diag.p;
  int* body_diag = (int*)ws.body_diag.p;
  if (in_rows < STEP_IN_DOUBLES) {
    // rows a partial upload does not carry read as zero (flat ground, no external heights): cleared once per batch size
    if (ws.zero_B != B) {
      CU(h, cudaMemsetAsync(step_in + b * in_rows, 0, b * (STEP_IN_DOUBLES - in_rows) * sizeof(double), st));
      ws.zero_B = B;
    }
  } else {
    ws.zero_B = -1;
  }
  CU(h, cudaMemcpyAsync(tick, t->tick, tb, cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(step_in, t->step_in, b * in_rows * sizeof(double), cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(body_tick_in, t->body_tick_in, tib, cudaMemcpyHostToDevice, st));
  // planner tick: out of place from the pristine state when the caller gives one (replays of the same tick), else in place
  const double* src = t->step_state_src_d ? t->step_state_src_d : t->step_state_d;
  if ((rc = go1mpc_step_timing_step_batch(h, t->n_sqp, B, tick, src, t->step_state_d, step_in, out38, step_diag, st))) return rc;
  // body tick on the resident records
  CU(h, body_record_expand_launch(B, nh, is, ts, os, t->tx_d, body_tick_in, t->body_out_d, body_in, h->sms, st));
  h->launches++;
  if ((rc = go1mpc_body_mpc_step_batch(h, nh, B, body_in, t->body_out_d, body_diag, st))) return rc;
  CU(h, compact_pack_launch(B, nh, os, ds, out38, step_diag, t->body_out_d, body_diag, t->compact_d, h->sms, st));
  h->launches++;
  if (t->out38) CU(h, cudaMemcpyAsync(t->out38, out38, ob, cudaMemcpyDeviceToHost, st));
  if (t->step_diag) CU(h, cudaMemcpyAsync(t->step_diag, step_diag, sdb, cudaMemcpyDeviceToHost, st));
  if (t->body_diag) CU(h, cudaMemcpyAsync(t->body_diag, body_diag, bdb, cudaMemcpyDeviceToHost, st));
  if (t->compact) CU(h, cudaMemcpyAsync(t->compact, t->compact_d, b * GO1MPC_COMPACT_DOUBLES * sizeof(double), cudaMemcpyDeviceToHost, st));
  return GO1MPC_OK;
}

// ------------------------------------------------------------------ stream ordering and CUDA-graph capture of tick sequences
int go1mpc_stream_wait(go1mpc_t* h, void* waiter, void* signaller) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  CU(h, cudaSetDevice(h->device));
  cudaEvent_t e = h->ev_pool[h->ev_next++ % h->ev_pool.size()];
  CU(h, cudaEventRecord(e, signaller ? (cudaStream_t)signaller : h->stream));
  CU(h, cudaStreamWaitEvent(waiter ? (cudaStream_t)waiter : h->stream, e, 0));
  return GO1MPC_OK;
}
int go1mpc_graph_capture_begin(go1mpc_t* h, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  CU(h, cudaSetDevice(h->device));
  CU(h, cudaStreamBeginCapture(stream ? (cudaStream_t)stream : h->stream, cudaStreamCaptureModeThreadLocal));
  return GO1MPC_OK;
}
int go1mpc_graph_capture_end(go1mpc_t* h, void* stream, void** graph_exec_out) {
  if (!h || !graph_exec_out) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  *graph_exec_out = nullptr;
  cudaGraph_t g = nullptr;
  CU(h, cudaStreamEndCapture(stream ? (cudaStream_t)stream : h->stream, &g));
  cudaGraphExec_t ge = nullptr;
  cudaError_t e = cudaGraphInstantiate(&ge, g, 0);
  cudaGraphDestroy(g);
  if (e != cudaSuccess) return cuda_fail(h, e, "cudaGraphInstantiate");
  cudaGraphUpload(ge, stream ? (cudaStream_t)stream : h->stream);      // so that the first launch does not pay for it
  *graph_exec_out = (void*)ge;
  return GO1MPC_OK;
}
int go1mpc_graph_launch(go1mpc_t* h, void* graph_exec, void* stream) {
  if (!h || !graph_exec) return GO1MPC_E_INVALID;
  CU(h, cudaSetDevice(h->device));
  CU(h, cudaGraphLaunch((cudaGraphExec_t)graph_exec, stream ? (cudaStream_t)stream : h->stream));
  return GO1MPC_OK;
}
int go1mpc_graph_destroy(go1mpc_t* h, void* graph_exec) {
  if (!h) return GO1MPC_E_INVALID;
  if (graph_exec) CU(h, cudaGraphExecDestroy((cudaGraphExec_t)graph_exec));
  return GO1MPC_OK;
}

int go1mpc_measure_dfma_peak(go1mpc_t* h, int ms, double* gflops) {
  if (!h || !gflops) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  CU(h, cudaSetDevice(h->device));
  double* sink;
  CU(h, cudaMalloc(&sink, sizeof(double)));
  cudaEvent_t e0, e1;
  CU(h, cudaEventCreate(&e0));
  CU(h, cudaEventCreate(&e1));
  const int grid = h->sms * 8, block = 256;
  int iters = 2000;
  double best = 0.0, elapsed_total = 0.0;
  CU(h, dfma_peak_launch(grid, block, 200, sink, h->stream));   // warm-up
  h->launches++;
  for (int rep = 0; rep < 64 && elapsed_total < ms; rep++) {
    CU(h, cudaEventRecord(e0, h->stream));
    CU(h, dfma_peak_launch(grid, block, iters, sink, h->stream));
    CU(h, cudaEventRecord(e1, h->stream));
    CU(h, cudaEventSynchronize(e1));
    h->launches++;
    float t_ms = 0.f;
    CU(h, cudaEventElapsedTime(&t_ms, e0, e1));
    elapsed_total += t_ms;
    double flops = (double)grid * block * (double)iters * 64.0 * 2.0;
    double gf = flops / (t_ms * 1e-3) * 1e-9;
    if (gf > best) best = gf;
    if (t_ms < 2.0f) iters *= 4;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(sink);
  *gflops = best;
  return GO1MPC_OK;
}

}  // extern "C"
