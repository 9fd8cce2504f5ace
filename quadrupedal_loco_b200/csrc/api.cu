// api.cu -- C ABI of libgo1mpc.so (include/go1mpc.h): handle, model tables, launches.
//
// Host side of the boundary.  No CPU compute path exists here: every entry point
// either launches the sm_100a kernels or fails with an error code.
#include <cuda_runtime.h>
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

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
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
  // one and the D2H copy of the one before that
  struct Lane { cudaStream_t stream = nullptr; DevBuf stage[12]; };
  static const int kLanes = 8;
  Lane lanes[8];
  unsigned lane_next = 0;
  // device-resident buffers the pipelined calls read AND write (planner state): the last
  // enqueued writer per buffer, so that a later call on another lane is ordered after it
  std::map<const void*, cudaEvent_t> last_writer;
  // per caller stream: {next, done} scheduler counters of the persistent body kernels and the hand-over list
  // {count, total, ids[kFlistCap]}.  Keyed by stream because launches on one stream are ordered, so a block is idle
  // again when the next launch on that stream starts; launches on different streams never share counters.
  struct StreamCtl { int* p = nullptr; };
  std::map<cudaStream_t, StreamCtl> ctl;
  // staging of go1mpc_control_tick_host_async, one set per caller stream (grown on demand): tick | step_in | body tick
  // records | expanded body records | out38 | planner diag | body diag
  struct TickWs { DevBuf b[7]; int zero_B = -1; };   // zero_B: batch size for which rows 10..19 of the planner inputs are known zero
  std::map<cudaStream_t, TickWs> tick_ws;
  cudaStream_t side = nullptr;     // side stream of the planner tick's out-of-place state copy
  bool phase_timing = false;       // go1mpc_body_phase_timing: events around the three launches of the body tick
  cudaEvent_t phase_ev[4] = {nullptr, nullptr, nullptr, nullptr};
  double* squat_d = nullptr;       // X_CoM_position_squat table of the planner node (host libm), built on first use
  struct NlpWs { DevBuf b[7]; };   // workspace of go1mpc_nlp_node_tick_batch, one per caller stream
  std::map<cudaStream_t, NlpWs> nlp_ws;
  // workspace of the gait stack entries, one per caller stream (grown on demand): sensor | /control2rtmpc/state |
  // walkdtime ints | cmd | start | body-MPC input records | planner mask of the clocked tick | reset count, flags and robot list |
  // farm copy count and lists
  struct StackWs { DevBuf b[9]; int zero_B = -1; };   // zero_B: batch size for which the control message's other slots are zero
  std::map<cudaStream_t, StackWs> stack_ws;
  struct ServoWs { DevBuf ch, reset; };   // servo torque tick: filtered channels [SERVO_TICKS_MAX][9][B], reset flags [B]
  std::map<cudaStream_t, ServoWs> servo_ws;
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
  // body_tri workspace, one per stream the entry point is called with (calls on one stream are ordered, so the
  // buffers are free again when the next call's first kernel starts); grown on demand
  struct TriWs { char* p = nullptr; int capB = 0; size_t off[6] = {0, 0, 0, 0, 0, 0}; size_t qctl_off = 0; };
  std::map<cudaStream_t, TriWs> tri_ws;
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

// scheduler counters + hand-over list of the stream `st` (allocated and zeroed on first use)
int get_ctl(go1mpc* h, cudaStream_t st, int** out) {
  auto it = h->ctl.find(st);
  if (it == h->ctl.end()) {
    if (h->ctl.size() >= 256) return fail(h, GO1MPC_E_UNSUPPORTED, "more than 256 distinct streams used with one handle");
    int* p = nullptr;
    const size_t bytes = sizeof(int) * (size_t)(kFlistCap + 4);
    CU(h, cudaMalloc((void**)&p, bytes));
    cudaError_t e = cudaMemset(p, 0, bytes);
    if (e != cudaSuccess) { cudaFree(p); return cuda_fail(h, e, "cudaMemset(stream control block)"); }
    it = h->ctl.emplace(st, go1mpc::StreamCtl{p}).first;
  }
  *out = it->second.p;
  return GO1MPC_OK;
}

int stage_buf2(go1mpc* h, DevBuf& b, size_t bytes, void** out);
int stage_buf(go1mpc* h, int slot, size_t bytes, void** out) { return stage_buf2(h, h->stage[slot], bytes, out); }
int stage_buf2(go1mpc* h, DevBuf& b, size_t bytes, void** out) {
  if (bytes > b.cap) {
    if (b.p) cudaFree(b.p);
    b.p = nullptr; b.cap = 0;
    size_t cap = bytes + bytes / 4 + 256;
    CU(h, cudaMalloc(&b.p, cap));
    b.cap = cap;
  }
  *out = b.p;
  return GO1MPC_OK;
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
  for (DevBuf& b : h->stage) if (b.p) cudaFree(b.p);
  for (auto& kv : h->ctl) if (kv.second.p) cudaFree(kv.second.p);
  for (auto& kv : h->tri_ws) if (kv.second.p) cudaFree(kv.second.p);
  for (auto& kv : h->last_writer) cudaEventDestroy(kv.second);
  for (auto& kv : h->tick_ws) for (DevBuf& b : kv.second.b) if (b.p) cudaFree(b.p);
  for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
  if (h->trtab_d) cudaFree(h->trtab_d);
  if (h->squat_d) cudaFree(h->squat_d);
  for (cudaEvent_t e : h->phase_ev) if (e) cudaEventDestroy(e);
  for (auto& kv : h->nlp_ws) for (DevBuf& b : kv.second.b) if (b.p) cudaFree(b.p);
  for (auto& kv : h->stack_ws) for (DevBuf& b : kv.second.b) if (b.p) cudaFree(b.p);
  for (auto& kv : h->servo_ws) for (DevBuf* b : {&kv.second.ch, &kv.second.reset}) if (b->p) cudaFree(b->p);
  for (auto& kv : h->stack_col_d) cudaFree(kv.second);
  for (auto& L : h->lanes) {
    for (DevBuf& b : L.stage) if (b.p) cudaFree(b.p);
    if (L.stream) cudaStreamDestroy(L.stream);
  }
  if (h->side) cudaStreamDestroy(h->side);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
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
  CU(h, cudaSetDevice(h->device));
  const size_t szd = sizeof(double), szi = sizeof(int), b = (size_t)B;
  void *dG, *dg0, *dCE = nullptr, *dce0 = nullptr, *dCI = nullptr, *dci0 = nullptr, *dx, *dcost, *dact, *dna, *dit, *dst;
  int rc;
  if ((rc = stage_buf(h, 0, b * n * n * szd, &dG))) return rc;
  if ((rc = stage_buf(h, 1, b * n * szd, &dg0))) return rc;
  if (p) { if ((rc = stage_buf(h, 2, b * n * p * szd, &dCE))) return rc; if ((rc = stage_buf(h, 3, b * p * szd, &dce0))) return rc; }
  if (m) { if ((rc = stage_buf(h, 4, b * n * m * szd, &dCI))) return rc; if ((rc = stage_buf(h, 5, b * m * szd, &dci0))) return rc; }
  if ((rc = stage_buf(h, 6, b * n * szd, &dx))) return rc;
  if ((rc = stage_buf(h, 7, b * szd, &dcost))) return rc;
  if ((rc = stage_buf(h, 8, b * (m + p + 1) * szi, &dact))) return rc;
  if ((rc = stage_buf(h, 9, b * szi, &dna))) return rc;
  if ((rc = stage_buf(h, 10, b * 6 * szi, &dit))) return rc;
  if ((rc = stage_buf(h, 11, b * szi, &dst))) return rc;
  cudaStream_t st = h->stream;
  CU(h, cudaMemcpyAsync(dG, G, b * n * n * szd, cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(dg0, g0, b * n * szd, cudaMemcpyHostToDevice, st));
  if (p) { CU(h, cudaMemcpyAsync(dCE, CE, b * n * p * szd, cudaMemcpyHostToDevice, st)); CU(h, cudaMemcpyAsync(dce0, ce0, b * p * szd, cudaMemcpyHostToDevice, st)); }
  if (m) { CU(h, cudaMemcpyAsync(dCI, CI, b * n * m * szd, cudaMemcpyHostToDevice, st)); CU(h, cudaMemcpyAsync(dci0, ci0, b * m * szd, cudaMemcpyHostToDevice, st)); }
  CU(h, cudaMemcpyAsync(dx, x, b * n * szd, cudaMemcpyHostToDevice, st));
  rc = go1mpc_qp_solve_batch(h, n, p, m, B, (double*)dG, (double*)dg0, (double*)dCE, (double*)dce0, (double*)dCI,
                             (double*)dci0, (double*)dx, (double*)dcost, (int*)dact, (int*)dna, (int*)dit, (int*)dst, st);
  if (rc) return rc;
  CU(h, cudaMemcpyAsync(x, dx, b * n * szd, cudaMemcpyDeviceToHost, st));
  if (cost) CU(h, cudaMemcpyAsync(cost, dcost, b * szd, cudaMemcpyDeviceToHost, st));
  if (active) CU(h, cudaMemcpyAsync(active, dact, b * (m + p) * szi, cudaMemcpyDeviceToHost, st));
  if (nactive) CU(h, cudaMemcpyAsync(nactive, dna, b * szi, cudaMemcpyDeviceToHost, st));
  if (iters) CU(h, cudaMemcpyAsync(iters, dit, b * 6 * szi, cudaMemcpyDeviceToHost, st));
  if (status) CU(h, cudaMemcpyAsync(status, dst, b * szi, cudaMemcpyDeviceToHost, st));
  CU(h, cudaStreamSynchronize(st));
  return GO1MPC_OK;
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
  const int is = go1mpc_body_in_stride(nh), os = go1mpc_body_out_stride(nh);
  if (body_fast_supported(nh) && !h->force_generic && h->body_mode != 4) {
    const Go1BodyMpcConfig& c = h->cfg.body;
    BodyKParams P;
    P.nh = nh; P.B = B; P.in_stride = is; P.out_stride = os; P.diag_stride = go1mpc_body_diag_stride(nh);
    P.tab_doubles = M->tab_doubles; P.warp_doubles = 0;
    P.cap_scale = h->cfg.qp_iter_cap_scale; P.gate = M->gate; P.nstepx = M->nstepx; P.nsum_mpc = M->nsum_mpc;
    P.in = in_d; P.out = out_d; P.diag = diag_d; P.tab = M->tab_d;
    int* ctl = nullptr;
    if ((rc = get_ctl(h, st, &ctl))) return rc;
    P.sched = ctl;
    P.flist = nullptr; P.flist_count = nullptr; P.flist_cap = 0;
    P.dt_mpc = c.dt_mpc; P.j_ini = c.j_ini; P.mass = c.mass; P.g = c.g; P.gama = c.gama_zmp;
    P.theta_lim = c.theta_lim; P.torque_lim = c.torque_lim;
    for (int k = 0; k < 4; k++) P.lamda[k] = c.lamda[k];
    if (body_tri_supported(nh) && (h->body_mode == 2 || (h->body_mode == 3 && B >= h->body_tri_min))) {
      if (h->tri_ws.size() >= 64 && h->tri_ws.find(st) == h->tri_ws.end()) {
        // a caller that keeps creating streams: drop the workspaces of the old ones (their work is done after the sync)
        CU(h, cudaDeviceSynchronize());
        for (auto& kv : h->tri_ws) if (kv.second.p) cudaFree(kv.second.p);
        h->tri_ws.clear();
      }
      go1mpc::TriWs& W = h->tri_ws[st];
      if (W.capB < B) {
        if (W.p) { CU(h, cudaStreamSynchronize(st)); cudaFree(W.p); W.p = nullptr; W.capB = 0; }
        const size_t bytes = body_tri_workspace_bytes(nh, B, W.off);
        W.qctl_off = bytes;
        CU(h, cudaMalloc((void**)&W.p, bytes + 16));
        CU(h, cudaMemsetAsync(W.p + W.qctl_off, 0, 16, st));
        W.capB = B;
      }
      P.tri_jb = (double*)(W.p + W.off[0]); P.tri_hs = (double*)(W.p + W.off[1]); P.tri_res = (double*)(W.p + W.off[2]);
      P.tri_queue = (int*)(W.p + W.off[3]); P.tri_qctl = (int*)(W.p + W.qctl_off); P.tri_meta = (int*)(W.p + W.off[4]); P.tri_fr = (double*)(W.p + W.off[5]);
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
  size_t smem = body_smem_bytes(nh, wpc, is, os, M->tab_doubles, &wd);
  while (wpc > 1 && smem > h->smem_optin / 2) { wpc >>= 1; smem = body_smem_bytes(nh, wpc, is, os, M->tab_doubles, &wd); }
  if (smem > h->smem_optin) return fail(h, GO1MPC_E_UNSUPPORTED, "body_mpc_step_batch: workspace exceeds shared memory");
  int occ = 0;
  CU(h, body_mpc_occupancy(wpc, smem, &occ));
  if (occ < 1) return fail(h, GO1MPC_E_UNSUPPORTED, "body_mpc_step_batch: kernel does not fit on an SM");
  int grid = (B + wpc - 1) / wpc;
  if (grid > h->sms * occ) grid = h->sms * occ;
  const Go1BodyMpcConfig& c = h->cfg.body;
  BodyKParams P;
  P.nh = nh; P.B = B; P.in_stride = is; P.out_stride = os; P.diag_stride = go1mpc_body_diag_stride(nh);
  P.tab_doubles = M->tab_doubles; P.warp_doubles = wd;
  P.cap_scale = h->cfg.qp_iter_cap_scale; P.gate = M->gate; P.nstepx = M->nstepx; P.nsum_mpc = M->nsum_mpc;
  P.in = in_d; P.out = out_d; P.diag = diag_d; P.tab = M->tab_d; P.sched = nullptr;
  P.flist = nullptr; P.flist_count = nullptr; P.flist_cap = 0;
  P.dt_mpc = c.dt_mpc; P.j_ini = c.j_ini; P.mass = c.mass; P.g = c.g; P.gama = c.gama_zmp;
  P.theta_lim = c.theta_lim; P.torque_lim = c.torque_lim;
  for (int k = 0; k < 4; k++) P.lamda[k] = c.lamda[k];
  if (duo) {
    int* ctl = nullptr;
    if ((rc = get_ctl(h, st, &ctl))) return rc;
    int* fl = ctl + 2;
    P.flist_count = fl; P.flist = fl + 2; P.flist_cap = kFlistCap;
    CU(h, body_duo_launch(P, h->sms, h->smem_optin, st));
    P.warp_doubles = wd;
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
  for (auto& kv : h->ctl) {
    int v = 0;
    CU(h, cudaMemcpy(&v, kv.second.p + 3, sizeof(int), cudaMemcpyDeviceToHost));
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
  for (auto& kv : h->tri_ws) {
    if (!kv.second.p) continue;
    int v = 0;
    CU(h, cudaMemcpy(&v, kv.second.p + kv.second.qctl_off + 8, sizeof(int), cudaMemcpyDeviceToHost));
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
  CU(h, cudaSetDevice(h->device));
  const size_t ib = (size_t)B * go1mpc_body_in_stride(nh) * sizeof(double);
  const size_t ob = (size_t)B * go1mpc_body_out_stride(nh) * sizeof(double);
  const size_t db = (size_t)B * go1mpc_body_diag_stride(nh) * sizeof(int);
  void *din, *dout, *ddiag = nullptr;
  int rc;
  if ((rc = stage_buf(h, 12, ib, &din))) return rc;
  if ((rc = stage_buf(h, 13, ob, &dout))) return rc;
  if (diag && (rc = stage_buf(h, 14, db, &ddiag))) return rc;
  cudaStream_t st = h->stream;
  CU(h, cudaMemcpyAsync(din, in, ib, cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(dout, out, ob, cudaMemcpyHostToDevice, st));   // out14 is in/out (gated ticks)
  rc = go1mpc_body_mpc_step_batch(h, nh, B, (const double*)din, (double*)dout, (int*)ddiag, st);
  if (rc) return rc;
  CU(h, cudaMemcpyAsync(out, dout, ob, cudaMemcpyDeviceToHost, st));
  if (diag) CU(h, cudaMemcpyAsync(diag, ddiag, db, cudaMemcpyDeviceToHost, st));
  CU(h, cudaStreamSynchronize(st));
  return GO1MPC_OK;
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
  CU(h, cudaSetDevice(h->device));
  const size_t b = (size_t)B;
  const size_t tb = b * sizeof(int), sb = b * STEP_STATE_DOUBLES * sizeof(double), ib = b * STEP_IN_DOUBLES * sizeof(double);
  const size_t ob = b * STEP_OUT_DOUBLES * sizeof(double), db = b * STEP_DIAG_INTS * sizeof(int);
  void *dt_, *ds, *di, *do_, *dd = nullptr;
  int rc;
  if ((rc = stage_buf(h, 0, tb, &dt_))) return rc;
  if ((rc = stage_buf(h, 1, sb, &ds))) return rc;
  if ((rc = stage_buf(h, 2, ib, &di))) return rc;
  if ((rc = stage_buf(h, 3, ob, &do_))) return rc;
  if (diag && (rc = stage_buf(h, 4, db, &dd))) return rc;
  cudaStream_t st = h->stream;
  CU(h, cudaMemcpyAsync(dt_, tick, tb, cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(ds, state, sb, cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(di, in, ib, cudaMemcpyHostToDevice, st));
  rc = go1mpc_step_timing_step_batch(h, n_sqp, B, (const int*)dt_, (const double*)ds, (double*)ds, (const double*)di, (double*)do_, (int*)dd, st);
  if (rc) return rc;
  CU(h, cudaMemcpyAsync(state, ds, sb, cudaMemcpyDeviceToHost, st));
  CU(h, cudaMemcpyAsync(out, do_, ob, cudaMemcpyDeviceToHost, st));
  if (diag) CU(h, cudaMemcpyAsync(diag, dd, db, cudaMemcpyDeviceToHost, st));
  CU(h, cudaStreamSynchronize(st));
  return GO1MPC_OK;
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
  CU(h, cudaSetDevice(h->device));
  const size_t b = (size_t)B, tb = b * sizeof(int), sb = b * STEP_STATE_DOUBLES * sizeof(double), ob = b * STEP_OUT_DOUBLES * sizeof(double);
  const size_t fb = b * FOOT_STATE_DOUBLES * sizeof(double), o18 = b * FOOT_OUT_DOUBLES * sizeof(double);
  void *dt_, *ds, *do_, *df, *d18, *drs = nullptr;
  int rc;
  if ((rc = stage_buf(h, 0, tb, &dt_))) return rc;
  if ((rc = stage_buf(h, 1, sb, &ds))) return rc;
  if ((rc = stage_buf(h, 3, ob, &do_))) return rc;
  if ((rc = stage_buf(h, 5, fb, &df))) return rc;
  if ((rc = stage_buf(h, 6, o18, &d18))) return rc;
  if (right_support && (rc = stage_buf(h, 7, tb, &drs))) return rc;
  void *dl0 = nullptr, *dstop = nullptr;
  const size_t lb = b * sizeof(double);
  if (lift0 && (rc = stage_buf(h, 8, lb, &dl0))) return rc;
  if (lift0 && stop && (rc = stage_buf(h, 9, lb, &dstop))) return rc;
  cudaStream_t st = h->stream;
  CU(h, cudaMemcpyAsync(dt_, tick, tb, cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(ds, state, sb, cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(do_, out38, ob, cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(df, foot, fb, cudaMemcpyHostToDevice, st));
  if (lift0) CU(h, cudaMemcpyAsync(dl0, lift0, lb, cudaMemcpyHostToDevice, st));
  if (dstop) CU(h, cudaMemcpyAsync(dstop, stop, lb, cudaMemcpyHostToDevice, st));
  rc = foot_enqueue(h, B, (const int*)dt_, (const double*)ds, (const double*)do_, (double*)df, (double*)d18, (int*)drs, st,
                    (double*)dl0, (const double*)dstop, lift0 ? go1mpc_nlp_t_end_footstep(h) : 0);
  if (rc) return rc;
  CU(h, cudaMemcpyAsync(foot, df, fb, cudaMemcpyDeviceToHost, st));
  CU(h, cudaMemcpyAsync(out18, d18, o18, cudaMemcpyDeviceToHost, st));
  if (right_support) CU(h, cudaMemcpyAsync(right_support, drs, tb, cudaMemcpyDeviceToHost, st));
  if (lift0) CU(h, cudaMemcpyAsync(lift0, dl0, lb, cudaMemcpyDeviceToHost, st));
  CU(h, cudaStreamSynchronize(st));
  return GO1MPC_OK;
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
  GrfKParams P;
  P.B = B; P.cap = h->cfg.qp_iter_cap_scale * (12 + 12 + 24) + 50; P.warp_doubles = 0;
  P.qp_alpha = 10000; P.qp_beta = 1000; P.qp_gama = 10; P.fz_max = 160; P.mu = 0.25;   // dynmics_compute.cpp:59-63
  P.in = in_d; P.out = out_d; P.diag = diag_d;
  CU(h, grf_force_opt_launch(P, h->sms, stream ? (cudaStream_t)stream : h->stream));
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
  P.B = B; P.swing_kp = 1; P.swing_kd = 0.01;   // dynmics_compute.cpp:37-38
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
  CU(h, cudaSetDevice(h->device));
  const size_t ib = (size_t)B * GRF_IN_DOUBLES * sizeof(double), ob = (size_t)B * GRF_OUT_DOUBLES * sizeof(double);
  const size_t db = (size_t)B * GRF_DIAG_INTS * sizeof(int);
  void *di, *do_, *dd = nullptr;
  int rc;
  if ((rc = stage_buf(h, 0, ib, &di))) return rc;
  if ((rc = stage_buf(h, 1, ob, &do_))) return rc;
  if (diag && (rc = stage_buf(h, 2, db, &dd))) return rc;
  cudaStream_t st = h->stream;
  CU(h, cudaMemcpyAsync(di, in, ib, cudaMemcpyHostToDevice, st));
  rc = go1mpc_grf_force_opt_batch(h, B, (const double*)di, (double*)do_, (int*)dd, st);
  if (rc) return rc;
  CU(h, cudaMemcpyAsync(out, do_, ob, cudaMemcpyDeviceToHost, st));
  if (diag) CU(h, cudaMemcpyAsync(diag, dd, db, cudaMemcpyDeviceToHost, st));
  CU(h, cudaStreamSynchronize(st));
  return GO1MPC_OK;
}
int go1mpc_grf_force_distribution_batch_host(go1mpc_t* h, int B, int gait_mode, double y_coefficient, const double* com_des,
                                             const double* leg_des, const double* F_force_des, const double* rfoot_des,
                                             const double* lfoot_des, double* F_leg_ref) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!com_des || !leg_des || !F_force_des || !rfoot_des || !lfoot_des || !F_leg_ref)
    return fail(h, GO1MPC_E_INVALID, "grf_force_distribution_batch_host: bad argument");
  CU(h, cudaSetDevice(h->device));
  const size_t d = (size_t)B * sizeof(double);
  const double* src[5] = {com_des, leg_des, F_force_des, rfoot_des, lfoot_des};
  const int rows[5] = {3, 12, 6, 3, 3};
  void* dev[6];
  int rc;
  cudaStream_t st = h->stream;
  for (int k = 0; k < 5; k++) {
    if ((rc = stage_buf(h, k, rows[k] * d, &dev[k]))) return rc;
    CU(h, cudaMemcpyAsync(dev[k], src[k], rows[k] * d, cudaMemcpyHostToDevice, st));
  }
  if ((rc = stage_buf(h, 5, 12 * d, &dev[5]))) return rc;
  rc = go1mpc_grf_force_distribution_batch(h, B, gait_mode, y_coefficient, (const double*)dev[0], (const double*)dev[1],
                                           (const double*)dev[2], (const double*)dev[3], (const double*)dev[4], (double*)dev[5], st);
  if (rc) return rc;
  CU(h, cudaMemcpyAsync(F_leg_ref, dev[5], 12 * d, cudaMemcpyDeviceToHost, st));
  CU(h, cudaStreamSynchronize(st));
  return GO1MPC_OK;
}
int go1mpc_grf_joint_torques_batch_host(go1mpc_t* h, int B, const double* jac, const int* swing, const double* p_des,
                                        const double* p_est, const double* pv_des, const double* pv_est,
                                        const double* F_leg_ref, long long F_elem_stride, long long F_robot_stride, double* tau) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!jac || !swing || !p_des || !p_est || !pv_des || !pv_est || !F_leg_ref || !tau || F_elem_stride < 0 || F_robot_stride < 0)
    return fail(h, GO1MPC_E_INVALID, "grf_joint_torques_batch_host: bad argument");
  CU(h, cudaSetDevice(h->device));
  const size_t d = (size_t)B * sizeof(double);
  const size_t fdoubles = (size_t)(11 * F_elem_stride + (B - 1) * F_robot_stride + 1);   // extent the strides address
  const void* src[7] = {jac, swing, p_des, p_est, pv_des, pv_est, F_leg_ref};
  const size_t bytes[7] = {36 * d, 4 * (size_t)B * sizeof(int), 12 * d, 12 * d, 12 * d, 12 * d, fdoubles * sizeof(double)};
  void* dev[8];
  int rc;
  cudaStream_t st = h->stream;
  for (int k = 0; k < 7; k++) {
    if ((rc = stage_buf(h, k, bytes[k], &dev[k]))) return rc;
    CU(h, cudaMemcpyAsync(dev[k], src[k], bytes[k], cudaMemcpyHostToDevice, st));
  }
  if ((rc = stage_buf(h, 7, 12 * d, &dev[7]))) return rc;
  rc = go1mpc_grf_joint_torques_batch(h, B, (const double*)dev[0], (const int*)dev[1], (const double*)dev[2], (const double*)dev[3],
                                      (const double*)dev[4], (const double*)dev[5], (const double*)dev[6], F_elem_stride,
                                      F_robot_stride, (double*)dev[7], st);
  if (rc) return rc;
  CU(h, cudaMemcpyAsync(tau, dev[7], 12 * d, cudaMemcpyDeviceToHost, st));
  CU(h, cudaStreamSynchronize(st));
  return GO1MPC_OK;
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
                     const double* rfoot_fb_d, const double* lfoot_fb_d, double* msg_d, const int* active_d, void* stream);
}
int go1mpc_nlp_node_tick_batch(go1mpc_t* h, int B, double* state_d, const int* walkdtime_d, const int* start_d, const int* cmd_d,
                               const double* rfoot_fb_d, const double* lfoot_fb_d, double* msg_d, void* stream) {
  return nlp_node_enqueue(h, B, state_d, walkdtime_d, start_d, cmd_d, rfoot_fb_d, lfoot_fb_d, msg_d, nullptr, stream);
}
namespace {
// active_d: [B] ints or null (= all); robots with 0 leave the node untouched (per-robot clocks of the gait stack)
int nlp_node_enqueue(go1mpc_t* h, int B, double* state_d, const int* walkdtime_d, const int* start_d, const int* cmd_d,
                     const double* rfoot_fb_d, const double* lfoot_fb_d, double* msg_d, const int* active_d, void* stream) {
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
  // per-stream workspace: tick | in | out38 | out18 | right_support | hz_co | lipm
  if (h->nlp_ws.size() >= 256 && h->nlp_ws.find(st) == h->nlp_ws.end())
    return fail(h, GO1MPC_E_UNSUPPORTED, "nlp_node_tick_batch: more than 256 distinct streams used with one handle");
  go1mpc::NlpWs& W = h->nlp_ws[st];
  const size_t need[7] = {(size_t)B * sizeof(int), (size_t)B * STEP_IN_DOUBLES * sizeof(double), (size_t)B * STEP_OUT_DOUBLES * sizeof(double),
                          (size_t)B * FOOT_OUT_DOUBLES * sizeof(double), (size_t)B * sizeof(int), (size_t)B * 8 * sizeof(double),
                          (size_t)B * 6 * sizeof(double)};
  for (int k = 0; k < 7; k++)
    if (W.b[k].cap < need[k]) {
      CU(h, cudaStreamSynchronize(st));
      if (W.b[k].p) CU(h, cudaFree(W.b[k].p));
      W.b[k].p = nullptr; W.b[k].cap = 0;
      CU(h, cudaMalloc(&W.b[k].p, need[k]));
      W.b[k].cap = need[k];
    }
  NlpKParams P;
  P.B = B;
  nlp_limits(h, &P.t_end, &P.walkdtime_max);
  P.dt = c.dt; P.dtx = kNlpDtx; P.height_offset_time = kNlpHeightOffsetTime; P.half_hip_width = c.half_hip_width;
  P.stepwidth0 = c.stepwidth0; P.mass = kNlpMass; P.rad = kNlpRad; P.ggg = c.ggg; P.z_c = c.hcom + kNlpHeightOffset;
  P.height_offset = kNlpHeightOffset; P.Wn = c.Wn;
  for (int q = 0; q < NLP_NTD_MAX; q++) { const double w = c.Wn * c.dt * (q + 1); P.sh_w[q] = sinh(w); P.ch_w[q] = cosh(w); }
  P.squat = h->squat_d; P.squat_n = kSquatN;
  P.node = state_d; P.walkdtime = walkdtime_d; P.start = start_d; P.cmd = cmd_d; P.rfoot_fb = rfoot_fb_d; P.lfoot_fb = lfoot_fb_d;
  P.tick = (int*)W.b[0].p; P.in = (double*)W.b[1].p; P.out38 = (double*)W.b[2].p; P.out18 = (double*)W.b[3].p;
  P.right_support = (int*)W.b[4].p; P.hz_co = (double*)W.b[5].p; P.lipm = (double*)W.b[6].p; P.msg = msg_d;
  P.active = active_d;
  CU(h, nlp_pre_launch(P, st));
  h->launches++;
  // the planner state is rows [0, 202) of the node, the swing-foot window rows [202, 234): same SoA stride B
  int rc = step_tick_enqueue(h, 3, B, P.tick, state_d, state_d, P.in, P.out38, nullptr, st, P.hz_co, P.lipm);
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
  CU(h, cudaSetDevice(h->device));
  const size_t b = (size_t)B, ib = b * sizeof(int), sb = b * NLP_NODE_DOUBLES * sizeof(double), fb = b * 3 * sizeof(double), mb = b * 100 * sizeof(double);
  void *ds, *dw, *dst_ = nullptr, *dc = nullptr, *drf = nullptr, *dlf = nullptr, *dm;
  int rc;
  if ((rc = stage_buf(h, 0, sb, &ds))) return rc;
  if ((rc = stage_buf(h, 1, ib, &dw))) return rc;
  if (start && (rc = stage_buf(h, 2, ib, &dst_))) return rc;
  if (cmd && (rc = stage_buf(h, 3, ib, &dc))) return rc;
  if (rfoot_fb && (rc = stage_buf(h, 4, fb, &drf))) return rc;
  if (lfoot_fb && (rc = stage_buf(h, 5, fb, &dlf))) return rc;
  if ((rc = stage_buf(h, 6, mb, &dm))) return rc;
  cudaStream_t st = h->stream;
  CU(h, cudaMemcpyAsync(ds, state, sb, cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(dw, walkdtime, ib, cudaMemcpyHostToDevice, st));
  if (start) CU(h, cudaMemcpyAsync(dst_, start, ib, cudaMemcpyHostToDevice, st));
  if (cmd) CU(h, cudaMemcpyAsync(dc, cmd, ib, cudaMemcpyHostToDevice, st));
  if (rfoot_fb) CU(h, cudaMemcpyAsync(drf, rfoot_fb, fb, cudaMemcpyHostToDevice, st));
  if (lfoot_fb) CU(h, cudaMemcpyAsync(dlf, lfoot_fb, fb, cudaMemcpyHostToDevice, st));
  rc = go1mpc_nlp_node_tick_batch(h, B, (double*)ds, (const int*)dw, (const int*)dst_, (const int*)dc, (const double*)drf,
                                  (const double*)dlf, (double*)dm, st);
  if (rc) return rc;
  CU(h, cudaMemcpyAsync(state, ds, sb, cudaMemcpyDeviceToHost, st));
  CU(h, cudaMemcpyAsync(msg, dm, mb, cudaMemcpyDeviceToHost, st));
  CU(h, cudaStreamSynchronize(st));
  return GO1MPC_OK;
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
  CU(h, cudaSetDevice(h->device));
  const size_t b = (size_t)B, sb = b * go1mpc_rt_node_state_doubles(nh) * sizeof(double), mb = b * 100 * sizeof(double);
  const size_t ib = b * sizeof(int), ab = b * 4 * sizeof(double), bib = b * go1mpc_body_in_stride(nh) * sizeof(double);
  const size_t bob = b * go1mpc_body_out_stride(nh) * sizeof(double);
  void *ds, *dm, *dc = nullptr, *da = nullptr, *dbi, *dbo, *dout;
  int rc;
  if ((rc = stage_buf(h, 0, sb, &ds))) return rc;
  if ((rc = stage_buf(h, 1, mb, &dm))) return rc;
  if (ctrl && (rc = stage_buf(h, 2, ib, &dc))) return rc;
  if (bodyangle_state && (rc = stage_buf(h, 3, ab, &da))) return rc;
  if ((rc = stage_buf(h, 4, bib, &dbi))) return rc;
  if ((rc = stage_buf(h, 5, bob, &dbo))) return rc;
  if ((rc = stage_buf(h, 6, mb, &dout))) return rc;
  cudaStream_t st = h->stream;
  CU(h, cudaMemcpyAsync(ds, state, sb, cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(dm, msg, mb, cudaMemcpyHostToDevice, st));
  if (ctrl) CU(h, cudaMemcpyAsync(dc, ctrl, ib, cudaMemcpyHostToDevice, st));
  if (bodyangle_state) CU(h, cudaMemcpyAsync(da, bodyangle_state, ab, cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(dbo, body_out, bob, cudaMemcpyHostToDevice, st));
  rc = go1mpc_rt_node_tick_batch(h, nh, B, (double*)ds, (const double*)dm, (const int*)dc, (const double*)da, (double*)dbi,
                                 (double*)dbo, nullptr, (double*)dout, nullptr, st);
  if (rc) return rc;
  CU(h, cudaMemcpyAsync(state, ds, sb, cudaMemcpyDeviceToHost, st));
  CU(h, cudaMemcpyAsync(body_out, dbo, bob, cudaMemcpyDeviceToHost, st));
  CU(h, cudaMemcpyAsync(out100, dout, mb, cudaMemcpyDeviceToHost, st));
  CU(h, cudaStreamSynchronize(st));
  return GO1MPC_OK;
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
int gait_stack_enqueue(go1mpc_t* h, int B, const Go1GaitStackTick* t, int* clock_d, void* stream, const char* name) {
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
  }
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  if (h->stack_ws.size() >= 256 && h->stack_ws.find(st) == h->stack_ws.end())
    return fail(h, GO1MPC_E_UNSUPPORTED, "more than 256 distinct streams used with one handle");
  go1mpc::StackWs& W = h->stack_ws[st];
  const size_t b = (size_t)B;
  const int nbuf = clock_d ? 7 : 6;
  const size_t bytes[7] = {b * GO1MPC_STACK_SENSOR_ROWS * sizeof(double), b * 25 * sizeof(double), b * sizeof(int), b * sizeof(int),
                           b * sizeof(int), b * go1mpc_body_in_stride(nh) * sizeof(double), b * sizeof(int)};
  void* d[7] = {};
  int rc;
  for (int k = 0; k < nbuf; k++) {
    const bool grow = bytes[k] > W.b[k].cap;
    if (grow) CU(h, cudaStreamSynchronize(st));     // growing: earlier work on this stream may still use the old buffer
    if ((rc = stage_buf2(h, W.b[k], bytes[k], &d[k]))) return rc;
    if (grow && k == 1) W.zero_B = -1;
  }
  double* ctl = (double*)d[1];
  if (W.zero_B != B) {
    // the 14 slots of /control2rtmpc/state the stack does not upload read as zero: cleared once per batch size
    CU(h, cudaMemsetAsync(ctl, 0, bytes[1], st));
    W.zero_B = B;
  }
  double* state = t->state_d;
  // device inputs are read in place; host inputs go up into the stream's staging buffers
  const double* sensor = t->sensor_d;
  if (!sensor) { CU(h, cudaMemcpyAsync(d[0], t->sensor, bytes[0], cudaMemcpyHostToDevice, st)); sensor = (const double*)d[0]; }
  // with per-robot clocks some robot may plan in any call, so cmd / start go up whenever they are given
  const bool planner = clock_d || t->planner;
  const int* cmd_d = t->cmd_d;
  const int* start_d = t->start_d;
  if (planner && t->cmd) { CU(h, cudaMemcpyAsync(d[3], t->cmd, bytes[3], cudaMemcpyHostToDevice, st)); cmd_d = (const int*)d[3]; }
  if (planner && t->start) { CU(h, cudaMemcpyAsync(d[4], t->start, bytes[4], cudaMemcpyHostToDevice, st)); start_d = (const int*)d[4]; }
  int* plan_d = (int*)d[6];
  if (clock_d)
    CU(h, gait_stack_clocked_pre_launch(B, clock_d, plan_d, state + GO1MPC_STACK_ROW_WALKDTIME * b, (int*)d[2], sensor, ctl, h->sms, st));
  else
    CU(h, gait_stack_pre_launch(B, t->planner ? 1 : 0, state + GO1MPC_STACK_ROW_WALKDTIME * b, (int*)d[2], sensor, ctl, h->sms, st));
  h->launches++;
  double* gait = state + GO1MPC_STACK_ROW_GAIT * b;
  double* rt2nrt = state + GO1MPC_STACK_ROW_RT2NRT * b;
  double* traj = state + GO1MPC_STACK_ROW_TRAJ * b;
  if (planner &&
      (rc = nlp_node_enqueue(h, B, state + GO1MPC_STACK_ROW_NLP * b, (const int*)d[2], start_d, cmd_d, rt2nrt + 22 * b, rt2nrt + 19 * b,
                             gait, clock_d ? plan_d : nullptr, st)))
    return rc;
  if ((rc = rt_node_enqueue(h, nh, B, state + GO1MPC_STACK_ROW_RT * b, gait, nullptr, nullptr, ctl, (double*)d[5], t->body_out_d, nullptr,
                            traj, rt2nrt, nullptr, st)))
    return rc;
  CU(h, gait_stack_pack_launch(S, B, gait, traj, t->rows_d, h->sms, st));
  h->launches++;
  if (t->rows) CU(h, cudaMemcpyAsync(t->rows, t->rows_d, b * n * sizeof(double), cudaMemcpyDeviceToHost, st));
  return GO1MPC_OK;
}
}  // namespace

int go1mpc_gait_stack_tick_host_async(go1mpc_t* h, int B, const Go1GaitStackTick* t, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  return gait_stack_enqueue(h, B, t, nullptr, stream, "gait_stack_tick_host_async");
}

int go1mpc_gait_stack_tick_clocked_async(go1mpc_t* h, int B, const Go1GaitStackClockedTick* t, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!t || !t->clock_d) return fail(h, GO1MPC_E_INVALID, "gait_stack_tick_clocked_async: bad argument");
  Go1GaitStackTick u;
  u.nh = t->nh; u.planner = 0; u.sensor = t->sensor; u.cmd = t->cmd; u.start = t->start; u.state_d = t->state_d;
  u.body_out_d = t->body_out_d; u.n_slots = t->n_slots; u.rows_d = t->rows_d; u.rows = t->rows;
  u.sensor_d = t->sensor_d; u.cmd_d = t->cmd_d; u.start_d = t->start_d;
  memcpy(u.slots, t->slots, sizeof u.slots);
  return gait_stack_enqueue(h, B, &u, t->clock_d, stream, "gait_stack_tick_clocked_async");
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
  if (h->stack_ws.size() >= 256 && h->stack_ws.find(st) == h->stack_ws.end())
    return fail(h, GO1MPC_E_UNSUPPORTED, "more than 256 distinct streams used with one handle");
  go1mpc::StackWs& W = h->stack_ws[st];
  // {count, 3 pad, flags[B], list[B]}
  const size_t b = (size_t)B, bytes = (4 + 2 * b) * sizeof(int);
  if (bytes > W.b[7].cap) CU(h, cudaStreamSynchronize(st));
  void* ws;
  int rc;
  if ((rc = stage_buf2(h, W.b[7], bytes, &ws))) return rc;
  StackResetParams P;
  P.B = B; P.rows = rows; P.out_stride = go1mpc_body_out_stride(nh);
  P.count = (int*)ws; P.reset = r->reset_d ? r->reset_d : P.count + 4; P.list = P.count + 4 + B;
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
  if (!D.clock_d != !S.clock_d || !D.servo_state_d != !S.servo_state_d || !D.force_state_d != !S.force_state_d)
    return fail(h, GO1MPC_E_INVALID, "farm_copy_async: clock_d, servo_state_d and force_state_d must be given on both sides or neither");
  if (((uintptr_t)D.body_out_d | (uintptr_t)S.body_out_d) & 15)
    return fail(h, GO1MPC_E_INVALID, "farm_copy_async: body_out_d must be 16-byte aligned");
  const int nh = c->nh;
  if (nh < 3 || nh > GO1MPC_BODY_NH_MAX) return fail(h, GO1MPC_E_UNSUPPORTED, "farm_copy_async: 3 <= nh <= 40");
  const int rows = go1mpc_gait_stack_state_doubles(nh), out_stride = go1mpc_body_out_stride(nh);
  // the kernels read the source while they write the destination: no destination block may share a byte with a source block
  auto blocks = [&](const Go1FarmColumns& F, uintptr_t* lo, uintptr_t* hi) {
    const size_t b = (size_t)F.B;
    const void* p[5] = {F.state_d, F.body_out_d, F.clock_d, F.servo_state_d, F.force_state_d};
    const size_t n[5] = {b * rows * sizeof(double), b * out_stride * sizeof(double), b * sizeof(int), b * SERVO_STATE_ROWS * sizeof(double),
                         b * SERVO_FORCE_ROWS * sizeof(double)};
    for (int k = 0; k < 5; k++) { lo[k] = (uintptr_t)p[k]; hi[k] = p[k] ? lo[k] + n[k] : lo[k]; }
  };
  uintptr_t dlo[5], dhi[5], slo[5], shi[5];
  blocks(D, dlo, dhi);
  blocks(S, slo, shi);
  for (int i = 0; i < 5; i++)
    for (int k = 0; k < 5; k++)
      if (dlo[i] < shi[k] && slo[k] < dhi[i])
        return fail(h, GO1MPC_E_INVALID, "farm_copy_async: a destination block overlaps a source block");
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  if (h->stack_ws.size() >= 256 && h->stack_ws.find(st) == h->stack_ws.end())
    return fail(h, GO1MPC_E_UNSUPPORTED, "more than 256 distinct streams used with one handle");
  go1mpc::StackWs& W = h->stack_ws[st];
  // {count, 3 pad, destination list[dst.B], source list[dst.B]}
  const size_t bytes = (4 + 2 * (size_t)D.B) * sizeof(int);
  if (bytes > W.b[8].cap) CU(h, cudaStreamSynchronize(st));
  void* ws;
  int rc;
  if ((rc = stage_buf2(h, W.b[8], bytes, &ws))) return rc;
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
  P.count = (int*)ws; P.dlist = P.count + 4; P.slist = P.count + 4 + D.B;
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
  P.jac = t->jac_d; P.foot_des = t->foot_des_d; P.iters = t->iters_d; P.ch = nullptr;
  CU(h, servo_stack_launch(P, st));
  h->launches++;
  if (t->q) CU(h, cudaMemcpyAsync(t->q, t->q_d, b * 12 * t->K * sizeof(double), cudaMemcpyDeviceToHost, st));
  return GO1MPC_OK;
}

// ------------------------------------------------------------------ servo torque tick: the servo stack + force QP + torque map
static_assert(GO1MPC_SERVO_FORCE_ROWS == SERVO_FORCE_ROWS, "servo force state layout");
int go1mpc_servo_torque_tick_async(go1mpc_t* h, int B, const Go1ServoTorqueTick* t, void* stream) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!t || !t->stack_state_d || !t->servo_state_d || !t->q_d || !t->force_state_d || !t->meas_d || !t->tau_d)
    return fail(h, GO1MPC_E_INVALID, "servo_torque_tick_async: bad argument");
  if (t->K < 1 || t->K > GO1MPC_SERVO_TICKS_MAX) return fail(h, GO1MPC_E_INVALID, "servo_torque_tick_async: 1 <= K <= 10");
  if (((uintptr_t)t->q_d | (uintptr_t)t->tau_d) & 7)
    return fail(h, GO1MPC_E_INVALID, "servo_torque_tick_async: q_d and tau_d must be 8-byte aligned");
  if (t->gait_mode < 101 || t->gait_mode > 103) return fail(h, GO1MPC_E_UNSUPPORTED, "servo_torque_tick_async: gait_mode 101, 102 or 103");
  if (t->reset && t->reset_d) return fail(h, GO1MPC_E_INVALID, "servo_torque_tick_async: at most one of reset / reset_d");
  if ((uintptr_t)t->reset_d & 3) return fail(h, GO1MPC_E_INVALID, "servo_torque_tick_async: reset_d must be 4-byte aligned");
  {
    const size_t b = (size_t)B, kb = b * 12 * t->K * sizeof(double);
    if (overlaps_written(t->reset_d, b * sizeof(int),
                         {{t->force_state_d, b * SERVO_FORCE_ROWS * sizeof(double)}, {t->servo_state_d, b * SERVO_STATE_ROWS * sizeof(double)},
                          {t->q_d, kb}, {t->tau_d, kb}}))
      return fail(h, GO1MPC_E_INVALID, "servo_torque_tick_async: reset_d overlaps force_state_d, servo_state_d, q_d or tau_d");
  }
  CU(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  if (h->servo_ws.size() >= 256 && h->servo_ws.find(st) == h->servo_ws.end())
    return fail(h, GO1MPC_E_UNSUPPORTED, "more than 256 distinct streams used with one handle");
  go1mpc::ServoWs& W = h->servo_ws[st];
  const size_t b = (size_t)B;
  // sized for K = GO1MPC_SERVO_TICKS_MAX, so that K changes do not reallocate; a growing buffer may still be read by the
  // stream's previous call
  const size_t chb = b * SERVO_TICKS_MAX * SERVO_LPF_CHANNELS * sizeof(double), rb = b * sizeof(int);
  if (chb > W.ch.cap || (t->reset && rb > W.reset.cap)) CU(h, cudaStreamSynchronize(st));
  void *ch, *rst = nullptr;
  int rc;
  if ((rc = stage_buf2(h, W.ch, chb, &ch))) return rc;
  if (t->reset && (rc = stage_buf2(h, W.reset, rb, &rst))) return rc;
  ServoStackKParams S;
  S.B = B; S.K = t->K; S.gait_mode = t->gait_mode;
  S.half_hip_width = h->cfg.step.half_hip_width; S.y_offset = t->y_offset;
  double k6[6];
  go1mpc_lpf_coefficients(1000.0, 3.0, k6);
  S.coef = LpfCoef{k6[0], k6[1], k6[2], k6[3], k6[4], k6[5]};
  S.gait = t->stack_state_d + GO1MPC_STACK_ROW_GAIT * b;
  S.traj = t->stack_state_d + GO1MPC_STACK_ROW_TRAJ * b;
  S.state = t->servo_state_d; S.q_out = t->q_d;
  S.jac = t->jac_d; S.foot_des = t->foot_des_d; S.iters = t->iters_d; S.ch = (double*)ch;
  ServoTorqueKParams P;
  P.g.B = B; P.g.cap = h->cfg.qp_iter_cap_scale * (12 + 12 + 24) + 50; P.g.warp_doubles = 0;
  P.g.qp_alpha = 10000; P.g.qp_beta = 1000; P.g.qp_gama = 10; P.g.fz_max = 160; P.g.mu = 0.25;   // as go1mpc_grf_force_opt_batch
  P.g.in = nullptr; P.g.out = nullptr; P.g.diag = nullptr;
  P.B = B; P.K = t->K; P.gait_mode = t->gait_mode;
  P.half_hip_width = S.half_hip_width; P.y_offset = t->y_offset; P.y_coefficient = t->y_coefficient;
  P.swing_kp = 1; P.swing_kd = 0.01;                                                               // as go1mpc_grf_joint_torques_batch
  P.gait = S.gait; P.traj = S.traj; P.homing = t->servo_state_d + SERVO_ROW_HOMING * b; P.ch = S.ch; P.q = t->q_d;
  P.meas = t->meas_d; P.reset = t->reset_d ? t->reset_d : (const int*)rst; P.force = t->force_state_d; P.tau = t->tau_d;
  P.grf = t->grf_d; P.grf_diag = t->grf_diag_d;
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
  const int is = go1mpc_body_in_stride(nh), os = go1mpc_body_out_stride(nh);
  const size_t ib = (size_t)B * is * sizeof(double), ob = (size_t)B * os * sizeof(double);
  const size_t db = (size_t)B * go1mpc_body_diag_stride(nh) * sizeof(int);
  go1mpc::Lane& L = h->lanes[h->lane_next++ % go1mpc::kLanes];
  void *din, *dout, *ddiag = nullptr;
  if ((rc = stage_buf2(h, L.stage[0], ib, &din))) return rc;
  if ((rc = stage_buf2(h, L.stage[1], ob, &dout))) return rc;
  if (diag && (rc = stage_buf2(h, L.stage[2], db, &ddiag))) return rc;
  // the previous outputs are only read by gated ticks (the reference returns its stale members):
  // upload them only when the batch has one
  bool gated = false;
  for (int b = 0; b < B && !gated; b++) {
    const int t = (int)in[(size_t)b * is + 27];
    gated = (t < M->gate) || !(t - M->gate < M->nsum_mpc - nh);
  }
  CU(h, cudaMemcpyAsync(din, in, ib, cudaMemcpyHostToDevice, L.stream));
  if (gated) CU(h, cudaMemcpyAsync(dout, out, ob, cudaMemcpyHostToDevice, L.stream));
  rc = go1mpc_body_mpc_step_batch(h, nh, B, (const double*)din, (double*)dout, (int*)ddiag, L.stream);
  if (rc) return rc;
  CU(h, cudaMemcpyAsync(out, dout, ob, cudaMemcpyDeviceToHost, L.stream));
  if (diag) CU(h, cudaMemcpyAsync(diag, ddiag, db, cudaMemcpyDeviceToHost, L.stream));
  return GO1MPC_OK;
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
  CU(h, cudaSetDevice(h->device));
  const int is = go1mpc_body_in_stride(nh), os = go1mpc_body_out_stride(nh), ts = go1mpc_body_tick_in_stride(nh);
  const size_t ib = (size_t)B * is * sizeof(double), tb = (size_t)B * ts * sizeof(double);
  const size_t tob = (size_t)B * GO1MPC_BODY_TICK_OUT * sizeof(double);
  const size_t db = (size_t)B * go1mpc_body_diag_stride(nh) * sizeof(int);
  go1mpc::Lane& L = h->lanes[h->lane_next++ % go1mpc::kLanes];
  void *drec, *dtick, *dto, *ddiag = nullptr;
  int rc;
  if ((rc = stage_buf2(h, L.stage[0], ib, &drec))) return rc;
  if ((rc = stage_buf2(h, L.stage[8], tb, &dtick))) return rc;
  if ((rc = stage_buf2(h, L.stage[9], tob, &dto))) return rc;
  if (diag && (rc = stage_buf2(h, L.stage[2], db, &ddiag))) return rc;
  CU(h, cudaMemcpyAsync(dtick, tick_in, tb, cudaMemcpyHostToDevice, L.stream));
  // consecutive ticks of the same instances sit on different lanes: order them through the resident records
  {
    auto it = h->last_writer.find((const void*)out_d);
    if (it != h->last_writer.end()) CU(h, cudaStreamWaitEvent(L.stream, it->second, 0));
  }
  CU(h, body_record_expand_launch(B, nh, is, ts, os, tx_d, (const double*)dtick, out_d, (double*)drec, h->sms, L.stream));
  h->launches++;
  rc = go1mpc_body_mpc_step_batch(h, nh, B, (const double*)drec, out_d, (int*)ddiag, L.stream);
  if (rc) return rc;
  CU(h, body_record_pack_launch(B, nh, os, out_d, (double*)dto, h->sms, L.stream));
  h->launches++;
  {
    cudaEvent_t& ev = h->last_writer[(const void*)out_d];
    if (!ev) CU(h, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CU(h, cudaEventRecord(ev, L.stream));
  }
  CU(h, cudaMemcpyAsync(tick_out, dto, tob, cudaMemcpyDeviceToHost, L.stream));
  if (diag) CU(h, cudaMemcpyAsync(diag, ddiag, db, cudaMemcpyDeviceToHost, L.stream));
  return GO1MPC_OK;
}

int go1mpc_step_timing_step_batch_host_async(go1mpc_t* h, int n_sqp, int B, const int* tick, const double* state_d,
                                             double* state_out_d, const double* in, double* out, int* diag) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!tick || !state_d || !state_out_d || !in || !out) return fail(h, GO1MPC_E_INVALID, "step_timing_step_batch_host_async: bad argument");
  CU(h, cudaSetDevice(h->device));
  const size_t b = (size_t)B;
  const size_t tb = b * sizeof(int), ib = b * STEP_IN_DOUBLES * sizeof(double);
  const size_t ob = b * STEP_OUT_DOUBLES * sizeof(double), db = b * STEP_DIAG_INTS * sizeof(int);
  go1mpc::Lane& L = h->lanes[h->lane_next++ % go1mpc::kLanes];
  void *dt_, *di, *do_, *dd = nullptr;
  int rc;
  if ((rc = stage_buf2(h, L.stage[3], tb, &dt_))) return rc;
  if ((rc = stage_buf2(h, L.stage[4], ib, &di))) return rc;
  if ((rc = stage_buf2(h, L.stage[5], ob, &do_))) return rc;
  if (diag && (rc = stage_buf2(h, L.stage[6], db, &dd))) return rc;
  // consecutive ticks of the same planners sit on different lanes: order them through the state buffers
  for (const void* key : {(const void*)state_d, (const void*)state_out_d}) {
    auto it = h->last_writer.find(key);
    if (it != h->last_writer.end()) CU(h, cudaStreamWaitEvent(L.stream, it->second, 0));
  }
  CU(h, cudaMemcpyAsync(dt_, tick, tb, cudaMemcpyHostToDevice, L.stream));
  CU(h, cudaMemcpyAsync(di, in, ib, cudaMemcpyHostToDevice, L.stream));
  rc = go1mpc_step_timing_step_batch(h, n_sqp, B, (const int*)dt_, state_d, state_out_d, (const double*)di, (double*)do_, (int*)dd, L.stream);
  if (rc) return rc;
  // the buffer read and the buffer written: a later call on another lane that WRITES the state this call read must come after
  // it too (write-after-read when state_out_d != state_d)
  for (const void* key : {(const void*)state_out_d, (const void*)state_d}) {
    cudaEvent_t& ev = h->last_writer[key];
    if (!ev) CU(h, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CU(h, cudaEventRecord(ev, L.stream));
    if (state_out_d == state_d) break;
  }
  CU(h, cudaMemcpyAsync(out, do_, ob, cudaMemcpyDeviceToHost, L.stream));
  if (diag) CU(h, cudaMemcpyAsync(diag, dd, db, cudaMemcpyDeviceToHost, L.stream));
  return GO1MPC_OK;
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

namespace {
// shared host staging for the two leg entries: ins[k] (bytes) up, outs[k] down
int leg_host(go1mpc* h, int B, bool ik, const double* a3, const double* b3, const int* leg, const double* bp, const double* br,
             double* o3, double* jac, int* iters) {
  const size_t b = (size_t)B, v3 = b * 3 * sizeof(double), v9 = b * 9 * sizeof(double), vi = b * sizeof(int);
  void *da, *db = nullptr, *dl, *dbp = nullptr, *dbr = nullptr, *do3, *dj = nullptr, *dit = nullptr;
  int rc;
  if ((rc = stage_buf(h, 0, v3, &da))) return rc;
  if (ik && (rc = stage_buf(h, 1, v3, &db))) return rc;
  if ((rc = stage_buf(h, 2, vi, &dl))) return rc;
  if (bp) { if ((rc = stage_buf(h, 3, v3, &dbp))) return rc; if ((rc = stage_buf(h, 4, v3, &dbr))) return rc; }
  if ((rc = stage_buf(h, 5, v3, &do3))) return rc;
  if (jac && (rc = stage_buf(h, 6, v9, &dj))) return rc;
  if (iters && (rc = stage_buf(h, 7, vi, &dit))) return rc;
  cudaStream_t st = h->stream;
  CU(h, cudaMemcpyAsync(da, a3, v3, cudaMemcpyHostToDevice, st));
  if (ik) CU(h, cudaMemcpyAsync(db, b3, v3, cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(dl, leg, vi, cudaMemcpyHostToDevice, st));
  if (bp) { CU(h, cudaMemcpyAsync(dbp, bp, v3, cudaMemcpyHostToDevice, st)); CU(h, cudaMemcpyAsync(dbr, br, v3, cudaMemcpyHostToDevice, st)); }
  if (ik) rc = go1mpc_leg_ik_batch(h, B, (double*)da, (double*)db, (int*)dl, (double*)dbp, (double*)dbr, (double*)do3, (double*)dj, (int*)dit, st);
  else rc = go1mpc_leg_fk_batch(h, B, (double*)da, (int*)dl, (double*)dbp, (double*)dbr, (double*)do3, (double*)dj, st);
  if (rc) return rc;
  CU(h, cudaMemcpyAsync(o3, do3, v3, cudaMemcpyDeviceToHost, st));
  if (jac) CU(h, cudaMemcpyAsync(jac, dj, v9, cudaMemcpyDeviceToHost, st));
  if (iters) CU(h, cudaMemcpyAsync(iters, dit, vi, cudaMemcpyDeviceToHost, st));
  CU(h, cudaStreamSynchronize(st));
  return GO1MPC_OK;
}
}  // namespace
int go1mpc_leg_fk_batch_host(go1mpc_t* h, int B, const double* q, const int* leg, const double* body_p, const double* body_r,
                             double* pos, double* jac) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!q || !leg || !pos || ((body_p == nullptr) != (body_r == nullptr))) return fail(h, GO1MPC_E_INVALID, "leg_fk_batch_host: bad argument");
  CU(h, cudaSetDevice(h->device));
  return leg_host(h, B, false, q, nullptr, leg, body_p, body_r, pos, jac, nullptr);
}
int go1mpc_leg_ik_batch_host(go1mpc_t* h, int B, const double* pdes, const double* qini, const int* leg, const double* body_p,
                             const double* body_r, double* q, double* jac, int* iters) {
  if (!h) return GO1MPC_E_INVALID;
  std::lock_guard<std::recursive_mutex> lk_(h->mu);
  if (B <= 0) return B == 0 ? GO1MPC_OK : GO1MPC_E_INVALID;
  if (!pdes || !qini || !leg || !q || ((body_p == nullptr) != (body_r == nullptr))) return fail(h, GO1MPC_E_INVALID, "leg_ik_batch_host: bad argument");
  CU(h, cudaSetDevice(h->device));
  return leg_host(h, B, true, pdes, qini, leg, body_p, body_r, q, jac, iters);
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
  if (h->tick_ws.size() >= 256 && h->tick_ws.find(st) == h->tick_ws.end())
    return fail(h, GO1MPC_E_UNSUPPORTED, "more than 256 distinct streams used with one handle");
  go1mpc::TickWs& W = h->tick_ws[st];
  const size_t b = (size_t)B;
  const int is = go1mpc_body_in_stride(nh), os = go1mpc_body_out_stride(nh), ts = go1mpc_body_tick_in_stride(nh), ds = go1mpc_body_diag_stride(nh);
  const size_t bytes[7] = {b * sizeof(int), b * STEP_IN_DOUBLES * sizeof(double), b * ts * sizeof(double), b * is * sizeof(double),
                           b * STEP_OUT_DOUBLES * sizeof(double), b * STEP_DIAG_INTS * sizeof(int), b * ds * sizeof(int)};
  void* d[7];
  int rc;
  const int in_rows = (t->step_in_rows > 0 && t->step_in_rows < STEP_IN_DOUBLES) ? t->step_in_rows : STEP_IN_DOUBLES;
  if (in_rows < STEP_IN_DOUBLES && (in_rows < 10 || h->cfg.step.ext_height))
    return fail(h, GO1MPC_E_INVALID, "control_tick_host_async: step_in_rows must cover the 10 sensor rows, and all 20 with cfg.step.ext_height");
  for (int k = 0; k < 7; k++) {
    const bool grow = bytes[k] > W.b[k].cap;
    if (grow) CU(h, cudaStreamSynchronize(st));     // growing: earlier work on this stream may still use the old buffer
    if ((rc = stage_buf2(h, W.b[k], bytes[k], &d[k]))) return rc;
    if (grow && k == 1) W.zero_B = -1;
  }
  if (in_rows < STEP_IN_DOUBLES) {
    // rows a partial upload does not carry read as zero (flat ground, no external heights): cleared once per batch size
    if (W.zero_B != B) {
      CU(h, cudaMemsetAsync((double*)d[1] + b * in_rows, 0, b * (STEP_IN_DOUBLES - in_rows) * sizeof(double), st));
      W.zero_B = B;
    }
  } else {
    W.zero_B = -1;
  }
  CU(h, cudaMemcpyAsync(d[0], t->tick, bytes[0], cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(d[1], t->step_in, b * in_rows * sizeof(double), cudaMemcpyHostToDevice, st));
  CU(h, cudaMemcpyAsync(d[2], t->body_tick_in, bytes[2], cudaMemcpyHostToDevice, st));
  // planner tick: out of place from the pristine state when the caller gives one (replays of the same tick), else in place
  const double* src = t->step_state_src_d ? t->step_state_src_d : t->step_state_d;
  if ((rc = go1mpc_step_timing_step_batch(h, t->n_sqp, B, (const int*)d[0], src, t->step_state_d, (const double*)d[1], (double*)d[4], (int*)d[5], st))) return rc;
  // body tick on the resident records
  CU(h, body_record_expand_launch(B, nh, is, ts, os, t->tx_d, (const double*)d[2], t->body_out_d, (double*)d[3], h->sms, st));
  h->launches++;
  if ((rc = go1mpc_body_mpc_step_batch(h, nh, B, (const double*)d[3], t->body_out_d, (int*)d[6], st))) return rc;
  CU(h, compact_pack_launch(B, nh, os, ds, (const double*)d[4], (const int*)d[5], t->body_out_d, (const int*)d[6], t->compact_d, h->sms, st));
  h->launches++;
  if (t->out38) CU(h, cudaMemcpyAsync(t->out38, d[4], bytes[4], cudaMemcpyDeviceToHost, st));
  if (t->step_diag) CU(h, cudaMemcpyAsync(t->step_diag, d[5], bytes[5], cudaMemcpyDeviceToHost, st));
  if (t->body_diag) CU(h, cudaMemcpyAsync(t->body_diag, d[6], bytes[6], cudaMemcpyDeviceToHost, st));
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
