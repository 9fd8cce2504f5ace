// body_tri.cu -- body-inclination MPC tick as three launches with register-resident solver state.
//
// Same contract as body_fast.cu / body_split.cu (replaces PRMPCClass::body_theta_mpc,
// RT/src/FastMPC/PRMPCClass.cpp:379-714, solve_body_rotation/Solve :799-849, Indexfind :716-738;
// QP = Eigen::QP::solve_quadprog2, RT/src/utils/EiQuadProg/EiQuadProg.cpp:172-491).
//
// body_split.cu showed WHY the warp-per-instance kernels sit at 5-10 % of the FP64 pipe: a step-2a
// pass of a 10-variable half costs ~900 warp instructions of which ~60 are DFMA -- one row per lane
// leaves every matrix-vector product 10 instructions long and surrounds it with shuffles, reductions,
// shared-memory round trips and loop control.  Here each phase gets the mapping that keeps lanes busy:
//
//   A  tri_setup_kernel   thread per instance: condensation (cpp:427-526), Cholesky of the NH x NH
//      Hessian block and J = L^-T fully unrolled in registers, unconstrained minimiser of both halves,
//      first slack evaluation.  A half with nothing violated is finished here (56 % of the bench
//      workload's instances never enter the active-set loop); the others are queued.
//   B  tri_solve_kernel   4 lanes per queued half (8 halves per warp): every lane holds 3 rows of J in
//      registers (static indexing, full unroll), d = J' n+ is an all-reduce over the 4 lanes, z, the
//      Householder update and the primal step are lane-local; R (packed) and the duals live in a
//      128-double shared-memory slice per group.  A group that finishes fetches the next queued half,
//      so the 8 groups of a warp stay busy whatever the iteration counts.  Logs as in body_split.cu.
//   C  tri_merge_kernel   thread per instance: replay of the reference's interleaving of the two halves
//      from the logs (ordered working set, counters, algorithmic flops), first-control clamp, roll-out
//      (cpp:567-655), output record and diagnostics.  Gated ticks are handled here.
//
// The halves are independent because G = blockdiag(H, H) and every constraint touches one half; the
// argument and the replay rule are spelled out at the top of body_split.cu.  What the replay cannot
// reproduce (infeasible / degenerate / non-PD / NaN halves, log overflow, a combined stopping test that
// would not have stopped) is handed, untouched, to body_fast_kernel in list mode.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <mutex>
#include "gi_warp.cuh"
#include "tma.cuh"
#include "kernels.h"

namespace go1 {

template <int NH>
struct TriDims {
  static constexpr int N = 2 * NH, M = 12 * NH;
  static constexpr int IN = (36 + 11 * NH + 1) & ~1;
  static constexpr int OUT = (18 + 2 * NH + 1 + 1) & ~1;
  static constexpr int TAB = (3 * NH * NH + 6 * NH + 1) & ~1;
  static constexpr int JB = NH * NH;                          // per instance: J row-major (entries c >= i valid)
  static constexpr int HS = (2 * NH + 2 + 1) & ~1;            // per half: x0 | pk | tol | f0
  static constexpr int FR = 24;                               // per instance, setup -> merge: theta 4 | measured 4 | zmp x 3 | zmp y 3 |
                                                              // com acc z 3 | i | bjx1 | bjx2 | tol | pad
  static constexpr int OMAX = 16, PMAX = 24;
  static constexpr int RES_D = NH + 4 + OMAX;                 // x | f psi_end R_norm dq_min | ssv
  static constexpr int RES_I = 4 + OMAX + PMAX;               // nout npass end_tol flag | ipv | plog
  static constexpr int RES = RES_D + (RES_I + 1) / 2;         // doubles per half
  static constexpr int RPK = (NH * (NH + 3) / 2 + 1) & ~1;    // packed R: column c holds rows 0..c+1
  static constexpr int V = (NH + 2) & ~1;                     // slot vectors: one spare slot for the pending constraint
  static constexpr int GSP = RPK + 3 * V + V / 2 + 4 * NH;    // R | rinv | u | xs | A (ints) | rot
};

__device__ __forceinline__ int* res_ints(double* res, int res_d) { return reinterpret_cast<int*>(res + res_d); }

// phase indices (cpp:406-417, Indexfind :716-738): first table entry the time has not reached
__device__ __forceinline__ int tri_index(const double* tx, double t) {
  int r = 27;
#pragma unroll
  for (int k = 26; k >= 0; k--) if (!(t >= tx[k])) r = k;
  return r;
}

template <int NH>
__device__ __forceinline__ void tri_finish(const BodyKParams& P, int b, const double* fr, const double* xr, const double* xp,
                                           double f_value, int iqc, int it_outer, int it_add, int it_drop, int it_l2a,
                                           unsigned flops, const int* Ac);
template <int NH>
__device__ __forceinline__ void tri_gated(const BodyKParams& P, int b, const double* rec);

// ======================================================================================= A: setup
constexpr int TRI_SETUP_THREADS = 64;

// The horizon model travels as a launch parameter: every index into it is a compile-time constant after
// unrolling, so its entries are constant-bank operands of the FMAs instead of loads.
template <int NH>
struct TriTab { double v[TriDims<NH>::TAB]; };

template <int NH>
__global__ void __launch_bounds__(TRI_SETUP_THREADS) tri_setup_kernel(const __grid_constant__ BodyKParams P, const __grid_constant__ TriTab<NH> T) {
  using D = TriDims<NH>;
  constexpr int N = D::N, M = D::M;
  // the block's input records are contiguous in HBM: ONE TMA bulk copy stages all of them (74.75 KB for 64)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* srec = reinterpret_cast<double*>(smem_raw);
  uint64_t* bar = reinterpret_cast<uint64_t*>(srec + (size_t)TRI_SETUP_THREADS * D::IN);
  const int b0 = blockIdx.x * TRI_SETUP_THREADS;
  const int nrec = min(TRI_SETUP_THREADS, P.B - b0);
  if (threadIdx.x == 0) { mbar_init(bar, 1); fence_mbar_init(); }
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t bytes = (uint32_t)((size_t)nrec * D::IN * sizeof(double));
    mbar_expect_tx(bar, bytes);
    tma_load_1d(srec, P.in + (size_t)b0 * D::IN, bytes, bar);
  }
  const double* tab = T.v;
  const double* ppu = tab;
  const double* gc0 = tab + NH * NH;
  const double* s2 = tab + 2 * NH * NH;
  const double* m1 = tab + 3 * NH * NH;
  const double* m2 = m1 + 2 * NH;
  const double* pps = m2 + 2 * NH;
  const int lane = threadIdx.x & 31;
  const int b = b0 + threadIdx.x;
  const double dt = P.dt_mpc;
  const double thmax = P.theta_lim;
  const double j_ini = P.j_ini, tq = P.torque_lim / P.j_ini;
  mbar_wait(bar, 0);

  bool live = false;
  int i = 0;
  const double* rec = srec + (size_t)(b < P.B ? threadIdx.x : 0) * D::IN;
  if (b < P.B) {
    i = (int)rec[27];
    if (!(i < P.gate)) { i -= P.gate; live = (i < P.nsum_mpc - NH); }
  }
  bool act0 = false, act1 = false, flag0 = false, flag1 = false, tol0 = false, done = false;
  double f00 = 0.0, psi0 = 0.0;
  if (b < P.B && !live) tri_gated<NH>(P, b, rec);
  bool need_merge = false;      // the instance has a queued half (or a flagged one): the merge kernel finishes it
  if (live) {
    const double* refs = rec + 36 + N;
    const int bjx1 = tri_index(rec, (i + 1) * dt), bjx2 = tri_index(rec, (i + NH) * dt);
    double* xpark = const_cast<double*>(rec) + 36;      // 2 NH doubles of shared memory owned by this thread
    double* fr = const_cast<double*>(rec);              // the step table is consumed: its slots carry the hand-over record
    {
      double t8[8];
#pragma unroll
      for (int k = 0; k < 8; k++) t8[k] = rec[28 + k];
#pragma unroll
      for (int k = 0; k < 8; k++) fr[k] = t8[k];
#pragma unroll
      for (int k = 0; k < 3; k++) { fr[8 + k] = refs[k]; fr[11 + k] = refs[NH + k]; fr[14 + k] = refs[8 * NH + k]; }
      fr[17] = (double)i; fr[18] = (double)bjx1; fr[19] = (double)bjx2;
    }
    const int t_yu = (i + 1) % P.nstepx;
    const bool left = (bjx1 < 2) || (bjx1 % 2 == 0);
    const bool sw = (bjx1 >= 2) && !((t_yu + NH - 1) < P.nstepx);
    const int t_yu_k = (t_yu + NH) - P.nstepx;

    // ---- Hessian block (cpp:511): H = 2 (gc0 + diag(gama/2 pth^2)); right-looking Cholesky in registers ----
    double L[NH][NH];     // lower triangle used
    double pth[NH];
    double tr = 0.0;
#pragma unroll
    for (int k = 0; k < NH; k++) pth[k] = j_ini / (P.mass * (refs[8 * NH + k] + P.g));
#pragma unroll
    for (int c = 0; c < NH; c++)
#pragma unroll
      for (int r = c; r < NH; r++) {
        double v = gc0[c * NH + r];
        if (r == c) { v = v + P.gama / 2 * (pth[c] * pth[c]); tr += 2 * v; }
        L[r][c] = 2 * v;
      }
    const double c1 = 2 * tr;
    double linv[NH];
    double c2 = 0.0;
    bool bad = false;
#pragma unroll
    for (int k = 0; k < NH; k++) {
      const double piv = L[k][k];
      if (!(piv > 0.0)) bad = true;            // <= 0 or NaN: the combined kernel deals with it
      const double rs = rsqrt(piv);
      linv[k] = rs; c2 += rs;
#pragma unroll
      for (int r = k; r < NH; r++) L[r][k] *= rs;
#pragma unroll
      for (int c = k + 1; c < NH; c++)
#pragma unroll
        for (int r = c; r < NH; r++) L[r][c] = fma(-L[r][k], L[c][k], L[r][c]);
    }
    c2 = 2 * c2;
    const double tol = M * EPS_D * c1 * c2 * 100.0;

    // ---- X = L^-1 in place, row by row (row i needs the original row i of L and the finished rows above);
    //      J = L^-T = X' goes to the instance's J buffer row-major, zeros below the diagonal, 16-byte stores ----
    fr[20] = tol;
#pragma unroll
    for (int i2 = 0; i2 < NH; i2++) {
      double t[NH];
#pragma unroll
      for (int j = 0; j < i2; j++) {
        double a = L[i2][j] * L[j][j];                   // k = j term: X(j,j) already holds 1 / L(j,j)
#pragma unroll
        for (int k = j + 1; k < i2; k++) a = fma(L[i2][k], L[k][j], a);
        t[j] = a;
      }
#pragma unroll
      for (int j = 0; j < i2; j++) L[i2][j] = -linv[i2] * t[j];
      L[i2][i2] = linv[i2];
    }
    {
      double2* jb2 = reinterpret_cast<double2*>(P.tri_jb + (size_t)b * D::JB);
#pragma unroll
      for (int r = 0; r < NH; r++)
#pragma unroll
        for (int c2i = 0; c2i < NH / 2; c2i++) {
          const int ca = 2 * c2i, cb = 2 * c2i + 1;      // J(r,c) = X(c,r) for c >= r
          jb2[(r * NH) / 2 + c2i] = make_double2(ca >= r ? L[ca][r] : 0.0, cb >= r ? L[cb][r] : 0.0);
        }
    }

    // ---- both halves: gradient (cpp:427-526), unconstrained minimiser, first slack scan ----
#pragma unroll 1
    for (int h = 0; h < 2; h++) {
      const double my0 = fr[2 * h], my1 = fr[1 + 2 * h];
      const double* bref = refs + (2 + h) * NH;
      double w[NH], pk[NH];
      double f0 = 0.0;
      double g0[NH];
#pragma unroll
      for (int k = 0; k < NH; k++) {
        const bool other = sw && (k >= NH - t_yu_k);
        const bool use_l = left ? !other : other;
        const double cop = h ? (use_l ? refs[6 * NH + k] : refs[4 * NH + k])      // half 1 (pitch accel) uses det_px
                             : (use_l ? refs[7 * NH + k] : refs[5 * NH + k]);     // half 0 (roll accel) uses det_py
        const double det = (h ? refs[k] : refs[NH + k]) - cop;
        pk[k] = fma(pps[k], my0, pps[NH + k] * my1);
        const double t1 = fma(m1[k], my0, m1[NH + k] * my1), t2 = fma(m2[k], my0, m2[NH + k] * my1);
        double t3 = 0.0;
#pragma unroll
        for (int j = 0; j < NH; j++) t3 = fma(s2[j * NH + k], bref[j], t3);
        g0[k] = ((t1 + t2) - t3) + (P.gama * (h ? -pth[k] : pth[k])) * det;
        w[k] = g0[k];
      }
      // x0 = -J (J' g0) with J' = X: two triangular products, no division
      {
        double d0[NH];
#pragma unroll
        for (int c = 0; c < NH; c++) {
          double a = L[c][0] * w[0];
#pragma unroll
          for (int r = 1; r <= c; r++) a = fma(L[c][r], w[r], a);
          d0[c] = a;
        }
#pragma unroll
        for (int r = 0; r < NH; r++) {
          double a = L[r][r] * d0[r];
#pragma unroll
          for (int c = r + 1; c < NH; c++) a = fma(L[c][r], d0[c], a);
          w[r] = a;
        }
      }
      double psi = 0.0, smin = 0.0;
      bool nan = false;
#pragma unroll
      for (int k = 0; k < NH; k++) {
        w[k] = -w[k];                      // x0
        xpark[h * NH + k] = w[k];
        nan = nan || (w[k] != w[k]);
        f0 = fma(g0[k], w[k], f0);
      }
      f0 *= 0.5;
#pragma unroll
      for (int k = 0; k < NH; k++) {
        double v = 0.0;
#pragma unroll
        for (int j = 0; j <= k; j++) v = fma(ppu[j * NH + k], w[j], v);
        const double n0 = (thmax - pk[k]) - v, n1 = v + (thmax + pk[k]);
        const double n2 = fma(-j_ini, w[k], tq), n3 = fma(j_ini, w[k], tq);
        psi += (fmin(0.0, n0) + fmin(0.0, n1)) + (fmin(0.0, n2) + fmin(0.0, n3));
        smin = fmin(smin, fmin(fmin(n0, n1), fmin(n2, n3)));
      }
      const bool over = fabs(psi) > tol;
      const bool active = !bad && !nan && over && (smin < 0.0);
      const size_t hid = 2 * (size_t)b + h;
      if (active) {
        double2* hs2 = reinterpret_cast<double2*>(P.tri_hs + hid * D::HS);
#pragma unroll
        for (int k = 0; k < NH / 2; k++) { hs2[k] = make_double2(w[2 * k], w[2 * k + 1]); hs2[NH / 2 + k] = make_double2(pk[2 * k], pk[2 * k + 1]); }
        hs2[NH] = make_double2(tol, f0);
      } else {
        double* rs_ = P.tri_res + hid * D::RES;
        int* ri = res_ints(rs_, D::RES_D);
        double2* rs2 = reinterpret_cast<double2*>(rs_);
#pragma unroll
        for (int k = 0; k < NH / 2; k++) rs2[k] = make_double2(w[2 * k], w[2 * k + 1]);
        rs2[NH / 2] = make_double2(f0, psi); rs2[NH / 2 + 1] = make_double2(1.0, CUDART_INF);
        ri[0] = 0; ri[1] = 0; ri[2] = over ? 0 : 1; ri[3] = (bad || nan || psi != psi) ? 1 : 0;
      }
      if (h == 0) act0 = active; else act1 = active;
      if (h == 0) flag0 = (bad || nan || psi != psi); else flag1 = (bad || nan || psi != psi);
      if (h == 0) { f00 = f0; psi0 = psi; tol0 = !over; }
      else if (!act0 && !active && !flag0 && !flag1) {
        // both halves finished here: the combined solve is one step-1 pass with nothing violated
        // (same validity rule as the merge kernel: a half that stopped on its tolerance with psi != 0 while the
        // SUM of both exceeds the tolerance is not reproducible here)
        const bool unsure = fabs(psi0 + psi) > tol && ((tol0 && psi0 != 0.0) || (!over && psi != 0.0));
        if (!unsure) {
          tri_finish<NH>(P, b, fr, xpark, xpark + NH, f00 + f0, 0, 1, 0, 0, 0,
                         (unsigned)gi_flops_setup(N, 0) + 2u * N * M, nullptr);
          done = true;
        }
      }
    }
    need_merge = !done;
    if (!done) {
      double2* frg = reinterpret_cast<double2*>(P.tri_fr + (size_t)b * D::FR);
#pragma unroll
      for (int k = 0; k < 11; k++) frg[k] = make_double2(fr[2 * k], fr[2 * k + 1]);
    }
  }
  // ---- queue the active halves (warp-aggregated) ----
  const unsigned m0 = __ballot_sync(FULL_MASK, act0), m1b = __ballot_sync(FULL_MASK, act1);
  const int n0 = __popc(m0), n1 = __popc(m1b);
  if (n0 + n1) {
    int base = 0;
    if (lane == 0) base = atomicAdd(P.tri_qctl, n0 + n1);
    base = __shfl_sync(FULL_MASK, base, 0);
    const unsigned below = (1u << lane) - 1u;
    if (act0) P.tri_queue[base + __popc(m0 & below)] = 2 * b;
    if (act1) P.tri_queue[base + n0 + __popc(m1b & below)] = 2 * b + 1;
  }
  // ---- list of the instances the merge kernel has to finish (compact: its CTAs are full whatever the finished share) ----
  const unsigned mm = __ballot_sync(FULL_MASK, need_merge);
  if (mm) {
    int base = 0;
    if (lane == 0) base = atomicAdd(P.tri_qctl + 3, __popc(mm));
    base = __shfl_sync(FULL_MASK, base, 0);
    if (need_merge) P.tri_meta[base + __popc(mm & ((1u << lane) - 1u))] = b;
  }
}

// ======================================================================================= B: active-set iteration
__device__ __forceinline__ double q4bc(double v, int src) { return __shfl_sync(FULL_MASK, v, src, 4); }
__device__ __forceinline__ double q4sum(double v) {
  v += __shfl_xor_sync(FULL_MASK, v, 2);
  v += __shfl_xor_sync(FULL_MASK, v, 1);
  return v;
}

#ifndef GO1_TRI_WARPS
#define GO1_TRI_WARPS 12
#endif
// A/B build knobs of the solve kernel: warps per CTA and, optionally, a register cap instead of the min-blocks bound
// (GO1_TRI_WPC=2 GO1_TRI_MAXNREG=144: 7 CTAs of 2 warps = 14 warps per SM with 148 bytes of spills)
#ifndef GO1_TRI_WPC
#define GO1_TRI_WPC 4
#endif
#ifdef GO1_TRI_MAXNREG
#define GO1_TRI_BOUNDS(WPC) __maxnreg__(GO1_TRI_MAXNREG)
#else
#define GO1_TRI_BOUNDS(WPC) __launch_bounds__(WPC * 32, GO1_TRI_WARPS / WPC)
#endif

template <int NH, int WPC>
__global__ void GO1_TRI_BOUNDS(WPC) tri_solve_kernel(BodyKParams P) {
  using D = TriDims<NH>;
  constexpr int RW = (NH + 3) / 4;          // rows of J per lane
  static_assert(RW >= 1 && RW <= 3 && NH % 2 == 0, "4 lanes per half, up to 3 rows of J per lane, rows moved 16 bytes at a time");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* smem = reinterpret_cast<double*>(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, gl = lane & 3;
  const unsigned gm = 0xfu << (g * 4);

  double* tab = smem;
  for (int i = threadIdx.x; i < NH * NH; i += blockDim.x) tab[i] = P.tab[i];   // ppu only
  const double* ppu = tab;
  double* gbase = smem + ((NH * NH + 1) & ~1) + (size_t)(warp * 8 + g) * D::GSP;
  double* Rp = gbase;                       // R(t,c) = Rp[c*(c+3)/2 + t], t <= c+1
  double* rinvs = Rp + D::RPK;
  double* us = rinvs + D::V;
  double* xs = us + D::V;
  int* As = reinterpret_cast<int*>(xs + D::V);
  double* rot = xs + D::V + D::V / 2;       // (cc, sn, xny, skip) per rotation
  __shared__ int nxt[WPC * 8];
  __syncthreads();

  const int count = *reinterpret_cast<volatile const int*>(P.tri_qctl);
  const double thmax = P.theta_lim;
  const double j_ini = P.j_ini, tq = P.torque_lim / P.j_ini;
  const double inf = CUDART_INF;

  int row[RW]; bool valid[RW];
#pragma unroll
  for (int m = 0; m < RW; m++) { row[m] = gl + 4 * m; valid[m] = row[m] < NH; if (!valid[m]) row[m] = NH - 1; }

  // per-lane state of the group's current half
  double Jr[RW][NH];
  double x[RW], pk[RW];
  unsigned inA = 0u;               // bit 4m+s: slot s of own variable m is in the working set
  int cur = -1, h = 0, iq = 0, nout = 0, npass = 0;
  bool fin = true, dead = false, need_l1 = true, flag = false, end_tol = false;
  double tol = 0.0, f_value = 0.0, R_norm = 1.0, dq_min = inf;
  int ip = 0, ip_blk = 0, ip_k = 0;
  double sip = 0.0, ip_sgn = 1.0;
  double* res = nullptr;
  int* resi = nullptr;

  for (unsigned guard = 0;; guard++) {
    if (guard > (1u << 22)) { if (lane == 0) atomicAdd(P.tri_qctl + 2, 1); break; }   // defensive: never spin forever
    // ---- groups that finished store their result and fetch the next queued half ----
    if (__any_sync(FULL_MASK, fin && !dead)) {
      if (fin && !dead) {
        if (cur >= 0) {
#pragma unroll
          for (int m = 0; m < RW; m++) if (valid[m]) res[row[m]] = x[m];
          if (gl == 0) {
            res[NH] = f_value; res[NH + 2] = R_norm; res[NH + 3] = dq_min;
            resi[0] = nout; resi[1] = npass; resi[2] = end_tol ? 1 : 0; resi[3] = flag ? 1 : 0;
          }
        }
        if (gl == 0) {
          const int q = atomicAdd(P.tri_qctl + 1, 1);
          nxt[warp * 8 + g] = (q < count) ? P.tri_queue[q] : -1;
        }
      }
      __syncwarp();
      if (fin && !dead) {
        cur = nxt[warp * 8 + g];
        if (cur < 0) dead = true;
        else {
          h = cur & 1;
          const double* jb = P.tri_jb + (size_t)(cur >> 1) * D::JB;
          const double* hs = P.tri_hs + (size_t)cur * D::HS;
#pragma unroll
          for (int m = 0; m < RW; m++) {
            const double2* jr = reinterpret_cast<const double2*>(jb + row[m] * NH);   // rows are 80 bytes: 16-byte aligned
#pragma unroll
            for (int j2 = 0; j2 < NH / 2; j2++) {
              const double2 v2 = jr[j2];
              Jr[m][2 * j2] = v2.x; Jr[m][2 * j2 + 1] = v2.y;
            }
            if (m == RW - 1 && !valid[m]) {
#pragma unroll
              for (int j = 0; j < NH; j++) Jr[m][j] = 0.0;
            }
            x[m] = valid[m] ? hs[row[m]] : 0.0;
            pk[m] = hs[NH + row[m]];
          }
          tol = hs[2 * NH]; f_value = hs[2 * NH + 1];
          res = P.tri_res + (size_t)cur * D::RES;
          resi = res_ints(res, D::RES_D);
          inA = 0u; iq = 0; nout = 0; npass = 0;
          fin = false; need_l1 = true; flag = false; end_tol = false;
          R_norm = 1.0; dq_min = inf;
        }
      }
    }
    if (__all_sync(FULL_MASK, dead)) break;
    const int cbase0 = (h << 1) * NH;        // constraint id = blk NH + k, blk = ((s>>1)<<2) | (h<<1) | (s&1)

    const bool g1 = need_l1 && !fin && !dead;
    if (__any_sync(FULL_MASK, g1)) {
      // ---- step 1 (cpp:282-320) and step 2 (cpp:322-342) ----
      if (g1) {
#pragma unroll
        for (int m = 0; m < RW; m++) if (valid[m]) xs[row[m]] = x[m];
      }
      __syncwarp();
      double xv[NH];
#pragma unroll
      for (int j = 0; j < NH; j++) xv[j] = xs[j];
      // slacks of the lane's variables; psi; the most negative eligible slack of the group and, among the
      // slacks equal to it, the lowest constraint id (the reference's strict '<' scan, cpp:322-342)
      double psi = 0.0, bv = inf;
      double sl[RW][4];
#pragma unroll
      for (int m = 0; m < RW; m++) {
        const int k = row[m];
        double v = 0.0;
#pragma unroll
        for (int j = 0; j < NH; j++) v = fma(ppu[j * NH + k], xv[j], v);   // zeros above the diagonal
        const unsigned bits = valid[m] ? (inA >> (4 * m)) : 0xfu;
        sl[m][0] = (thmax - pk[m]) - v; sl[m][1] = v + (thmax + pk[m]);
        sl[m][2] = fma(-j_ini, x[m], tq); sl[m][3] = fma(j_ini, x[m], tq);
        // min(0, s) as a select: fmin() carries IEEE NaN handling that costs 8 instructions a piece (NaN in x is
        // screened by the merge kernel); up and low slack of one angle cannot both be negative, nor both torque slacks
        const double pa = sl[m][0] < sl[m][1] ? sl[m][0] : sl[m][1], pt = sl[m][2] < sl[m][3] ? sl[m][2] : sl[m][3];
        const double p4 = (pa < 0.0 ? pa : 0.0) + (pt < 0.0 ? pt : 0.0);
        psi += valid[m] ? p4 : 0.0;
#pragma unroll
        for (int s4 = 0; s4 < 4; s4++) {
          if (bits & (1u << s4)) sl[m][s4] = inf;          // in the working set (or a padding row): not eligible
          bv = sl[m][s4] < bv ? sl[m][s4] : bv;
        }
      }
      psi = q4sum(psi);
      { const double o2 = __shfl_xor_sync(FULL_MASK, bv, 2); bv = o2 < bv ? o2 : bv; }
      { const double o1 = __shfl_xor_sync(FULL_MASK, bv, 1); bv = o1 < bv ? o1 : bv; }
      int bi = 0x7fffffff;
#pragma unroll
      for (int m = RW - 1; m >= 0; m--) {
        const int c0 = cbase0 + row[m];
        // ids of a variable ascend with the slot: test in descending order so the lowest match survives
        if (sl[m][3] == bv) bi = min(bi, c0 + 5 * NH);
        if (sl[m][2] == bv) bi = min(bi, c0 + 4 * NH);
        if (sl[m][1] == bv) bi = min(bi, c0 + NH);
        if (sl[m][0] == bv) bi = min(bi, c0);
      }
      bi = min(bi, __shfl_xor_sync(FULL_MASK, bi, 2));
      bi = min(bi, __shfl_xor_sync(FULL_MASK, bi, 1));
      if (g1) {
        if (gl == 0) res[NH + 1] = psi;       // psi at the last step 1 of the half: stored as it is found, not held
        if (!(fabs(psi) > tol)) { fin = true; end_tol = true; if (psi != psi) flag = true; }
        else if (!(bv < 0.0)) fin = true;
        else if (nout >= D::OMAX) { fin = true; flag = true; }
        else {
          ip = bi; sip = bv;
          if (gl == 0) { res[NH + 4 + nout] = bv; resi[4 + nout] = bi; As[iq] = bi; us[iq] = 0.0; }
          nout++;
          ip_blk = ip / NH; ip_k = ip - ip_blk * NH;
          ip_sgn = (ip_blk & 1) ? 1.0 : -1.0;
          need_l1 = false;
        }
      }
      __syncwarp();
    }
    if (!fin && !dead && npass >= D::PMAX) { fin = true; flag = true; }
    const bool run = !fin && !dead;
    if (!__any_sync(FULL_MASK, run)) continue;

    // ---- step 2a (cpp:349-386); groups that do not run compute along and commit nothing ----
    double np_[RW];
#pragma unroll
    for (int m = 0; m < RW; m++) {
      double v = 0.0;
      if (ip_blk < 4) { if (row[m] <= ip_k) v = ip_sgn * ppu[row[m] * NH + ip_k]; }
      else if (row[m] == ip_k) v = ip_sgn * j_ini;
      np_[m] = valid[m] ? v : 0.0;
    }
    // d = J' n+: partial sums over the lane's rows, all-reduced over the 4 lanes
    double d[NH];
#pragma unroll
    for (int j = 0; j < NH; j++) {
      double a = Jr[0][j] * np_[0];
#pragma unroll
      for (int m = 1; m < RW; m++) a = fma(Jr[m][j], np_[m], a);
      d[j] = a;
    }
#pragma unroll
    for (int j = 0; j < NH; j++) d[j] = q4sum(d[j]);
    // z = J[:, iq:] d[iq:], |d2|^2, d_iq
    double z[RW];
    double dd = 0.0, diq = 0.0;
#pragma unroll
    for (int m = 0; m < RW; m++) z[m] = 0.0;
#pragma unroll
    for (int j = 0; j < NH; j++) {
      const double dj = (j >= iq) ? d[j] : 0.0;            // select, not branch: the halves of a warp differ in iq
#pragma unroll
      for (int m = 0; m < RW; m++) z[m] = fma(Jr[m][j], dj, z[m]);
      dd = fma(dj, dj, dd);
      xs[j] = d[j];                                        // every lane of the group stores the same value
    }
    diq = xs[iq];                                          // slot NH exists (V > NH): iq = NH reads a stale, unused value
    double zz = 0.0, zn = 0.0;
#pragma unroll
    for (int m = 0; m < RW; m++) { zz = fma(z[m], z[m], zz); zn = fma(z[m], np_[m], zn); }
    zz = q4sum(zz); zn = q4sum(zn);
    // d[0:iq) would be the new column of R if this pass ends in an add: stored now (column iq is not read before it
    // is added), so that r = R^-1 d[0:iq) can overwrite it in place -- 20 registers less (168 -> 12 warps/SM is the
    // solve kernel's occupancy limit).  Every lane of the group solves redundantly (d is replicated).
    if (gl == 0 && iq < NH) {
#pragma unroll
      for (int tt = 0; tt < NH; tt++) if (tt < iq) Rp[iq * (iq + 3) / 2 + tt] = d[tt];
    }
#pragma unroll
    for (int c = NH - 1; c >= 0; c--) {
      if (c < iq) {
        const double rc = d[c] * rinvs[c];
        d[c] = rc;
#pragma unroll
        for (int t = 0; t < c; t++) d[t] = fma(-rc, Rp[c * (c + 3) / 2 + t], d[t]);
      }
    }
    double (&r)[NH] = d;      // entries below iq now hold r, entries from iq on are still d2
    // ratio test (cpp:360-367): arg-min of u_k / r_k over r_k > 0 by cross-multiplication (strict '<', first
    // slot wins, as the reference's scan), no division
    double ub = 0.0, rb = -1.0; int kb = -1;
#pragma unroll
    for (int k = 0; k < NH; k++) {
      const double uk = us[k];
      const bool take = (k < iq) && (r[k] > 0.0) && (kb < 0 || uk * rb < ub * r[k]);
      if (take) { ub = uk; rb = r[k]; kb = k; }
    }
    // step lengths.  One division instruction: group lane 0 -> t2 = -s_ip / z.n+, lane 1 -> Householder scale,
    // lane 2 -> t1 = u_l / r_l
    const double inrm = (dd > 0.0) ? rsqrt(dd) : 0.0;      // 1 / |d2|
    const double nrm = dd * inrm;                           // |d2|
    double num = ub, den = rb;
    if (gl == 0) { num = -sip; den = zn; }
    if (gl == 1) { num = 1.0; den = nrm * (nrm + fabs(diq)); }
    const double quo = num / den;
    const double q0 = q4bc(quo, 0);                         // (shuffles stay outside group-dependent conditions)
    const double t2 = (fabs(zz) > EPS_D) ? q0 : inf;
    const double tau = q4bc(quo, 1);
    const double q2 = q4bc(quo, 2);
    const double t1 = (kb >= 0) ? q2 : inf;
    const int l = As[kb >= 0 ? kb : 0];
    const double uiq = us[iq];
    const double t = fmin(t1, t2);
    const bool go = run && (t < inf);
    const bool prim = go && !(t2 >= inf);                  // case (iii); go && !prim: case (ii), dual step
    const bool full = prim && (t == t2);
    const bool dropg = go && !full;
    if (run && !go) { fin = true; flag = true; }           // case (i): infeasible (or NaN)
    __syncwarp();                                           // all reads of us / R above precede the writes below
    if (go && gl == 0) {
#pragma unroll
      for (int k = 0; k < NH; k++) if (k < iq) us[k] = fma(-t, r[k], us[k]);
      us[iq] = uiq + t;
    }
    if (prim) {
#pragma unroll
      for (int m = 0; m < RW; m++) x[m] = fma(t, z[m], x[m]);
      f_value += t * zn * (0.5 * t + uiq);
    }
    if (full) {
      // ---- add_constraint (cpp:30-93) as ONE Householder reflection H = I - tau v v', v = d2 + sigma e_iq ----
      const double sigma = (diq < 0.0) ? -nrm : nrm;
      if (nrm != 0.0) {
        // v overwrites d in place (entries below iq -- r, no longer needed -- become 0)
#pragma unroll
        for (int j = 0; j < NH; j++) d[j] = (j > iq) ? d[j] : ((j == iq) ? diq + sigma : 0.0);
#pragma unroll
        for (int m = 0; m < RW; m++) {
          double w = 0.0;
#pragma unroll
          for (int j = 0; j < NH; j++) w = fma(Jr[m][j], d[j], w);
          const double sw2 = tau * w;
#pragma unroll
          for (int j = 0; j < NH; j++) Jr[m][j] = fma(-sw2, d[j], Jr[m][j]);
        }
      }
      const double dq = (nrm != 0.0) ? -sigma : diq;           // new R(iq,iq)
      if (gl == 0) {
        Rp[iq * (iq + 3) / 2 + iq] = dq;
        rinvs[iq] = (nrm != 0.0) ? ((diq < 0.0) ? inrm : -inrm) : 1.0 / dq;
        resi[4 + D::OMAX + npass] = ip;
      }
      iq++;
      npass++;
      if (fabs(dq) <= EPS_D * R_norm) { fin = true; flag = true; }   // degenerate: combined kernel
      R_norm = fmax(R_norm, fabs(dq));
      dq_min = fmin(dq_min, fabs(dq));
      {
        const int slot = ((ip_blk >> 2) << 1) | (ip_blk & 1);
        if (gl == (ip_k & 3)) inA |= 1u << (4 * (ip_k >> 2) + slot);
      }
      need_l1 = true;
    }
    __syncwarp();
    if (!__any_sync(FULL_MASK, dropg)) continue;
    // ---- delete_constraint(l) (cpp:95-170) after a dual or a partial step: rare, the one group-divergent
    //      region; the group's lane 0 updates R, all lanes rotate their rows of J ----
    if (dropg) {
      {
        const int lblk = l / NH, lk = l - lblk * NH;
        const int slot = ((lblk >> 2) << 1) | (lblk & 1);
        if (gl == (lk & 3)) inA &= ~(1u << (4 * (lk >> 2) + slot));
      }
      int qq = -1;
      for (int k = iq - 1; k >= 0; k--) if (As[k] == l) qq = k;
      __syncwarp(gm);
      if (qq < 0) { fin = true; flag = true; }   // l not in the working set: UB in the reference
      else {
        if (gl == 0) {
          for (int k = qq; k < iq; k++) { As[k] = As[k + 1]; us[k] = us[k + 1]; }   // slot iq holds ip and its u
          for (int c = qq; c < iq - 1; c++)
            for (int tt = 0; tt <= c + 1; tt++) Rp[c * (c + 3) / 2 + tt] = Rp[(c + 1) * (c + 4) / 2 + tt];
          resi[4 + D::OMAX + npass] = 0x10000 | l;
        }
        iq--;
        npass++;
        if (gl == 0) {
          for (int j = qq; j < iq; j++) {
            double cc = Rp[j * (j + 3) / 2 + j], sn = Rp[j * (j + 3) / 2 + j + 1];
            // h = |(cc, sn)| through one rsqrt (the reference's overflow-safe distance(), EiQuadProg.hpp:100-118,
            // agrees to rounding at these magnitudes), one division for xny
            const double h2 = fma(cc, cc, sn * sn);
            if (h2 == 0.0) { rot[4 * j + 3] = 1.0; continue; }
            const double rh = rsqrt(h2), hh = h2 * rh;
            cc = cc * rh; sn = sn * rh;
            Rp[j * (j + 3) / 2 + j + 1] = 0.0;
            Rp[j * (j + 3) / 2 + j] = (cc < 0.0) ? -hh : hh;
            if (cc < 0.0) { cc = -cc; sn = -sn; }
            const double xny = sn / (1.0 + cc);
            for (int c = j + 1; c < iq; c++) {
              double* cp = Rp + c * (c + 3) / 2;
              const double t1j = cp[j], t2j = cp[j + 1];
              const double a = fma(t2j, sn, t1j * cc);
              cp[j] = a;
              cp[j + 1] = fma(xny, t1j + a, -t2j);
            }
            rot[4 * j] = cc; rot[4 * j + 1] = sn; rot[4 * j + 2] = xny; rot[4 * j + 3] = 0.0;
          }
        }
        __syncwarp(gm);
        for (int k = qq + gl; k < iq; k += 4) rinvs[k] = 1.0 / Rp[k * (k + 3) / 2 + k];
        for (int j = qq; j < iq; j++) {
          if (rot[4 * j + 3] != 0.0) continue;
          const double cc = rot[4 * j], sn = rot[4 * j + 1], xny = rot[4 * j + 2];
#pragma unroll
          for (int jj = 0; jj < NH - 1; jj++)
            if (jj == j) {
#pragma unroll
              for (int m = 0; m < RW; m++) {
                const double t1j = Jr[m][jj], t2j = Jr[m][jj + 1];
                const double a = fma(t2j, sn, t1j * cc);
                Jr[m][jj] = a;
                Jr[m][jj + 1] = fma(xny, a + t1j, -t2j);
              }
            }
        }
        if (prim) {
          // partial step: recompute the slack of ip at the new x (a dual step keeps s_ip)
#pragma unroll
          for (int m = 0; m < RW; m++) if (valid[m]) xs[row[m]] = x[m];
          __syncwarp(gm);
          if (ip_blk < 4) {
            double v = 0.0;
            for (int j = 0; j <= ip_k; j++) v = fma(ppu[j * NH + ip_k], xs[j], v);
            const double pkk = P.tri_hs[(size_t)cur * D::HS + NH + ip_k];
            sip = (ip_blk & 1) ? v + (thmax + pkk) : (thmax - pkk) - v;
          } else {
            sip = (ip_blk & 1) ? fma(j_ini, xs[ip_k], tq) : fma(-j_ini, xs[ip_k], tq);
          }
        }
      }
    }
    __syncwarp();
  }
}

// ======================================================================================= C: merge + outputs
// Output stage shared by the setup kernel (instances whose halves both finish there, gated ticks) and the merge
// kernel: first-control clamp (cpp:567-625), roll-out (cpp:629-655), output record, diagnostics.
// xr / xp: the NH accelerations of the roll / pitch half.
template <int NH>
__device__ __forceinline__ void tri_finish(const BodyKParams& P, int b, const double* fr, const double* xr, const double* xp,
                                           double f_value, int iqc, int it_outer, int it_add, int it_drop, int it_l2a,
                                           unsigned flops, const int* Ac) {
  using D = TriDims<NH>;
  constexpr int N = D::N;
  static_assert(D::OUT % 2 == 0 && N % 2 == 0, "the output record is stored 16 bytes at a time");
  const double dt = P.dt_mpc, b0 = dt * dt / 2, b1 = dt;
  const double thmax = P.theta_lim, thmin = -P.theta_lim;
  const double j_ini = P.j_ini;
  const double thx0 = fr[0], thx1 = fr[1], thy0 = fr[2], thy1 = fr[3];
  double o[18];              // head of the output record, built in registers (one thread writes a whole record:
                             // 16-byte stores halve the number of uncoalesced store instructions)
  double xa[3], ya[3];
#pragma unroll
  for (int k = 0; k < 3; k++) { xa[k] = xr[k]; ya[k] = xp[k]; }
  const double arow_x = thx0 + dt * thx1, arow_y = thy0 + dt * thy1;
  {
    const double nx0 = arow_x + b0 * xa[0];
    if (nx0 > thmax) xa[0] = (thmax - arow_x) / b0;
    else if (nx0 < thmin) xa[0] = (thmin - arow_x) / b0;
    const double ny0 = arow_y + b0 * ya[0];
    if (ny0 > thmax) ya[0] = (thmax - arow_y) / b0;
    else if (ny0 < thmin) ya[0] = (thmin - arow_y) / b0;
  }
#pragma unroll
  for (int ax = 0; ax < 2; ax++) {
    const double a0 = ax ? ya[0] : xa[0], a1 = ax ? ya[1] : xa[1], a2 = ax ? ya[2] : xa[2];
    const double p0 = ax ? thy0 : thx0, v0 = ax ? thy1 : thx1;
    const double lam_p = P.lamda[2 * ax], lam_v = P.lamda[2 * ax + 1];
    const double bs_p = fr[4 + 2 * ax], bs_v = fr[5 + 2 * ax];
    double pkk = (p0 + dt * v0) + b0 * a0, vk = v0 + b1 * a0;
    o[14 + 2 * ax] = lam_p * bs_p + (1 - lam_p) * pkk;
    o[15 + 2 * ax] = lam_v * bs_v + (1 - lam_v) * vk;
    o[0 + ax] = pkk;
    double pn = (pkk + dt * vk) + b0 * a1; vk = vk + b1 * a1; pkk = pn;
    o[6 + ax] = pkk;
    pn = (pkk + dt * vk) + b0 * a2; pkk = pn;
    o[10 + ax] = pkk;
    o[2 + ax] = j_ini * a0;
  }
#pragma unroll
  for (int k = 0; k < 3; k++) {
    // cpp:651-652 ZMP consistent with the planned angular acceleration (steps 0..2)
    const double den = P.mass * (P.g + fr[14 + k]);
    const int oo = (k == 0) ? 4 : (k == 1 ? 8 : 12);
    o[oo] = fr[8 + k] - j_ini * ya[k] / den;
    o[oo + 1] = fr[11 + k] + j_ini * xa[k] / den;
  }
  double2* og = reinterpret_cast<double2*>(P.out + (size_t)b * D::OUT);
#pragma unroll
  for (int k = 0; k < 9; k++) og[k] = make_double2(o[2 * k], o[2 * k + 1]);
  og[9] = make_double2(xa[0], xr[1]);
#pragma unroll
  for (int k = 1; k < NH / 2; k++) og[9 + k] = make_double2(xr[2 * k], xr[2 * k + 1]);
  og[9 + NH / 2] = make_double2(ya[0], xp[1]);
#pragma unroll
  for (int k = 1; k < NH / 2; k++) og[9 + NH / 2 + k] = make_double2(xp[2 * k], xp[2 * k + 1]);
  og[9 + NH] = make_double2(f_value, 0.0);
  if (P.diag) {
    int dgv[10 + N];
    dgv[0] = ST_OK; dgv[1] = iqc;
    dgv[2] = it_outer; dgv[3] = it_add; dgv[4] = it_drop; dgv[5] = 0;
    dgv[6] = (int)fr[18]; dgv[7] = (int)fr[19]; dgv[8] = it_l2a; dgv[9] = (int)flops;
#pragma unroll
    for (int k = 0; k < N; k++) dgv[10 + k] = (Ac != nullptr && k < iqc) ? Ac[k] : -1;
    int* dg = P.diag + (size_t)b * P.diag_stride;
    if ((P.diag_stride & 1) == 0 && ((uintptr_t)P.diag & 7) == 0) {
      int2* dg2 = reinterpret_cast<int2*>(dg);
#pragma unroll
      for (int k = 0; k < (10 + N) / 2; k++) dg2[k] = make_int2(dgv[2 * k], dgv[2 * k + 1]);
    } else {
#pragma unroll
      for (int k = 0; k < 10 + N; k++) dg[k] = dgv[k];
    }
  }
}

// gated tick: the reference returns its stale members (out14 stays); state and V_ini unchanged
template <int NH>
__device__ __forceinline__ void tri_gated(const BodyKParams& P, int b, const double* rec) {
  using D = TriDims<NH>;
  constexpr int N = D::N;
  double* outg = P.out + (size_t)b * D::OUT;
#pragma unroll
  for (int k = 0; k < 4; k++) outg[14 + k] = rec[28 + k];
  for (int k = 0; k < N; k++) outg[18 + k] = rec[36 + k];
  outg[18 + N] = 0.0;
  if (D::OUT > 19 + N) outg[19 + N] = 0.0;
  if (P.diag) {
    int* dg = P.diag + (size_t)b * P.diag_stride;
    dg[0] = -1;
    for (int k = 1; k < 10; k++) dg[k] = 0;
    for (int k = 0; k < N; k++) dg[10 + k] = -1;
  }
}

constexpr int TRI_MERGE_THREADS = 64;

template <int NH>
__global__ void __launch_bounds__(TRI_MERGE_THREADS) tri_merge_kernel(BodyKParams P) {
  using D = TriDims<NH>;
  constexpr int N = D::N, M = D::M, RSTR = D::RES + 2;     // 432-byte rows: 16-byte aligned for TMA, 12 banks apart
  constexpr int FSTR = D::FR + 2;
  static_assert((D::RES * sizeof(double)) % 16 == 0 && (D::FR * sizeof(double)) % 16 == 0, "records move as TMA bulk copies");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sres = reinterpret_cast<double*>(smem_raw);      // roll records [thread], pitch records [thread], hand-over records
  double* sfr = sres + (size_t)2 * TRI_MERGE_THREADS * RSTR;
  uint64_t* bar = reinterpret_cast<uint64_t*>(sfr + (size_t)TRI_MERGE_THREADS * FSTR);
  const int tid = threadIdx.x;
  const int idx = blockIdx.x * TRI_MERGE_THREADS + tid;
  if (idx == 0) { P.tri_qctl[0] = 0; P.tri_qctl[1] = 0; }  // queue counters for the next call on this stream (the merge count
                                                           // is cleared by a memset node behind this kernel: every CTA reads it)
  const int cnt = *reinterpret_cast<volatile const int*>(P.tri_qctl + 3);
  const bool mine = idx < cnt;                              // the setup kernel's list of unfinished instances, compact
  const int b = mine ? P.tri_meta[idx] : 0;
  if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
  const int nmine = __syncthreads_count(mine);
  if (nmine == 0) return;
  // every thread fetches its own records (2 x 416 + 192 bytes) with TMA onto one mbarrier: no other global load
  if (tid == 0) mbar_expect_tx(bar, (uint32_t)(nmine * (2 * D::RES + D::FR) * sizeof(double)));
  if (mine) {
    const double* src = P.tri_res + (size_t)2 * b * D::RES;
    tma_load_1d(sres + (size_t)tid * RSTR, src, (uint32_t)(D::RES * sizeof(double)), bar);
    tma_load_1d(sres + (size_t)(TRI_MERGE_THREADS + tid) * RSTR, src + D::RES, (uint32_t)(D::RES * sizeof(double)), bar);
    tma_load_1d(sfr + (size_t)tid * FSTR, P.tri_fr + (size_t)b * D::FR, (uint32_t)(D::FR * sizeof(double)), bar);
  }
  if (!mine) return;
  mbar_wait(bar, 0);
  const double* fr = sfr + (size_t)tid * FSTR;
  const double* rx = sres + (size_t)tid * RSTR;
  const double* ry = sres + (size_t)(TRI_MERGE_THREADS + tid) * RSTR;
  const int* ix = reinterpret_cast<const int*>(rx + D::RES_D);
  const int* iy = reinterpret_cast<const int*>(ry + D::RES_D);
  const double tol = fr[20];
  bool flag = ix[3] || iy[3];
  const double psi_x = rx[NH + 1], psi_y = ry[NH + 1];
  if (fabs(psi_x + psi_y) > tol && ((ix[2] && psi_x != 0.0) || (iy[2] && psi_y != 0.0))) flag = true;
  if (fmin(rx[NH + 3], ry[NH + 3]) <= EPS_D * fmax(rx[NH + 2], ry[NH + 2])) flag = true;
  for (int k = 0; k < NH; k++) if (rx[k] != rx[k] || ry[k] != ry[k]) flag = true;
  // ---- replay of the combined iteration (EiQuadProg.cpp:282-342 decides which half moves) ----
  const int nout_x = ix[0], nout_y = iy[0];
  const int np_x = ix[1], np_y = iy[1];
  bool broken = nout_x < 0 || nout_x > D::OMAX || nout_y < 0 || nout_y > D::OMAX || np_x < 0 || np_x > D::PMAX || np_y < 0 || np_y > D::PMAX;
  const double* ssx = rx + NH + 4; const double* ssy = ry + NH + 4;
  const int* ipx = ix + 4; const int* ipy = iy + 4;
  const int* plx = ix + 4 + D::OMAX; const int* ply = iy + 4 + D::OMAX;
  int Ac[N];
  int iqc = 0, it_outer = 0, it_add = 0, it_drop = 0, it_l2a = 0;
  unsigned flops = (unsigned)gi_flops_setup(N, 0);
  int ox = 0, oy = 0, px = 0, py = 0;
  while (!flag) {
    it_outer++;
    flops += 2u * N * M;
    const bool hx = ox < nout_x, hy = oy < nout_y;
    if ((!hx && !hy) || broken) break;
    bool pickx = hx;
    if (hx && hy) {
      const double a = ssx[ox], c = ssy[oy];
      pickx = (a < c) || (a == c && ipx[ox] < ipy[oy]);
    }
    for (;;) {
      if (pickx ? (px >= np_x) : (py >= np_y)) { broken = true; break; }   // a log that does not end in an add
      const int e = pickx ? plx[px++] : ply[py++];
      it_l2a++;
      flops += 2u * N * N + 2u * N * (N - iqc) + (unsigned)(iqc * iqc) + 4u * N + 2u * iqc;
      if (!(e & 0x10000)) {
        flops += 6u * N * (unsigned)(N - iqc - 1 > 0 ? N - iqc - 1 : 0);
        if (iqc < N) Ac[iqc] = e;
        iqc++; it_add++;
        break;
      }
      const int l = e & 0xffff;
      int qq = 0;
      for (int k = iqc - 1; k >= 0; k--) if (Ac[k] == l) qq = k;
      for (int k = qq; k < iqc - 1; k++) Ac[k] = Ac[k + 1];
      iqc--; it_drop++;
      flops += 3u * (unsigned)((iqc - qq) * (iqc - qq)) + 6u * N * (unsigned)(iqc - qq);
    }
    if (pickx) ox++; else oy++;
  }
  if (flag || broken) {      // not reproducible from the logs: the combined kernel takes the instance
    const int slot = atomicAdd(P.flist_count, 1);
    if (slot < P.flist_cap) P.flist[slot] = b;
    return;
  }
  tri_finish<NH>(P, b, fr, rx, ry, rx[NH] + ry[NH], iqc, it_outer, it_add, it_drop, it_l2a, flops, Ac);
}

// ======================================================================================= host side
bool body_tri_supported(int nh);
size_t body_tri_workspace_bytes(int nh, int B, size_t off[6]) {
  if (!body_tri_supported(nh)) return 0;
  using D = TriDims<10>;        // sized for the largest supported horizon: a stream's workspace serves every horizon
  size_t o = 0;
  off[0] = o; o += (size_t)B * D::JB * sizeof(double);
  off[1] = o; o += (size_t)2 * B * D::HS * sizeof(double);
  off[2] = o; o += (size_t)2 * B * D::RES * sizeof(double);
  off[3] = o; o += ((size_t)2 * B * sizeof(int) + 15) & ~(size_t)15;
  off[4] = o; o += ((size_t)B * sizeof(int) + 15) & ~(size_t)15;
  off[5] = o; o += (size_t)B * D::FR * sizeof(double);
  return o;
}

bool body_tri_supported(int nh) { return nh == 10 || nh == 4; }

template <int NH>
static cudaError_t tri_launch_nh(const BodyKParams& P, const double* tab_host, int sms, cudaStream_t st, cudaEvent_t* phase_ev) {
  using D = TriDims<NH>;
  constexpr int WPC = GO1_TRI_WPC;
  if (P.in_stride != D::IN || P.out_stride != D::OUT || P.tab_doubles != D::TAB) return cudaErrorInvalidValue;
  const int blocks = (P.B + TRI_SETUP_THREADS - 1) / TRI_SETUP_THREADS;
  const size_t ssmem = (size_t)TRI_SETUP_THREADS * D::IN * sizeof(double) + 16;
  // function attributes (opt-in dynamic shared memory) and occupancy are per device: one slot per device ordinal
  const size_t smem = (size_t)(((NH * NH + 1) & ~1) + WPC * 8 * D::GSP) * sizeof(double);
  const size_t msmem = (size_t)TRI_MERGE_THREADS * (2 * (D::RES + 2) + D::FR + 2) * sizeof(double) + 16;
  int dev_ = 0;
  cudaGetDevice(&dev_);
  dev_ &= 63;
  // per-device cache of the opt-in attributes and the solve kernel's occupancy; handles on several host threads
  // may launch concurrently, so the first use per device is serialised
  static std::mutex cache_mu;
  static int occ_[64] = {};
  int occ;
  {
    std::lock_guard<std::mutex> lk(cache_mu);
    if (occ_[dev_] == 0) {
      cudaError_t e = cudaFuncSetAttribute(tri_setup_kernel<NH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssmem);
      if (e != cudaSuccess) return e;
      e = cudaFuncSetAttribute(tri_solve_kernel<NH, WPC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
      e = cudaFuncSetAttribute(tri_merge_kernel<NH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem);
      if (e != cudaSuccess) return e;
      int o = 0;
      e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, tri_solve_kernel<NH, WPC>, WPC * 32, smem);
      if (e != cudaSuccess) return e;
      if (o < 1) return cudaErrorLaunchOutOfResources;
      occ_[dev_] = o;
    }
    occ = occ_[dev_];
  }
  TriTab<NH> T;
  memcpy(T.v, tab_host, sizeof(T.v));
  // phase_ev (optional, 4 events): recorded around the three launches, for bench.py's per-kernel roofline
  if (phase_ev) cudaEventRecord(phase_ev[0], st);
  tri_setup_kernel<NH><<<blocks, TRI_SETUP_THREADS, ssmem, st>>>(P, T);
  if (phase_ev) cudaEventRecord(phase_ev[1], st);
  int grid = (2 * P.B + WPC * 8 - 1) / (WPC * 8);
  {
    // A/B knob (GO1MPC_TRI_OCC = resident solve CTAs per SM the grid is sized for): smaller grids leave room for the solve
    // kernels of other streams and give every group several halves to balance its iteration counts over
    static const int occ_env = [] { const char* e = getenv("GO1MPC_TRI_OCC"); return e ? atoi(e) : 0; }();
    if (occ_env > 0 && occ_env < occ) occ = occ_env;
  }
  if (grid > sms * occ) grid = sms * occ;
  tri_solve_kernel<NH, WPC><<<grid, WPC * 32, smem, st>>>(P);
  if (phase_ev) cudaEventRecord(phase_ev[2], st);
  tri_merge_kernel<NH><<<(P.B + TRI_MERGE_THREADS - 1) / TRI_MERGE_THREADS, TRI_MERGE_THREADS, msmem, st>>>(P);
  cudaMemsetAsync(P.tri_qctl + 3, 0, sizeof(int), st);
  if (phase_ev) cudaEventRecord(phase_ev[3], st);
  return cudaGetLastError();
}

cudaError_t body_tri_launch(BodyKParams P, const double* tab_host, int sms, cudaStream_t st, cudaEvent_t* phase_ev) {
  switch (P.nh) {
    case 4: return tri_launch_nh<4>(P, tab_host, sms, st, phase_ev);       // the reference's own horizon (PRMPCClass.h:34)
    case 10: return tri_launch_nh<10>(P, tab_host, sms, st, phase_ev);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace go1
