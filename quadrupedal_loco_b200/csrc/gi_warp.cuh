// gi_warp.cuh -- warp-cooperative Goldfarb-Idnani dual active-set QP core (sm_100a, FP64).
//
// One warp solves one problem; all of the solver's state (J = L^-T, R, the
// duals, the working set) lives in that warp's slice of shared memory and never
// touches HBM.  Control flow is warp-uniform: every branch is taken on values
// that all 32 lanes hold identically (butterfly reductions, then a lane-0
// broadcast), so the data-dependent goto structure of the reference becomes a
// three-phase loop without divergence.
//
// Algorithm and every tie rule / tolerance follow the reference solver
//   Eigen::QP::solve_quadprog2  RT/src/utils/EiQuadProg/EiQuadProg.cpp:172-491
//   add_constraint :30-93, delete_constraint :95-170, helpers EiQuadProg.hpp:100-134
// (RT = unitree_ros/rt_mpc_qp).  What is re-designed for the GPU:
//   * lanes own rows of J for z = J2 d and for the Givens sweeps, and columns of
//     J for d = J' n+ (J is stored with an odd leading dimension so both access
//     patterns are shared-memory bank-conflict free);
//   * the chain of n-q-1 Givens rotations of add_constraint is replaced by one
//     Householder reflection built from the z already computed in step 2a (an
//     equivalent orthogonal update of the null-space basis, one parallel pass);
//   * the working-set membership vectors iai/iaexcl are per-lane bit masks in
//     registers (constraint c lives in lane c&31, bit c>>5);
//   * n+ is produced by a policy object, so a front-end with structured
//     constraints (body MPC) never materialises CI; the policy also gives the
//     non-zero range of n+ so d = J' n+ skips exact zeros.
// Rounding therefore differs from the CPU oracle in the last bits (FMA
// contraction, reduction trees); parity is checked at 1e-9 relative on x with
// an identical active set and identical iteration counters.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>

namespace go1 {

// The three multiply-adds below that the code writes as a*b+c follow the including file's -fmad setting: contracted in the
// default build (qp_dense.cu, body_*.cu, grf_qp.cu), rounded twice in the -fmad=false build of step_timing.cu.  A file built
// with -fmad=false that must reproduce the contracting build's bits (servo_torque.cu: grf_qp.cu's force QP) defines
// GO1_GI_FMA before the first include, which writes them as fma().
#ifdef GO1_GI_FMA
#define GI_MAD(a, b, c) fma((a), (b), (c))
#else
#define GI_MAD(a, b, c) ((a) * (b) + (c))
#endif

constexpr unsigned FULL_MASK = 0xffffffffu;
constexpr double EPS_D = 2.220446049250313e-16;

// status codes, numerically identical to include/go1mpc.h
enum { ST_OK = 0, ST_NOT_PD = 1, ST_INFEASIBLE = 2, ST_ITER_CAP = 3, ST_NAN = 4, ST_EQ_DEP = 5 };

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
  return __shfl_sync(FULL_MASK, v, 0);
}
// minimum value, lowest index among equal minima (the reference's strict '<' scan)
__device__ __forceinline__ void warp_argmin(double& v, int& idx) {
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    double ov = __shfl_xor_sync(FULL_MASK, v, o);
    int oi = __shfl_xor_sync(FULL_MASK, idx, o);
    if (ov < v || (ov == v && oi < idx)) { v = ov; idx = oi; }
  }
  v = __shfl_sync(FULL_MASK, v, 0);
  idx = __shfl_sync(FULL_MASK, idx, 0);
}

// The same arg-min with three integer warp reductions (REDUX): doubles are mapped to
// order-preserving unsigned 64-bit keys and reduced high word first.
__device__ __forceinline__ void warp_argmin_redux(double& v, int& idx) {
  unsigned long long k = (unsigned long long)__double_as_longlong(v);
  k ^= (k >> 63) ? 0xffffffffffffffffull : 0x8000000000000000ull;
  const unsigned hi = (unsigned)(k >> 32), lo = (unsigned)k;
  const unsigned mhi = __reduce_min_sync(FULL_MASK, hi);
  const unsigned mlo = __reduce_min_sync(FULL_MASK, hi == mhi ? lo : 0xffffffffu);
  const bool win = (hi == mhi) && (lo == mlo);
  idx = (int)__reduce_min_sync(FULL_MASK, win ? (unsigned)idx : 0xffffffffu);
  unsigned long long m = ((unsigned long long)mhi << 32) | mlo;
  m ^= (m >> 63) ? 0x8000000000000000ull : 0xffffffffffffffffull;
  v = __longlong_as_double((long long)m);
}

// EiQuadProg.hpp:100-118
__device__ __forceinline__ double gi_hypot(double a, double b) {
  double a1 = fabs(a), b1 = fabs(b), t;
  if (a1 > b1) { t = b1 / a1; return a1 * sqrt(GI_MAD(t, t, 1.0)); }
  if (b1 > a1) { t = a1 / b1; return b1 * sqrt(GI_MAD(t, t, 1.0)); }
  return a1 * sqrt(2.0);
}

// Per-warp workspace: pointers into the warp's shared-memory slice.
struct GiWs {
  int n, p, m, ld;      // ld: odd leading dimension of J and R (>= n)
  int ms;               // constraints the step-2 scan must look at (<= m; rows >= ms are identically 0)
  double* J;            // n x ld, column-major: J(i,j) = J[j*ld + i]
  double* R;            // n x ld, column-major upper triangular
  double* s;            // ms
  double *x, *xold, *z, *d, *np, *r, *u, *uold;  // n + 2 each
  double* rot;          // 4 * (n + 2): (cc, ss, xny, skip) per rotation
  int *A, *Aold;        // n + 2 each
};

__host__ __device__ inline int gi_ld(int n) { return n | 1; }
// doubles needed for one warp's workspace (ints are packed at the end)
__host__ __device__ inline int gi_ws_doubles(int n, int m) {
  int ld = gi_ld(n), v = n + 2;
  int d = 2 * n * ld + m + 8 * v + 4 * v;
  int ints = 2 * v;
  d += (ints + 1) / 2;
  return (d + 1) & ~1;  // even: keeps 16-byte alignment of what follows
}
__device__ inline void gi_ws_carve(GiWs& w, double* base, int n, int p, int m) {
  int ld = gi_ld(n), v = n + 2;
  w.n = n; w.p = p; w.m = m; w.ld = ld; w.ms = m;
  w.J = base; base += n * ld;
  w.R = base; base += n * ld;
  w.s = base; base += m;
  w.x = base; base += v;  w.xold = base; base += v;  w.z = base; base += v;
  w.d = base; base += v;  w.np = base; base += v;    w.r = base; base += v;
  w.u = base; base += v;  w.uold = base; base += v;
  w.rot = base; base += 4 * v;
  w.A = reinterpret_cast<int*>(base);
  w.Aold = w.A + v;
}

// d = J' n+ over the non-zero range [klo,khi) of n+     (EiQuadProg.hpp:121-124)
__device__ __forceinline__ void gi_compute_d(const GiWs& w, int klo, int khi, int lane) {
  for (int j = lane; j < w.n; j += 32) {
    const double* col = w.J + j * w.ld;
    double acc = 0.0;
    for (int k = klo; k < khi; k++) acc = fma(col[k], w.np[k], acc);
    w.d[j] = acc;
  }
  __syncwarp();
}
// z = J[:, iq:] d[iq:]                                    (EiQuadProg.hpp:126-129)
__device__ __forceinline__ void gi_update_z(const GiWs& w, int iq, int lane) {
  for (int k = lane; k < w.n; k += 32) {
    double acc = 0.0;
    for (int j = iq; j < w.n; j++) acc = fma(w.J[j * w.ld + k], w.d[j], acc);
    w.z[k] = acc;
  }
  __syncwarp();
}
// r[0..iq) = R[0..iq,0..iq)^-1 d[0..iq), column-oriented  (EiQuadProg.hpp:131-134)
__device__ __forceinline__ void gi_update_r(const GiWs& w, int iq, int lane) {
  for (int t = lane; t < iq; t += 32) w.r[t] = w.d[t];
  __syncwarp();
  for (int i = iq - 1; i >= 0; i--) {
    double ri = w.r[i] / w.R[i * w.ld + i];
    __syncwarp();
    for (int t = lane; t < i; t += 32) w.r[t] = fma(-ri, w.R[i * w.ld + t], w.r[t]);
    if (lane == 0) w.r[i] = ri;
    __syncwarp();
  }
}

// EiQuadProg.cpp:30-93.  The reference zeroes d[iq+1:] with a chain of n-iq-1 Givens rotations of J's
// trailing columns; any orthogonal map sending d2 = d[iq:] to a multiple of e_0 yields an equivalent
// null-space basis, so ONE Householder reflection H = I - tau v v', v = d2 + sigma e_0,
// sigma = sign(d_iq)|d2| is used: J2 <- J2 - tau (J2 v) v' with J2 v = z + sigma J(:,iq), where
// z = J2 d2 is still in w.z from step 2a -- a single dependency-free pass, rows per lane.
// On return d[iq_old] = -sigma, d[j > iq_old] = 0, R(:, iq_old) = d[0..iq_old].
__device__ inline bool gi_add_constraint(const GiWs& w, int& iq, double& R_norm, int lane) {
  const int n = w.n, ld = w.ld;
  double dd = 0.0;
  for (int j = iq + lane; j < n; j += 32) dd = fma(w.d[j], w.d[j], dd);
  dd = warp_sum(dd);
  const double nrm = sqrt(dd);
  const double diq = w.d[iq];
  const double sigma = (diq < 0.0) ? -nrm : nrm;
  __syncwarp();
  if (nrm != 0.0) {
    const double tau = 1.0 / (nrm * (nrm + fabs(diq)));
    const double viq = diq + sigma;
    for (int k = lane; k < n; k += 32) {
      const double sw = tau * fma(sigma, w.J[iq * ld + k], w.z[k]);
      w.J[iq * ld + k] = fma(-sw, viq, w.J[iq * ld + k]);
      for (int j = iq + 1; j < n; j++) w.J[j * ld + k] = fma(-sw, w.d[j], w.J[j * ld + k]);
    }
    __syncwarp();
    if (lane == 0) w.d[iq] = -sigma;
    for (int j = iq + 1 + lane; j < n; j += 32) w.d[j] = 0.0;
  }
  __syncwarp();
  iq++;
  for (int t = lane; t < iq; t += 32) w.R[(iq - 1) * ld + t] = w.d[t];
  const double dq = w.d[iq - 1];
  __syncwarp();
  if (fabs(dq) <= EPS_D * R_norm) return false;  // degenerate
  R_norm = fmax(R_norm, fabs(dq));
  return true;
}

// EiQuadProg.cpp:95-170.  Returns false when l is not in A[p..iq) (UB in the reference).
__device__ inline bool gi_delete_constraint(const GiWs& w, int& iq, int l, int lane, int& qq) {
  const int n = w.n, ld = w.ld, p = w.p;
  qq = -1;
  for (int base = p; base < iq; base += 32) {
    int i = base + lane;
    unsigned hit = __ballot_sync(FULL_MASK, i < iq && w.A[i] == l);
    if (hit) { qq = base + __ffs(hit) - 1; break; }
  }
  if (qq < 0) return false;
  // shift A, u down by one (ascending chunks: read, sync, write)
  for (int base = qq; base < iq - 1; base += 32) {
    int i = base + lane;
    int a = 0; double uu = 0.0;
    if (i < iq - 1) { a = w.A[i + 1]; uu = w.u[i + 1]; }
    __syncwarp();
    if (i < iq - 1) { w.A[i] = a; w.u[i] = uu; }
    __syncwarp();
  }
  // R columns shift left; lane t touches row t only
  for (int i = qq; i < iq - 1; i++)
    for (int t = lane; t < n; t += 32) w.R[i * ld + t] = w.R[(i + 1) * ld + t];
  if (lane == 0) {
    w.A[iq - 1] = w.A[iq]; w.u[iq - 1] = w.u[iq];
    w.A[iq] = 0; w.u[iq] = 0.0;
  }
  for (int t = lane; t < iq; t += 32) w.R[(iq - 1) * ld + t] = 0.0;
  iq--;
  __syncwarp();
  if (iq == 0) return true;
  for (int j = qq; j < iq; j++) {
    double cc = w.R[j * ld + j], ss = w.R[j * ld + j + 1];
    double h = gi_hypot(cc, ss);
    __syncwarp();
    if (h == 0.0) continue;
    cc = cc / h; ss = ss / h;
    if (lane == 0) { w.R[j * ld + j + 1] = 0.0; w.R[j * ld + j] = (cc < 0.0) ? -h : h; }
    if (cc < 0.0) { cc = -cc; ss = -ss; }
    double xny = ss / (1.0 + cc);
    for (int k = j + 1 + lane; k < iq; k += 32) {
      double t1 = w.R[k * ld + j], t2 = w.R[k * ld + j + 1];
      double a = fma(t2, ss, t1 * cc);
      w.R[k * ld + j] = a;
      w.R[k * ld + j + 1] = fma(xny, t1 + a, -t2);
    }
    for (int k = lane; k < n; k += 32) {
      double t1 = w.J[j * ld + k], t2 = w.J[(j + 1) * ld + k];
      double a = fma(t2, ss, t1 * cc);
      w.J[j * ld + k] = a;
      w.J[(j + 1) * ld + k] = fma(xny, a + t1, -t2);
    }
    __syncwarp();
  }
  return true;
}

// In-place lower Cholesky of the n x n matrix in w.R (ld = w.ld), unblocked
// left-looking, lanes own rows.  Returns false when not PD.
__device__ inline bool gi_llt(const GiWs& w, int n, int lane) {
  const int ld = w.ld;
  double* L = w.R;
  for (int k = 0; k < n; k++) {
    // v_i = L(i,k) - sum_{j<k} L(i,j) L(k,j) for rows i >= k
    for (int i = k + lane; i < n; i += 32) {
      double t = 0.0;
      for (int j = 0; j < k; j++) t = fma(L[j * ld + i], L[j * ld + k], t);
      L[k * ld + i] = L[k * ld + i] - t;
    }
    __syncwarp();
    double x = L[k * ld + k];
    __syncwarp();
    if (!(x > 0.0) && !(x != x)) return false;  // x <= 0 (NaN passes through, as in the reference)
    double sq = sqrt(x);
    for (int i = k + lane; i < n; i += 32) L[k * ld + i] = (i == k) ? sq : L[k * ld + i] / sq;
    __syncwarp();
  }
  return true;
}

// J = L^-T for the leading nb x nb block of L (in w.R), written at J(off.., off..);
// lanes own columns.  J must have been zeroed.
__device__ inline void gi_inv_lt(const GiWs& w, int nb, int off, int lane) {
  const int ld = w.ld;
  const double* L = w.R;
  for (int c = lane; c < nb; c += 32) {
    double* col = w.J + (off + c) * ld + off;
    for (int i = c; i >= 0; i--) {
      double t = 0.0;
      for (int k = i + 1; k <= c; k++) t = fma(L[i * ld + k], col[k], t);
      col[i] = ((i == c ? 1.0 : 0.0) - t) / L[i * ld + i];
    }
  }
  __syncwarp();
}

// Constraint policy concept:
//   void eval_s(const GiWs& w, int lane, double& psi_part)  -- s[c] for the lane's constraints c = lane + 32 t
//   void load_np(const GiWs& w, int ip, int lane, int& klo, int& khi) -- n+ = CI(:, ip) into w.np (ends with __syncwarp)
//   double eval_one(const GiWs& w, int ip, int lane)        -- CI(:,ip).x + ci0(ip), warp-uniform result
//   void load_eq(const GiWs& w, int i, int lane, bool& allzero) -- n+ = CE(:, i)   (only used when p > 0)
//   double ce0(int i)
// it_l2a counts passes through step 2a; flops is the ALGORITHMIC flop count of the dense
// reference algorithm for the path this problem took (SURVEY.md section 8d formula, one
// multiply-add = 2 flop) -- what bench.py's roofline uses, not the instructions executed.
struct GiResult { double f; int iq; int status; int it_outer, it_add, it_drop, it_degen, it_l2a; unsigned long long flops; };

__host__ __device__ inline unsigned long long gi_flops_setup(int n, int p) {
  unsigned long long N = n;
  return N * N * N / 3 + N * N * N / 3 + 2 * N * N + (unsigned long long)p * 4 * N * N;
}

// Main loop.  Requires: w.J = L^-T, w.R = 0, w.x = unconstrained minimiser, res.f = its cost.
template <class Pol>
__device__ inline void gi_loop(const GiWs& w, Pol& pol, double c1, double c2, int cap, GiResult& res, int lane) {
  const int n = w.n, m = w.m, me = w.p;
  const double inf = CUDART_INF;
  double R_norm = 1.0, f_value = res.f;
  int iq = 0, status = ST_OK;
  int it_outer = 0, it_add = 0, it_drop = 0, it_degen = 0, it_l2a = 0, qq = 0;
  unsigned long long flops = res.flops;
  unsigned inA = 0u, excl = 0u;  // bit t <-> constraint lane + 32 t

  for (int t = lane; t < n + 2; t += 32) { w.u[t] = 0.0; w.uold[t] = 0.0; w.A[t] = 0; w.Aold[t] = 0; w.r[t] = 0.0; }
  __syncwarp();

  // EiQuadProg.cpp:236-276 equality constraints
  for (int i = 0; i < me; i++) {
    bool allzero;
    pol.load_eq(w, i, lane, allzero);
    if (allzero) continue;
    gi_compute_d(w, 0, n, lane);
    gi_update_z(w, iq, lane);
    gi_update_r(w, iq, lane);
    double zz = 0.0, zn = 0.0, nx = 0.0;
    for (int k = lane; k < n; k += 32) { zz = fma(w.z[k], w.z[k], zz); zn = fma(w.z[k], w.np[k], zn); nx = fma(w.np[k], w.x[k], nx); }
    zz = warp_sum(zz); zn = warp_sum(zn); nx = warp_sum(nx);
    double t2 = 0.0;
    if (fabs(zz) > EPS_D) t2 = (-nx - pol.ce0(i)) / zn;
    for (int k = lane; k < n; k += 32) w.x[k] = fma(t2, w.z[k], w.x[k]);
    for (int k = lane; k < iq; k += 32) w.u[k] = fma(-t2, w.r[k], w.u[k]);
    if (lane == 0) { w.u[iq] = t2; w.A[i] = -i - 1; }
    f_value = GI_MAD(0.5 * (t2 * t2), zn, f_value);
    __syncwarp();
    if (!gi_add_constraint(w, iq, R_norm, lane)) { status = ST_EQ_DEP; goto done; }
  }

  {
    enum { PH_L1, PH_L2, PH_L2A };
    int phase = PH_L1, ip = 0, l = 0, passes = 0, klo = 0, khi = n;
    double ss = 0.0;
    for (;;) {
      if (phase == PH_L1) {
        // EiQuadProg.cpp:282-320
        it_outer++;
        flops += 2ull * n * m;
        for (int i = me; i < iq; i++) { int c = w.A[i]; if ((c & 31) == lane) inA |= 1u << (c >> 5); }
        excl = 0u;
        double psi = 0.0;
        pol.eval_s(w, lane, psi);
        psi = warp_sum(psi);
        ss = 0.0; ip = 0;
        __syncwarp();
        if (fabs(psi) <= m * EPS_D * c1 * c2 * 100.0) break;
        for (int t = lane; t < iq; t += 32) { w.uold[t] = w.u[t]; w.Aold[t] = w.A[t]; }
        for (int k = lane; k < n; k += 32) w.xold[k] = w.x[k];
        __syncwarp();
        phase = PH_L2;
      }
      if (phase == PH_L2) {
        // EiQuadProg.cpp:322-342: most negative eligible s, first index wins
        double bv = ss; int bi = 0x7fffffff;
        for (int c = lane, t = 0; c < w.ms; c += 32, t++) {
          double sv = w.s[c];
          if (sv < bv && !((inA >> t) & 1u) && !((excl >> t) & 1u)) { bv = sv; bi = c; }
        }
        warp_argmin_redux(bv, bi);
        if (bv < ss) { ss = bv; ip = bi; }
        if (ss >= 0.0) break;
        pol.load_np(w, ip, lane, klo, khi);
        if (lane == 0) { w.u[iq] = 0.0; w.A[iq] = ip; }
        __syncwarp();
        phase = PH_L2A;
      }
      // PH_L2A: EiQuadProg.cpp:349-490
      if (++passes > cap) { status = ST_ITER_CAP; break; }
      it_l2a++;
      flops += 2ull * n * n + 2ull * n * (n - iq) + (unsigned long long)iq * iq + 4ull * n + 2ull * iq;
      gi_compute_d(w, klo, khi, lane);
      gi_update_z(w, iq, lane);
      gi_update_r(w, iq, lane);
      // step lengths
      double t1 = inf; int kmin = 0x7fffffff;
      for (int k = me + lane; k < iq; k += 32) {
        double rk = w.r[k];
        if (rk > 0.0) { double tmp = w.u[k] / rk; if (tmp < t1) { t1 = tmp; kmin = k; } }
      }
      warp_argmin_redux(t1, kmin);
      l = (kmin != 0x7fffffff && t1 < inf) ? w.A[kmin] : 0;
      double zz = 0.0, zn = 0.0;
      for (int k = lane; k < n; k += 32) { zz = fma(w.z[k], w.z[k], zz); zn = fma(w.z[k], w.np[k], zn); }
      zz = warp_sum(zz); zn = warp_sum(zn);
      double t2 = (fabs(zz) > EPS_D) ? (-w.s[ip] / zn) : inf;
      double t = fmin(t1, t2);
      if (t >= inf) { status = ST_INFEASIBLE; f_value = inf; break; }      // case (i)
      if (t2 >= inf) {                                                      // case (ii): dual step
        for (int k = lane; k < iq; k += 32) w.u[k] = fma(-t, w.r[k], w.u[k]);
        if (lane == 0) w.u[iq] += t;
        if ((l & 31) == lane) inA &= ~(1u << (l >> 5));
        __syncwarp();
        if (!gi_delete_constraint(w, iq, l, lane, qq)) { status = ST_ITER_CAP; break; }
        it_drop++;
        flops += 3ull * (iq - qq) * (iq - qq) + 6ull * n * (iq - qq);
        continue;
      }
      // case (iii): step in primal and dual space
      double uiq = w.u[iq];
      __syncwarp();
      for (int k = lane; k < n; k += 32) w.x[k] = fma(t, w.z[k], w.x[k]);
      f_value = GI_MAD(t * zn, GI_MAD(0.5, t, uiq), f_value);
      for (int k = lane; k < iq; k += 32) w.u[k] = fma(-t, w.r[k], w.u[k]);
      if (lane == 0) w.u[iq] = uiq + t;
      __syncwarp();
      if (t == t2) {
        flops += 6ull * n * (n - iq - 1 > 0 ? n - iq - 1 : 0);
        if (!gi_add_constraint(w, iq, R_norm, lane)) {
          // EiQuadProg.cpp:444-462 degenerate: exclude ip, restore the state saved at l1
          it_degen++;
          if ((ip & 31) == lane) excl |= 1u << (ip >> 5);
          if (!gi_delete_constraint(w, iq, ip, lane, qq)) { status = ST_ITER_CAP; break; }
          inA = 0u;
          for (int t3 = lane; t3 < iq; t3 += 32) { w.A[t3] = w.Aold[t3]; w.u[t3] = w.uold[t3]; }
          for (int k = lane; k < n; k += 32) w.x[k] = w.xold[k];
          __syncwarp();
          for (int i = 0; i < iq; i++) { int c = w.A[i]; if (c >= 0 && (c & 31) == lane) inA |= 1u << (c >> 5); }
          phase = PH_L2;
          continue;
        }
        it_add++;
        if ((ip & 31) == lane) inA |= 1u << (ip >> 5);
        phase = PH_L1;
        continue;
      }
      // partial step: drop l, recompute s(ip), stay in 2a   (EiQuadProg.cpp:477-490)
      if ((l & 31) == lane) inA &= ~(1u << (l >> 5));
      if (!gi_delete_constraint(w, iq, l, lane, qq)) { status = ST_ITER_CAP; break; }
      it_drop++;
      flops += 3ull * (iq - qq) * (iq - qq) + 6ull * n * (iq - qq);
      {
        double sv = pol.eval_one(w, ip, lane);
        if (lane == 0) w.s[ip] = sv;
        __syncwarp();
      }
    }
  }
done:
  res.f = f_value; res.iq = iq; res.status = status;
  res.it_outer = it_outer; res.it_add = it_add; res.it_drop = it_drop; res.it_degen = it_degen;
  res.it_l2a = it_l2a; res.flops = flops;
}

}  // namespace go1
