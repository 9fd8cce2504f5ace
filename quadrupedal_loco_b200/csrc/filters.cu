// filters.cu -- the servo loop's signal filters for B robots x C channels, one thread per (channel, robot).
//
// Replaces (GO1 = unitree_ros/go1_rt_control):
//   butterworthLPF::filter            GO1/src/Filter/butterworthLPF.cpp:104-121 (coefficients: init :82-100, on the host)
//   ButterworthFilter::ForceFilter    GO1/src/Filter/butterworth_filter.cpp:37-69
// go1_servo runs 28 butterworthLPF objects on slots of the /MPC/Gait message every 1 kHz tick (servo.cpp:579-610, 898-931):
// here the C channels of a call are message slots, the state of all objects is one SoA buffer [5][C][B] (call counter, y_p,
// y_pp, x_p, x_pp) and a launch filters every channel of every robot.  Pure streaming: 7 doubles in, 6 out per sample, HBM
// bound.  Compiled with -fmad=false, the reference's left-to-right sums: bit-identical to the CPU oracle.
#include <cuda_runtime.h>
#include "kernels.h"
#include "servo_math.cuh"   // lpf_step

namespace go1 {

__global__ void __launch_bounds__(256) lpf_kernel(LpfKParams P) {
  const size_t B = (size_t)P.B, CB = (size_t)P.C * B;
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < CB; t += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(t / B);
    const size_t b = t - (size_t)c * B;
    const double* in = P.in + (size_t)(P.in_rows ? P.in_rows[c] : c) * B + b;
    double* S = P.state + t;
    const double y = *in;
    LpfState s{S[0], S[CB], S[2 * CB], S[3 * CB], S[4 * CB]};
    const bool counting = !(s.i > 2);
    const double out = lpf_step(P.coef[c], s, y);
    if (counting) S[0] = s.i;
    S[2 * CB] = s.y_pp; S[CB] = s.y_p; S[4 * CB] = s.x_pp; S[3 * CB] = s.x_p;
    P.out[t] = out;
  }
}

// state [6][C][B]: count | raw[0] raw[1] | filtered[0..2]
__global__ void __launch_bounds__(256) force_filter_kernel(int B, int C, const double* in, double* state, double* out) {
  const size_t CB = (size_t)C * B;
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < CB; t += (size_t)gridDim.x * blockDim.x) {
    double* S = state + t;
    const double x = in[t];
    const double cnt = S[0];
    double r0 = S[CB], r1 = S[2 * CB], f0 = S[3 * CB], f1 = S[4 * CB], f2 = S[5 * CB];
    if (cnt == 0) {
      f2 = x; r1 = x; S[0] = 1;
    } else if (cnt == 1) {
      f1 = f2; f2 = x; r0 = r1; r1 = x; S[0] = 2;
    } else {
      r0 = r1; r1 = x;
      f0 = f1; f1 = f2;
      f2 = 0.0 * r1 + 0.0521 * r0 - (-1.6498) * f1 - 0.7022 * f0;
    }
    S[CB] = r0; S[2 * CB] = r1; S[3 * CB] = f0; S[4 * CB] = f1; S[5 * CB] = f2;
    out[t] = f2;
  }
}

static int filter_grid(size_t n, int sms) {
  size_t g = (n + 255) / 256;
  const size_t cap = (size_t)sms * 8;
  return (int)(g < cap ? (g ? g : 1) : cap);
}
cudaError_t lpf_launch(LpfKParams P, int sms, cudaStream_t st) {
  lpf_kernel<<<filter_grid((size_t)P.B * P.C, sms), 256, 0, st>>>(P);
  return cudaGetLastError();
}
cudaError_t force_filter_launch(int B, int C, const double* in, double* state, double* out, int sms, cudaStream_t st) {
  force_filter_kernel<<<filter_grid((size_t)B * C, sms), 256, 0, st>>>(B, C, in, state, out);
  return cudaGetLastError();
}

}  // namespace go1
