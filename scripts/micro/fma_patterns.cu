// The two FMA-heavy phases of the fused step kernel as packed (FFMA2) and as scalar (FFMA) code: cycles per pixel pair
// and scheduler with 4 warps per scheduler.  (a) gradient accumulation acc[c][i] += e_c * phi_i (all vector registers):
// one sum per pixel column (packed or scalar) or both pixels of the pair folded into one sum, (b) polynomial forward u_c = sum_i q[c][i] * phi_i with the coefficients in uniform registers.
#include <cstdio>
#include <cuda_runtime.h>
#define ITERS 4096
struct Coef { float q[30]; };
template <int V>
__global__ void __launch_bounds__(512, 1) pat_kernel(Coef cf, float* out, long long* cyc) {
  const float x0 = 1.f + threadIdx.x * 1e-6f;
  float2 phi[9], e[3], acc[27];
  float sphi[18], se[6], sacc[54];
#pragma unroll
  for (int i = 0; i < 9; ++i) { phi[i] = make_float2(x0 + i * 0.01f, x0 - i * 0.01f); sphi[2 * i] = phi[i].x; sphi[2 * i + 1] = phi[i].y; }
#pragma unroll
  for (int c = 0; c < 3; ++c) { e[c] = make_float2(1e-3f * (c + 1) + x0 * 1e-4f, -1e-3f * (c + 1) - x0 * 2e-4f); se[2 * c] = e[c].x; se[2 * c + 1] = e[c].y; }
#pragma unroll
  for (int i = 0; i < 27; ++i) { acc[i] = make_float2(0.f, 0.f); sacc[2 * i] = 0.f; sacc[2 * i + 1] = 0.f; }
  __shared__ float2 sh[9][512];
#pragma unroll
  for (int i = 0; i < 9; ++i) sh[i][threadIdx.x] = phi[i];
  volatile float2* vsh = &sh[0][0];
  __syncthreads();
  const long long t0 = clock64();
  for (int it = 0; it < ITERS; ++it) {
    if (V == 0) {          // packed accumulate: 27 FFMA2 per pair
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < 9; ++i) acc[c * 9 + i] = __ffma2_rn(e[c], phi[i], acc[c * 9 + i]);
    } else if (V == 1) {   // scalar accumulate: 54 FFMA per pair
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < 9; ++i) {
          sacc[2 * (c * 9 + i)] = fmaf(se[2 * c], sphi[2 * i], sacc[2 * (c * 9 + i)]);
          sacc[2 * (c * 9 + i) + 1] = fmaf(se[2 * c + 1], sphi[2 * i + 1], sacc[2 * (c * 9 + i) + 1]);
        }
    } else if (V == 2) {   // packed polynomial forward: 27 FFMA2 (uniform coefficient) per pair
      float2 u[3];
#pragma unroll
      for (int i = 0; i < 9; ++i) { phi[i].x = vsh[i * 512 + threadIdx.x].x; phi[i].y = vsh[i * 512 + threadIdx.x].y; }
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        u[c] = __ffma2_rn(make_float2(cf.q[c * 10], cf.q[c * 10]), phi[0], make_float2(cf.q[c * 10 + 9], cf.q[c * 10 + 9]));
#pragma unroll
        for (int i = 1; i < 9; ++i) u[c] = __ffma2_rn(make_float2(cf.q[c * 10 + i], cf.q[c * 10 + i]), phi[i], u[c]);
      }
      acc[0] = __fadd2_rn(acc[0], u[0]); acc[1] = __fadd2_rn(acc[1], u[1]); acc[2] = __fadd2_rn(acc[2], u[2]);
    } else if (V == 3) {   // scalar polynomial forward: 54 FFMA per pair
      float u[6];
#pragma unroll
      for (int i = 0; i < 9; ++i) { sphi[2 * i] = vsh[i * 512 + threadIdx.x].x; sphi[2 * i + 1] = vsh[i * 512 + threadIdx.x].y; }
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float t = fmaf(cf.q[c * 10], sphi[h], cf.q[c * 10 + 9]);
#pragma unroll
          for (int i = 1; i < 9; ++i) t = fmaf(cf.q[c * 10 + i], sphi[2 * i + h], t);
          u[2 * c + h] = t;
        }
#pragma unroll
      for (int k = 0; k < 6; ++k) sacc[k] += u[k];
    } else if (V == 4) {   // mixed accumulate: channel 0 packed, channels 1, 2 scalar
#pragma unroll
      for (int i = 0; i < 9; ++i) acc[i] = __ffma2_rn(e[0], phi[i], acc[i]);
#pragma unroll
      for (int c = 1; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < 9; ++i) {
          sacc[2 * (c * 9 + i)] = fmaf(se[2 * c], sphi[2 * i], sacc[2 * (c * 9 + i)]);
          sacc[2 * (c * 9 + i) + 1] = fmaf(se[2 * c + 1], sphi[2 * i + 1], sacc[2 * (c * 9 + i) + 1]);
        }
    } else if (V == 5) {   // folded accumulate: 54 FFMA per pair into 27 sums, acc = fma(e.y, phi.y, fma(e.x, phi.x, acc))
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < 9; ++i)
          sacc[c * 9 + i] = fmaf(se[2 * c + 1], sphi[2 * i + 1], fmaf(se[2 * c], sphi[2 * i], sacc[c * 9 + i]));
    }
  }
  const long long t1 = clock64();
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 27; ++i) s += acc[i].x + acc[i].y + sacc[2 * i] + sacc[2 * i + 1];
#pragma unroll
  for (int i = 0; i < 9; ++i) s += phi[i].x + phi[i].y + sphi[2 * i] + sphi[2 * i + 1];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
  if (threadIdx.x == 0) cyc[blockIdx.x] = t1 - t0;
}
template <int V>
static void run(const char* name, float* out, long long* cyc) {
  Coef cf;
  for (int i = 0; i < 30; ++i) cf.q[i] = 0.01f * (i % 7) - 0.02f;
  pat_kernel<V><<<148, 512>>>(cf, out, cyc);
  pat_kernel<V><<<148, 512>>>(cf, out, cyc);
  cudaDeviceSynchronize();
  long long h[148];
  cudaMemcpy(h, cyc, sizeof(h), cudaMemcpyDeviceToHost);
  double m = 0;
  for (int i = 0; i < 148; ++i) m += (double)h[i] / 148;
  printf("%-52s %7.2f cycles per pixel pair per scheduler (%s)\n", name, m / (4.0 * ITERS), cudaGetErrorString(cudaGetLastError()));
}
int main() {
  float* out; long long* cyc;
  cudaMalloc(&out, 148 * 512 * 4); cudaMalloc(&cyc, 148 * 8);
  run<0>("accumulate 3x9, packed (27 FFMA2 r,r,r)", out, cyc);
  run<1>("accumulate 3x9, scalar (54 FFMA r,r,r)", out, cyc);
  run<5>("accumulate 3x9, folded (54 FFMA r,r,r, 27 sums)", out, cyc);
  run<4>("accumulate 3x9, 1 channel packed + 2 scalar", out, cyc);
  run<2>("polynomial forward, packed (27 FFMA2 r,u,r)", out, cyc);
  run<3>("polynomial forward, scalar (54 FFMA r,u,r)", out, cyc);
  return 0;
}
