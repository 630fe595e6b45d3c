// Issue rates of the fp32 instruction forms the fused step kernel is made of (cycles per warp instruction per SM
// sub-partition, 8 warps per scheduler, 8 independent chains per thread):  nvcc -arch=sm_100a -o fma_rates fma_rates.cu
#include <cstdio>
#include <cuda_runtime.h>
typedef unsigned long long u64;
__constant__ float c_coef[4] = {1.0001f, 0.9999f, 1.0002f, 0.9998f};
#define REP 8
#define ITERS 2048
template <int V>
__global__ void __launch_bounds__(1024, 1) rate_kernel(float s, float t, u64* out, long long* cyc) {
  float a[REP], b[REP];
  u64 p[REP], q[REP];
  const float x0 = 1.f + threadIdx.x * 1e-6f;
  const u64 ss = ((u64)__float_as_uint(s) << 32) | __float_as_uint(s);
  const float su = c_coef[(int)t & 3];
#pragma unroll
  for (int i = 0; i < REP; ++i) {
    a[i] = x0 + i; b[i] = 0.999f + i * 1e-7f + threadIdx.x * 1e-9f;
    p[i] = ((u64)__float_as_uint(x0) << 32) | __float_as_uint(x0 + i); q[i] = ((u64)__float_as_uint(0.999f + threadIdx.x * 1e-9f) << 32) | __float_as_uint(0.9991f + i * 1e-6f);
  }
  __syncthreads();
  const long long t0 = clock64();
  for (int it = 0; it < ITERS; ++it) {
#pragma unroll
    for (int i = 0; i < REP; ++i) {
      if (V == 0) asm volatile("fma.rn.f32 %0, %0, %1, %2;" : "+f"(a[i]) : "f"(b[i]), "f"(b[(i + 1) % REP]));
      if (V == 1) asm volatile("fma.rn.f32 %0, %0, 0f3F7FF972, %1;" : "+f"(a[i]) : "f"(b[i]));
      if (V == 2) asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(p[i]) : "l"(q[i]), "l"(q[(i + 1) % REP]));
      if (V == 3) asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(p[i]) : "l"(q[i]), "l"(ss));
      if (V == 4) asm volatile("mul.rn.f32x2 %0, %0, %1;" : "+l"(p[i]) : "l"(q[i]));
      if (V == 5) asm volatile("add.sat.f32 %0, %0, %1;" : "+f"(a[i]) : "f"(b[i]));
      if (V == 6) { asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(p[i]) : "l"(q[i]), "l"(q[(i + 1) % REP]));
                    asm volatile("max.f32 %0, %0, %1;" : "+f"(a[i]) : "f"(b[i])); }
      if (V == 7) { asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(p[i]) : "l"(q[i]), "l"(q[(i + 1) % REP]));
                    asm volatile("add.f32 %0, %0, %1;" : "+f"(a[i]) : "f"(b[i])); }
      if (V == 8) asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(a[i]));
      if (V == 9) { asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(p[i]) : "l"(q[i]), "l"(ss));
                    asm volatile("max.f32 %0, %0, %1;" : "+f"(a[i]) : "f"(b[i])); }
      if (V == 10) asm volatile("add.f32 %0, %0, %1;" : "+f"(a[i]) : "f"(b[i]));
      if (V == 11) asm volatile("max.f32 %0, %0, %1;" : "+f"(a[i]) : "f"(b[i]));
      if (V == 12) asm volatile("add.rn.f32x2 %0, %0, %1;" : "+l"(p[i]) : "l"(q[i]));
      if (V == 13) { asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(p[i]) : "l"(q[i]), "l"(q[(i + 1) % REP]));
                     asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(q[i]) : "l"(p[i]), "l"(ss));
                     asm volatile("max.f32 %0, %0, %1;" : "+f"(a[i]) : "f"(b[i])); }
      // a coefficient from the constant bank: the step kernel reads it as FFMA R,R,UR,R; in this short loop ptxas keeps it in
      // a vector register instead, read through the operand reuse cache (no register-bank read either way)
      if (V == 14) a[i] = fmaf(a[i], su, b[i]);
    }
  }
  const long long t1 = clock64();
  u64 acc = 0;
#pragma unroll
  for (int i = 0; i < REP; ++i) acc += p[i] + q[i] + __float_as_uint(a[i]) + __float_as_uint(b[i]);
  out[blockIdx.x * blockDim.x + threadIdx.x] = acc + (u64)t;
  if (threadIdx.x == 0) cyc[blockIdx.x] = t1 - t0;
}
template <int V>
static void run(const char* name, int per_iter, u64* out, long long* cyc) {
  rate_kernel<V><<<148, 1024>>>(1.0001f, 0.f, out, cyc);
  rate_kernel<V><<<148, 1024>>>(1.0001f, 0.f, out, cyc);
  cudaDeviceSynchronize();
  long long h[148];
  cudaMemcpy(h, cyc, sizeof(h), cudaMemcpyDeviceToHost);
  double m = 0;
  for (int i = 0; i < 148; ++i) m += (double)h[i] / 148;
  const double warp_inst_per_smsp = 8.0 * ITERS * REP * per_iter;     // 32 warps per SM = 8 per scheduler
  printf("%-44s %6.3f cycles per warp instruction per scheduler (%s)\n", name, m / warp_inst_per_smsp, cudaGetErrorString(cudaGetLastError()));
}
int main() {
  u64* out; long long* cyc;
  cudaMalloc(&out, 148 * 1024 * 8); cudaMalloc(&cyc, 148 * 8);
  run<0>("FFMA  R,R,R", 1, out, cyc);
  run<1>("FFMA  R,imm,R", 1, out, cyc);
  run<14>("FFMA  R,coefficient (R.reuse),R", 1, out, cyc);
  run<2>("FFMA2 R,R,R", 1, out, cyc);
  run<3>("FFMA2 R,uniform pair,R", 1, out, cyc);
  run<4>("FMUL2 R,R", 1, out, cyc);
  run<12>("FADD2 R,R", 1, out, cyc);
  run<10>("FADD  R,R", 1, out, cyc);
  run<5>("FADD.SAT R,R", 1, out, cyc);
  run<11>("FMNMX R,R", 1, out, cyc);
  run<8>("MUFU.EX2", 1, out, cyc);
  run<6>("FFMA2 rrr + FMNMX (per pair)", 2, out, cyc);
  run<7>("FFMA2 rrr + FADD (per pair)", 2, out, cyc);
  run<9>("FFMA2 r,u,r + FMNMX (per pair)", 2, out, cyc);
  run<13>("2 FFMA2 + FMNMX (per triple)", 3, out, cyc);
  return 0;
}
