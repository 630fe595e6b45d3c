// Shared device/host helpers for the reconfigisp_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/reconfigisp_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "reconfigisp_b200 is written for sm_100a (B200) only"
#endif

namespace risp {

// ---- error plumbing -------------------------------------------------------------------
void set_error(const char* fmt, ...);
int check_launch(const char* what);  // cudaGetLastError() -> RISP_OK / RISP_E_CUDA
int sm_count();

#define RISP_REQUIRE(cond, code, ...)          \
  do {                                         \
    if (!(cond)) {                             \
      ::risp::set_error(__VA_ARGS__);          \
      return (code);                           \
    }                                          \
  } while (0)

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline cudaStream_t as_stream(risp_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
static inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }

// ---- chain descriptor passed by value (lands in the constant bank) ---------------------
struct ChainDesc {
  int S;
  int op[RISP_MAX_STAGES];
  int off[RISP_MAX_STAGES];
  int iarg[RISP_MAX_STAGES];
};

int op_param_count(int op, int iarg);  // -1 for an unknown op
bool op_has_bwd(int op);
// validates and fills d; returns RISP_OK or error. P_needed = max(off+count).
int make_chain(ChainDesc* d, const int* ops, const int* off, const int* iarg, int S, int* P_needed);

#ifdef __CUDACC__
// ---- streaming loads / stores (read-once data: keep it out of L1) -------------------------
__device__ __forceinline__ float4 ld_stream4(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ float2 ld_stream2(const float* p) {
  float2 v;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream1(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void st_stream4(float* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_stream2(float* p, float2 v) {
  asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1,%2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float sat01(float v) { return __saturatef(v); }   // one .SAT instruction (NaN -> 0)
// 8-bit display code of tensor2bgr (utils/util.py:118-135): trunc(clip(fl32(v*255), 0, 255)), NaN -> 0, the codes of
// risp_to_u8_hwc.  Same value as fl32(sat(v)*255) (sat first or clip after the rounded product: both give 0 / 255 outside
// [0,1] and the same product inside), truncated without F2I: adding 2^23 rounding toward zero leaves trunc(x) in the low
// mantissa bits for 0 <= x < 2^23.  FMUL + FADD.RZ on the FMA pipe instead of a conversion on the quarter-rate XU pipe, which
// the gamma's lg2 / ex2 already load (the difference of two codes cancels the exponent bits).
__device__ __forceinline__ int u8_code(float v) {
  return __float_as_int(__fadd_rz(__fmul_rn(__saturatef(v), 255.f), 8388608.f)) - 0x4B000000;
}
// squared code differences of 4 pixels of one channel: <= 4 * 255^2, exact in 32 bits
__device__ __forceinline__ uint32_t sq_codes4(float4 y, float4 t) {
  const int d0 = u8_code(y.x) - u8_code(t.x), d1 = u8_code(y.y) - u8_code(t.y);
  const int d2 = u8_code(y.z) - u8_code(t.z), d3 = u8_code(y.w) - u8_code(t.w);
  return (uint32_t)(d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3);
}
__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// torch.clamp backward mask is inclusive on both ends
__device__ __forceinline__ float in01(float v) { return (v >= 0.f && v <= 1.f) ? 1.f : 0.f; }
#endif

// Accumulator slot layout shared by the chain / pipeline / mixed-op backward kernels:
//   stage s small slot j -> s*4 + j ; big op coefficient k -> 24 + k ; 54 = loss ; 55 = spare
#define RISP_NSLOT 56
#define RISP_SLOT_BIG 24
#define RISP_SLOT_LOSS 54
struct SlotList {
  int n;
  short dst[96];
  short slot[96];
};
void chain_slot_list(const ChainDesc& d, SlotList* m);

// Deterministic second-stage reduction (one warp per entry, fixed order):
//   out[r][dst[e]] = scale * sum_b partial[(r*B + b)*NS + slot[e]]   ; sum_rows also sums over r into row 0
int finalize_partials(const float* partial, float* out, int R, int B, int NS, int P, const short* dst,
                      const short* slot, int n, float scale, bool sum_rows, cudaStream_t st);

// Same reduction for many slots at once, two levels in one launch (see risp_api.cu).  `scratch_ws` holds
// finalize_rows_workspace(R, NS) bytes.  Writes ALL P entries of every output row (unmapped ones become 0) and, when
// loss_out is given (sum_rows only), loss_out[0] = loss_scale * sum(partial[..][loss_slot]).
constexpr int kFinBlocks = 64;
size_t finalize_rows_workspace(int R, int NS);
int finalize_rows(const float* partial, void* scratch_ws, float* out, float* loss_out, int R, int B, int NS, int P,
                  const short* dst, const short* slot, int n, float scale, float loss_scale, int loss_slot, bool sum_rows,
                  cudaStream_t st);

// Integer sums of the evaluation kernels: out[r] = sum_b partial[r*B + b] (risp_metric.cu).  Exact, so any order gives the
// same bits.
int finalize_sse(const unsigned long long* partial, long long* out, int R, int B, cudaStream_t st);

}  // namespace risp
