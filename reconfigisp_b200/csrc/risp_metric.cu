// Evaluation metric of the reference (test.py / test_split.py: tensor2bgr -> psnr per image) on the device.
//
// Both images are quantised as tensor2bgr does (utils/util.py:118-135: clip(x*255, 0, 255) truncated to uint8) and the
// squared differences of the 8-bit codes are summed per image.  They are integers, so the sum is exact (64 bits: a 12 MP
// frame can reach 3 * 12e6 * 255^2 > 2^32) and the same whatever the grid or the order of the additions.  The host turns
// it into PSNR (reconfigisp_b200/metrics.py).  risp_sse_u8 takes any fp32 pair; risp_pipeline_eval (risp_pipeline.cu)
// computes the same sum inside the pipeline kernels, from raw, without writing the image.
#include "risp_common.cuh"

namespace risp {

constexpr int kMetricThreads = 256;

__device__ __forceinline__ uint32_t sq_code(float y, float t) {
  const int d = u8_code(y) - u8_code(t);
  return (uint32_t)(d * d);
}

__device__ __forceinline__ unsigned long long block_sum_u64(unsigned long long v) {
  __shared__ unsigned long long part[kMetricThreads / 32];
  v = warp_sum_u64(v);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = v;
  __syncthreads();
  v = 0;
  if (threadIdx.x < 32) {
    v = threadIdx.x < kMetricThreads / 32 ? part[threadIdx.x] : 0ull;
    v = warp_sum_u64(v);
  }
  return v;     // valid in thread 0
}

// grid (blocks per image, N): each block sums a grid-stride share of one image's C*H*W values and adds it to out[n].
// vec: y and gt have the same alignment modulo 16 bytes, so the body of every image is read as float4 (a scalar head up to
// the first 16-byte boundary, a scalar tail after the last one)
__global__ void __launch_bounds__(kMetricThreads)
sse_u8_kernel(const float* __restrict__ y, const float* __restrict__ gt, unsigned long long* __restrict__ out,
              long long per_image, int vec) {
  const long long n = blockIdx.y;
  const float* __restrict__ yp = y + n * per_image;
  const float* __restrict__ gp = gt + n * per_image;
  long long head = per_image, nv = 0;
  if (vec) {
    head = (long long)(((16u - (uint32_t)(reinterpret_cast<uintptr_t>(yp) & 15u)) & 15u) >> 2);
    if (head > per_image) head = per_image;
    nv = (per_image - head) >> 2;
  }
  const long long tid = (long long)blockIdx.x * kMetricThreads + threadIdx.x, nth = (long long)gridDim.x * kMetricThreads;
  unsigned long long s = 0;
  for (long long i = tid; i < head; i += nth) s += sq_code(yp[i], gp[i]);
  const float* yv = yp + head;
  const float* gv = gp + head;
  for (long long i = tid; i < nv; i += nth) s += sq_codes4(ld_stream4(yv + 4 * i), ld_stream4(gv + 4 * i));
  for (long long i = head + 4 * nv + tid; i < per_image; i += nth) s += sq_code(yp[i], gp[i]);
  s = block_sum_u64(s);
  if (threadIdx.x == 0) atomicAdd(out + n, s);     // integer addition: exact in any order
}

// out[r] = sum_b partial[r*B + b]: one block per row
__global__ void __launch_bounds__(kMetricThreads)
finalize_sse_kernel(const unsigned long long* __restrict__ partial, long long* __restrict__ out, int B) {
  const unsigned long long* p = partial + (long long)blockIdx.x * B;
  unsigned long long s = 0;
  for (int b = threadIdx.x; b < B; b += kMetricThreads) s += p[b];
  s = block_sum_u64(s);
  if (threadIdx.x == 0) out[blockIdx.x] = (long long)s;
}

int finalize_sse(const unsigned long long* partial, long long* out, int R, int B, cudaStream_t st) {
  finalize_sse_kernel<<<R, kMetricThreads, 0, st>>>(partial, out, B);
  return check_launch("finalize_sse_kernel");
}

}  // namespace risp

using namespace risp;

extern "C" int risp_sse_u8(const float* y, const float* gt, long long* sse_out, int N, int C, int H, int W,
                           risp_stream_t stream) {
  RISP_REQUIRE(y && gt && sse_out, RISP_E_INVALID, "risp_sse_u8: y, gt and sse_out must be non-null");
  RISP_REQUIRE(N > 0 && C > 0 && H > 0 && W > 0, RISP_E_INVALID, "risp_sse_u8: bad shape (%d,%d,%d,%d)", N, C, H, W);
  RISP_REQUIRE(N <= 65535, RISP_E_INVALID, "risp_sse_u8: batch %d > 65535", N);
  RISP_REQUIRE((reinterpret_cast<uintptr_t>(y) & 3u) == 0 && (reinterpret_cast<uintptr_t>(gt) & 3u) == 0 &&
                   (reinterpret_cast<uintptr_t>(sse_out) & 7u) == 0,
               RISP_E_ALIGN, "risp_sse_u8: y / gt must be 4-byte and sse_out 8-byte aligned");
  cudaStream_t st = as_stream(stream);
  const long long per_image = (long long)C * H * W;
  const int vec = ((reinterpret_cast<uintptr_t>(y) ^ reinterpret_cast<uintptr_t>(gt)) & 15u) == 0 ? 1 : 0;
  // about 8 resident blocks per SM over the whole batch, and at least 4 float4 per thread
  long long bx = cdiv(per_image, (long long)kMetricThreads * 16);
  const long long cap = cdiv((long long)sm_count() * 8, N);
  if (bx > cap) bx = cap;
  if (bx < 1) bx = 1;
  if (cudaMemsetAsync(sse_out, 0, sizeof(long long) * (size_t)N, st) != cudaSuccess) {
    set_error("risp_sse_u8: memset failed");
    return RISP_E_CUDA;
  }
  sse_u8_kernel<<<dim3((unsigned)bx, (unsigned)N), kMetricThreads, 0, st>>>(
      y, gt, reinterpret_cast<unsigned long long*>(sse_out), per_image, vec);
  return check_launch("sse_u8_kernel");
}
