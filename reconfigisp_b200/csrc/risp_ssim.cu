// Per-image SSIM of the 8-bit images on the device (the reference's get_ssim: skimage compare_ssim(a, b, multichannel=True)
// with its defaults on the tensor2bgr codes; the definition is stated in oracle/metrics_oracle.py and the header).
//
// Both operands are quantised as tensor2bgr does (u8_code), so every window moment is an integer.  For each interior pixel
// the five 7x7 sums Sa, Sb, Saa, Sbb, Sab are formed in int32, and so are the four terms of the ratio
//   P1 = 2 Sa Sb, Q1 = Sa^2 + Sb^2, P2 = 2 (49 Sab - Sa Sb), Q2 = 49 (Saa + Sbb) - Q1        (all < 3.2e8)
// before any rounding: in fp32 the differences 49 Saa - Sa^2 cancel on flat regions.  The ratio
// S = (P1 + c1)(P2 + c2) / ((Q1 + c1)(Q2 + c2)) is then fp32 with a correctly rounded division, so identical images give
// exactly 1 and swapped operands the same bits.  rint(S * 2^32) is summed per image in 64-bit integers: exact, so the sum has
// the same bits whatever the grid, the row chunking or the order of the additions.
//
// Register marching as in the guided filter (risp_stencil.cu, gmarch): a warp owns a strip of 128 loaded columns (4 per lane;
// lanes 0 and 31 are halo only, so 120 output columns) and walks a chunk of interior rows.  Each lane keeps the VERTICAL 7-row
// sums of its 4 columns in registers (one row enters, one leaves per step; the leaving row is read again, from L1 / L2), and
// the 7-wide HORIZONTAL sum is gathered from the two neighbouring lanes by shuffles.  No shared memory, no barrier.  Only
// interior pixels are produced, so no window leaves the frame.  Three quantities are carried: Sa | Sb << 16 packed in one
// word (both < 2^16), Saa + Sbb (only their sum enters Q2) and Sab, so a step costs 18 shuffles per lane.
#include "risp_common.cuh"

namespace risp {
namespace ssim {

constexpr int kWarps = 4, kOutCols = 120, kMinRows = 48;
constexpr float kC1 = 15612.5025f;        // 49^2 (0.01 * 255)^2
constexpr float kC2 = 137644.92f;         // 49 * 48 (0.03 * 255)^2

__device__ __forceinline__ float comp(const float4& v, int i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }
__device__ __forceinline__ int byte_of(uint32_t w, int j) { return (int)__byte_perm(w, 0u, 0x4440u | (uint32_t)j); }

// One row of a lane's 4 columns, as loaded: gt (fp32, or with GS one word of 4 codes of a frame store) for KC channels, and y
// as fp32 (NCHW), as the 12 interleaved bytes of 4 BGR pixels (NHWC, vector path, KC == 3) or as one word of 4 codes per
// channel (NHWC, scalar path).
template <int LAYOUT, int KC, bool VEC, bool GS>
struct Row {
  static constexpr bool kU8 = LAYOUT == RISP_IMG_U8_NHWC;
  float4 g[GS ? 1 : KC];
  uint32_t g8[GS ? KC : 1];
  float4 yf[kU8 ? 1 : KC];
  uint32_t y8[kU8 ? (VEC ? 3 : KC) : 1];
};

__device__ __forceinline__ float ld_or0(const float* __restrict__ row, int c, int W) {
  return (c >= 0 && c < W) ? __ldg(row + c) : 0.f;
}
__device__ __forceinline__ float4 ld4(const float* __restrict__ row, int c, int W, bool vec) {
  if (vec) return (c >= 0 && c < W) ? __ldg(reinterpret_cast<const float4*>(row + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
  return make_float4(ld_or0(row, c, W), ld_or0(row, c + 1, W), ld_or0(row, c + 2, W), ld_or0(row, c + 3, W));
}

// Row q, columns [c, c+4) (c % 4 == 0), channels ch0 .. ch0+KC-1 of image n (with GS: gt is the GT store and gn the frame
// of image n in it).  Columns outside the frame read 0; they only feed lanes whose outputs lie outside the interior.  With VEC
// (W % 4 == 0, aligned operands) a lane is wholly inside or wholly outside the frame.
template <int LAYOUT, int KC, bool VEC, bool GS>
__device__ __forceinline__ void load_row(Row<LAYOUT, KC, VEC, GS>& r, const void* __restrict__ y, const float* __restrict__ gt,
                                         long long n, long long gn, int ch0, int C, int H, int W, int q, int c) {
  if constexpr (GS) {
#pragma unroll
    for (int k = 0; k < KC; ++k) {
      const unsigned char* __restrict__ row = reinterpret_cast<const unsigned char*>(gt) + (((gn * C + ch0 + k) * H) + q) * (long long)W;
      uint32_t w = 0;
      if constexpr (VEC) {
        if (c >= 0 && c < W) w = __ldg(reinterpret_cast<const uint32_t*>(row + c));
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (c + i >= 0 && c + i < W) w |= (uint32_t)__ldg(row + c + i) << (8 * i);
      }
      r.g8[k] = w;
    }
  } else {
#pragma unroll
    for (int k = 0; k < KC; ++k) r.g[k] = ld4(gt + (((n * C + ch0 + k) * H) + q) * (long long)W, c, W, VEC);
  }
  if constexpr (LAYOUT == RISP_IMG_F32_NCHW) {
#pragma unroll
    for (int k = 0; k < KC; ++k)
      r.yf[k] = ld4(static_cast<const float*>(y) + (((n * C + ch0 + k) * H) + q) * (long long)W, c, W, VEC);
  } else {
    const unsigned char* __restrict__ row = static_cast<const unsigned char*>(y) + ((n * H + q) * (long long)W) * C;
    if constexpr (VEC) {
      static_assert(KC == 3, "the vector NHWC path reads all three channels of 4 pixels");
      const bool in = c >= 0 && c < W;
      const uint32_t* p = reinterpret_cast<const uint32_t*>(row + 3ll * c);
#pragma unroll
      for (int j = 0; j < 3; ++j) r.y8[j] = in ? __ldg(p + j) : 0u;
    } else {
#pragma unroll
      for (int k = 0; k < KC; ++k) {
        uint32_t w = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (c + i >= 0 && c + i < W) w |= (uint32_t)__ldg(row + (long long)(c + i) * C + ch0 + k) << (8 * i);
        r.y8[k] = w;
      }
    }
  }
}

// the codes of channel k, column i of a loaded row
template <int LAYOUT, int KC, bool VEC, bool GS>
__device__ __forceinline__ int code_y(const Row<LAYOUT, KC, VEC, GS>& r, int k, int i) {
  if constexpr (LAYOUT == RISP_IMG_F32_NCHW) return u8_code(comp(r.yf[k], i));
  else if constexpr (VEC) return byte_of(r.y8[(3 * i + k) >> 2], (3 * i + k) & 3);
  else return byte_of(r.y8[k], i);
}
// a stored GT code is its own tensor2bgr code (trunc(clip(fl32(fl32(c/255)*255), 0, 255)) == c for all 256 codes)
template <int LAYOUT, int KC, bool VEC, bool GS>
__device__ __forceinline__ int code_g(const Row<LAYOUT, KC, VEC, GS>& r, int k, int i) {
  if constexpr (GS) return byte_of(r.g8[k], i);
  else return u8_code(comp(r.g[k], i));
}

// 7-wide window sums of a per-column quantity: columns i-3 .. i+3 of the lane's 4 columns, the outer ones from the
// neighbouring lanes (their suffix / prefix sums).  Lanes 0 and 31 receive their own values; they produce no output.
__device__ __forceinline__ void hsum7(const int (&v)[4], int (&o)[4]) {
  const int t = v[0] + v[1] + v[2] + v[3];
  const int l3 = __shfl_up_sync(0xffffffffu, v[3], 1);
  const int l23 = __shfl_up_sync(0xffffffffu, v[2] + v[3], 1);
  const int l123 = __shfl_up_sync(0xffffffffu, v[1] + v[2] + v[3], 1);
  const int r0 = __shfl_down_sync(0xffffffffu, v[0], 1);
  const int r01 = __shfl_down_sync(0xffffffffu, v[0] + v[1], 1);
  const int r012 = __shfl_down_sync(0xffffffffu, v[0] + v[1] + v[2], 1);
  o[0] = l123 + t;
  o[1] = l23 + t + r0;
  o[2] = l3 + t + r01;
  o[3] = t + r012;
}

// rint(S * 2^32) of one pixel from its window sums: s = Sa | Sb << 16, q = Saa + Sbb, x = Sab
__device__ __forceinline__ long long ssim_fixed(int s, int q, int x) {
  const int sa = s & 0xffff, sb = s >> 16;
  const int ab = sa * sb;
  const int q1 = sa * sa + sb * sb;
  const int p1 = 2 * ab, p2 = 2 * (49 * x - ab), q2 = 49 * q - q1;
  const float num = __fmul_rn(__fadd_rn((float)p1, kC1), __fadd_rn((float)p2, kC2));
  const float den = __fmul_rn(__fadd_rn((float)q1, kC1), __fadd_rn((float)q2, kC2));
  return __float2ll_rn(__fmul_rn(__fdiv_rn(num, den), 4294967296.f));
}

// grid (cdiv(strips, kWarps), min(chunks * groups, 65535), N); groups = C / KC channel groups.  Work item t of blockIdx.y's
// stride is (row chunk t / groups, channel group t % groups): the channel groups of one chunk are neighbours, so with
// KC < C on the NHWC operand the other channels' bytes are still in L2.
// GS: gt is a store of G frames of 8-bit planar codes and image n is scored against frame pos[n].y (a record that is not a
// whole frame of the store sets *status and adds nothing).
template <int LAYOUT, int KC, bool VEC, bool GS>
__global__ void __launch_bounds__(kWarps * 32)
ssim_u8_kernel(const void* __restrict__ y, const float* __restrict__ gt, unsigned long long* __restrict__ out, int C, int H,
               int W, int strips, int rows_per_chunk, int items, const int4* __restrict__ pos, int G, int* status) {
  const int lane = threadIdx.x & 31;
  const int strip = blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (strip >= strips) return;                                      // whole warps only
  const long long n = blockIdx.z;
  long long gn = n;
  if constexpr (GS) {
    const int4 rec = pos[n];
    if (rec.y < 0 || rec.y >= G || rec.z != 0 || rec.w != 0) {
      if (threadIdx.x == 0) *status = 1;
      return;
    }
    gn = rec.y;
  }
  const int groups = C / KC;
  const int c = strip * kOutCols - 4 + lane * 4;                    // first of the lane's 4 columns
  bool valid[4];                                                    // interior output columns of this lane
#pragma unroll
  for (int i = 0; i < 4; ++i) valid[i] = lane >= 1 && lane <= 30 && c + i >= 3 && c + i < W - 3;
  unsigned long long acc = 0;
  for (int t = blockIdx.y; t < items; t += gridDim.y) {
    const int ch0 = (t % groups) * KC;
    const int ra = 3 + (t / groups) * rows_per_chunk, rb = min(H - 3, ra + rows_per_chunk);
    int vs[KC][4], vq[KC][4], vx[KC][4];                            // vertical 7-row sums: Sa | Sb << 16, Saa + Sbb, Sab
#pragma unroll
    for (int k = 0; k < KC; ++k)
#pragma unroll
      for (int i = 0; i < 4; ++i) vs[k][i] = vq[k][i] = vx[k][i] = 0;
    Row<LAYOUT, KC, VEC, GS> rin, rout;
    for (int d = -3; d <= 3; ++d) {
      load_row(rin, y, gt, n, gn, ch0, C, H, W, ra + d, c);
#pragma unroll
      for (int k = 0; k < KC; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int a = code_y(rin, k, i), b = code_g(rin, k, i);
          vs[k][i] += a + (b << 16);
          vq[k][i] += a * a + b * b;
          vx[k][i] += a * b;
        }
    }
    for (int r = ra; r < rb; ++r) {
      const bool more = r + 1 < rb;
      if (more) {                                                   // in flight while row r is scored
        load_row(rin, y, gt, n, gn, ch0, C, H, W, r + 4, c);
        load_row(rout, y, gt, n, gn, ch0, C, H, W, r - 3, c);
      }
#pragma unroll
      for (int k = 0; k < KC; ++k) {
        int hs[4], hq[4], hx[4];
        hsum7(vs[k], hs);
        hsum7(vq[k], hq);
        hsum7(vx[k], hx);
#pragma unroll
        for (int i = 0; i < 4; ++i) {        // every output lane computes all 4 pixels: a select, not a branch
          const long long v = ssim_fixed(hs[i], hq[i], hx[i]);
          acc += valid[i] ? (unsigned long long)v : 0ull;
        }
      }
      if (more) {
#pragma unroll
        for (int k = 0; k < KC; ++k)
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int a = code_y(rin, k, i), b = code_g(rin, k, i);
            const int ao = code_y(rout, k, i), bo = code_g(rout, k, i);
            vs[k][i] += (a + (b << 16)) - (ao + (bo << 16));
            vq[k][i] += (a * a + b * b) - (ao * ao + bo * bo);
            vx[k][i] += a * b - ao * bo;
          }
      }
    }
  }
  acc = warp_sum_u64(acc);
  if (lane == 0 && acc != 0) atomicAdd(out + n, acc);               // integer addition: exact in any order
}

template <int LAYOUT, int KC, bool VEC, bool GS = false>
static int launch(const void* y, const float* gt, long long* out, int N, int C, int H, int W, cudaStream_t st,
                  const int4* pos = nullptr, int G = 0, int* status = nullptr) {
  const int strips = (int)cdiv(W - 3, kOutCols), bx = (int)cdiv(strips, kWarps), groups = C / KC;
  // about 32 warps per SM over the whole batch, at least kMinRows rows per chunk (a chunk start costs 6 extra rows)
  const long long want = cdiv((long long)sm_count() * 32, (long long)strips * N * groups);
  int rows = (int)cdiv(H - 6, want < 1 ? 1 : want);
  if (rows < kMinRows) rows = kMinRows;
  const long long items = cdiv(H - 6, rows) * (long long)groups;     // <= C (H-6) < 2^31
  const unsigned gy = (unsigned)(items < 65535 ? items : 65535);
  ssim_u8_kernel<LAYOUT, KC, VEC, GS><<<dim3((unsigned)bx, gy, (unsigned)N), kWarps * 32, 0, st>>>(
      y, gt, reinterpret_cast<unsigned long long*>(out), C, H, W, strips, rows, (int)items, pos, G, status);
  return check_launch("ssim_u8_kernel");
}

}  // namespace ssim
}  // namespace risp

using namespace risp;

extern "C" int risp_ssim_u8(const void* y, int y_layout, const float* gt, long long* ssim_sum_out, int N, int C, int H,
                            int W, risp_stream_t stream) {
  RISP_REQUIRE(y && gt && ssim_sum_out, RISP_E_INVALID, "risp_ssim_u8: y, gt and ssim_sum_out must be non-null");
  RISP_REQUIRE(y_layout == RISP_IMG_F32_NCHW || y_layout == RISP_IMG_U8_NHWC, RISP_E_INVALID,
               "risp_ssim_u8: unknown y_layout %d", y_layout);
  RISP_REQUIRE(N >= 1 && N <= 65535, RISP_E_INVALID, "risp_ssim_u8: batch %d outside [1, 65535]", N);
  RISP_REQUIRE(C > 0, RISP_E_INVALID, "risp_ssim_u8: C = %d", C);
  RISP_REQUIRE(H >= 7 && W >= 7, RISP_E_INVALID, "risp_ssim_u8: the 7x7 window needs H and W >= 7, got %d x %d", H, W);
  RISP_REQUIRE((long long)C * (H - 6) * (W - 6) < (1ll << 31), RISP_E_INVALID,
               "risp_ssim_u8: C (H-6)(W-6) = %lld interior values must stay below 2^31", (long long)C * (H - 6) * (W - 6));
  const uintptr_t py = reinterpret_cast<uintptr_t>(y), pg = reinterpret_cast<uintptr_t>(gt);
  RISP_REQUIRE((pg & 3u) == 0 && (y_layout != RISP_IMG_F32_NCHW || (py & 3u) == 0) &&
                   (reinterpret_cast<uintptr_t>(ssim_sum_out) & 7u) == 0,
               RISP_E_ALIGN, "risp_ssim_u8: fp32 operands must be 4-byte and ssim_sum_out 8-byte aligned");
  cudaStream_t st = as_stream(stream);
  if (cudaMemsetAsync(ssim_sum_out, 0, sizeof(long long) * (size_t)N, st) != cudaSuccess) {
    set_error("risp_ssim_u8: memset failed");
    return RISP_E_CUDA;
  }
  // vector loads: every row of every plane starts on a 16-byte (fp32) / 4-byte (NHWC bytes) boundary
  const bool vec = W % 4 == 0 && (pg & 15u) == 0;
  if (y_layout == RISP_IMG_F32_NCHW) {
    return vec && (py & 15u) == 0 ? ssim::launch<RISP_IMG_F32_NCHW, 1, true>(y, gt, ssim_sum_out, N, C, H, W, st)
                                  : ssim::launch<RISP_IMG_F32_NCHW, 1, false>(y, gt, ssim_sum_out, N, C, H, W, st);
  }
  if (C == 3) {       // one warp reads all three channels of its pixels: the interleaved bytes are fetched once
    return vec && (py & 3u) == 0 ? ssim::launch<RISP_IMG_U8_NHWC, 3, true>(y, gt, ssim_sum_out, N, C, H, W, st)
                                 : ssim::launch<RISP_IMG_U8_NHWC, 3, false>(y, gt, ssim_sum_out, N, C, H, W, st);
  }
  return ssim::launch<RISP_IMG_U8_NHWC, 1, false>(y, gt, ssim_sum_out, N, C, H, W, st);
}

extern "C" int risp_ssim_u8_store(const void* y, int y_layout, const unsigned char* gt_store, int G, const int* pos, int* status,
                                  long long* ssim_sum_out, int N, int H, int W, risp_stream_t stream) {
  RISP_REQUIRE(y && gt_store && pos && status && ssim_sum_out, RISP_E_INVALID,
               "risp_ssim_u8_store: y, gt_store, pos, status and ssim_sum_out must be non-null");
  RISP_REQUIRE(y_layout == RISP_IMG_F32_NCHW || y_layout == RISP_IMG_U8_NHWC, RISP_E_INVALID,
               "risp_ssim_u8_store: unknown y_layout %d", y_layout);
  RISP_REQUIRE(N >= 1 && N <= 65535 && G >= 1, RISP_E_INVALID, "risp_ssim_u8_store: batch %d outside [1, 65535] or G = %d", N, G);
  RISP_REQUIRE(H >= 7 && W >= 7, RISP_E_INVALID, "risp_ssim_u8_store: the 7x7 window needs H and W >= 7, got %d x %d", H, W);
  RISP_REQUIRE(3ll * (H - 6) * (W - 6) < (1ll << 31), RISP_E_INVALID,
               "risp_ssim_u8_store: 3 (H-6)(W-6) = %lld interior values must stay below 2^31", 3ll * (H - 6) * (W - 6));
  const uintptr_t py = reinterpret_cast<uintptr_t>(y), pg = reinterpret_cast<uintptr_t>(gt_store);
  RISP_REQUIRE((y_layout != RISP_IMG_F32_NCHW || (py & 3u) == 0) && (reinterpret_cast<uintptr_t>(ssim_sum_out) & 7u) == 0 &&
                   aligned16(pos),
               RISP_E_ALIGN, "risp_ssim_u8_store: fp32 y must be 4-byte, ssim_sum_out 8-byte and pos 16-byte aligned");
  cudaStream_t st = as_stream(stream);
  if (cudaMemsetAsync(ssim_sum_out, 0, sizeof(long long) * (size_t)N, st) != cudaSuccess) {
    set_error("risp_ssim_u8_store: memset failed");
    return RISP_E_CUDA;
  }
  // vector loads: every GT row starts on a 4-byte boundary and every fp32 / NHWC row of y on a 16- / 4-byte one
  const bool vec = W % 4 == 0 && (pg & 3u) == 0;
  const float* gt = reinterpret_cast<const float*>(gt_store);
  const int4* p = reinterpret_cast<const int4*>(pos);
  if (y_layout == RISP_IMG_F32_NCHW)
    return vec && (py & 15u) == 0 ? ssim::launch<RISP_IMG_F32_NCHW, 1, true, true>(y, gt, ssim_sum_out, N, 3, H, W, st, p, G, status)
                                  : ssim::launch<RISP_IMG_F32_NCHW, 1, false, true>(y, gt, ssim_sum_out, N, 3, H, W, st, p, G, status);
  return vec && (py & 3u) == 0 ? ssim::launch<RISP_IMG_U8_NHWC, 3, true, true>(y, gt, ssim_sum_out, N, 3, H, W, st, p, G, status)
                               : ssim::launch<RISP_IMG_U8_NHWC, 3, false, true>(y, gt, ssim_sum_out, N, 3, H, W, st, p, G, status);
}
