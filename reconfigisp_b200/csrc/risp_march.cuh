// Register-marching window kernels for small stencils on planar images (median 3x3, bilateral window 3, unsharp mask 5x5).
//
// A warp owns a 128-column strip of NP planes and walks down a chunk of rows; every lane keeps the (2*HL+1) x (4+2*HL)
// window of its 4 output pixels in registers.  A new row costs one coalesced 128-bit load per lane and plane, the
// horizontal halo comes from the neighbouring lanes by shuffle (the strip's end lanes read theirs from memory, the frame
// border rule applied to their own columns), the vertical halo stays in registers and the next row is always in flight.
// No shared memory, no barrier, each input element is fetched from HBM once (chunk seams: twice, from L2).
// Requires W % 4 == 0 and 16-byte aligned planes; other shapes take the shared-memory tile kernels of risp_stencil.cu.
#pragma once
#include "risp_common.cuh"

namespace risp {
namespace march {

enum { REFLECT101 = 0, REPLICATE = 1 };
constexpr int kWarps = 4, kStrip = 128;

template <int BORDER>
__device__ __forceinline__ int brow(int r, int H) {
  if (BORDER == REPLICATE) return r < 0 ? 0 : (r >= H ? H - 1 : r);
  return r < 0 ? -r : (r >= H ? 2 * H - 2 - r : r);      // H >= HL + 1 is checked on the host
}

template <int HL> struct Row;
template <> struct Row<1> { float4 v; float l, r; };
template <> struct Row<2> { float4 v; float2 l, r; };

template <int HL>
__device__ __forceinline__ void row_issue(Row<HL>& q, const float* __restrict__ rp, int W, int c0, bool active, int lane) {
  q.v = active ? ld_stream4(rp + c0) : make_float4(0.f, 0.f, 0.f, 0.f);
  if constexpr (HL == 1) {
    q.l = 0.f; q.r = 0.f;
    if (active && lane == 0 && c0 > 0) q.l = __ldg(rp + c0 - 1);
    if (active && lane == 31 && c0 + 4 < W) q.r = __ldg(rp + c0 + 4);
  } else {
    q.l = make_float2(0.f, 0.f); q.r = make_float2(0.f, 0.f);
    if (active && lane == 0 && c0 > 0) q.l = __ldg(reinterpret_cast<const float2*>(rp + c0 - 2));
    if (active && lane == 31 && c0 + 4 < W) q.r = __ldg(reinterpret_cast<const float2*>(rp + c0 + 4));
  }
}

// dst[0 .. 4+2*HL) = columns c0-HL .. c0+3+HL of the row, frame border rule BORDER at the two ends
template <int HL, int BORDER>
__device__ __forceinline__ void row_finish(float (&dst)[4 + 2 * HL], const Row<HL>& q, int W, int c0, bool active, int lane) {
  const unsigned full = 0xffffffffu;
  const float4 v = q.v;
  const bool first = (c0 == 0), last = active && (c0 + 4 >= W);
  if constexpr (HL == 1) {
    float l = __shfl_up_sync(full, v.w, 1), r = __shfl_down_sync(full, v.x, 1);
    if (lane == 0) l = first ? (BORDER == REPLICATE ? v.x : v.y) : q.l;
    if (last) r = (BORDER == REPLICATE) ? v.w : v.z;
    else if (lane == 31) r = q.r;
    dst[0] = l; dst[1] = v.x; dst[2] = v.y; dst[3] = v.z; dst[4] = v.w; dst[5] = r;
  } else {
    float l0 = __shfl_up_sync(full, v.z, 1), l1 = __shfl_up_sync(full, v.w, 1);
    float r0 = __shfl_down_sync(full, v.x, 1), r1 = __shfl_down_sync(full, v.y, 1);
    if (lane == 0) {
      l0 = first ? (BORDER == REPLICATE ? v.x : v.z) : q.l.x;      // col -2 -> 2
      l1 = first ? (BORDER == REPLICATE ? v.x : v.y) : q.l.y;      // col -1 -> 1
    }
    if (last) { r0 = (BORDER == REPLICATE) ? v.w : v.z; r1 = (BORDER == REPLICATE) ? v.w : v.y; }   // cols W, W+1 -> W-2, W-3
    else if (lane == 31) { r0 = q.r.x; r1 = q.r.y; }
    dst[0] = l0; dst[1] = l1; dst[2] = v.x; dst[3] = v.y; dst[4] = v.z; dst[5] = v.w; dst[6] = r0; dst[7] = r1;
  }
}

// F: struct with  __device__ void operator()(const float (&w)[NP][2*HL+1][4+2*HL], float (&out)[NP][4], int zp) const
constexpr int kMarchDepth = 3;
template <int HL, int NP, int BORDER, class F, int D = kMarchDepth>
__global__ void __launch_bounds__(kWarps * 32)
march_kernel(const float* __restrict__ x, float* __restrict__ y, int H, int W, int rows_per_chunk, F f) {
  constexpr int WR = 2 * HL + 1, WC = 4 + 2 * HL;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int strip = blockIdx.x * kWarps + wid;
  if (strip * kStrip >= W) return;
  const int c0 = strip * kStrip + lane * 4;
  const bool active = c0 < W;
  const int zp = blockIdx.z;
  const long long plane = (long long)H * W;
  const float* __restrict__ xb = x + (long long)zp * NP * plane;
  float* __restrict__ yb = y + (long long)zp * NP * plane;
  const int ra = blockIdx.y * rows_per_chunk, rb = min(H, ra + rows_per_chunk);
  float w[NP][WR][WC];
  Row<HL> qq[D][NP];           // D rows in flight per warp: at ~32 warps per SM one 512-byte row per warp does not cover the HBM latency
#pragma unroll
  for (int j = 0; j < WR - 1; ++j) {
    const long long ro = (long long)brow<BORDER>(ra - HL + j, H) * W;
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      row_issue<HL>(qq[0][p], xb + p * plane + ro, W, c0, active, lane);
      row_finish<HL, BORDER>(w[p][j], qq[0][p], W, c0, active, lane);
    }
  }
#pragma unroll
  for (int d = 0; d < D; ++d) {
    const long long ro = (long long)brow<BORDER>(ra + d + HL, H) * W;      // rows past the chunk are loaded and dropped
#pragma unroll
    for (int p = 0; p < NP; ++p) row_issue<HL>(qq[d][p], xb + p * plane + ro, W, c0, active, lane);
  }
  for (int r = ra; r < rb; ++r) {
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      row_finish<HL, BORDER>(w[p][WR - 1], qq[0][p], W, c0, active, lane);
#pragma unroll
      for (int d = 0; d + 1 < D; ++d) qq[d][p] = qq[d + 1][p];
    }
    if (r + D < rb) {
      const long long ro = (long long)brow<BORDER>(r + D + HL, H) * W;
#pragma unroll
      for (int p = 0; p < NP; ++p) row_issue<HL>(qq[D - 1][p], xb + p * plane + ro, W, c0, active, lane);
    }
    float out[NP][4];
    f(w, out, zp);
    if (active) {
#pragma unroll
      for (int p = 0; p < NP; ++p)
        st_stream4(yb + p * plane + (long long)r * W + c0, make_float4(out[p][0], out[p][1], out[p][2], out[p][3]));
    }
#pragma unroll
    for (int p = 0; p < NP; ++p)
#pragma unroll
      for (int j = 0; j < WR - 1; ++j)
#pragma unroll
        for (int i = 0; i < WC; ++i) w[p][j][i] = w[p][j + 1][i];
  }
}

struct Geom { dim3 grid; int rows_per_chunk; };
static inline Geom geometry(int H, int W, int Z) {
  const int bx = (int)cdiv(cdiv(W, kStrip), kWarps);
  long long want = (long long)sm_count() * 8;                 // CTAs: ~8 per SM
  long long chunks = cdiv(want, (long long)bx * Z);
  int rows = (int)cdiv(H, chunks < 1 ? 1 : chunks);
  rows = rows < 8 ? 8 : (rows > 96 ? 96 : rows);
  Geom g;
  g.rows_per_chunk = rows;
  g.grid = dim3((unsigned)bx, (unsigned)cdiv(H, rows), (unsigned)Z);
  return g;
}

static inline bool usable(const void* x, const void* y, int H, int W, int HL) {
  return (W % 4 == 0) && aligned16(x) && aligned16(y) && H > HL && W >= 4 + 0 * HL && cdiv(H, 8) <= 65535;
}

}  // namespace march
}  // namespace risp
