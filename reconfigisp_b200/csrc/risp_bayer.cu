// Bayer-domain index work (bit-exact): RGGB pack / unpack, PixelShuffle(2) and its adjoint,
// the adjoint of nearest-neighbour demosaic, and the black-level + CFA white-balance stage.
// References: srcnn_demosaic_arch.py:39-43, path_14l_bayer_arch.py:48,71-75 (pack / PixelShuffle),
// tools_origin.py:265-286 (DemosaicNearest is differentiable: its adjoint feeds alpha_bayer),
// data/preprocessing/generate_rggb2bgr_imgs_SID_Sony.py:50 (black level).
#include "risp_common.cuh"

namespace risp {

constexpr int kT = 256;

// (N,C,H,W) -> (N,4C,H/2,W/2), out channel c*4 + dy*2 + dx.   One thread: 4 output columns (8 input columns).
template <bool VEC>
__global__ void __launch_bounds__(kT)
unshuffle2_kernel(const float* __restrict__ in, float* __restrict__ out, int H, int W, long long total) {
  const int h2 = H / 2, w2 = W / 2;
  const int per_row = VEC ? w2 / 4 : w2;
  for (long long t = (long long)blockIdx.x * kT + threadIdx.x; t < total; t += (long long)gridDim.x * kT) {
    const int xq = (int)(t % per_row);
    long long rest = t / per_row;
    const int y = (int)(rest % h2);
    const long long nc = rest / h2;                       // n*C + c
    const float* src = in + (nc * H + 2 * y) * (long long)W;
    float* dst = out + (nc * 4 * h2 + y) * (long long)w2;
    const long long cs = (long long)h2 * w2;               // output channel stride
    if (VEC) {
      const int x = xq * 4;
      float4 a0 = ld_stream4(src + 2 * x), a1 = ld_stream4(src + 2 * x + 4);
      float4 b0 = ld_stream4(src + W + 2 * x), b1 = ld_stream4(src + W + 2 * x + 4);
      st_stream4(dst + x, make_float4(a0.x, a0.z, a1.x, a1.z));
      st_stream4(dst + cs + x, make_float4(a0.y, a0.w, a1.y, a1.w));
      st_stream4(dst + 2 * cs + x, make_float4(b0.x, b0.z, b1.x, b1.z));
      st_stream4(dst + 3 * cs + x, make_float4(b0.y, b0.w, b1.y, b1.w));
    } else {
      const int x = xq;
      dst[x] = src[2 * x]; dst[cs + x] = src[2 * x + 1];
      dst[2 * cs + x] = src[W + 2 * x]; dst[3 * cs + x] = src[W + 2 * x + 1];
    }
  }
}

// (N,4C,H/2,W/2) -> (N,C,H,W)
template <bool VEC>
__global__ void __launch_bounds__(kT)
shuffle2_kernel(const float* __restrict__ in, float* __restrict__ out, int H, int W, long long total) {
  const int h2 = H / 2, w2 = W / 2;
  const int per_row = VEC ? w2 / 4 : w2;
  for (long long t = (long long)blockIdx.x * kT + threadIdx.x; t < total; t += (long long)gridDim.x * kT) {
    const int xq = (int)(t % per_row);
    long long rest = t / per_row;
    const int y = (int)(rest % h2);
    const long long nc = rest / h2;
    float* dst = out + (nc * H + 2 * y) * (long long)W;
    const float* src = in + (nc * 4 * h2 + y) * (long long)w2;
    const long long cs = (long long)h2 * w2;
    if (VEC) {
      const int x = xq * 4;
      float4 c0 = ld_stream4(src + x), c1 = ld_stream4(src + cs + x);
      float4 c2 = ld_stream4(src + 2 * cs + x), c3 = ld_stream4(src + 3 * cs + x);
      st_stream4(dst + 2 * x, make_float4(c0.x, c1.x, c0.y, c1.y));
      st_stream4(dst + 2 * x + 4, make_float4(c0.z, c1.z, c0.w, c1.w));
      st_stream4(dst + W + 2 * x, make_float4(c2.x, c3.x, c2.y, c3.y));
      st_stream4(dst + W + 2 * x + 4, make_float4(c2.z, c3.z, c2.w, c3.w));
    } else {
      const int x = xq;
      dst[2 * x] = src[x]; dst[2 * x + 1] = src[cs + x];
      dst[W + 2 * x] = src[2 * cs + x]; dst[W + 2 * x + 1] = src[3 * cs + x];
    }
  }
}

static int grid_for(long long total) {
  long long g = cdiv(total, kT);
  long long cap = (long long)sm_count() * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

template <bool SHUFFLE>
static int run_shuffle(const char* who, const float* in, float* out, int N, int C, int H, int W, cudaStream_t st) {
  RISP_REQUIRE(in && out && N > 0 && C > 0 && H > 0 && W > 0, RISP_E_INVALID, "%s: bad arguments", who);
  RISP_REQUIRE(H % 2 == 0 && W % 2 == 0, RISP_E_INVALID, "%s: H and W must be even (got %dx%d)", who, H, W);
  bool vec = (W % 8 == 0) && aligned16(in) && aligned16(out);
  long long total = (long long)N * C * (H / 2) * (vec ? W / 8 : W / 2);
  int g = grid_for(total);
  if (SHUFFLE) {
    if (vec) shuffle2_kernel<true><<<g, kT, 0, st>>>(in, out, H, W, total);
    else shuffle2_kernel<false><<<g, kT, 0, st>>>(in, out, H, W, total);
  } else {
    if (vec) unshuffle2_kernel<true><<<g, kT, 0, st>>>(in, out, H, W, total);
    else unshuffle2_kernel<false><<<g, kT, 0, st>>>(in, out, H, W, total);
  }
  return check_launch(who);
}

// adjoint of nearest demosaic: one thread per 2x2 cell
__global__ void __launch_bounds__(kT)
nearest_bwd_kernel(const float* __restrict__ dbgr, float* __restrict__ draw, int H, int W, long long cells) {
  const int w2 = W / 2, h2 = H / 2;
  const long long plane = (long long)H * W;
  for (long long t = (long long)blockIdx.x * kT + threadIdx.x; t < cells; t += (long long)gridDim.x * kT) {
    const int j = (int)(t % w2);
    long long rest = t / w2;
    const int i = (int)(rest % h2);
    const long long n = rest / h2;
    const float* gB = dbgr + n * 3 * plane + (long long)(2 * i) * W + 2 * j;
    const float* gG = gB + plane;
    const float* gR = gB + 2 * plane;
    float2 b0 = ld_stream2(gB), b1 = ld_stream2(gB + W);
    float2 g0 = ld_stream2(gG), g1 = ld_stream2(gG + W);
    float2 r0 = ld_stream2(gR), r1 = ld_stream2(gR + W);
    float* o = draw + n * plane + (long long)(2 * i) * W + 2 * j;
    st_stream2(o, make_float2((r0.x + r0.y) + (r1.x + r1.y), g0.x + g0.y));
    st_stream2(o + W, make_float2(g1.x + g1.y, (b0.x + b0.y) + (b1.x + b1.y)));
  }
}

// ---- black level + per-site gain ---------------------------------------------------------------------
__device__ __forceinline__ float blc_px(float x, float bl, float inv, float g) {
  return sat01(fmaxf(x - bl, 0.f) * inv * g);
}

__global__ void __launch_bounds__(kT)
blc_wb_fwd_kernel(const float* __restrict__ raw, float* __restrict__ out, int H, int W,
                  const float* __restrict__ params, int pstride) {
  const int n = blockIdx.y;
  const float* p = params + (long long)n * pstride;
  const float bl = p[0], inv = 1.f / (1.f - bl);
  const long long plane = (long long)H * W;
  const int wq = W / 2;
  const long long pairs = plane / 2;
  for (long long t = (long long)blockIdx.x * kT + threadIdx.x; t < pairs; t += (long long)gridDim.x * kT) {
    const int row = (int)(t / wq);
    const float g0 = p[1 + (row & 1) * 2], g1 = p[2 + (row & 1) * 2];
    float2 v = ld_stream2(raw + n * plane + 2 * t);
    st_stream2(out + n * plane + 2 * t, make_float2(blc_px(v.x, bl, inv, g0), blc_px(v.y, bl, inv, g1)));
  }
}

__global__ void __launch_bounds__(kT)
blc_wb_bwd_kernel(const float* __restrict__ raw, const float* __restrict__ dout, float* __restrict__ draw,
                  float* __restrict__ partial, int H, int W, const float* __restrict__ params, int pstride) {
  const int n = blockIdx.y;
  const float* p = params + (long long)n * pstride;
  const float bl = p[0], inv = 1.f / (1.f - bl);
  const long long plane = (long long)H * W;
  const int wq = W / 2;
  const long long pairs = plane / 2;
  float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  for (long long t = (long long)blockIdx.x * kT + threadIdx.x; t < pairs; t += (long long)gridDim.x * kT) {
    const int row = (int)(t / wq);
    const int odd = row & 1;
    float2 v = ld_stream2(raw + n * plane + 2 * t);
    float2 d = ld_stream2(dout + n * plane + 2 * t);
    float xs[2] = {v.x, v.y}, ds[2] = {d.x, d.y}, o[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const float g = p[1 + odd * 2 + k];
      const float tt = fmaxf(xs[k] - bl, 0.f);
      const float e = ds[k] * in01(tt * inv * g);
      const float pass = (xs[k] - bl >= 0.f) ? 1.f : 0.f;
      o[k] = e * inv * g * pass;
      const float dgain = e * tt * inv;
      if (odd) { if (k) acc[4] += dgain; else acc[3] += dgain; }
      else     { if (k) acc[2] += dgain; else acc[1] += dgain; }
      acc[0] += e * g * (tt * inv * inv - pass * inv);
    }
    if (draw) st_stream2(draw + n * plane + 2 * t, make_float2(o[0], o[1]));
  }
  __shared__ float red[kT / 32][5];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    float v = warp_sum(acc[k]);
    if (lane == 0) red[wid][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < 5) {
    float v = 0.f;
    for (int w = 0; w < kT / 32; ++w) v += red[w][threadIdx.x];
    partial[((long long)n * gridDim.x + blockIdx.x) * 8 + threadIdx.x] = v;
  }
}

static int blc_blocks(int N, int H, int W) {
  long long pairs = (long long)H * W / 2;
  long long g = cdiv(pairs, (long long)kT * 4);
  long long cap = (long long)sm_count() * 8 / N;
  if (cap < 8) cap = 8;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace risp

using namespace risp;

extern "C" int risp_pack_rggb(const float* raw, float* packed, int N, int H, int W, risp_stream_t s) {
  return run_shuffle<false>("risp_pack_rggb", raw, packed, N, 1, H, W, as_stream(s));
}
extern "C" int risp_unpack_rggb(const float* packed, float* raw, int N, int H, int W, risp_stream_t s) {
  return run_shuffle<true>("risp_unpack_rggb", packed, raw, N, 1, H, W, as_stream(s));
}
extern "C" int risp_pixel_shuffle2(const float* in, float* out, int N, int C, int H, int W, risp_stream_t s) {
  return run_shuffle<true>("risp_pixel_shuffle2", in, out, N, C, H, W, as_stream(s));
}
extern "C" int risp_pixel_unshuffle2(const float* in, float* out, int N, int C, int H, int W, risp_stream_t s) {
  return run_shuffle<false>("risp_pixel_unshuffle2", in, out, N, C, H, W, as_stream(s));
}

extern "C" int risp_demosaic_bwd(const float* raw, const float* dbgr, float* draw, int N, int H, int W, int kind,
                                 float clip_hi, risp_stream_t stream) {
  (void)raw; (void)clip_hi;
  RISP_REQUIRE(dbgr && draw && N > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0, RISP_E_INVALID,
               "risp_demosaic_bwd: bad arguments");
  RISP_REQUIRE(kind == RISP_DM_NEAREST, RISP_E_UNSUPPORTED,
               "risp_demosaic_bwd: only the nearest-neighbour demosaic is differentiable in the reference "
               "(bilinear / laplacian are Origin* stages, tools_origin.py:445-509)");
  RISP_REQUIRE((reinterpret_cast<uintptr_t>(dbgr) & 7) == 0 && (reinterpret_cast<uintptr_t>(draw) & 7) == 0, RISP_E_ALIGN,
               "risp_demosaic_bwd: pointers must be 8-byte aligned");
  long long cells = (long long)N * (H / 2) * (W / 2);
  nearest_bwd_kernel<<<grid_for(cells), kT, 0, as_stream(stream)>>>(dbgr, draw, H, W, cells);
  return check_launch("nearest_bwd_kernel");
}

extern "C" int risp_bayer_blc_wb_fwd(const float* raw, float* out, int N, int H, int W, const float* params,
                                     int param_stride, risp_stream_t stream) {
  RISP_REQUIRE(raw && out && params && N > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0, RISP_E_INVALID,
               "risp_bayer_blc_wb_fwd: bad arguments");
  RISP_REQUIRE(param_stride == 0 || param_stride >= 5, RISP_E_INVALID, "risp_bayer_blc_wb_fwd: param_stride");
  dim3 grid(blc_blocks(N, H, W), N);
  blc_wb_fwd_kernel<<<grid, kT, 0, as_stream(stream)>>>(raw, out, H, W, params, param_stride);
  return check_launch("blc_wb_fwd_kernel");
}

extern "C" size_t risp_bayer_blc_wb_bwd_workspace(int N, int H, int W) {
  if (N <= 0 || H <= 0 || W <= 0) return 0;
  return (size_t)N * blc_blocks(N, H, W) * 8 * sizeof(float);
}

extern "C" int risp_bayer_blc_wb_bwd(const float* raw, const float* dout, float* draw, float* dparams, int N, int H,
                                     int W, const float* params, int param_stride, void* workspace,
                                     size_t workspace_bytes, risp_stream_t stream) {
  RISP_REQUIRE(raw && dout && dparams && params && N > 0 && H % 2 == 0 && W % 2 == 0, RISP_E_INVALID,
               "risp_bayer_blc_wb_bwd: bad arguments");
  RISP_REQUIRE(param_stride == 0 || param_stride >= 5, RISP_E_INVALID, "risp_bayer_blc_wb_bwd: param_stride");
  RISP_REQUIRE(workspace && workspace_bytes >= risp_bayer_blc_wb_bwd_workspace(N, H, W), RISP_E_WORKSPACE,
               "risp_bayer_blc_wb_bwd: workspace too small");
  cudaStream_t st = as_stream(stream);
  int B = blc_blocks(N, H, W);
  dim3 grid(B, N);
  float* partial = static_cast<float*>(workspace);
  blc_wb_bwd_kernel<<<grid, kT, 0, st>>>(raw, dout, draw, partial, H, W, params, param_stride);
  int rc = check_launch("blc_wb_bwd_kernel");
  if (rc != RISP_OK) return rc;
  const short idx[5] = {0, 1, 2, 3, 4};
  int P = param_stride == 0 ? 5 : param_stride;
  if (cudaMemsetAsync(dparams, 0, sizeof(float) * (size_t)P * (param_stride == 0 ? 1 : N), st) != cudaSuccess) {
    set_error("risp_bayer_blc_wb_bwd: memset failed");
    return RISP_E_CUDA;
  }
  return finalize_partials(partial, dparams, N, B, 8, P, idx, idx, 5, 1.f, param_stride == 0, st);
}

// ---- device-side input codec: integer sensor / display codes -> fp32 in [0,1] ---------------------------
// The reference's loaders decode 16-bit PNG Bayer frames and 8-bit ground truth on the HOST and ship fp32
// (x/1023. s7isp_rggb2bgr_dataset.py:123, x/16383. sid_sony_ratio_rggb2bgr_dataset.py:133, gt/255. :134),
// i.e. 16 B/px over PCIe.  Shipping the codes (2 + 3 B/px) and normalising here cuts the host->device
// volume 3.2x; the arithmetic is the same single fp32 multiply... the loaders use a DIVISION, so this does too.
namespace risp {
template <typename T>
__global__ void __launch_bounds__(256)
decode_kernel(const T* __restrict__ src, float* __restrict__ dst, long long n, float denom) {
  const long long nv = n / 4;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < nv; i += (long long)gridDim.x * 256) {
    float v[4];
    if (sizeof(T) == 2) {
      const uint2 t = *reinterpret_cast<const uint2*>(src + 4 * i);
      v[0] = (float)(t.x & 0xffffu); v[1] = (float)(t.x >> 16); v[2] = (float)(t.y & 0xffffu); v[3] = (float)(t.y >> 16);
    } else {
      const unsigned t = *reinterpret_cast<const unsigned*>(src + 4 * i);
      v[0] = (float)(t & 0xffu); v[1] = (float)((t >> 8) & 0xffu); v[2] = (float)((t >> 16) & 0xffu); v[3] = (float)(t >> 24);
    }
    st_stream4(dst + 4 * i, make_float4(__fdiv_rn(v[0], denom), __fdiv_rn(v[1], denom), __fdiv_rn(v[2], denom), __fdiv_rn(v[3], denom)));
  }
  for (long long i = nv * 4 + (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
    dst[i] = __fdiv_rn((float)src[i], denom);
}
}  // namespace risp

extern "C" int risp_decode_codes(const void* src, float* dst, long long n, int bytes_per_code, float denom,
                                 risp_stream_t stream) {
  RISP_REQUIRE(src && dst && n > 0 && denom > 0.f, RISP_E_INVALID, "risp_decode_codes: bad arguments");
  RISP_REQUIRE(bytes_per_code == 1 || bytes_per_code == 2, RISP_E_INVALID, "risp_decode_codes: 1 or 2 bytes per code");
  RISP_REQUIRE((reinterpret_cast<uintptr_t>(src) & 7) == 0 && aligned16(dst), RISP_E_ALIGN, "risp_decode_codes: alignment");
  long long g = cdiv(n / 4 + 1, 256);
  long long cap = (long long)sm_count() * 16;
  int grid = (int)(g > cap ? cap : g);
  if (bytes_per_code == 2)
    decode_kernel<unsigned short><<<grid, 256, 0, as_stream(stream)>>>(static_cast<const unsigned short*>(src), dst, n, denom);
  else
    decode_kernel<unsigned char><<<grid, 256, 0, as_stream(stream)>>>(static_cast<const unsigned char*>(src), dst, n, denom);
  return check_launch("decode_kernel");
}

namespace risp {
// Crop + decode of a batch of records: the loader's random crop, after the PCIe hop or out of a frame store in HBM.
// Record r = (frame a, frame b, y0, x0) crops store a (pa planes per frame, codes of T) and store b (pb planes per frame,
// 8-bit codes) at the same origin:  da[r][p] = a[frame a][p][y0:y0+h, x0:x0+w] / denom_a, and db likewise from b.
// Records may be device data the host never sees, so each block checks its own: a record out of range, or odd where
// `odd` asks for even origins (the CFA phase of a Bayer crop), sets *status and is skipped; nothing outside the stores is read.
struct CropJob {
  const void* a;
  const unsigned char* b;
  float* da;
  float* db;
  const int4* pos;       // DEVICE records; null: the single record (0, 0, y0, x0)
  int fa, fb;            // frames in each store
  int pa, pb;            // planes per frame (pb = 0: no second store)
  int H, W, h, w, y0, x0;
  int odd;               // origin bits that must be clear: 1 for a Bayer crop, 0 for any origin
  float denom_a, denom_b;
  int* status;           // nullable when pos is null (the host checked the one record)
};

// One plane of one record.  s: the crop's first code, d: the output plane.  VEC: four columns per item and one 16-byte
// store (w % 4 == 0, d 16-byte aligned).  An item's row and column advance by a constant stride: no division in the loop.
template <typename T, bool VEC>
__device__ __forceinline__ void crop_plane(const T* __restrict__ s, float* __restrict__ d, int W, int h, int w, float denom) {
  constexpr int V = VEC ? 4 : 1;
  const int wq = w / V;
  const int start = blockIdx.x * 256 + threadIdx.x, step = gridDim.x * 256;
  int y = start / wq, x = start - y * wq;
  const int dy = step / wq, dx = step - dy * wq;
  while (y < h) {
    const T* p = s + (long long)y * W + x * V;
    float* o = d + (long long)y * w + x * V;
    if (VEC)
      st_stream4(o, make_float4(__fdiv_rn((float)__ldg(p), denom), __fdiv_rn((float)__ldg(p + 1), denom),
                                __fdiv_rn((float)__ldg(p + 2), denom), __fdiv_rn((float)__ldg(p + 3), denom)));
    else
      *o = __fdiv_rn((float)__ldg(p), denom);
    x += dx;
    y += dy;
    if (x >= wq) { x -= wq; ++y; }
  }
}

// grid: x = blocks per output plane, y = records * (pa + pb) output planes
template <typename T, bool VEC>
__global__ void __launch_bounds__(256)
crop_decode_kernel(const CropJob j) {
  const int planes = j.pa + j.pb;
  const int r = blockIdx.y / planes, p = blockIdx.y - r * planes;
  const int4 rec = j.pos ? j.pos[r] : make_int4(0, 0, j.y0, j.x0);
  if (rec.x < 0 || rec.x >= j.fa || (j.pb && (rec.y < 0 || rec.y >= j.fb)) || rec.z < 0 || rec.w < 0 ||
      rec.z > j.H - j.h || rec.w > j.W - j.w || ((rec.z | rec.w) & j.odd)) {
    if (j.status && threadIdx.x == 0) *j.status = 1;
    return;
  }
  const long long plane_in = (long long)j.H * j.W, plane_out = (long long)j.h * j.w, off = (long long)rec.z * j.W + rec.w;
  if (p < j.pa)
    crop_plane<T, VEC>(static_cast<const T*>(j.a) + ((long long)rec.x * j.pa + p) * plane_in + off,
                       j.da + ((long long)r * j.pa + p) * plane_out, j.W, j.h, j.w, j.denom_a);
  else
    crop_plane<unsigned char, VEC>(j.b + ((long long)rec.y * j.pb + p - j.pa) * plane_in + off,
                                   j.db + ((long long)r * j.pb + p - j.pa) * plane_out, j.W, j.h, j.w, j.denom_b);
}

// At most max(16 blocks per SM, one block per output plane) blocks; each block strides over its plane.
static int launch_crops(const CropJob& j, int records, int bytes_per_code, cudaStream_t st) {
  const bool vec = j.w % 4 == 0 && aligned16(j.da) && (j.pb == 0 || aligned16(j.db));
  const int planes = records * (j.pa + j.pb);
  long long g = cdiv((long long)j.h * (vec ? j.w / 4 : j.w), 256), cap = (long long)sm_count() * 16 / planes;
  if (cap < 1) cap = 1;
  dim3 grid((unsigned)(g > cap ? cap : g), (unsigned)planes);
  if (bytes_per_code == 2) {
    if (vec) crop_decode_kernel<unsigned short, true><<<grid, 256, 0, st>>>(j);
    else crop_decode_kernel<unsigned short, false><<<grid, 256, 0, st>>>(j);
  } else {
    if (vec) crop_decode_kernel<unsigned char, true><<<grid, 256, 0, st>>>(j);
    else crop_decode_kernel<unsigned char, false><<<grid, 256, 0, st>>>(j);
  }
  return check_launch("crop_decode_kernel");
}
}  // namespace risp

extern "C" int risp_crop_decode(const void* src, float* dst, int planes, int H, int W, int y0, int x0, int h, int w,
                                int bytes_per_code, float denom, int require_even, risp_stream_t stream) {
  RISP_REQUIRE(src && dst && planes > 0 && planes <= 65535 && H > 0 && W > 0 && h > 0 && w > 0 && denom > 0.f, RISP_E_INVALID,
               "risp_crop_decode: bad arguments");
  RISP_REQUIRE(y0 >= 0 && x0 >= 0 && y0 + h <= H && x0 + w <= W, RISP_E_INVALID, "risp_crop_decode: crop %dx%d at (%d,%d) leaves the %dx%d frame",
               h, w, y0, x0, H, W);
  RISP_REQUIRE(bytes_per_code == 1 || bytes_per_code == 2, RISP_E_INVALID, "risp_crop_decode: 1 or 2 bytes per code");
  RISP_REQUIRE(!require_even || ((y0 % 2 == 0) && (x0 % 2 == 0)), RISP_E_ALIGN,
               "risp_crop_decode: a Bayer crop must start on an even row and column (CFA phase), got (%d,%d)", y0, x0);
  CropJob j{};
  j.a = src; j.da = dst; j.fa = 1; j.pa = planes;
  j.H = H; j.W = W; j.h = h; j.w = w; j.y0 = y0; j.x0 = x0;
  j.odd = require_even ? 1 : 0;
  j.denom_a = denom;
  return launch_crops(j, 1, bytes_per_code, as_stream(stream));
}

extern "C" int risp_sample_crops(const void* raw_store, int raw_bytes_per_code, int F, const unsigned char* gt_store, int G,
                                 int H, int W, const int* pos, int B, int h, int w, float white_level, float* img_out,
                                 float* gt_out, int* status, risp_stream_t stream) {
  RISP_REQUIRE(raw_store && pos && img_out && status && F > 0 && H > 0 && W > 0 && B > 0 && h > 0 && w > 0 && white_level > 0.f,
               RISP_E_INVALID, "risp_sample_crops: bad arguments");
  RISP_REQUIRE(!gt_out || (gt_store && G > 0), RISP_E_INVALID, "risp_sample_crops: gt_out needs gt_store and G > 0");
  RISP_REQUIRE(raw_bytes_per_code == 1 || raw_bytes_per_code == 2, RISP_E_INVALID, "risp_sample_crops: 1 or 2 bytes per raw code");
  RISP_REQUIRE(h <= H && w <= W, RISP_E_INVALID, "risp_sample_crops: a %dx%d crop does not fit the %dx%d frames", h, w, H, W);
  RISP_REQUIRE((long long)B * (gt_out ? 4 : 1) <= 65535, RISP_E_INVALID, "risp_sample_crops: %d records are too many for one launch", B);
  RISP_REQUIRE(aligned16(pos), RISP_E_ALIGN, "risp_sample_crops: pos must be 16-byte aligned");
  CropJob j{};
  j.a = raw_store; j.da = img_out; j.fa = F; j.pa = 1;
  if (gt_out) { j.b = gt_store; j.db = gt_out; j.fb = G; j.pb = 3; }
  j.pos = reinterpret_cast<const int4*>(pos);
  j.H = H; j.W = W; j.h = h; j.w = w;
  j.odd = 1;
  j.denom_a = white_level; j.denom_b = 255.f;
  j.status = status;
  return launch_crops(j, B, raw_bytes_per_code, as_stream(stream));
}
