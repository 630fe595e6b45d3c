// Fused raw -> BGR pipeline: demosaic head + per-pixel stage chain (+ MSE loss and parameter
// gradients) in ONE pass over the frame.   risp_demosaic_fwd / risp_pipeline_fwd / risp_pipeline_mse_step
//
// Reference: the containers run one full-image pass per stage and keep every intermediate
// (isp_universal.py:210-232, origin_universal.py:143-161); proxy tuning adds MSELoss + backward
// (isp_model.py:128-142).  Here a frame costs 16 B/px forward (read raw 4, write BGR 12) and
// 16 B/px for the whole tuning step (read raw 4 + GT 12; nothing is written but ~100 floats).
//
// Design: "register-marching" stencil.  One warp owns a 128-column strip and walks down a chunk of
// rows; each lane holds the (2*HL+1) x (4+2*HL) raw window of its 4 output pixels in registers.
// A new raw row costs one coalesced 128-bit load per lane; the horizontal halo comes from the
// neighbouring lanes by warp shuffle (only lanes 0/31 touch memory for it), the vertical halo stays
// in registers.  No shared memory, no block barrier, and the next row (raw and GT) is always in
// flight while the current one is being computed.  Borders are reflect-101, which preserves the
// CFA phase.  Requires H even and W % 4 == 0 (reference frames: 48..4000, all multiples of 4).
#include "risp_common.cuh"
#include "risp_stage.cuh"

#include <stdlib.h>
#include <type_traits>

namespace risp {

constexpr int kWarpsPerBlock = 4;
constexpr int kStripCols = 128;  // columns per warp

template <int HL> struct RawRow;  // one lane's share of one raw row, before the halo exchange
template <> struct RawRow<1> { float4 v; float l, r; };
template <> struct RawRow<2> { float4 v; float2 l, r; };

__device__ __forceinline__ int reflect101(int r, int H) { return r < 0 ? -r : (r >= H ? 2 * H - 2 - r : r); }

// issue the loads of row `row` (already reflected) -- no dependent instruction here
template <int HL>
__device__ __forceinline__ void row_issue(RawRow<HL>& q, const float* __restrict__ img, int row, int W, int c0,
                                          bool active, int lane) {
  const float* rp = img + (long long)row * W;
  q.v = active ? __ldg(reinterpret_cast<const float4*>(rp + c0)) : make_float4(0.f, 0.f, 0.f, 0.f);
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

// the same row out of a frame store of ES-byte codes (ES = 2: 16-bit, 1: 8-bit): the codes are loaded here and decoded in
// row_decode, after the loads have been issued
template <int HL> struct CodeRow { uint2 v; uint32_t l, r; };   // 4 codes (ES = 1: v.x only); HL halo codes each side
template <int HL, int ES>
__device__ __forceinline__ void row_issue_codes(CodeRow<HL>& q, const unsigned char* __restrict__ img, int row, int W, int c0,
                                                bool active, int lane) {
  const unsigned char* rp = img + (long long)row * W * ES;
  q.v = make_uint2(0u, 0u); q.l = 0u; q.r = 0u;
  if (active) {
    if constexpr (ES == 2) q.v = __ldg(reinterpret_cast<const uint2*>(rp + 2 * c0));
    else q.v.x = __ldg(reinterpret_cast<const uint32_t*>(rp + c0));
  }
  // HL codes at c0-HL and at c0+4: 2-byte aligned (c0 % 4 == 0)
  auto ld = [&](int c) -> uint32_t {
    if constexpr (ES == 2) return HL == 1 ? (uint32_t)__ldg(reinterpret_cast<const unsigned short*>(rp + 2 * c))
                                          : __ldg(reinterpret_cast<const uint32_t*>(rp + 2 * c));
    else return HL == 1 ? (uint32_t)__ldg(rp + c) : (uint32_t)__ldg(reinterpret_cast<const unsigned short*>(rp + c));
  };
  if (active && lane == 0 && c0 > 0) q.l = ld(c0 - HL);
  if (active && lane == 31 && c0 + 4 < W) q.r = ld(c0 + 4);
}
// the same row of a crop: img is the crop's first code in frames of `stride` codes per row (W: the crop's width).  The crop's
// origin is only even, so the 4 codes are loaded as two halves (4 / 2-byte aligned) instead of one 8 / 4-byte vector; the
// halo codes at c0-HL and c0+4 stay 2-byte aligned
template <int HL, int ES>
__device__ __forceinline__ void row_issue_crop_codes(CodeRow<HL>& q, const unsigned char* __restrict__ img, int row, int stride,
                                                     int W, int c0, bool active, int lane) {
  const unsigned char* rp = img + (long long)row * stride * ES;
  q.v = make_uint2(0u, 0u); q.l = 0u; q.r = 0u;
  if (active) {
    if constexpr (ES == 2)
      q.v = make_uint2(__ldg(reinterpret_cast<const uint32_t*>(rp + 2 * c0)), __ldg(reinterpret_cast<const uint32_t*>(rp + 2 * c0 + 4)));
    else
      q.v.x = (uint32_t)__ldg(reinterpret_cast<const unsigned short*>(rp + c0)) |
              ((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(rp + c0 + 2)) << 16);
  }
  auto ld = [&](int c) -> uint32_t {
    if constexpr (ES == 2) return HL == 1 ? (uint32_t)__ldg(reinterpret_cast<const unsigned short*>(rp + 2 * c))
                                          : __ldg(reinterpret_cast<const uint32_t*>(rp + 2 * c));
    else return HL == 1 ? (uint32_t)__ldg(rp + c) : (uint32_t)__ldg(reinterpret_cast<const unsigned short*>(rp + c));
  };
  if (active && lane == 0 && c0 > 0) q.l = ld(c0 - HL);
  if (active && lane == 31 && c0 + 4 < W) q.r = ld(c0 + 4);
}
template <int HL, int ES>
__device__ __forceinline__ RawRow<HL> row_decode(const CodeRow<HL>& q, float wl) {
  constexpr int B = 8 * ES;                 // bits per code
  constexpr uint32_t M = (1u << B) - 1u;
  RawRow<HL> o;
  const uint32_t c1 = ES == 2 ? q.v.x >> 16 : (q.v.x >> 8) & M, c2 = ES == 2 ? q.v.y & M : (q.v.x >> 16) & M,
                 c3 = ES == 2 ? q.v.y >> 16 : q.v.x >> 24;
  o.v = make_float4(decode_code(q.v.x & M, wl), decode_code(c1, wl), decode_code(c2, wl), decode_code(c3, wl));
  if constexpr (HL == 1) {
    o.l = decode_code(q.l, wl); o.r = decode_code(q.r, wl);
  } else {
    o.l = make_float2(decode_code(q.l & M, wl), decode_code(q.l >> B, wl));
    o.r = make_float2(decode_code(q.r & M, wl), decode_code(q.r >> B, wl));
  }
  return o;
}

// halo exchange: dst[0 .. 4+2*HL) = columns c0-HL .. c0+3+HL of the row
template <int HL>
__device__ __forceinline__ void row_finish(float (&dst)[4 + 2 * HL], const RawRow<HL>& q, int W, int c0,
                                           bool active, int lane) {
  const unsigned full = 0xffffffffu;
  const float4 v = q.v;
  const bool first = (c0 == 0), last = active && (c0 + 4 >= W);
  if constexpr (HL == 1) {
    float l = __shfl_up_sync(full, v.w, 1), r = __shfl_down_sync(full, v.x, 1);
    if (lane == 0) l = first ? v.y : q.l;          // col -1 -> col 1
    if (last) r = v.z;                             // col W  -> col W-2
    else if (lane == 31) r = q.r;
    dst[0] = l; dst[1] = v.x; dst[2] = v.y; dst[3] = v.z; dst[4] = v.w; dst[5] = r;
  } else {
    float l0 = __shfl_up_sync(full, v.z, 1), l1 = __shfl_up_sync(full, v.w, 1);
    float r0 = __shfl_down_sync(full, v.x, 1), r1 = __shfl_down_sync(full, v.y, 1);
    const float2 ql = q.l, qr = q.r;
    if (lane == 0) { l0 = first ? v.z : ql.x; l1 = first ? v.y : ql.y; }   // cols -2,-1 -> 2,1
    if (last) { r0 = v.z; r1 = v.y; }                                       // cols W,W+1 -> W-2,W-3
    else if (lane == 31) { r0 = qr.x; r1 = qr.y; }
    dst[0] = l0; dst[1] = l1; dst[2] = v.x; dst[3] = v.y; dst[4] = v.z; dst[5] = v.w; dst[6] = r0; dst[7] = r1;
  }
}

// ---- demosaic of 4 pixels from the register window --------------------------------------------------
// w[j][i]: row r-HL+j, column c0-HL+i.  `odd` = row parity (warp-uniform).  c0 is even, so pixel k has
// column parity k&1.   Sites: (even,even)=R (even,odd)=G1 (odd,even)=G2 (odd,odd)=B.
template <int DM, int HL>
__device__ __forceinline__ void demosaic4(const float (&w)[2 * HL + 1][4 + 2 * HL], bool odd, float clip_hi, Px<4>& out) {
  float (&B)[4] = out.b; float (&G)[4] = out.g; float (&R)[4] = out.r;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int x = HL + k;            // window column of the pixel
    const bool xo = (k & 1);
    const float c = w[HL][x];
    if (DM == RISP_DM_NEAREST) {
      // R,B replicated over the 2x2 cell; G from the same row (oracle/SPEC.md)
      if (!odd) {
        R[k] = xo ? w[HL][x - 1] : c;
        G[k] = xo ? c : w[HL][x + 1];
        B[k] = xo ? w[HL + 1][x] : w[HL + 1][x + 1];
      } else {
        R[k] = xo ? w[HL - 1][x - 1] : w[HL - 1][x];
        G[k] = xo ? w[HL][x - 1] : c;
        B[k] = xo ? c : w[HL][x + 1];
      }
    } else if (DM == RISP_DM_BILINEAR) {
      const float cross = (w[HL - 1][x] + w[HL + 1][x]) + (w[HL][x - 1] + w[HL][x + 1]);
      const float diag = (w[HL - 1][x - 1] + w[HL - 1][x + 1]) + (w[HL + 1][x - 1] + w[HL + 1][x + 1]);
      const float hor = 0.5f * (w[HL][x - 1] + w[HL][x + 1]);
      const float ver = 0.5f * (w[HL - 1][x] + w[HL + 1][x]);
      const bool at_g = (odd != xo);
      G[k] = at_g ? c : 0.25f * cross;
      if (!odd) { R[k] = xo ? hor : c;           B[k] = xo ? ver : 0.25f * diag; }
      else      { R[k] = xo ? 0.25f * diag : ver; B[k] = xo ? c : hor; }
    } else {  // Malvar-He-Cutler 5x5
      const float n1 = w[HL - 1][x], s1 = w[HL + 1][x], e1 = w[HL][x + 1], w1 = w[HL][x - 1];
      const float n2 = w[HL - 2][x], s2 = w[HL + 2][x], e2 = w[HL][x + 2], w2 = w[HL][x - 2];
      const float dg = (w[HL - 1][x - 1] + w[HL - 1][x + 1]) + (w[HL + 1][x - 1] + w[HL + 1][x + 1]);
      const float f_g = 0.125f * (4.f * c + 2.f * ((n1 + s1) + (e1 + w1)) - ((n2 + s2) + (e2 + w2)));
      const float f_row = 0.125f * (5.f * c + 4.f * (e1 + w1) - dg - (e2 + w2) + 0.5f * (n2 + s2));
      const float f_col = 0.125f * (5.f * c + 4.f * (n1 + s1) - dg - (n2 + s2) + 0.5f * (e2 + w2));
      const float f_dg = 0.125f * (6.f * c + 2.f * dg - 1.5f * ((n2 + s2) + (e2 + w2)));
      float rr, gg, bb;
      if (!odd) { rr = xo ? f_row : c;    gg = xo ? c : f_g; bb = xo ? f_col : f_dg; }
      else      { rr = xo ? f_dg : f_col; gg = xo ? f_g : c; bb = xo ? c : f_row; }
      R[k] = fminf(fmaxf(rr, 0.f), clip_hi); G[k] = fminf(fmaxf(gg, 0.f), clip_hi);
      B[k] = fminf(fmaxf(bb, 0.f), clip_hi);
    }
  }
}

// EVAL: the forward of MODE_FWD, then the squared 8-bit code differences to the GT (per-image PSNR numerator); writes no y
// EVAL_S16 / EVAL_U8: EVAL reading a frame store (16-bit / 8-bit raw codes, 8-bit planar GT codes; frames named by records)
// STEP_S16 / STEP_U8: STEP (MSE target, not dy) on h x w crops of a frame store (crops named by records)
enum { MODE_FWD = 0, MODE_STEP = 1, MODE_EVAL = 2, MODE_EVAL_S16 = 3, MODE_EVAL_U8 = 4, MODE_STEP_S16 = 5, MODE_STEP_U8 = 6 };
constexpr bool is_store(int mode) { return mode == MODE_EVAL_S16 || mode == MODE_EVAL_U8 || mode == MODE_STEP_S16 || mode == MODE_STEP_U8; }
constexpr bool is_eval(int mode) { return mode == MODE_EVAL || mode == MODE_EVAL_S16 || mode == MODE_EVAL_U8; }
constexpr bool is_step(int mode) { return mode == MODE_STEP || mode == MODE_STEP_S16 || mode == MODE_STEP_U8; }

// 4 GT codes of a crop row (2-byte aligned: the crop's origin is even) decoded as the sampler decodes them, code / 255
__device__ __forceinline__ float4 gt_codes4(const unsigned char* __restrict__ p) {
  const uint32_t v = (uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p)) |
                     ((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p + 2)) << 16);
  return make_float4(decode_code(v & 0xffu, 255.f), decode_code((v >> 8) & 0xffu, 255.f), decode_code((v >> 16) & 0xffu, 255.f),
                     decode_code(v >> 24, 255.f));
}
// the 3 planes of a crop's GT row (o: offset of the lane's first pixel in the first plane, fplane: codes per frame plane)
__device__ __forceinline__ void crop_gt_row(const unsigned char* __restrict__ sgt, long long fplane, long long o, float4& b,
                                            float4& g, float4& r) {
  b = gt_codes4(sgt + o); g = gt_codes4(sgt + fplane + o); r = gt_codes4(sgt + 2 * fplane + o);
}

// packed-fp32 / constant-bank kernels for the pre-instantiated signatures (risp_fused.cu)
bool fused_handles(const ChainDesc& d, int N, int param_stride, int H, int W);
int fused_partial_rows_per_frame(int N);
int fused_launch(int mode, const float* raw, const float* gt, float* y, float* partial, const float* params, int pstride,
                 int N, int H, int W, int dm_kind, float clip_hi, const ChainDesc& d, cudaStream_t st, int* rows_per_frame);
int fused_eval_launch(const float* raw, const float* gt, unsigned char* u8, unsigned long long* partial, const float* params,
                      int pstride, int N, int H, int W, int dm_kind, float clip_hi, const ChainDesc& d, cudaStream_t st,
                      int* rows_per_frame);
int fused_eval_store_launch(const void* raw_store, int raw_bpc, int F, const unsigned char* gt_store, int G, const int* pos,
                            int* status, float white_level, unsigned char* u8, unsigned long long* partial, const float* params,
                            int pstride, int N, int H, int W, int dm_kind, float clip_hi, const ChainDesc& d, cudaStream_t st,
                            int* rows_per_frame);
int fused_step_store_launch(bool l1, const void* raw_store, int raw_bpc, int F, const unsigned char* gt_store, int G, int H,
                            int W, const int* pos, int* status, float white_level, float* partial, const float* params,
                            int pstride, int N, int h, int w, int dm_kind, float clip_hi, const ChainDesc& d, cudaStream_t st,
                            int* rows_per_frame);

struct PipeArgs {
  const float* raw;   // (N,1,H,W)
  const float* gt;    // (N,3,H,W)   MODE_STEP
  float* y;           // (N,3,H,W)   nullable in MODE_STEP
  float* partial;     // MODE_STEP: [N][warps_per_image][RISP_NSLOT]
  const float* params;
  int pstride;
  int H, W, rows_per_chunk;
  float clip_hi;
  int gt_is_dy;       // MODE_STEP: `gt` holds dL/dy (container-level backward) instead of the target
  unsigned char* u8;  // MODE_EVAL: (N,H,W,3) 8-bit codes of y, nullable
  unsigned long long* sse;   // MODE_EVAL: [N][warps_per_image] sums of squared code differences
  // store modes: image n is raw frame pos[n].x of `store` against the 8-bit planar GT frame pos[n].y of `gstore`
  const unsigned char* store;
  const unsigned char* gstore;
  const int4* pos;
  int* status;        // set when a record is not a whole frame (eval) / a crop (step) of the stores; that image adds nothing
  float white_level;
  int F, G;
};

// resident CTAs per SM the kernels are compiled for (register cap)
constexpr int kStepMinBlocks = 2;   // backward-carrying kernels of the pre-instantiated signatures (the generic one: 1)
constexpr int kFwdMinBlocks = 4;
constexpr int kEvalMinBlocks = 3;   // the forward's registers plus the GT row in flight: 4 CTAs (128 registers) spill
constexpr int kPairUnroll = 2;
// One raw row in flight per warp in the forward-only kernel: measured on B200 (12 MP x 4, bilinear + 4 stages), two rows
// took 0.242 ms against 0.234 ms for one -- the kernel is not latency-bound.

template <int DM, int MODE, unsigned SIG, bool BIGG>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, is_step(MODE) ? ((SIG == 0) ? 1 : kStepMinBlocks)
                                                    : is_eval(MODE) ? kEvalMinBlocks : kFwdMinBlocks)
pipeline_kernel(PipeArgs a, ChainDesc d, const int2 frame) {   // frame: store step modes, (H, W) of the stores' frames
  using SG = Sig<SIG>;
  constexpr int SMAX = SG::S;
  constexpr bool BIG = SG::generic ? BIGG : SG::big_c();
  constexpr int HL = (DM == RISP_DM_MALVAR) ? 2 : 1;
  constexpr int WR = 2 * HL + 1, WC = 4 + 2 * HL;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int strip = blockIdx.x * kWarpsPerBlock + wid;
  const int n = blockIdx.z;
  const int H = a.H, W = a.W;
  const int c0 = strip * kStripCols + lane * 4;
  const bool active = c0 < W;
  const int ra = blockIdx.y * a.rows_per_chunk;
  const int rb = min(H, ra + a.rows_per_chunk);
  const long long plane = (long long)H * W;
  constexpr bool ST = is_store(MODE);
  constexpr bool CROP = ST && is_step(MODE);               // store step modes: the image is a crop of a frame
  constexpr int ES = (MODE == MODE_EVAL_S16 || MODE == MODE_STEP_S16) ? 2 : 1;      // store modes: bytes per raw code
  bool ok = true;                                          // store modes: the record names a whole frame / crop of the stores
  const unsigned char* __restrict__ simg = nullptr;        // store modes: the raw frame's codes and the GT frame's planes
  const unsigned char* __restrict__ sgt = nullptr;         // (store step modes: their codes at the crop's origin)
  if constexpr (CROP) {
    const int4 rec = a.pos[n];
    ok = crop_record(rec, a.F, a.G, frame.x, frame.y, H, W);
    if (!ok && threadIdx.x == 0) *a.status = 1;
    const long long fplane = (long long)frame.x * frame.y, org = ok ? (long long)rec.z * frame.y + rec.w : 0;
    simg = a.store + ((ok ? rec.x : 0) * fplane + org) * ES;
    sgt = a.gstore + (ok ? rec.y : 0) * 3 * fplane + org;
  } else if constexpr (ST) {
    const int4 rec = a.pos[n];
    ok = whole_frame_record(rec, a.F, a.G);
    if (!ok && threadIdx.x == 0) *a.status = 1;
    simg = a.store + (long long)(ok ? rec.x : 0) * plane * ES;
    sgt = a.gstore + (long long)(ok ? rec.y : 0) * 3 * plane;
  }
  const float* __restrict__ img = ST ? nullptr : a.raw + (long long)n * plane;
  const float* __restrict__ prow = a.params + (long long)n * a.pstride;
  const float* __restrict__ gtb = (MODE != MODE_FWD) ? a.gt + (long long)n * 3 * plane : nullptr;
  float* __restrict__ yb = a.y ? a.y + (long long)n * 3 * plane : nullptr;

  float accS[SMAX][RISP_SMALL_ACC];
  float2 accB[RISP_BIG_ACC];
  float loss = 0.f;
  unsigned long long sse = 0;     // MODE_EVAL: this lane's sum of squared code differences
  if (is_step(MODE)) {
#pragma unroll
    for (int s = 0; s < SMAX; ++s)
#pragma unroll
      for (int j = 0; j < RISP_SMALL_ACC; ++j) accS[s][j] = 0.f;
#pragma unroll
    for (int k = 0; k < RISP_BIG_ACC; ++k) accB[k] = make_float2(0.f, 0.f);
  }

  if (strip * kStripCols < W && (!ST || ok)) {   // warp-uniform: the whole strip is outside the frame otherwise
    float w[WR][WC];
    std::conditional_t<ST, CodeRow<HL>, RawRow<HL>> q;     // store modes: codes, decoded when the row is finished
#pragma unroll
    for (int j = 0; j < WR - 1; ++j) {
      if constexpr (ST) {
        if constexpr (CROP) row_issue_crop_codes<HL, ES>(q, simg, reflect101(ra - HL + j, H), frame.y, W, c0, active, lane);
        else row_issue_codes<HL, ES>(q, simg, reflect101(ra - HL + j, H), W, c0, active, lane);
        row_finish<HL>(w[j], row_decode<HL, ES>(q, a.white_level), W, c0, active, lane);
      } else {
        row_issue<HL>(q, img, reflect101(ra - HL + j, H), W, c0, active, lane);
        row_finish<HL>(w[j], q, W, c0, active, lane);
      }
    }
    if constexpr (CROP) row_issue_crop_codes<HL, ES>(q, simg, reflect101(ra + HL, H), frame.y, W, c0, active, lane);
    else if constexpr (ST) row_issue_codes<HL, ES>(q, simg, reflect101(ra + HL, H), W, c0, active, lane);
    else row_issue<HL>(q, img, reflect101(ra + HL, H), W, c0, active, lane);
    float4 gB = make_float4(0.f, 0.f, 0.f, 0.f), gG = gB, gR = gB;   // GT of the row being computed, fetched one row ahead
    if (MODE == MODE_STEP && active) {
      const long long o = (long long)ra * W + c0;
      gB = ld_stream4(gtb + o); gG = ld_stream4(gtb + plane + o); gR = ld_stream4(gtb + 2 * plane + o);
    }
    if constexpr (CROP) {
      if (active) crop_gt_row(sgt, (long long)frame.x * frame.y, (long long)ra * frame.y + c0, gB, gG, gR);
    }
    for (int r = ra; r < rb; ++r) {
      if constexpr (ST) row_finish<HL>(w[WR - 1], row_decode<HL, ES>(q, a.white_level), W, c0, active, lane);
      else row_finish<HL>(w[WR - 1], q, W, c0, active, lane);
      const float4 tB = gB, tG = gG, tR = gR;
      float4 eB, eG, eR;         // MODE_EVAL: GT of this row
      [[maybe_unused]] uint32_t sB, sG, sR;   // store modes: its 4 codes per plane
      if constexpr (is_eval(MODE)) {
        // requested before the demosaic and the chain it waits behind (a row-ahead prefetch as in MODE_STEP keeps two GT
        // rows live and spills)
        if (active) {
          const long long o = (long long)r * W + c0;
          if constexpr (ST) {
            sB = __ldg(reinterpret_cast<const uint32_t*>(sgt + o)); sG = __ldg(reinterpret_cast<const uint32_t*>(sgt + plane + o));
            sR = __ldg(reinterpret_cast<const uint32_t*>(sgt + 2 * plane + o));
          } else {
            eB = ld_stream4(gtb + o); eG = ld_stream4(gtb + plane + o); eR = ld_stream4(gtb + 2 * plane + o);
          }
        }
      }
      if (r + 1 < rb) {
        if constexpr (CROP) row_issue_crop_codes<HL, ES>(q, simg, reflect101(r + 1 + HL, H), frame.y, W, c0, active, lane);
        else if constexpr (ST) row_issue_codes<HL, ES>(q, simg, reflect101(r + 1 + HL, H), W, c0, active, lane);
        else row_issue<HL>(q, img, reflect101(r + 1 + HL, H), W, c0, active, lane);
        if (MODE == MODE_STEP && active) {
          const long long o = (long long)(r + 1) * W + c0;
          gB = ld_stream4(gtb + o); gG = ld_stream4(gtb + plane + o); gR = ld_stream4(gtb + 2 * plane + o);
        }
        if constexpr (CROP) {
          if (active) crop_gt_row(sgt, (long long)frame.x * frame.y, (long long)(r + 1) * frame.y + c0, gB, gG, gR);
        }
      }
      Px<4> px;
      demosaic4<DM, HL>(w, (r & 1) != 0, a.clip_hi, px);
      if constexpr (is_eval(MODE)) {
#pragma unroll
        for (int s = 0; s < SMAX; ++s)
          if (SG::live(d, s)) stage_fwd(SG::op(d, s), SG::iarg(d, s), prow + d.off[s], px);
        if (active) {
          const float4 yB = make_float4(px.b[0], px.b[1], px.b[2], px.b[3]), yG = make_float4(px.g[0], px.g[1], px.g[2], px.g[3]),
                       yR = make_float4(px.r[0], px.r[1], px.r[2], px.r[3]);
          if constexpr (ST) sse += sq_codes4_u8(yB, sB) + sq_codes4_u8(yG, sG) + sq_codes4_u8(yR, sR);
          else sse += sq_codes4(yB, eB) + sq_codes4(yG, eG) + sq_codes4(yR, eR);
          if (a.u8) {        // (H,W,3) BGR bytes of the lane's 4 pixels: 12 contiguous bytes, 4-byte aligned (c0 % 4 == 0)
            uint32_t b[4], g[4], rr[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) { b[k] = u8_code(px.b[k]); g[k] = u8_code(px.g[k]); rr[k] = u8_code(px.r[k]); }
            uint32_t* po = reinterpret_cast<uint32_t*>(a.u8 + (((long long)n * H + r) * W + c0) * 3);
            po[0] = b[0] | (g[0] << 8) | (rr[0] << 16) | (b[1] << 24);
            po[1] = g[1] | (rr[1] << 8) | (b[2] << 16) | (g[2] << 24);
            po[2] = rr[2] | (b[3] << 8) | (g[3] << 16) | (rr[3] << 24);
          }
        }
      } else if (MODE == MODE_FWD) {
#pragma unroll
        for (int s = 0; s < SMAX; ++s)
          if (SG::live(d, s)) stage_fwd(SG::op(d, s), SG::iarg(d, s), prow + d.off[s], px);
      } else {
        // Backward-carrying mode: the 4 pixels of the lane are processed as two sequential PAIRS so that
        // only one pair's saved activations / gradients are live at a time (register pressure decides the
        // occupancy of this kernel).  The pair is selected with a warp-uniform predicate, not an index.
        const float gtB[4] = {tB.x, tB.y, tB.z, tB.w}, gtG[4] = {tG.x, tG.y, tG.z, tG.w},
                    gtR[4] = {tR.x, tR.y, tR.z, tR.w};
#pragma unroll kPairUnroll
        for (int h = 0; h < 2; ++h) {
          const bool hi = (h != 0);
          Px<2> saved[SMAX + 1];        // saved[s] = input of stage s, saved[s+1] = its output
          Px<2> cur, tgt;
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            cur.b[k] = hi ? px.b[2 + k] : px.b[k]; cur.g[k] = hi ? px.g[2 + k] : px.g[k]; cur.r[k] = hi ? px.r[2 + k] : px.r[k];
            tgt.b[k] = hi ? gtB[2 + k] : gtB[k]; tgt.g[k] = hi ? gtG[2 + k] : gtG[k]; tgt.r[k] = hi ? gtR[2 + k] : gtR[k];
          }
          saved[0] = cur;
#pragma unroll
          for (int s = 0; s < SMAX; ++s) {
            if (SG::live(d, s)) {
              stage_fwd(SG::op(d, s), SG::iarg(d, s), prow + d.off[s], cur);
              saved[s + 1] = cur;
            }
          }
          if (yb) {
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              if (hi) { px.b[2 + k] = cur.b[k]; px.g[2 + k] = cur.g[k]; px.r[2 + k] = cur.r[k]; }
              else { px.b[k] = cur.b[k]; px.g[k] = cur.g[k]; px.r[k] = cur.r[k]; }
            }
          }
          Px<2> dd;
          if (a.gt_is_dy) {
            dd = tgt;
          } else {
            // d loss / d y up to the constant 2/numel, applied by the finaliser
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              dd.b[k] = active ? cur.b[k] - tgt.b[k] : 0.f; dd.g[k] = active ? cur.g[k] - tgt.g[k] : 0.f;
              dd.r[k] = active ? cur.r[k] - tgt.r[k] : 0.f;
              loss = fmaf(dd.b[k], dd.b[k], fmaf(dd.g[k], dd.g[k], fmaf(dd.r[k], dd.r[k], loss)));
            }
          }
#pragma unroll
          for (int s = SMAX - 1; s >= 0; --s)
            if (SG::live(d, s)) stage_bwd<2, BIG>(SG::op(d, s), SG::iarg(d, s), prow + d.off[s], saved[s], saved[s + 1], dd, accS[s], accB);
        }
      }
      if (yb && active) {
        const long long o = (long long)r * W + c0;
        st_stream4(yb + o, make_float4(px.b[0], px.b[1], px.b[2], px.b[3]));
        st_stream4(yb + plane + o, make_float4(px.g[0], px.g[1], px.g[2], px.g[3]));
        st_stream4(yb + 2 * plane + o, make_float4(px.r[0], px.r[1], px.r[2], px.r[3]));
      }
#pragma unroll
      for (int j = 0; j < WR - 1; ++j)
#pragma unroll
        for (int i = 0; i < WC; ++i) w[j][i] = w[j + 1][i];
    }
  }

  if (is_step(MODE)) {
    const int warps_per_image = gridDim.y * gridDim.x * kWarpsPerBlock;
    const int widx = (blockIdx.y * gridDim.x + blockIdx.x) * kWarpsPerBlock + wid;
    float* __restrict__ out = a.partial + ((long long)n * warps_per_image + widx) * RISP_NSLOT;
#pragma unroll
    for (int s = 0; s < RISP_MAX_STAGES; ++s) {
#pragma unroll
      for (int j = 0; j < RISP_SMALL_ACC; ++j) {
        float v = 0.f;
        if (s < SMAX) { if (SG::live(d, s)) v = warp_sum(accS[s < SMAX ? s : 0][j]); }
        if (lane == 0) out[s * RISP_SMALL_ACC + j] = v;
      }
    }
#pragma unroll
    for (int k = 0; k < RISP_BIG_ACC; ++k) {
      float v0 = BIG ? warp_sum(accB[k].x) : 0.f, v1 = BIG ? warp_sum(accB[k].y) : 0.f;
      if (lane == 0) { out[RISP_SLOT_BIG + 2 * k] = v0; out[RISP_SLOT_BIG + 2 * k + 1] = v1; }
    }
    float v = warp_sum(loss);
    if (lane == 0) { out[RISP_SLOT_LOSS] = v; out[RISP_SLOT_LOSS + 1] = 0.f; }
  }
  if constexpr (is_eval(MODE)) {    // every warp writes its row, also one whose strip lies outside the frame
    const int warps_per_image = gridDim.y * gridDim.x * kWarpsPerBlock;
    const int widx = (blockIdx.y * gridDim.x + blockIdx.x) * kWarpsPerBlock + wid;
    const unsigned long long v = warp_sum_u64(sse);
    if (lane == 0) a.sse[(long long)n * warps_per_image + widx] = v;
  }
}

struct PipeGeom { int strips_x, chunks, rows_per_chunk, warps_per_image; };

static PipeGeom pipe_geometry(int N, int H, int W) {
  PipeGeom g;
  int strips = (int)cdiv(W, kStripCols);
  g.strips_x = (int)cdiv(strips, kWarpsPerBlock);
  // enough warps to fill 148 SMs x ~24 resident warps, but chunks of >= 8 rows so the vertical halo
  // (2*HL re-read rows per chunk, served by L2) stays small
  long long want_warps = (long long)sm_count() * 32;
  long long per_image = cdiv(want_warps, N);
  int chunks = (int)cdiv(per_image, (long long)g.strips_x * kWarpsPerBlock);
  int rows = (int)cdiv(H, chunks < 1 ? 1 : chunks);
  if (rows < 8) rows = 8;
  if (rows > 64) rows = 64;
  rows = (rows + 1) & ~1;
  g.rows_per_chunk = rows;
  g.chunks = (int)cdiv(H, rows);
  g.warps_per_image = g.chunks * g.strips_x * kWarpsPerBlock;
  return g;
}

template <int MODE>
static int launch_pipeline(const PipeArgs& a, const ChainDesc& d, int N, int dm_kind, bool big, cudaStream_t st,
                           int2 frame = int2{0, 0}) {
  PipeGeom g = pipe_geometry(N, a.H, a.W);
  PipeArgs b = a;
  b.rows_per_chunk = g.rows_per_chunk;
  dim3 grid(g.strips_x, g.chunks, N), block(kWarpsPerBlock * 32);
  const unsigned sig = chain_signature(d);
  bool done = false;
  // the evaluation mode has the generic instantiation only: the same stage_fwd arithmetic, 3 kernels instead of 15
#define RISP_PIPE_SIG(DMK, SG)                                                       \
  if constexpr (!is_eval(MODE)) {                                                    \
    if (!done && sig == (SG)) {                                                      \
      pipeline_kernel<DMK, MODE, (SG), false><<<grid, block, 0, st>>>(b, d, frame);  \
      done = true;                                                                   \
    }                                                                                \
  }
#define RISP_PIPE(DMK)                                                               \
  do {                                                                               \
    RISP_PIPE_SIG(DMK, RISP_SIG_A) RISP_PIPE_SIG(DMK, RISP_SIG_B) RISP_PIPE_SIG(DMK, RISP_SIG_C) RISP_PIPE_SIG(DMK, RISP_SIG_D) \
    if (!done) {                                                                     \
      if constexpr (is_eval(MODE)) pipeline_kernel<DMK, MODE, 0u, false><<<grid, block, 0, st>>>(b, d, frame);    \
      else if (big) pipeline_kernel<DMK, MODE, 0u, true><<<grid, block, 0, st>>>(b, d, frame); \
      else pipeline_kernel<DMK, MODE, 0u, false><<<grid, block, 0, st>>>(b, d, frame);      \
    }                                                                                \
  } while (0)
  switch (dm_kind) {
    case RISP_DM_NEAREST: RISP_PIPE(RISP_DM_NEAREST); break;
    case RISP_DM_BILINEAR: RISP_PIPE(RISP_DM_BILINEAR); break;
    case RISP_DM_MALVAR: RISP_PIPE(RISP_DM_MALVAR); break;
    default: set_error("unknown demosaic kind %d", dm_kind); return RISP_E_INVALID;
  }
#undef RISP_PIPE
#undef RISP_PIPE_SIG
  return check_launch("pipeline_kernel");
}

// RISP_FUSED=0 in the environment keeps every chain on the interpreter-style kernels of this file (A/B measurements)
static bool use_fused() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("RISP_FUSED"); v = (e && e[0] == '0') ? 0 : 1; }
  return v != 0;
}

static int check_frame(const char* who, const void* raw, int N, int H, int W) {
  RISP_REQUIRE(raw && N > 0 && H >= 4 && W >= 4, RISP_E_INVALID, "%s: bad frame arguments", who);
  RISP_REQUIRE(H % 2 == 0 && W % 4 == 0, RISP_E_ALIGN, "%s: needs H even and W %% 4 == 0 (got %dx%d)", who, H, W);
  RISP_REQUIRE(aligned16(raw), RISP_E_ALIGN, "%s: raw must be 16-byte aligned", who);
  RISP_REQUIRE(N <= 65535, RISP_E_INVALID, "%s: batch %d > 65535", who, N);
  return RISP_OK;
}

}  // namespace risp

using namespace risp;

extern "C" int risp_pipeline_fwd(const float* raw, float* y, int N, int H, int W, int dm_kind, float dm_clip_hi,
                                 const int* ops, const int* param_off, const int* iarg, int S, const float* params,
                                 int param_stride, risp_stream_t stream) {
  int rc = check_frame("risp_pipeline_fwd", raw, N, H, W);
  if (rc != RISP_OK) return rc;
  RISP_REQUIRE(y && aligned16(y), RISP_E_ALIGN, "risp_pipeline_fwd: y must be non-null and 16-byte aligned");
  ChainDesc d;
  int P = 0;
  rc = make_chain(&d, ops, param_off, iarg, S, &P);
  if (rc != RISP_OK) return rc;
  RISP_REQUIRE(P == 0 || params, RISP_E_INVALID, "risp_pipeline_fwd: chain needs %d parameters but params is null", P);
  RISP_REQUIRE(param_stride == 0 || param_stride >= P, RISP_E_INVALID, "risp_pipeline_fwd: param_stride %d < %d", param_stride, P);
  if (use_fused()) {
    ChainDesc df = d;
    if (S == 0) { df.S = 1; df.op[0] = RISP_OP_SKIP; df.off[0] = 0; df.iarg[0] = 0; }     // demosaic only
    rc = fused_launch(0, raw, nullptr, y, nullptr, params, param_stride, N, H, W, dm_kind, dm_clip_hi, df, as_stream(stream), nullptr);
    if (rc != 1) return rc;
  }
  PipeArgs a{raw, nullptr, y, nullptr, params, param_stride, H, W, 0, dm_clip_hi, 0};
  return launch_pipeline<MODE_FWD>(a, d, N, dm_kind, false, as_stream(stream));
}

extern "C" int risp_demosaic_fwd(const float* raw, float* bgr, int N, int H, int W, int kind, float clip_hi,
                                 risp_stream_t stream) {
  return risp_pipeline_fwd(raw, bgr, N, H, W, kind, clip_hi, nullptr, nullptr, nullptr, 0, nullptr, 0, stream);
}

extern "C" size_t risp_pipeline_eval_workspace(int N, int H, int W) {
  if (N <= 0 || H <= 0 || W <= 0) return 0;
  size_t rows = (size_t)pipe_geometry(N, H, W).warps_per_image;
  const size_t frows = (size_t)fused_partial_rows_per_frame(N);
  if (frows > rows) rows = frows;
  return (size_t)N * rows * sizeof(unsigned long long);
}

// Per-image sum of squared 8-bit code differences between the pipeline's output and gt, without writing the image: the same
// dispatch as risp_pipeline_fwd (packed kernel when it takes the chain, else the interpreter), so the codes are that entry
// point's codes under either setting of RISP_FUSED.
extern "C" int risp_pipeline_eval(const float* raw, const float* gt, unsigned char* u8_out, long long* sse_out, int N, int H,
                                  int W, int dm_kind, float dm_clip_hi, const int* ops, const int* param_off, const int* iarg,
                                  int S, const float* params, int param_stride, void* workspace, size_t workspace_bytes,
                                  risp_stream_t stream) {
  const char* who = "risp_pipeline_eval";
  int rc = check_frame(who, raw, N, H, W);
  if (rc != RISP_OK) return rc;
  RISP_REQUIRE(gt && sse_out, RISP_E_INVALID, "%s: gt and sse_out must be non-null", who);
  RISP_REQUIRE(aligned16(gt), RISP_E_ALIGN, "%s: gt must be 16-byte aligned", who);
  RISP_REQUIRE((reinterpret_cast<uintptr_t>(sse_out) & 7u) == 0, RISP_E_ALIGN, "%s: sse_out must be 8-byte aligned", who);
  RISP_REQUIRE((reinterpret_cast<uintptr_t>(u8_out) & 3u) == 0, RISP_E_ALIGN, "%s: u8_out must be 4-byte aligned", who);
  RISP_REQUIRE(dm_kind == RISP_DM_NEAREST || dm_kind == RISP_DM_BILINEAR || dm_kind == RISP_DM_MALVAR, RISP_E_INVALID,
               "%s: unknown demosaic kind %d", who, dm_kind);
  ChainDesc d;
  int P = 0;
  rc = make_chain(&d, ops, param_off, iarg, S, &P);
  if (rc != RISP_OK) return rc;
  RISP_REQUIRE(P == 0 || params, RISP_E_INVALID, "%s: chain needs %d parameters but params is null", who, P);
  RISP_REQUIRE(param_stride == 0 || param_stride >= P, RISP_E_INVALID, "%s: param_stride %d < %d", who, param_stride, P);
  RISP_REQUIRE(workspace, RISP_E_INVALID, "%s: workspace is null", who);
  const size_t need = risp_pipeline_eval_workspace(N, H, W);
  RISP_REQUIRE(workspace_bytes >= need, RISP_E_WORKSPACE, "%s: workspace %zu < %zu", who, workspace_bytes, need);
  cudaStream_t st = as_stream(stream);
  unsigned long long* partial = static_cast<unsigned long long*>(workspace);
  int rows = 0;
  rc = 1;
  if (use_fused()) {
    ChainDesc df = d;
    if (S == 0) { df.S = 1; df.op[0] = RISP_OP_SKIP; df.off[0] = 0; df.iarg[0] = 0; }     // demosaic only
    rc = fused_eval_launch(raw, gt, u8_out, partial, params, param_stride, N, H, W, dm_kind, dm_clip_hi, df, st, &rows);
  }
  if (rc == 1) {
    PipeArgs a{raw, gt, nullptr, nullptr, params, param_stride, H, W, 0, dm_clip_hi, 0, u8_out, partial};
    rc = launch_pipeline<MODE_EVAL>(a, d, N, dm_kind, false, st);
    rows = pipe_geometry(N, H, W).warps_per_image;
  }
  if (rc != RISP_OK) return rc;
  return finalize_sse(partial, sse_out, N, rows, st);
}

// risp_pipeline_eval on frames of stores of codes: image n is raw frame pos[n].x (decoded as the sampler decodes it) against
// GT frame pos[n].y, whose codes are compared as they are.  The same dispatch as risp_pipeline_eval, so the codes and sums
// are that entry point's on the decoded batch under either setting of RISP_FUSED.
extern "C" int risp_pipeline_eval_store(const void* raw_store, int raw_bytes_per_code, int F, const unsigned char* gt_store,
                                        int G, int H, int W, const int* pos, int N, float white_level, int* status,
                                        unsigned char* u8_out, long long* sse_out, int dm_kind, float dm_clip_hi,
                                        const int* ops, const int* param_off, const int* iarg, int S, const float* params,
                                        int param_stride, void* workspace, size_t workspace_bytes, risp_stream_t stream) {
  const char* who = "risp_pipeline_eval_store";
  RISP_REQUIRE(raw_store && gt_store && pos && status && sse_out, RISP_E_INVALID,
               "%s: raw_store, gt_store, pos, status and sse_out must be non-null", who);
  RISP_REQUIRE(raw_bytes_per_code == 1 || raw_bytes_per_code == 2, RISP_E_INVALID, "%s: 1 or 2 bytes per raw code", who);
  RISP_REQUIRE(F > 0 && G > 0 && N > 0 && N <= 65535 && H >= 4 && W >= 4 && white_level > 0.f, RISP_E_INVALID,
               "%s: bad store arguments (F %d, G %d, N %d, %dx%d, white_level %g)", who, F, G, N, H, W, (double)white_level);
  RISP_REQUIRE(H % 2 == 0 && W % 4 == 0, RISP_E_ALIGN, "%s: needs H even and W %% 4 == 0 (got %dx%d)", who, H, W);
  RISP_REQUIRE((long long)F * H * W < (1ll << 40) && (long long)G * 3 * H * W < (1ll << 40), RISP_E_INVALID,
               "%s: stores of %d / %d frames of %dx%d are too large", who, F, G, H, W);
  RISP_REQUIRE(aligned16(raw_store) && aligned16(gt_store) && aligned16(pos), RISP_E_ALIGN,
               "%s: raw_store, gt_store and pos must be 16-byte aligned", who);
  RISP_REQUIRE((reinterpret_cast<uintptr_t>(sse_out) & 7u) == 0, RISP_E_ALIGN, "%s: sse_out must be 8-byte aligned", who);
  RISP_REQUIRE((reinterpret_cast<uintptr_t>(u8_out) & 3u) == 0, RISP_E_ALIGN, "%s: u8_out must be 4-byte aligned", who);
  RISP_REQUIRE(dm_kind == RISP_DM_NEAREST || dm_kind == RISP_DM_BILINEAR || dm_kind == RISP_DM_MALVAR, RISP_E_INVALID,
               "%s: unknown demosaic kind %d", who, dm_kind);
  ChainDesc d;
  int P = 0;
  int rc = make_chain(&d, ops, param_off, iarg, S, &P);
  if (rc != RISP_OK) return rc;
  RISP_REQUIRE(P == 0 || params, RISP_E_INVALID, "%s: chain needs %d parameters but params is null", who, P);
  RISP_REQUIRE(param_stride == 0 || param_stride >= P, RISP_E_INVALID, "%s: param_stride %d < %d", who, param_stride, P);
  RISP_REQUIRE(workspace, RISP_E_INVALID, "%s: workspace is null", who);
  const size_t need = risp_pipeline_eval_workspace(N, H, W);
  RISP_REQUIRE(workspace_bytes >= need, RISP_E_WORKSPACE, "%s: workspace %zu < %zu", who, workspace_bytes, need);
  cudaStream_t st = as_stream(stream);
  unsigned long long* partial = static_cast<unsigned long long*>(workspace);
  int rows = 0;
  rc = 1;
  if (use_fused()) {
    ChainDesc df = d;
    if (S == 0) { df.S = 1; df.op[0] = RISP_OP_SKIP; df.off[0] = 0; df.iarg[0] = 0; }     // demosaic only
    rc = fused_eval_store_launch(raw_store, raw_bytes_per_code, F, gt_store, G, pos, status, white_level, u8_out, partial,
                                 params, param_stride, N, H, W, dm_kind, dm_clip_hi, df, st, &rows);
  }
  if (rc == 1) {
    PipeArgs a{nullptr, nullptr, nullptr, nullptr, params, param_stride, H, W, 0, dm_clip_hi, 0, u8_out, partial,
               static_cast<const unsigned char*>(raw_store), gt_store, reinterpret_cast<const int4*>(pos), status,
               white_level, F, G};
    rc = raw_bytes_per_code == 2 ? launch_pipeline<MODE_EVAL_S16>(a, d, N, dm_kind, false, st)
                                 : launch_pipeline<MODE_EVAL_U8>(a, d, N, dm_kind, false, st);
    rows = pipe_geometry(N, H, W).warps_per_image;
  }
  if (rc != RISP_OK) return rc;
  return finalize_sse(partial, sse_out, N, rows, st);
}

extern "C" size_t risp_pipeline_step_workspace(int N, int H, int W, int P) {
  (void)P;
  if (N <= 0 || H <= 0 || W <= 0) return 0;
  PipeGeom g = pipe_geometry(N, H, W);
  size_t rows = (size_t)g.warps_per_image;
  const size_t frows = (size_t)fused_partial_rows_per_frame(N);
  if (frows > rows) rows = frows;
  return (size_t)N * rows * RISP_NSLOT * sizeof(float) + finalize_rows_workspace(N, RISP_NSLOT);
}

// the inputs of the store steps: N crops of H x W (the step's geometry) out of frame stores of FH x FW frames
struct StepStore {
  const void* raw;
  int bpc, F;
  const unsigned char* gt;
  int G, FH, FW;
  const int* pos;
  float white_level;
  int* status;
};

static int check_store_step(const char* who, const StepStore& s, float* loss_out, int N, int h, int w) {
  RISP_REQUIRE(s.raw && s.gt && s.pos && s.status && loss_out, RISP_E_INVALID,
               "%s: raw_store, gt_store, pos, status and loss_out must be non-null", who);
  RISP_REQUIRE(s.bpc == 1 || s.bpc == 2, RISP_E_INVALID, "%s: 1 or 2 bytes per raw code", who);
  RISP_REQUIRE(s.F > 0 && s.G > 0 && N > 0 && N <= 65535 && h >= 4 && w >= 4 && h <= s.FH && w <= s.FW && s.white_level > 0.f,
               RISP_E_INVALID, "%s: bad store arguments (F %d, G %d, N %d, %dx%d crops of %dx%d frames, white_level %g)", who, s.F,
               s.G, N, h, w, s.FH, s.FW, (double)s.white_level);
  RISP_REQUIRE((long long)s.F * s.FH * s.FW < (1ll << 40) && (long long)s.G * 3 * s.FH * s.FW < (1ll << 40), RISP_E_INVALID,
               "%s: stores of %d / %d frames of %dx%d are too large", who, s.F, s.G, s.FH, s.FW);
  // the packed kernels read the stores through tensor maps (16-byte aligned base, rows of a 16-byte multiple); both kernels
  // march 4-column lanes down row pairs
  RISP_REQUIRE(s.FW % 16 == 0 && w % 4 == 0 && h % 2 == 0 && aligned16(s.raw) && aligned16(s.gt) && aligned16(s.pos),
               RISP_E_UNSUPPORTED, "%s: needs 16-byte aligned stores and pos, frames with W %% 16 == 0 and crops with w %% 4 == 0 "
               "and h even (got %dx%d crops of %dx%d frames)", who, h, w, s.FH, s.FW);
  return RISP_OK;
}

// gt_is_dy: gt holds dL/dy (risp_pipeline_bwd).  store (nullable): the store steps, whose raw and gt come from the stores
static int pipeline_step_impl(const char* who, bool gt_is_dy, bool l1, const float* raw, const float* gt, float* y_out,
                              float* loss_out, float* dparams, int N, int H, int W, int dm_kind, float dm_clip_hi,
                              const int* ops, const int* param_off, const int* iarg, int S, const float* params,
                              int param_stride, int P, void* workspace, size_t workspace_bytes, risp_stream_t stream,
                              const StepStore* store = nullptr) {
  int rc = store ? check_store_step(who, *store, loss_out, N, H, W) : check_frame(who, raw, N, H, W);
  if (rc != RISP_OK) return rc;
  RISP_REQUIRE(store || (gt && aligned16(gt) && (gt_is_dy || loss_out)), RISP_E_ALIGN, "%s: gt/dy/loss_out null or unaligned", who);
  RISP_REQUIRE(!y_out || aligned16(y_out), RISP_E_ALIGN, "%s: y_out must be 16-byte aligned", who);
  ChainDesc d;
  int Pn = 0;
  rc = make_chain(&d, ops, param_off, iarg, S, &Pn);
  if (rc != RISP_OK) return rc;
  bool big = false;
  for (int s = 0; s < S; ++s) {
    RISP_REQUIRE(op_has_bwd(ops[s]), RISP_E_UNSUPPORTED, "%s: op %d is forward-only", who, ops[s]);
    big = big || op_is_big(ops[s]);
  }
  RISP_REQUIRE(Pn <= P, RISP_E_INVALID, "%s: chain needs %d parameters, P=%d", who, Pn, P);
  RISP_REQUIRE(Pn == 0 || (params && dparams), RISP_E_INVALID, "%s: null params/dparams", who);
  RISP_REQUIRE(param_stride == 0 || param_stride >= P, RISP_E_INVALID, "%s: param_stride %d < P %d", who, param_stride, P);
  size_t need = risp_pipeline_step_workspace(N, H, W, P);
  RISP_REQUIRE(workspace && workspace_bytes >= need, RISP_E_WORKSPACE, "%s: workspace %zu < %zu", who, workspace_bytes, need);
  cudaStream_t st = as_stream(stream);
  PipeGeom g = pipe_geometry(N, H, W);
  float* partial = static_cast<float*>(workspace);
  void* fin_ws = reinterpret_cast<char*>(workspace) + (need - finalize_rows_workspace(N, RISP_NSLOT));
  int frows = 0;
  RISP_REQUIRE(!l1 || (P > 0 && use_fused() && fused_handles(d, N, param_stride, H, W)), RISP_E_UNSUPPORTED,
               "%s: the fused L1 step exists for the pre-instantiated chain signatures only (run the unfused path)", who);
  if (P > 0 && use_fused())
    rc = store ? fused_step_store_launch(l1, store->raw, store->bpc, store->F, store->gt, store->G, store->FH, store->FW,
                                         store->pos, store->status, store->white_level, partial, params, param_stride, N, H,
                                         W, dm_kind, dm_clip_hi, d, st, &frows)
               : fused_launch(gt_is_dy ? 2 : (l1 ? 3 : 1), raw, gt, y_out, partial, params, param_stride, N, H, W, dm_kind,
                              dm_clip_hi, d, st, &frows);
  else
    rc = 1;
  if (rc == 1 && store) {
    PipeArgs a{nullptr, nullptr, nullptr, partial, params, param_stride, H, W, 0, dm_clip_hi, 0, nullptr, nullptr,
               static_cast<const unsigned char*>(store->raw), store->gt, reinterpret_cast<const int4*>(store->pos),
               store->status, store->white_level, store->F, store->G};
    rc = store->bpc == 2 ? launch_pipeline<MODE_STEP_S16>(a, d, N, dm_kind, big, st, int2{store->FH, store->FW})
                         : launch_pipeline<MODE_STEP_U8>(a, d, N, dm_kind, big, st, int2{store->FH, store->FW});
  } else if (rc == 1) {
    PipeArgs a{raw, gt, y_out, partial, params, param_stride, H, W, 0, dm_clip_hi, gt_is_dy ? 1 : 0};
    rc = launch_pipeline<MODE_STEP>(a, d, N, dm_kind, big, st);
  } else if (rc == RISP_OK) {
    g.warps_per_image = frows;
  }
  if (rc != RISP_OK) return rc;
  const double numel = (double)N * 3.0 * H * W;
  const bool shared_row = (param_stride == 0);
  if (N > 64 || P == 0) {
    // rare shapes: the one-warp-per-entry finaliser
    if (!gt_is_dy) {
      const short loss_dst = 0, loss_slot = RISP_SLOT_LOSS;
      rc = finalize_partials(partial, loss_out, N, g.warps_per_image, RISP_NSLOT, 1, &loss_dst, &loss_slot, 1,
                             (float)(1.0 / numel), true, st);
      if (rc != RISP_OK) return rc;
    }
    if (P == 0) return RISP_OK;
    if (cudaMemsetAsync(dparams, 0, sizeof(float) * (size_t)P * (shared_row ? 1 : N), st) != cudaSuccess) {
      set_error("%s: memset failed", who);
      return RISP_E_CUDA;
    }
    SlotList m;
    chain_slot_list(d, &m);
    return finalize_partials(partial, dparams, N, g.warps_per_image, RISP_NSLOT, P, m.dst, m.slot, m.n,
                             gt_is_dy ? 1.f : (float)((l1 ? 1.0 : 2.0) / numel), shared_row, st);
  }
  // loss and every parameter gradient in one launch (the loss rides along when all frames share one parameter row)
  const bool loss_inline = !gt_is_dy && shared_row;
  if (!gt_is_dy && !loss_inline) {
    const short loss_dst = 0, loss_slot = RISP_SLOT_LOSS;
    rc = finalize_partials(partial, loss_out, N, g.warps_per_image, RISP_NSLOT, 1, &loss_dst, &loss_slot, 1,
                           (float)(1.0 / numel), true, st);
    if (rc != RISP_OK) return rc;
  }
  SlotList m;
  chain_slot_list(d, &m);
  return finalize_rows(partial, fin_ws, dparams, loss_inline ? loss_out : nullptr, N, g.warps_per_image, RISP_NSLOT, P, m.dst,
                       m.slot, m.n, gt_is_dy ? 1.f : (float)((l1 ? 1.0 : 2.0) / numel), (float)(1.0 / numel), RISP_SLOT_LOSS, shared_row, st);
}

extern "C" int risp_pipeline_mse_step(const float* raw, const float* gt, float* y_out, float* loss_out, float* dparams,
                                      int N, int H, int W, int dm_kind, float dm_clip_hi, const int* ops,
                                      const int* param_off, const int* iarg, int S, const float* params,
                                      int param_stride, int P, void* workspace, size_t workspace_bytes,
                                      risp_stream_t stream) {
  return pipeline_step_impl("risp_pipeline_mse_step", false, false, raw, gt, y_out, loss_out, dparams, N, H, W, dm_kind,
                            dm_clip_hi, ops, param_off, iarg, S, params, param_stride, P, workspace, workspace_bytes,
                            stream);
}

extern "C" int risp_pipeline_bwd(const float* raw, const float* dy, float* dparams, int N, int H, int W, int dm_kind,
                                 float dm_clip_hi, const int* ops, const int* param_off, const int* iarg, int S,
                                 const float* params, int param_stride, int P, void* workspace, size_t workspace_bytes,
                                 risp_stream_t stream) {
  return pipeline_step_impl("risp_pipeline_bwd", true, false, raw, dy, nullptr, nullptr, dparams, N, H, W, dm_kind, dm_clip_hi,
                            ops, param_off, iarg, S, params, param_stride, P, workspace, workspace_bytes, stream);
}

extern "C" int risp_pipeline_l1_step(const float* raw, const float* gt, float* y_out, float* loss_out, float* dparams,
                                     int N, int H, int W, int dm_kind, float dm_clip_hi, const int* ops,
                                     const int* param_off, const int* iarg, int S, const float* params,
                                     int param_stride, int P, void* workspace, size_t workspace_bytes,
                                     risp_stream_t stream) {
  return pipeline_step_impl("risp_pipeline_l1_step", false, true, raw, gt, y_out, loss_out, dparams, N, H, W, dm_kind,
                            dm_clip_hi, ops, param_off, iarg, S, params, param_stride, P, workspace, workspace_bytes,
                            stream);
}

// The MSE / L1 step on N crops of h x w out of frame stores (see the header): the dispatch and the finaliser of
// risp_pipeline_mse_step / risp_pipeline_l1_step, with raw and gt read as codes.
extern "C" int risp_pipeline_mse_step_store(const void* raw_store, int raw_bytes_per_code, int F, const unsigned char* gt_store,
                                            int G, int H, int W, const int* pos, int N, float white_level, int* status, int h,
                                            int w, float* loss_out, float* dparams, int dm_kind, float dm_clip_hi,
                                            const int* ops, const int* param_off, const int* iarg, int S, const float* params,
                                            int param_stride, int P, void* workspace, size_t workspace_bytes,
                                            risp_stream_t stream) {
  const StepStore s{raw_store, raw_bytes_per_code, F, gt_store, G, H, W, pos, white_level, status};
  return pipeline_step_impl("risp_pipeline_mse_step_store", false, false, nullptr, nullptr, nullptr, loss_out, dparams, N, h,
                            w, dm_kind, dm_clip_hi, ops, param_off, iarg, S, params, param_stride, P, workspace,
                            workspace_bytes, stream, &s);
}

extern "C" int risp_pipeline_l1_step_store(const void* raw_store, int raw_bytes_per_code, int F, const unsigned char* gt_store,
                                           int G, int H, int W, const int* pos, int N, float white_level, int* status, int h,
                                           int w, float* loss_out, float* dparams, int dm_kind, float dm_clip_hi,
                                           const int* ops, const int* param_off, const int* iarg, int S, const float* params,
                                           int param_stride, int P, void* workspace, size_t workspace_bytes,
                                           risp_stream_t stream) {
  const StepStore s{raw_store, raw_bytes_per_code, F, gt_store, G, H, W, pos, white_level, status};
  return pipeline_step_impl("risp_pipeline_l1_step_store", false, true, nullptr, nullptr, nullptr, loss_out, dparams, N, h,
                            w, dm_kind, dm_clip_hi, ops, param_off, iarg, S, params, param_stride, P, workspace,
                            workspace_bytes, stream, &s);
}
