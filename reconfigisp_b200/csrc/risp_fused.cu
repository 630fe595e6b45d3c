// Fused raw -> BGR pipeline on packed fp32 with constant-bank parameters: the kernels behind
// risp_pipeline_fwd / risp_pipeline_mse_step / risp_pipeline_bwd for the pre-instantiated chain signatures.
//
// Reference: isp_universal.py:210-232 / origin_universal.py:143-161 (one full-image pass per stage) and the
// proxy-tuning step isp_model.py:128-142 (forward, MSELoss, backward).  Here: one pass, 16 B/px.
//
// Shape of the kernel (see DESIGN.md §4):
//   * persistent CTAs (one wave: SMs x resident CTAs), each walking a static list of (row chunk, 128-column strip)
//     items of ONE frame -> accumulators live in registers for the whole kernel, one reduction per warp, and the
//     summation order is fixed (bit-reproducible gradients);
//   * a warp owns a 128-column strip and marches down the rows with the demosaic window in registers (horizontal halo
//     by shuffle), two rows per loop trip so the CFA row parity is a compile-time constant;
//   * the chain runs on pixel PAIRS with FFMA2/FMUL2/FADD2, coefficients from uniform registers; the FMA-heavy sites of the
//     backward-carrying kernels use scalar FFMA and accumulate both pixels of a pair into one sum (risp_fused.cuh).
#include "risp_fused.cuh"

#include <cuda.h>
#include <array>
#include <map>
#include <mutex>
#include <stdlib.h>

namespace risp {
namespace fused {

__constant__ float g_cpar[kCSlots][kCRows][kCRowFloats];

// STEP: MSE loss; STEP_L1: L1 loss (isp_model.py:44-49); EVAL: inference arithmetic + squared 8-bit code differences to the GT
enum { MODE_FWD = 0, MODE_STEP = 1, MODE_BWD = 2, MODE_STEP_L1 = 3, MODE_EVAL = 4 };
// A CTA is one warp (32 threads), so everything but the lane index is CTA-uniform (uniform datapath, no R2UR).  The warp
// owns a strip of kStrip columns.
constexpr int kStrip = 128;

struct FusedArgs {
  const float* raw;     // (N,1,H,W)
  const float* gt;      // (N,3,H,W): target (STEP) or dL/dy (BWD)
  float* y;             // (N,3,H,W), nullable except in FWD
  float* partial;       // [N][cpf][RISP_NSLOT]
  const float* params;  // raw parameter rows (epilogue of the folded gain)
  int pstride;
  int H, W;
  int rows_per_chunk, chunks, strip_blocks, cpf;   // cpf = CTAs per frame
  float clip_hi;
  int slot;
  unsigned char* u8;    // EVAL: (N,H,W,3) 8-bit codes of y, nullable
  unsigned long long* sse;   // EVAL: [N][cpf] sums of squared code differences
  // narrow items (backward-carrying kernels): the last strip of a frame, nw = 32 or 64 columns wide (0: none), marched by
  // 128/nw lane groups on as many row pairs at once; the strip_blocks full strips lie to its left
  int nw, nrows_per_chunk, nchunks;
};

// ---- preparation: derived constants of every parameter row ---------------------------------------------------------
__global__ void fused_prep_kernel(const float* __restrict__ params, int pstride, ChainDesc d, float* __restrict__ cslot) {
  if (threadIdx.x != 0) return;
  const float* p = params + (long long)blockIdx.x * pstride;
  float* c = cslot + (long long)blockIdx.x * kCRowFloats;
  const EffChain e = eff_from_ops(d.op, d.iarg, d.S);
  for (int k = 0; k < e.n; ++k) {
    float* o = c + e.coff[k];
    const float* q = p + d.off[e.src[k]];
    switch (e.op[k]) {
      case RISP_OP_GAMMA: o[0] = q[0]; break;     // gm (the block stays 2 floats wide: fop_csize)
      case RISP_OP_GAIN: o[0] = q[0]; o[1] = q[1]; o[2] = q[2]; o[3] = 0.f; break;
      case RISP_OP_POLY10:
      case FOP_POLYG: {
        float gm[10];
        if (e.op[k] == FOP_POLYG) {
          const float* g = p + d.off[e.src[k] - 1];
          const float gb = g[0], gg = g[1], gr = g[2];
          gm[0] = gb * gb; gm[1] = gg * gg; gm[2] = gr * gr; gm[3] = gb * gg; gm[4] = gb * gr; gm[5] = gg * gr;
          gm[6] = gb; gm[7] = gg; gm[8] = gr; gm[9] = 1.f;
        } else {
          for (int i = 0; i < 10; ++i) gm[i] = 1.f;
        }
        for (int cc = 0; cc < 3; ++cc)
          for (int i = 0; i < 10; ++i) o[cc * 10 + i] = q[cc * 10 + i] * gm[i];
        for (int cc = 0; cc < 3; ++cc)
          for (int i = 0; i < 3; ++i) o[30 + cc * 3 + i] = 2.f * o[cc * 10 + i];
        o[39] = 0.f;
      } break;
      case RISP_OP_GTM: {
        // knots y_0 = 0, y_k = q[k-1], y_4 = 1;  s_k = (y_{k+1} - y_k) * 4
        const float y1 = q[0], y2 = q[1], y3 = q[2];
        const float s0 = (y1 - 0.f) * 4.f, s1 = (y2 - y1) * 4.f, s2 = (y3 - y2) * 4.f, s3 = (1.f - y3) * 4.f;
        o[0] = s0; o[1] = s1 - s0; o[2] = s2 - s1; o[3] = s3 - s2;
        const bool in_range = (y1 >= 0.f && y1 <= 1.f) && (y2 >= 0.f && y2 <= 1.f) && (y3 >= 0.f && y3 <= 1.f);
        o[5] = in_range ? 0.f : 1.f;
        o[6] = 0.f; o[7] = 0.f;
        // table form: out = s_k x + a_k on segment k, a_k = y_k - x_k s_k
        o[8] = 0.f; o[9] = y1 - 0.25f * s1; o[10] = y2 - 0.5f * s2; o[11] = y3 - 0.75f * s3;
        o[12] = s0; o[13] = s1; o[14] = s2; o[15] = s3;
      } break;
      default: break;
    }
  }
}

// ---- per-warp row ring in shared memory, filled by bulk async copies (TMA, 1-D) ----------------------------------------
// Each warp owns a ring of D row records: [raw strip with a 4-column pad on both sides | GT B | GT G | GT R].  One elected
// lane issues the copies of a whole row (cp.async.bulk ... mbarrier::complete_tx) D - 2*HL - 1 rows ahead of the row being
// computed, so 3-5 rows (2 KB each) per warp are in flight without a single register: enough bytes in flight for HBM
// (Little's law wants ~40 KB per SM) at 8 warps per SM.  Lanes read their window with LDS: 128-bit own columns plus the two
// halo columns, whose offsets fold the reflect-101 frame border (column -1 -> 1, column W -> W-2) -- no shuffles, no
// register window, no prefetch registers.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t mbar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred P1;\n\tmbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\tselp.u32 %0, 1, 0, P1;\n\t}\n"
               : "=r"(ok) : "r"(mbar), "r"(parity) : "memory");
  return ok != 0;
}
// bounded wait: a protocol bug must trap (and fail the launch) instead of hanging the device
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
  for (uint32_t spin = 0; !mbar_try(mbar, parity); ++spin)
    if (spin > (1u << 26)) __trap();
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P1;\n\telect.sync _|P1, 0xffffffff;\n\tselp.u32 %0, 1, 0, P1;\n\t}\n" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ float4 lds4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float lds1(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts4(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// tensor-map TMA: one instruction moves a (columns x rows x planes) box; out-of-bounds elements arrive as zeros
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, int x, int y, int z, uint32_t mbar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
               ::"r"(dst), "l"(tm), "r"(x), "r"(y), "r"(z), "r"(mbar) : "memory");
}

constexpr int kPad = 4;            // floats of halo pad on each side of the raw strip
template <int MODE>
struct RingCfg {
  static constexpr int D = 4;                                            // records per warp (power of 2)
  // rows per record = rows per TMA box.  A TMA instruction costs the SM's copy engine ~150 cycles whatever its size
  // (measured: 1 KB boxes deliver 1.9 TB/s chip-wide), so the inference kernel, which has nothing but the copies to wait
  // for, uses 4-row boxes; the backward-carrying kernels are issue-bound and keep the smaller ring
  static constexpr int RR = (MODE == MODE_FWD) ? 4 : 2;
  static constexpr int RAWROWB = (kStrip + 2 * kPad) * 4;                // 544 B: one raw row of the box
  static constexpr int RAWB = (RR * RAWROWB + 127) / 128 * 128;          // RR rows, padded to a 128-B multiple
  static constexpr int GTPLANEB = RR * kStrip * 4;
  static constexpr int GTB = (MODE == MODE_FWD) ? 0 : 3 * GTPLANEB;  // [plane][row][128]
  static constexpr int RECB = RAWB + GTB;                                // multiple of 128
  static constexpr int WARPB = D * RECB;
  static constexpr int TBLOFF = (WARPB + D * 8 + 63) / 64 * 64;       // tone-curve tables (one per stage slot)
  static constexpr int SMEM = TBLOFF + ((MODE == MODE_FWD) ? 0 : RISP_MAX_STAGES * kGtmTableBytes) + 128;  // records + mbarriers + tables + alignment slack
};

__device__ __forceinline__ int reflect101(int r, int H) { return r < 0 ? -r : (r >= H ? 2 * H - 2 - r : r); }

// ---- demosaic of the lane's 4 pixels; row parity is a template parameter (no selects) ---------------------------------
// w[RO + j][i]: raw row r-HL+j, column c0-HL+i.  Sites: (even,even)=R (even,odd)=G1 (odd,even)=G2 (odd,odd)=B.
template <int DM, int HL, int RO, bool ODD, int WRT, bool PK>
__device__ __forceinline__ void demosaic4(const float (&w)[WRT][4 + 2 * HL], float clip_hi, P2& lo, P2& hi) {
  float B[4], G[4], R[4];
  constexpr int M = RO + HL;     // window row of the pixel's own raw row
  if constexpr (DM == RISP_DM_BILINEAR && PK) {   // PK: the chain starts with packed arithmetic on the pairs (gain / polynomial)
    // The 0.5 / 0.25 / 1 weights are applied by ONE packed multiply per output pair (constant pair from the uniform
    // datapath): a pair like (raw, 0.5*sum) then leaves the demosaic as the result of an arithmetic instruction.  A pair
    // that is a plain pack of a raw window value and a computed value is re-packed by ptxas at every use (it
    // rematerialises the two moves instead of keeping the 64-bit register live: 12 MOV per pixel in the step kernel).
    // Same values bit for bit: x*1 is exact, the other products are the ones the scalar form computes.
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int x = HL + k;
      const bool xo = (k & 1);
      const float c = w[M][x];
      if (ODD != xo) {   // green site
        const float hor = w[M][x - 1] + w[M][x + 1], ver = w[M - 1][x] + w[M + 1][x];
        G[k] = c;
        if (!ODD) { R[k] = hor; B[k] = ver; } else { R[k] = ver; B[k] = hor; }
      } else {
        const float cross = (w[M - 1][x] + w[M + 1][x]) + (w[M][x - 1] + w[M][x + 1]);
        const float diag = (w[M - 1][x - 1] + w[M - 1][x + 1]) + (w[M + 1][x - 1] + w[M + 1][x + 1]);
        G[k] = cross;
        if (!ODD) { R[k] = c; B[k] = diag; } else { R[k] = diag; B[k] = c; }
      }
    }
    // weights of (even column, odd column): even rows R G / odd rows G B
    const float2 sb = ODD ? make_float2(0.5f, 1.f) : make_float2(0.25f, 0.5f);
    const float2 sg = ODD ? make_float2(1.f, 0.25f) : make_float2(0.25f, 1.f);
    const float2 sr = ODD ? make_float2(0.5f, 0.25f) : make_float2(1.f, 0.5f);
    lo.b = __fmul2_rn(make_float2(B[0], B[1]), sb); lo.g = __fmul2_rn(make_float2(G[0], G[1]), sg); lo.r = __fmul2_rn(make_float2(R[0], R[1]), sr);
    hi.b = __fmul2_rn(make_float2(B[2], B[3]), sb); hi.g = __fmul2_rn(make_float2(G[2], G[3]), sg); hi.r = __fmul2_rn(make_float2(R[2], R[3]), sr);
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int x = HL + k;
      const bool xo = (k & 1);
      const float c = w[M][x];
      if constexpr (DM == RISP_DM_NEAREST) {
        if (!ODD) { R[k] = xo ? w[M][x - 1] : c; G[k] = xo ? c : w[M][x + 1]; B[k] = xo ? w[M + 1][x] : w[M + 1][x + 1]; }
        else      { R[k] = xo ? w[M - 1][x - 1] : w[M - 1][x]; G[k] = xo ? w[M][x - 1] : c; B[k] = xo ? c : w[M][x + 1]; }
      } else if constexpr (DM == RISP_DM_BILINEAR) {
        const bool at_g = (ODD != xo);
        if (at_g) {
          const float hor = 0.5f * (w[M][x - 1] + w[M][x + 1]);
          const float ver = 0.5f * (w[M - 1][x] + w[M + 1][x]);
          G[k] = c;
          if (!ODD) { R[k] = hor; B[k] = ver; } else { R[k] = ver; B[k] = hor; }
        } else {
          const float cross = (w[M - 1][x] + w[M + 1][x]) + (w[M][x - 1] + w[M][x + 1]);
          const float diag = (w[M - 1][x - 1] + w[M - 1][x + 1]) + (w[M + 1][x - 1] + w[M + 1][x + 1]);
          G[k] = 0.25f * cross;
          if (!ODD) { R[k] = c; B[k] = 0.25f * diag; } else { R[k] = 0.25f * diag; B[k] = c; }
        }
      } else {  // Malvar-He-Cutler 5x5
        const float n1 = w[M - 1][x], s1 = w[M + 1][x], e1 = w[M][x + 1], w1 = w[M][x - 1];
        const float n2 = w[M - 2][x], s2 = w[M + 2][x], e2 = w[M][x + 2], w2 = w[M][x - 2];
        const float dg = (w[M - 1][x - 1] + w[M - 1][x + 1]) + (w[M + 1][x - 1] + w[M + 1][x + 1]);
        float rr, gg, bb;
        const bool at_g = (ODD != xo);
        if (at_g) {
          const float f_row = 0.125f * (5.f * c + 4.f * (e1 + w1) - dg - (e2 + w2) + 0.5f * (n2 + s2));
          const float f_col = 0.125f * (5.f * c + 4.f * (n1 + s1) - dg - (n2 + s2) + 0.5f * (e2 + w2));
          gg = c;
          if (!ODD) { rr = f_row; bb = f_col; } else { rr = f_col; bb = f_row; }
        } else {
          const float f_g = 0.125f * (4.f * c + 2.f * ((n1 + s1) + (e1 + w1)) - ((n2 + s2) + (e2 + w2)));
          const float f_dg = 0.125f * (6.f * c + 2.f * dg - 1.5f * ((n2 + s2) + (e2 + w2)));
          gg = f_g;
          if (!ODD) { rr = c; bb = f_dg; } else { rr = f_dg; bb = c; }
        }
        R[k] = fminf(fmaxf(rr, 0.f), clip_hi); G[k] = fminf(fmaxf(gg, 0.f), clip_hi); B[k] = fminf(fmaxf(bb, 0.f), clip_hi);
      }
    }
    lo.b = make_float2(B[0], B[1]); lo.g = make_float2(G[0], G[1]); lo.r = make_float2(R[0], R[1]);
    hi.b = make_float2(B[2], B[3]); hi.g = make_float2(G[2], G[3]); hi.r = make_float2(R[2], R[3]);
  }
}

// ---- the chain on one pixel pair: forward, loss, backward (compile-time recursion over the effective stages) ----------
template <unsigned SIG>
__host__ __device__ constexpr bool per_channel_from(int k) {     // stages k.. never mix channels
  constexpr EffChain E = Eff<SIG>::e;
  for (int i = k; i < E.n; ++i)
    if (E.op[i] == RISP_OP_POLY10 || E.op[i] == FOP_POLYG) return false;
  return true;
}

// stages K.. on ONE channel C of the pair (gamma / gain / tone curve): forward, loss term, backward.  Keeping a channel's
// whole tail together makes its saved state transient (a few registers) instead of live across all three channels.
// NOMASK: stage K is a gamma whose clamp mask the caller merges with its own (see the polynomial's channel-major form)
template <unsigned SIG, int K, int MODE, int C, bool NOMASK = false>
struct Tail {
  static constexpr EffChain E = Eff<SIG>::e;
  static constexpr bool SC = !per_channel_from<SIG>(0);    // scalar fp32 sites: chains with the polynomial (risp_fused.cuh)
  static __device__ __forceinline__ float2 go(float2 x, float2 tgt, const float* __restrict__ cp, float2* acc, float2& loss,
                                              float2& yout, bool slow, float lane_w, uint32_t tbl) {
    if constexpr (K == E.n) {
      yout = x;
      if constexpr (MODE == MODE_BWD) return tgt;
      // d loss / d y up to the constant 2/numel (applied by the finaliser).  lane_w = 1 for lanes inside the frame (1*x - t is
      // exactly x - t) and 0 for the lanes of the last strip that hang over the right edge (their t is 0): no divergent branch
      const float2 dd = SC ? make_float2(fmaf(lane_w, x.x, -tgt.x), fmaf(lane_w, x.y, -tgt.y))
                           : __ffma2_rn(make_float2(lane_w, lane_w), x, make_float2(-tgt.x, -tgt.y));
      if constexpr (MODE == MODE_STEP_L1) {      // nn.L1Loss: sum |y - t| ; gradient sign(y - t) (0 at equality), 1/numel later
        acc_add<SC>(loss, make_float2(fabsf(dd.x), fabsf(dd.y)));
        return make_float2((dd.x > 0.f ? 1.f : 0.f) - (dd.x < 0.f ? 1.f : 0.f), (dd.y > 0.f ? 1.f : 0.f) - (dd.y < 0.f ? 1.f : 0.f));
      }
      acc_fma<SC>(loss, dd, dd);
      return dd;
    } else {
      constexpr int OP = E.op[K];
      constexpr bool IN01 = (K > 0) && fop_out01(E.op[K > 0 ? K - 1 : 0]);
      constexpr bool NEED_DX = (K > 0);
      const float* c = cp + E.coff[K];
      float2* a = acc + E.aoff[K];
      if constexpr (OP == RISP_OP_SKIP) {
        return Tail<SIG, K + 1, MODE, C>::go(x, tgt, cp, acc, loss, yout, slow, lane_w, tbl);
      } else if constexpr (OP == RISP_OP_GAMMA) {
        float2 l2;
        const float gm = c[0];
        const float2 y = gamma_fwd2<IN01>(x, gm, l2);
        const float2 d = Tail<SIG, K + 1, MODE, C>::go(y, tgt, cp, acc, loss, yout, slow, lane_w, tbl);
        return gamma_bwd2<IN01, NEED_DX, true, NOMASK, SC>(x, y, l2, d, gm, a[0]);
      } else if constexpr (OP == RISP_OP_GAIN) {
        const float2 y = mul2s(x, c[C]);
        const float2 d = Tail<SIG, K + 1, MODE, C>::go(y, tgt, cp, acc, loss, yout, slow, lane_w, tbl);
        a[C] = fma2(d, x, a[C]);
        return NEED_DX ? mul2s(d, c[C]) : zero2();
      } else {
        static_assert(OP == RISP_OP_GTM && IN01, "packed path: unsupported per-channel op");
        float2 slope, m = zero2();
        const float2 y = gtm_fwd2<true>(x, c, slope, slow, m, tbl + K * kGtmTableBytes);
        float2 d = Tail<SIG, K + 1, MODE, C>::go(y, tgt, cp, acc, loss, yout, slow, lane_w, tbl);
        if (slow) d = mul2(d, m);
        return gtm_bwd2<NEED_DX, SC>(x, slope, d, a);
      }
    }
  }
};

template <unsigned SIG, int K, int MODE>
struct Run {
  static constexpr EffChain E = Eff<SIG>::e;
  static __device__ __forceinline__ P2 go(const P2& x, const P2& tgt, const float* __restrict__ cp, float2* acc, float2& loss,
                                          P2& yout, bool slow, float lane_w, uint32_t tbl) {
    if constexpr (per_channel_from<SIG>(K)) {
      P2 d;
      d.b = Tail<SIG, K, MODE, 0>::go(x.b, tgt.b, cp, acc, loss, yout.b, slow, lane_w, tbl);
      d.g = Tail<SIG, K, MODE, 1>::go(x.g, tgt.g, cp, acc, loss, yout.g, slow, lane_w, tbl);
      d.r = Tail<SIG, K, MODE, 2>::go(x.r, tgt.r, cp, acc, loss, yout.r, slow, lane_w, tbl);
      return d;
    } else {
      constexpr int OP = E.op[K];
      constexpr bool IN01 = (K > 0) && fop_out01(E.op[K > 0 ? K - 1 : 0]);
      constexpr bool NEED_DX = (K > 0);
      const float* c = cp + E.coff[K];
      float2* a = acc + E.aoff[K];
      if constexpr (OP == RISP_OP_GAMMA) {
        GammaSaved sv;
        const float gm = c[0];
        const P2 y = gamma_fwd<IN01>(x, gm, sv);
        const P2 d = Run<SIG, K + 1, MODE>::go(y, tgt, cp, acc, loss, yout, slow, lane_w, tbl);
        return gamma_bwd<IN01, NEED_DX, true>(sv, d, gm, a[0]);
      } else if constexpr ((OP == RISP_OP_POLY10 || OP == FOP_POLYG) && !NEED_DX && per_channel_from<SIG>(K + 1)) {
        // channel-major: the monomials are the only cross-channel state; each output channel then runs its polynomial
        // row, its whole tail, the loss and the way back, and accumulates e_c * phi straight away
        float2 phi[9];
        phi[0] = mul2(x.b, x.b); phi[1] = mul2(x.g, x.g); phi[2] = mul2(x.r, x.r);
        phi[3] = mul2(x.b, x.g); phi[4] = mul2(x.b, x.r); phi[5] = mul2(x.g, x.r);
        phi[6] = x.b; phi[7] = x.g; phi[8] = x.r;
        auto channel = [&](auto ctag, float2 tg, float2& yo) {
          constexpr int C = decltype(ctag)::value;
          float2 u = make_float2(fmaf(c[C * 10], phi[0].x, c[C * 10 + 9]), fmaf(c[C * 10], phi[0].y, c[C * 10 + 9]));
#pragma unroll
          for (int i = 1; i < 9; ++i) u = make_float2(fmaf(c[C * 10 + i], phi[i].x, u.x), fmaf(c[C * 10 + i], phi[i].y, u.y));
          const float2 y = sat2(u);
          // a gamma directly behind the polynomial masks its gradient with [y >= eps]; together with the clamp mask
          // [0 <= u <= 1] that is [eps <= u <= 1] <=> max(sat(u), eps) == u: one compare on the value gamma computes anyway
          constexpr bool GNEXT = (K + 1 < E.n) && (E.op[K + 1 < E.n ? K + 1 : K] == RISP_OP_GAMMA);
          const float2 d = Tail<SIG, K + 1, MODE, C, GNEXT>::go(y, tg, cp, acc, loss, yo, slow, lane_w, tbl);
          float2 e;
          if constexpr (GNEXT) {
            const float2 xc = make_float2(fmaxf(y.x, RISP_GAMMA_EPS), fmaxf(y.y, RISP_GAMMA_EPS));
            e = sel2(xc.x == u.x, xc.y == u.y, d);
          } else {
            e = sel2(u.x == y.x, u.y == y.y, d);     // clamp mask, inclusive: u in [0,1] <=> sat(u) == u
          }
#pragma unroll
          for (int i = 0; i < 9; ++i) acc_fma<true>(a[C * 10 + i], e, phi[i]);
          acc_add<true>(a[C * 10 + 9], e);
        };
        channel(std::integral_constant<int, 0>{}, tgt.b, yout.b);
        channel(std::integral_constant<int, 1>{}, tgt.g, yout.g);
        channel(std::integral_constant<int, 2>{}, tgt.r, yout.r);
        P2 z; z.b = zero2(); z.g = zero2(); z.r = zero2();
        return z;
      } else {
        // a gain or tone curve in front of a cross-channel stage: no instantiated signature has one (Tail runs them)
        static_assert(OP == RISP_OP_POLY10 || OP == FOP_POLYG, "packed path: unsupported effective op");
        PolySaved sv;
        const P2 y = poly_fwd(x, c, sv);
        const P2 d = Run<SIG, K + 1, MODE>::go(y, tgt, cp, acc, loss, yout, slow, lane_w, tbl);
        return poly_bwd<NEED_DX>(sv, d, c, a);
      }
    }
  }
};

template <unsigned SIG, int K>
struct Fwd {
  static constexpr EffChain E = Eff<SIG>::e;
  static __device__ __forceinline__ P2 go(const P2& x, const float* __restrict__ cp, bool slow) {
    if constexpr (K == E.n) {
      return x;
    } else {
      constexpr int OP = E.op[K];
      constexpr bool IN01 = (K > 0) && fop_out01(E.op[K > 0 ? K - 1 : 0]);
      const float* c = cp + E.coff[K];
      P2 y;
      if constexpr (OP == RISP_OP_SKIP) { y = x; }
      else if constexpr (OP == RISP_OP_GAMMA) { GammaSaved sv; y = gamma_fwd<IN01>(x, c[0], sv); }
      else if constexpr (OP == RISP_OP_GAIN) { y = gain_fwd(x, c); }
      else if constexpr (OP == RISP_OP_POLY10 || OP == FOP_POLYG) { PolySaved sv; y = poly_fwd(x, c, sv); }
      else { y = gtm_fwd(x, c, slow); }
      return Fwd<SIG, K + 1>::go(y, cp, slow);
    }
  }
};

template <unsigned SIG>
__device__ __forceinline__ bool chain_slow(const float* __restrict__ cp) {
  constexpr EffChain E = Eff<SIG>::e;
  bool slow = false;
#pragma unroll
  for (int k = 0; k < E.n; ++k)
    if (E.op[k] == RISP_OP_GTM) slow = slow || (cp[E.coff[k] + 5] != 0.f);
  return slow;
}

constexpr int kStepMinBlocks = 8;    // resident CTAs per SM the kernels are compiled for (register cap)
constexpr int kFwdMinBlocks = 16;
constexpr int kMaxRows = 256;        // rows per item at most

// NARROW: the kernel also runs narrow items (a.nw != 0); a separate instantiation, so that the kernels of frames without
// them keep their register allocation
template <int DM, int MODE, unsigned SIG, bool NARROW>
__global__ void __launch_bounds__(32, (MODE == MODE_FWD) ? kFwdMinBlocks : kStepMinBlocks)
fused_kernel(FusedArgs a, ChainDesc d, const __grid_constant__ CUtensorMap tm_raw, const __grid_constant__ CUtensorMap tm_gt,
             const __grid_constant__ CUtensorMap tm_rawn, const __grid_constant__ CUtensorMap tm_gtn) {
  constexpr EffChain E = Eff<SIG>::e;
  constexpr int HL = (DM == RISP_DM_MALVAR) ? 2 : 1;
  constexpr int WR = 2 * HL + 1, WC = 4 + 2 * HL;
  constexpr int NACC = (MODE == MODE_FWD || MODE == MODE_EVAL || E.nacc == 0) ? 1 : E.nacc;
  constexpr int NCST = E.ncst > 0 ? E.ncst : 1;
  static_assert(E.ncst <= kCRowFloats, "the chain's derived constants must fit one row of the constant slot");
  constexpr bool PKDM = E.n > 0 && (E.op[0] == RISP_OP_POLY10 || E.op[0] == FOP_POLYG || E.op[0] == RISP_OP_GAIN);
  using RC = RingCfg<MODE>;
  constexpr int D = RC::D;
  extern __shared__ unsigned char smem_raw[];
  const int lane = threadIdx.x;
  const int n = blockIdx.y, j0 = blockIdx.x;       // frame, CTA within the frame (both uniform)
  const int H = a.H, W = a.W;
  const long long plane = (long long)H * W;
  float* __restrict__ yb = a.y ? a.y + (long long)n * 3 * plane : nullptr;
  // derived constants of this frame's parameter row (written by fused_prep_kernel earlier on the stream): they enter the
  // packed instructions as broadcast scalars from uniform registers
  float cst[NCST];
  {
    const float* __restrict__ crow = &g_cpar[a.slot][a.pstride ? n : 0][0];
#pragma unroll
    for (int i = 0; i < NCST; ++i) cst[i] = crow[i];
  }
  const float* cp = cst;
  const bool slow = chain_slow<SIG>(cp);

  // ---- ring set-up -------------------------------------------------------------------------------------------------
  const uint32_t ring = (smem_u32(smem_raw) + 127u) & ~127u;
  const uint32_t bars = ring + RC::WARPB;
  const uint32_t tbl = ring + RC::TBLOFF;        // 64-byte aligned (the ring is 128-byte aligned)
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < D; ++s) mbar_init(bars + 8 * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if constexpr (MODE != MODE_FWD && MODE != MODE_EVAL) {
#pragma unroll
      for (int k = 0; k < E.n; ++k)
        if (E.op[k] == RISP_OP_GTM) gtm_table_fill(tbl + k * kGtmTableBytes, cp + E.coff[k]);
    }
  }
  __syncwarp();
  unsigned gcount = 0;        // records issued before the current item

  float2 acc[NACC];
  float2 loss = zero2();
  unsigned long long sse = 0;     // EVAL: this lane's sum of squared code differences (64 bits: exact for any geometry)
#pragma unroll
  for (int i = 0; i < NACC; ++i) acc[i] = zero2();

  // where a lane's 4 pixels sit in the records of the current item (backward-carrying kernels)
  struct LanePos {
    uint32_t own, oL0, oL1, oR0, oR1;   // raw-row byte offsets: own columns; halo columns c0-HL, c0-1, c0+4, c0+5
    uint32_t gt;                        // GT-row byte offset of the own columns
    int c0;                             // first column
    int dr;                             // row of the lane's pixels relative to the row the warp computes
    bool active;                        // a pixel of this item: inside the frame and the item's rows
    float lane_w;                       // active ? 1 : 0
  };
  // ---- backward-carrying kernels (issue-bound): a private window per row read with plain LDS ----
  // one row: read the window (wa(j): shared-memory address of its raw row j) and the GT row, demosaic, chain, store.
  // Narrow items: the lane's row may belong to another item while its GT is real data: such a lane's target is zeroed so
  // that it adds exactly nothing.
  auto do_row = [&](auto odd_tag, auto slow_tag, auto narrow_tag, int r, auto wa, uint32_t gta, const LanePos& L) {
    constexpr bool ODD = decltype(odd_tag)::value;
    constexpr bool slow = decltype(slow_tag)::value;     // shadows the run-time flag: the chain's branches on it fold away
    float w[WR][WC];
#pragma unroll
    for (int j = 0; j < WR; ++j) {
      const uint32_t rj = wa(j);
      const float4 v = lds4(rj + L.own);
      if constexpr (HL == 1) {
        w[j][0] = lds1(rj + L.oL0); w[j][1] = v.x; w[j][2] = v.y; w[j][3] = v.z; w[j][4] = v.w; w[j][5] = lds1(rj + L.oR0);
      } else {
        w[j][0] = lds1(rj + L.oL0); w[j][1] = lds1(rj + L.oL1);
        w[j][2] = v.x; w[j][3] = v.y; w[j][4] = v.z; w[j][5] = v.w;
        w[j][6] = lds1(rj + L.oR0); w[j][7] = lds1(rj + L.oR1);
      }
    }
    P2 lo, hi;
    demosaic4<DM, HL, 0, ODD, WR, PKDM>(w, a.clip_hi, lo, hi);
    P2 ylo, yhi;
    if constexpr (MODE == MODE_EVAL) {
      // the inference arithmetic (Fwd, not Run): the codes are those of risp_pipeline_fwd's image, byte for byte
      ylo = Fwd<SIG, 0>::go(lo, cp, slow);
      yhi = Fwd<SIG, 0>::go(hi, cp, slow);
      const float4 yB = make_float4(ylo.b.x, ylo.b.y, yhi.b.x, yhi.b.y), yG = make_float4(ylo.g.x, ylo.g.y, yhi.g.x, yhi.g.y),
                   yR = make_float4(ylo.r.x, ylo.r.y, yhi.r.x, yhi.r.y);
      // lanes beyond the right edge compute garbage from zero-filled raw (a zero pixel is not zero after the chain): masked
      if (L.active) {
        const uint32_t s = sq_codes4(yB, lds4(gta + L.gt)) + sq_codes4(yG, lds4(gta + RC::GTPLANEB + L.gt)) +
                           sq_codes4(yR, lds4(gta + 2 * RC::GTPLANEB + L.gt));
        sse += s;
        if (a.u8) {      // (H,W,3) BGR bytes of the lane's 4 pixels: 12 contiguous bytes, 4-byte aligned (c0 % 4 == 0)
          const uint32_t b0 = u8_code(yB.x), b1 = u8_code(yB.y), b2 = u8_code(yB.z), b3 = u8_code(yB.w);
          const uint32_t g0 = u8_code(yG.x), g1 = u8_code(yG.y), g2 = u8_code(yG.z), g3 = u8_code(yG.w);
          const uint32_t r0 = u8_code(yR.x), r1 = u8_code(yR.y), r2 = u8_code(yR.z), r3 = u8_code(yR.w);
          uint32_t* po = reinterpret_cast<uint32_t*>(a.u8 + (((long long)n * H + r + L.dr) * W + L.c0) * 3);
          po[0] = b0 | (g0 << 8) | (r0 << 16) | (b1 << 24);
          po[1] = g1 | (r1 << 8) | (b2 << 16) | (g2 << 24);
          po[2] = r2 | (b3 << 8) | (g3 << 16) | (r3 << 24);
        }
      }
    } else {
      constexpr bool narrow_item = decltype(narrow_tag)::value;
      float4 tg[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        tg[c] = lds4(gta + c * RC::GTPLANEB + L.gt);
        if constexpr (narrow_item) {
          if (!L.active) tg[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      P2 tlo, thi;
      tlo.b = make_float2(tg[0].x, tg[0].y); tlo.g = make_float2(tg[1].x, tg[1].y); tlo.r = make_float2(tg[2].x, tg[2].y);
      thi.b = make_float2(tg[0].z, tg[0].w); thi.g = make_float2(tg[1].z, tg[1].w); thi.r = make_float2(tg[2].z, tg[2].w);
      Run<SIG, 0, MODE>::go(lo, tlo, cp, acc, loss, ylo, slow, L.lane_w, tbl);
      Run<SIG, 0, MODE>::go(hi, thi, cp, acc, loss, yhi, slow, L.lane_w, tbl);
    }
    if (MODE != MODE_EVAL && yb && L.active) {
      float* po = yb + (size_t)(r + L.dr) * W + L.c0;
      st_stream4(po, make_float4(ylo.b.x, ylo.b.y, yhi.b.x, yhi.b.y));
      st_stream4(po + plane, make_float4(ylo.g.x, ylo.g.y, yhi.g.x, yhi.g.y));
      st_stream4(po + 2 * plane, make_float4(ylo.r.x, ylo.r.y, yhi.r.x, yhi.r.y));
    }
  };

  const int items = a.chunks * a.strip_blocks;
  for (int item = j0; item < items; item += a.cpf) {
    const int chunk = item / a.strip_blocks, strip = item - chunk * a.strip_blocks;
    const int c0s = strip * kStrip;                 // first column of the strip
    const int c0 = c0s + lane * 4;
    const bool active = c0 < W;                     // columns beyond the frame arrive as zeros (TMA out-of-bounds fill)
    const bool first = (c0 == 0), last = active && (c0 + 4 >= W);
    const float lane_w = active ? 1.f : 0.f;
    const int ra = chunk * a.rows_per_chunk;
    const int rb = min(H, ra + a.rows_per_chunk);
    constexpr int RR = RC::RR;
    const int rbase = ra - RR;                      // record k of the item holds physical rows rbase + RR*k .. + RR-1
    const int nrec = (rb - ra + RR - 1) / RR + 2;

    auto issue = [&](int k) {        // one elected lane: the two TMA boxes of record k
      const unsigned g = gcount + (unsigned)k;
      const uint32_t rec = ring + (g & (D - 1)) * RC::RECB, bar = bars + (g & (D - 1)) * 8;
      const bool has_gt = (MODE != MODE_FWD) && (k >= 1) && (k < nrec - 1);
      mbar_expect_tx(bar, (uint32_t)(RR * RC::RAWROWB) + (has_gt ? (uint32_t)RC::GTB : 0u));
      tma_load_3d(rec, &tm_raw, c0s - kPad, rbase + RR * k, n, bar);
      if (has_gt) tma_load_3d(rec + RC::RAWB, &tm_gt, c0s, rbase + RR * k, 3 * n, bar);
    };
    auto wait_rec = [&](int k) {
      const unsigned g = gcount + (unsigned)k;
      mbar_wait(bars + (g & (D - 1)) * 8, (g / D) & 1u);
    };
    // shared-memory address of physical raw row q (reflect-101 at the frame border) -- uniform
    auto row_addr = [&](int q) -> uint32_t {
      const int qq = reflect101(q, H);
      const int rel = qq - rbase;
      const unsigned g = gcount + (unsigned)(rel / RR);
      return ring + (g & (D - 1)) * RC::RECB + (uint32_t)(rel % RR) * RC::RAWROWB;
    };
    if (elect_one()) {
      for (int k = 0; k < D && k < nrec; ++k) issue(k);
    }
    __syncwarp();
    wait_rec(0);
    wait_rec(1);

    // lane offsets inside a raw row (bytes): own 4 columns; the strip's first / last lane reads its outer halo from the
    // record (frame border folded into the offset), every other lane gets it from its neighbour by shuffle
    const uint32_t own = (uint32_t)(kPad + lane * 4) * 4u;
    const bool endL = (lane == 0), endR = (lane == 31) || last;
    const uint32_t oL0 = own + (first ? (HL == 1 ? 4 : 8) : -4 * HL);    // column c0-HL   (reflect: -1 -> 1, -2 -> 2)
    const uint32_t oL1 = own + (first ? 4 : -4);                         // column c0-1    (HL == 2 only)
    const uint32_t oR0 = own + (last ? 8 : 16);                          // column c0+4    (reflect: W -> W-2)
    const uint32_t oR1 = own + (last ? 4 : 20);                          // column c0+5    (reflect: W+1 -> W-3)

    if constexpr (MODE != MODE_FWD) {
      // ---- backward-carrying kernels: 2-row records ----
      const LanePos L{own, oL0, oL1, oR0, oR1, (uint32_t)lane * 16u, c0, 0, active, lane_w};

      // iteration m computes rows r = ra + 2(m-1) (even) and r+1 (odd) from records m-1, m, m+1.
      // The loop exists twice, with the tone curve's slow flag (a knot outside [0,1]: final clamp active) as a compile-time
      // constant: two uniform branches per pixel pair and channel would otherwise cut the chain into ~25 basic blocks per
      // trip, and the scheduler cannot interleave the two pairs / the FMA-heavy and the ALU/XU phases across them.
      auto rows_loop = [&](auto slow_tag) {
      for (int m = 1; m < nrec - 1; ++m) {
        const int r = ra + 2 * (m - 1);
        wait_rec(m + 1);
        const unsigned gB = gcount + (unsigned)m;
        const uint32_t recA = ring + ((gB - 1) & (D - 1)) * RC::RECB, recB = ring + (gB & (D - 1)) * RC::RECB,
                       recC = ring + ((gB + 1) & (D - 1)) * RC::RECB;
        uint32_t we[WR], wo[WR];
        if (r >= HL && r + 1 + HL < H) {           // interior: static places
          if constexpr (HL == 1) {
            we[0] = recA + RC::RAWROWB; we[1] = recB; we[2] = recB + RC::RAWROWB;
            wo[0] = recB; wo[1] = recB + RC::RAWROWB; wo[2] = recC;
          } else {
            we[0] = recA; we[1] = recA + RC::RAWROWB; we[2] = recB; we[3] = recB + RC::RAWROWB; we[4] = recC;
            wo[0] = recA + RC::RAWROWB; wo[1] = recB; wo[2] = recB + RC::RAWROWB; wo[3] = recC; wo[4] = recC + RC::RAWROWB;
          }
        } else {                                   // first / last rows of the frame: reflected rows
  #pragma unroll
          for (int j = 0; j < WR; ++j) { we[j] = row_addr(r - HL + j); wo[j] = row_addr(r + 1 - HL + j); }
        }
        do_row(std::false_type{}, slow_tag, std::false_type{}, r, [&](int j) { return we[j]; }, recB + RC::RAWB, L);
        do_row(std::true_type{}, slow_tag, std::false_type{}, r + 1, [&](int j) { return wo[j]; }, recB + RC::RAWB + kStrip * 4, L);
        __syncwarp();                              // every lane has read record m-1: its slot may be refilled
        if (m - 1 + D < nrec) {
          if (elect_one()) issue(m - 1 + D);
        }
      }
      };
      if (slow) rows_loop(std::true_type{}); else rows_loop(std::false_type{});
    } else {
      // ---- inference kernel (memory-bound): RR-row records, one shared window per row pair, halo by shuffle ---------
      float w[WR + 1][WC];                                        // raw rows r-HL .. r+1+HL of the current row pair
      auto load_row = [&](float* dst, uint32_t ra_) {            // one raw row of the window: columns c0-HL .. c0+3+HL
        const unsigned full = 0xffffffffu;
        const float4 v = lds4(ra_ + own);
        if constexpr (HL == 1) {
          float l = __shfl_up_sync(full, v.w, 1), r = __shfl_down_sync(full, v.x, 1);
          if (endL) l = lds1(ra_ + oL0);
          if (endR) r = lds1(ra_ + oR0);
          dst[0] = l; dst[1] = v.x; dst[2] = v.y; dst[3] = v.z; dst[4] = v.w; dst[5] = r;
        } else {
          float l0 = __shfl_up_sync(full, v.z, 1), l1 = __shfl_up_sync(full, v.w, 1);
          float r0 = __shfl_down_sync(full, v.x, 1), r1 = __shfl_down_sync(full, v.y, 1);
          if (endL) { l0 = lds1(ra_ + oL0); l1 = lds1(ra_ + oL1); }
          if (endR) { r0 = lds1(ra_ + oR0); r1 = lds1(ra_ + oR1); }
          dst[0] = l0; dst[1] = l1; dst[2] = v.x; dst[3] = v.y; dst[4] = v.z; dst[5] = v.w; dst[6] = r0; dst[7] = r1;
        }
      };

      // one row from the register window w[RO .. RO+WR): demosaic, chain, store
      auto do_row = [&](auto ro_tag, auto odd_tag, int r) {
        constexpr int RO = decltype(ro_tag)::value;
        constexpr bool ODD = decltype(odd_tag)::value;
        P2 lo, hi;
        demosaic4<DM, HL, RO, ODD, WR + 1, PKDM>(w, a.clip_hi, lo, hi);
        const P2 ylo = Fwd<SIG, 0>::go(lo, cp, slow), yhi = Fwd<SIG, 0>::go(hi, cp, slow);
        if (active) {
          float* po = yb + (size_t)r * W + c0;
          st_stream4(po, make_float4(ylo.b.x, ylo.b.y, yhi.b.x, yhi.b.y));
          st_stream4(po + plane, make_float4(ylo.g.x, ylo.g.y, yhi.g.x, yhi.g.y));
          st_stream4(po + 2 * plane, make_float4(ylo.r.x, ylo.r.y, yhi.r.x, yhi.r.y));
        }
      };

      // iteration m computes the RR rows of record m (pairs of an even and an odd row) from records m-1, m, m+1
      for (int m = 1; m < nrec - 1; ++m) {
        const int R0 = ra + RR * (m - 1);
        wait_rec(m + 1);
        const unsigned gB = gcount + (unsigned)m;
        const uint32_t recA = ring + ((gB - 1) & (D - 1)) * RC::RECB, recB = ring + (gB & (D - 1)) * RC::RECB,
                       recC = ring + ((gB + 1) & (D - 1)) * RC::RECB;
        const bool interior = (R0 >= HL) && (R0 + RR - 1 + HL < H);
  #pragma unroll
        for (int p = 0; p < RR / 2; ++p) {
          const int r = R0 + 2 * p;
          if (r < rb) {
            uint32_t wa[WR + 1];
  #pragma unroll
            for (int j = 0; j < WR + 1; ++j) {
              const int idx = 2 * p - HL + j;          // row of the window relative to record m (static)
              wa[j] = (idx < 0) ? recA + (uint32_t)(RR + idx) * RC::RAWROWB
                    : (idx >= RR) ? recC + (uint32_t)(idx - RR) * RC::RAWROWB : recB + (uint32_t)idx * RC::RAWROWB;
            }
            if (!interior) {                           // first / last rows of the frame: reflected rows
  #pragma unroll
              for (int j = 0; j < WR + 1; ++j) wa[j] = row_addr(r - HL + j);
            }
            // the WR+1 rows are read once and serve both output rows
  #pragma unroll
            for (int j = 0; j < WR + 1; ++j) load_row(w[j], wa[j]);
            do_row(std::integral_constant<int, 0>{}, std::false_type{}, r);
            do_row(std::integral_constant<int, 1>{}, std::true_type{}, r + 1);
          }
        }
        __syncwarp();                              // every lane has read record m-1: its slot may be refilled
        if (m - 1 + D < nrec) {
          if (elect_one()) issue(m - 1 + D);
        }
      }
    }
    gcount += (unsigned)nrec;
  }

  if constexpr (MODE != MODE_FWD && NARROW) {
    // ---- narrow items: the frame's last strip when it is nw = 32 or 64 columns wide (or less) ------------------------
    // A full-width warp would issue its whole row loop for 8 or 16 useful lanes.  Here the warp splits into G = 128/nw
    // groups of nw/4 lanes; a record holds 2G rows ((nw + kPad) x 2G raw box, nw x 2G x 3 GT box: no more bytes than a
    // full record) and group g computes rows 2g, 2g+1 of it, so every lane still runs an even and then an odd row.  The
    // window rows are per lane (reflect-101 folded in as in row_addr).  A CTA's narrow items come after its full ones:
    // item t goes to CTA cpf-1 - t % cpf, the CTAs with the fewest full items.
    const int nw = a.nw;
    const int sh = (nw == 32) ? 3 : 2;              // log2 of the rows per record (2G)
    const int RRn = 1 << sh;
    const int grp = lane >> (6 - sh), li = lane & ((1 << (6 - sh)) - 1);
    const int c0s = a.strip_blocks * kStrip, c0 = c0s + 4 * li;
    const uint32_t rowb = (uint32_t)(nw + kPad) * 4u;
    const bool incol = c0 < W, first = (c0 == 0), last = incol && (c0 + 4 >= W);
    LanePos L;
    L.own = (uint32_t)(kPad + 4 * li) * 4u;
    L.oL0 = L.own + (first ? (HL == 1 ? 4 : 8) : -4 * HL);
    L.oL1 = L.own + (first ? 4 : -4);
    // a lane with c0 + 4 < W is never the last of its group (W <= c0s + nw).  Lanes past the frame read inside their row
    // as well: past the last row of a 64-wide box lie pad bytes that no copy writes (stale data, possibly NaN)
    const bool fold = last || !incol;
    L.oR0 = L.own + (fold ? 8 : 16);
    L.oR1 = L.own + (fold ? 4 : 20);
    L.c0 = c0;
    L.dr = 2 * grp;
    const uint32_t gt_even = (uint32_t)(2 * grp * nw + 4 * li) * 4u;
    for (int t = a.cpf - 1 - j0; t < a.nchunks; t += a.cpf) {
      const int ra = t * a.nrows_per_chunk;
      const int rb = min(H, ra + a.nrows_per_chunk);
      const int rbase = ra - RRn;                   // record k holds rows rbase + RRn*k .. + RRn-1
      const int nrec = (rb - ra + RRn - 1) / RRn + 2;
      auto issue = [&](int k) {
        const unsigned g = gcount + (unsigned)k;
        const uint32_t rec = ring + (g & (D - 1)) * RC::RECB, bar = bars + (g & (D - 1)) * 8;
        const bool has_gt = (k >= 1) && (k < nrec - 1);
        mbar_expect_tx(bar, (uint32_t)RRn * rowb + (has_gt ? (uint32_t)RC::GTB : 0u));
        tma_load_3d(rec, &tm_rawn, c0s - kPad, rbase + RRn * k, n, bar);
        if (has_gt) tma_load_3d(rec + RC::RAWB, &tm_gtn, c0s, rbase + RRn * k, 3 * n, bar);
      };
      auto wait_rec = [&](int k) {
        const unsigned g = gcount + (unsigned)k;
        mbar_wait(bars + (g & (D - 1)) * 8, (g / D) & 1u);
      };
      auto row_addr = [&](int q) -> uint32_t {      // per lane
        const int rel = reflect101(q, H) - rbase;
        const unsigned g = gcount + (unsigned)(rel >> sh);
        return ring + (g & (D - 1)) * RC::RECB + (uint32_t)(rel & (RRn - 1)) * rowb;
      };
      if (elect_one()) {
        for (int k = 0; k < D && k < nrec; ++k) issue(k);
      }
      __syncwarp();
      wait_rec(0);
      wait_rec(1);
      auto rows_loop = [&](auto slow_tag) {
        for (int m = 1; m < nrec - 1; ++m) {
          const int R = ra + RRn * (m - 1);         // group g computes rows R + 2g, R + 2g + 1
          // a group past the item's last row is masked.  Its window rows, reflected at the frame's last row, still lie in
          // the records m-1 .. m+1 (R <= H-2, so a reflected row is >= R - 2G + 1): loaded frame data, finite
          L.active = incol && R + L.dr < rb;
          L.lane_w = L.active ? 1.f : 0.f;
          L.gt = gt_even;
          wait_rec(m + 1);
          const uint32_t gta = ring + ((gcount + (unsigned)m) & (D - 1)) * RC::RECB + RC::RAWB;
          // window rows are computed where they are read: per-lane addresses live across the chain would cost registers
          do_row(std::false_type{}, slow_tag, std::true_type{}, R, [&](int j) { return row_addr(R + L.dr - HL + j); }, gta, L);
          L.gt = gt_even + (uint32_t)nw * 4u;
          do_row(std::true_type{}, slow_tag, std::true_type{}, R + 1, [&](int j) { return row_addr(R + L.dr + 1 - HL + j); }, gta, L);
          __syncwarp();                              // every lane has read record m-1: its slot may be refilled
          if (m - 1 + D < nrec) {
            if (elect_one()) issue(m - 1 + D);
          }
        }
      };
      if (slow) rows_loop(std::true_type{}); else rows_loop(std::false_type{});
      gcount += (unsigned)nrec;
    }
  }

  if constexpr (MODE == MODE_EVAL) {
    const unsigned long long tot = warp_sum_u64(sse);
    if (lane == 0) a.sse[(long long)n * a.cpf + j0] = tot;
  } else if constexpr (MODE != MODE_FWD) {
    // ---- epilogue: one partial row per warp, slot layout of risp_common.cuh ------------------------------------------
    float tot[NACC];
#pragma unroll
    for (int i = 0; i < NACC; ++i) tot[i] = warp_sum(acc[i].x + acc[i].y);
    const float lsum = warp_sum(loss.x + loss.y);
    if (lane == 0) {
      float* __restrict__ out = a.partial + ((long long)n * a.cpf + j0) * RISP_NSLOT;
#pragma unroll
      for (int i = 0; i < RISP_NSLOT; ++i) out[i] = 0.f;
      out[RISP_SLOT_LOSS] = lsum;
      const float* __restrict__ prow = a.params + (long long)n * a.pstride;
      float scale = 1.f;        // product of the uniform factors deferred by the stages downstream
#pragma unroll
      for (int k = E.n - 1; k >= 0; --k) {
        const float* t = tot + E.aoff[k];
        const int src = E.src[k];
        if (E.op[k] == RISP_OP_GAMMA) {
          out[src * RISP_SMALL_ACC] = t[0] * RISP_LN2 * scale;
          scale *= cp[E.coff[k]];
        } else if (E.op[k] == RISP_OP_GAIN) {
#pragma unroll
          for (int i = 0; i < 3; ++i) out[src * RISP_SMALL_ACC + i] = t[i] * scale;
        } else if (E.op[k] == RISP_OP_GTM) {
          out[src * RISP_SMALL_ACC + 0] = 4.f * ((t[0] - 2.f * t[1]) + t[2]) * scale;
          out[src * RISP_SMALL_ACC + 1] = 4.f * ((t[1] - 2.f * t[2]) + t[3]) * scale;
          out[src * RISP_SMALL_ACC + 2] = 4.f * (t[2] - 2.f * t[3]) * scale;
        } else if (E.op[k] == RISP_OP_POLY10) {
#pragma unroll
          for (int i = 0; i < 30; ++i) out[RISP_SLOT_BIG + i] = t[i] * scale;
        } else if (E.op[k] == FOP_POLYG) {
          // S[c][i] = sum e_c phi_i(x0)  ->  d/dq[c][i] = gmon_i S ,  d/dg = sum q (d gmon / d g) S
          const float* g = prow + d.off[src - 1];
          const float* qq = prow + d.off[src];
          const float gb = g[0], gg = g[1], gr = g[2];
          const float gmon[10] = {gb * gb, gg * gg, gr * gr, gb * gg, gb * gr, gg * gr, gb, gg, gr, 1.f};
          const float dgb[10] = {2.f * gb, 0.f, 0.f, gg, gr, 0.f, 1.f, 0.f, 0.f, 0.f};
          const float dgg[10] = {0.f, 2.f * gg, 0.f, gb, 0.f, gr, 0.f, 1.f, 0.f, 0.f};
          const float dgr[10] = {0.f, 0.f, 2.f * gr, 0.f, gb, gg, 0.f, 0.f, 1.f, 0.f};
          float sb = 0.f, sg = 0.f, sr = 0.f;
#pragma unroll
          for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int i = 0; i < 10; ++i) {
              const float s = t[c * 10 + i] * scale;
              out[RISP_SLOT_BIG + c * 10 + i] = gmon[i] * s;
              const float qs = qq[c * 10 + i] * s;
              sb = fmaf(qs, dgb[i], sb); sg = fmaf(qs, dgg[i], sg); sr = fmaf(qs, dgr[i], sr);
            }
          out[(src - 1) * RISP_SMALL_ACC + 0] = sb; out[(src - 1) * RISP_SMALL_ACC + 1] = sg; out[(src - 1) * RISP_SMALL_ACC + 2] = sr;
        }
      }
    }
  }
}

// ---- host side ---------------------------------------------------------------------------------------------------------
struct Geometry { int rows_per_chunk, chunks, strip_blocks, cpf, grid, nw, nrows_per_chunk, nchunks; };

// Critical path of a layout, in row units: a full item of rf rows costs rf + rr + 2 (it also loads a lead-in record and
// fills the pipeline), a narrow item of rn rows 2 * rn / (2G) + rr + 2.  CTA j runs full items j, j + cpf, .. < F, then
// narrow items cpf-1-j, 2cpf-1-j, .. < Nn.  Both counts are step functions of j (at F % cpf and cpf - Nn % cpf), so the
// extremes are on those steps.  Returns the largest cost over all CTAs; *narrow_max: the largest over CTAs with a narrow item.
static long long layout_cost(long long F, long long cf, long long Nn, long long cn, long long cpf, long long* narrow_max) {
  const long long js[6] = {0, F % cpf - 1, F % cpf, cpf - Nn % cpf - 1, cpf - Nn % cpf, cpf - 1};
  long long worst = 0, nworst = 0;
  for (long long j : js) {
    if (j < 0 || j >= cpf) continue;
    const long long nf = F > j ? cdiv(F - j, cpf) : 0, u = cpf - 1 - j, nn = Nn > u ? cdiv(Nn - u, cpf) : 0;
    const long long c = nf * cf + nn * cn;
    worst = c > worst ? c : worst;
    if (nn > 0 && c > nworst) nworst = c;
  }
  *narrow_max = nworst;
  return worst;
}

static Geometry geometry_uncached(int N, int H, int W, int ctas_per_sm, int rr, int max_rows, bool narrow) {
  Geometry g{};
  const int rem = W % kStrip;
  g.nw = (narrow && rem > 0 && rem <= 64) ? (rem <= 32 ? 32 : 64) : 0;
  g.strip_blocks = g.nw ? W / kStrip : (int)cdiv(W, kStrip);     // items are (row chunk, strip): one warp per CTA
  const int slots = sm_count() * ctas_per_sm;
  g.cpf = slots / N < 1 ? 1 : slots / N;
  if (g.nw) {
    // rows per full and per narrow chunk: least critical path, then the narrow items' CTAs least loaded (the cost of a
    // narrow row is the least certain), then fewest items
    const int rrn = 2 * (kStrip / g.nw);
    long long best = -1, best_n = 0, best_items = 0;
    for (int rf = rr; rf <= max_rows; rf += rr) {
      if ((rf > H || g.strip_blocks == 0) && rf > rr) break;
      const long long F = cdiv(H, rf) * g.strip_blocks, cf = rf + rr + 2;
      for (int rn = rrn;; rn += rrn) {
        const long long Nn = cdiv(H, rn), cn = 2 * (rn / rrn) + rr + 2;
        if (best >= 0 && cn > best) break;          // grows with rn
        const long long cpf = F + Nn < g.cpf ? F + Nn : g.cpf;
        long long nmax;
        const long long c = layout_cost(F, cf, Nn, cn, cpf, &nmax);
        if (best < 0 || c < best || (c == best && (nmax < best_n || (nmax == best_n && F + Nn < best_items)))) {
          best = c; best_n = nmax; best_items = F + Nn;
          g.rows_per_chunk = rf; g.nrows_per_chunk = rn;
        }
        if (rn >= H) break;
      }
    }
    g.chunks = g.strip_blocks ? (int)cdiv(H, g.rows_per_chunk) : 0;
    g.nchunks = (int)cdiv(H, g.nrows_per_chunk);
    const long long items = (long long)g.chunks * g.strip_blocks + g.nchunks;
    if (items < g.cpf) g.cpf = (int)items;
    g.grid = N * g.cpf;
    return g;
  }
  // rows per chunk: minimise rounds * (rows + per-item overhead); an item costs ~3 extra rows (window fill, exposed latency)
  long long best = -1;
  int best_rows = rr;
  for (int rows = rr; rows <= max_rows; rows += rr) {        // whole records (rr rows each)
    if (rows > H && rows > rr) break;
    const int chunks = (int)cdiv(H, rows);
    const long long items = (long long)chunks * g.strip_blocks;
    const long long rounds = cdiv(items, g.cpf);
    const long long cost = rounds * (rows + rr + 2);   // an item also loads a lead-in record and fills the pipeline
    if (best < 0 || cost < best || (cost == best && rows > best_rows)) { best = cost; best_rows = rows; }
  }
  g.rows_per_chunk = best_rows;
  g.chunks = (int)cdiv(H, best_rows);
  const long long items = (long long)g.chunks * g.strip_blocks;
  if (items < g.cpf) g.cpf = (int)items;
  g.grid = N * g.cpf;
  return g;
}

// the narrow layout's search visits thousands of layouts: it runs once per shape, later launches look the result up
static Geometry geometry(int N, int H, int W, int ctas_per_sm, int rr, int max_rows, bool narrow) {
  static std::mutex mu;
  static std::map<std::array<int, 7>, Geometry> cache;
  const std::array<int, 7> key{N, H, W, ctas_per_sm, rr, max_rows, narrow ? 1 : 0};
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(key);
  if (it == cache.end()) it = cache.emplace(key, geometry_uncached(N, H, W, ctas_per_sm, rr, max_rows, narrow)).first;
  return it->second;
}

static std::mutex g_slot_mu;
static cudaStream_t g_slot_stream[kCSlots];
static int g_slot_used = 0;

// one constant slot per stream: prep kernel and consumer are ordered by the stream, so a slot is never rewritten while
// an earlier launch on that stream still reads it.  More than kCSlots distinct streams share the last slot (documented).
static int slot_of(cudaStream_t st) {
  std::lock_guard<std::mutex> lk(g_slot_mu);
  for (int i = 0; i < g_slot_used; ++i)
    if (g_slot_stream[i] == st) return i;
  if (g_slot_used < kCSlots) { g_slot_stream[g_slot_used] = st; return g_slot_used++; }
  return kCSlots - 1;
}

static float* cpar_device_ptr() {
  static float* p = nullptr;
  if (!p) {
    void* q = nullptr;
    if (cudaGetSymbolAddress(&q, g_cpar) == cudaSuccess) p = static_cast<float*>(q);
  }
  return p;
}

template <int DM, int MODE, unsigned SIG, bool NARROW>
static int resident_ctas() {
  static int n = 0;
  if (n == 0) {
    cudaFuncSetAttribute(fused_kernel<DM, MODE, SIG, NARROW>, cudaFuncAttributeMaxDynamicSharedMemorySize, RingCfg<MODE>::SMEM);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, fused_kernel<DM, MODE, SIG, NARROW>, 32, RingCfg<MODE>::SMEM) != cudaSuccess || n < 1) n = 1;
  }
  return n;
}

// ---- tensor maps (driver entry point resolved through the runtime: no -lcuda) ------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}
// fp32 tensor (W, H, Z) with rows of W floats, box (bx, by, bz); out-of-bounds elements read as zero
static int make_map(CUtensorMap* tm, const float* base, int W, int H, long long Z, int bx, int by, int bz) {
  EncodeTiledFn fn = encode_fn();
  RISP_REQUIRE(fn, RISP_E_CUDA, "fused pipeline: cuTensorMapEncodeTiled is not available");
  const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)Z};
  const cuuint64_t strides[2] = {(cuuint64_t)W * 4, (cuuint64_t)W * H * 4};
  const cuuint32_t box[3] = {(cuuint32_t)bx, (cuuint32_t)by, (cuuint32_t)bz};
  const cuuint32_t estr[3] = {1u, 1u, 1u};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  RISP_REQUIRE(r == CUDA_SUCCESS, RISP_E_CUDA, "fused pipeline: cuTensorMapEncodeTiled failed (%d) for %dx%dx%lld", (int)r, W, H, Z);
  return RISP_OK;
}

template <int DM, int MODE, unsigned SIG>
static int launch_one(FusedArgs a, const ChainDesc& d, int N, cudaStream_t st, int* rows_per_frame) {
  // RISP_FUSED_STEP_ROWS: cap of the rows per item of the backward-carrying and evaluation kernels (many short items)
  static const int cap = [] { const char* e = MODE == MODE_FWD ? nullptr : getenv("RISP_FUSED_STEP_ROWS"); return e ? atoi(e) : 0; }();
  // narrow items where the kernel that runs them keeps the occupancy of the one that does not
  bool narrow = false;
  if constexpr (MODE != MODE_FWD) narrow = resident_ctas<DM, MODE, SIG, true>() == resident_ctas<DM, MODE, SIG, false>();
  const Geometry g = geometry(N, a.H, a.W, resident_ctas<DM, MODE, SIG, false>(), RingCfg<MODE>::RR,
                              cap >= RingCfg<MODE>::RR ? cap : kMaxRows, narrow);
  if (rows_per_frame) *rows_per_frame = g.cpf;
  a.rows_per_chunk = g.rows_per_chunk; a.chunks = g.chunks; a.strip_blocks = g.strip_blocks; a.cpf = g.cpf;
  a.nw = g.nw; a.nrows_per_chunk = g.nrows_per_chunk; a.nchunks = g.nchunks;
  CUtensorMap tm_raw, tm_gt, tm_rawn, tm_gtn;
  int rc = make_map(&tm_raw, a.raw, a.W, a.H, N, kStrip + 2 * kPad, RingCfg<MODE>::RR, 1);
  if (rc != RISP_OK) return rc;
  if (MODE != MODE_FWD) {
    rc = make_map(&tm_gt, a.gt, a.W, a.H, 3ll * N, kStrip, RingCfg<MODE>::RR, 3);
    if (rc != RISP_OK) return rc;
  } else {
    tm_gt = tm_raw;
  }
  if (g.nw) {     // narrow boxes: 4 pad columns on the left only (the strip ends at the frame's right edge), 2G rows
    const int rrn = 2 * (kStrip / g.nw);
    static_assert(RingCfg<MODE_STEP>::RAWB >= 36 * 8 * 4 && RingCfg<MODE_STEP>::RAWB >= 68 * 4 * 4 &&
                  RingCfg<MODE_STEP>::GTB == 3 * 32 * 8 * 4 && RingCfg<MODE_STEP>::GTB == 3 * 64 * 4 * 4,
                  "a narrow record must fit the ring's record");
    rc = make_map(&tm_rawn, a.raw, a.W, a.H, N, g.nw + kPad, rrn, 1);
    if (rc != RISP_OK) return rc;
    rc = make_map(&tm_gtn, a.gt, a.W, a.H, 3ll * N, g.nw, rrn, 3);
    if (rc != RISP_OK) return rc;
  } else {
    tm_rawn = tm_raw; tm_gtn = tm_gt;
  }
  if constexpr (MODE != MODE_FWD) {
    if (g.nw) {
      fused_kernel<DM, MODE, SIG, true><<<dim3(g.cpf, N), 32, RingCfg<MODE>::SMEM, st>>>(a, d, tm_raw, tm_gt, tm_rawn, tm_gtn);
      return check_launch("fused_kernel");
    }
  }
  fused_kernel<DM, MODE, SIG, false><<<dim3(g.cpf, N), 32, RingCfg<MODE>::SMEM, st>>>(a, d, tm_raw, tm_gt, tm_rawn, tm_gtn);
  return check_launch("fused_kernel");
}

template <int MODE>
static int dispatch(const FusedArgs& a, const ChainDesc& d, int N, int dm_kind, cudaStream_t st, int* rows_per_frame) {
  const unsigned sig = chain_signature(d);
#define RISP_F_SIG(DMK, SG) if (sig == (SG)) return launch_one<DMK, MODE, (SG)>(a, d, N, st, rows_per_frame);
#define RISP_F_DM(DMK) RISP_F_SIG(DMK, RISP_SIG_A) RISP_F_SIG(DMK, RISP_SIG_B) RISP_F_SIG(DMK, RISP_SIG_C) RISP_F_SIG(DMK, RISP_SIG_D) \
  if constexpr (MODE == MODE_FWD || MODE == MODE_EVAL) { RISP_F_SIG(DMK, RISP_SIG_SKIP) }
  switch (dm_kind) {
    case RISP_DM_NEAREST: RISP_F_DM(RISP_DM_NEAREST) break;
    case RISP_DM_BILINEAR: RISP_F_DM(RISP_DM_BILINEAR) break;
    case RISP_DM_MALVAR: RISP_F_DM(RISP_DM_MALVAR) break;
    default: break;
  }
#undef RISP_F_DM
#undef RISP_F_SIG
  return 1;   // not handled
}

// derived constants of every parameter row into the stream's constant slot, ahead of the kernel that reads them
static int prep_constants(const float* params, int pstride, int N, const ChainDesc& d, cudaStream_t st, int* slot) {
  float* cbase = cpar_device_ptr();
  RISP_REQUIRE(cbase, RISP_E_CUDA, "fused pipeline: cannot resolve the constant parameter block");
  *slot = slot_of(st);
  fused_prep_kernel<<<pstride ? N : 1, 32, 0, st>>>(params, pstride, d, cbase + (size_t)*slot * kCRows * kCRowFloats);
  return check_launch("fused_prep_kernel");
}

}  // namespace fused

// true if the packed kernels take this chain (a pre-instantiated signature, parameter rows fit a constant slot)
bool fused_handles(const ChainDesc& d, int N, int param_stride, int H, int W) {
  if ((long long)H * W * 3 >= (1ll << 31)) return false;     // 32-bit element offsets inside a frame
  const unsigned sig = chain_signature(d);
  if (sig != RISP_SIG_A && sig != RISP_SIG_B && sig != RISP_SIG_C && sig != RISP_SIG_D && sig != RISP_SIG_SKIP) return false;
  if (param_stride != 0 && N > fused::kCRows) return false;
  return fused::eff_from_ops(d.op, d.iarg, d.S).ok;
}

// partial rows the step / backward kernels write: [N][rows_per_frame][RISP_NSLOT]
int fused_partial_rows_per_frame(int N) {
  // the largest grid any instantiation may use: 32 resident CTAs per SM is the hardware bound
  int slots = sm_count() * 32;
  return slots / N < 1 ? 1 : slots / N;
}

// evaluation mode: inference arithmetic, squared 8-bit code differences to gt -> partial[N][*rows_per_frame], optional 8-bit
// HWC image.  Returns RISP_OK, an error, or 1 when the chain is not handled.
int fused_eval_launch(const float* raw, const float* gt, unsigned char* u8, unsigned long long* partial, const float* params,
                      int pstride, int N, int H, int W, int dm_kind, float clip_hi, const ChainDesc& d, cudaStream_t st,
                      int* rows_per_frame) {
  using namespace fused;
  if (!fused_handles(d, N, pstride, H, W)) return 1;
  int slot;
  const int rc = prep_constants(params, pstride, N, d, st, &slot);
  if (rc != RISP_OK) return rc;
  const FusedArgs a{raw, gt, nullptr, nullptr, params, pstride, H, W, 0, 0, 0, 0, clip_hi, slot, u8, partial};
  return dispatch<MODE_EVAL>(a, d, N, dm_kind, st, rows_per_frame);
}

// mode: 0 forward, 1 MSE step, 2 backward with upstream dy, 3 L1 step.  Returns RISP_OK, an error, or 1 when the chain is not handled.
// *rows_per_frame (nullable) receives the number of partial rows per frame actually written (modes 1-3).
int fused_launch(int mode, const float* raw, const float* gt, float* y, float* partial, const float* params, int pstride,
                 int N, int H, int W, int dm_kind, float clip_hi, const ChainDesc& d, cudaStream_t st, int* rows_per_frame) {
  using namespace fused;
  if (!fused_handles(d, N, pstride, H, W)) return 1;
  int slot;
  const int rc = prep_constants(params, pstride, N, d, st, &slot);
  if (rc != RISP_OK) return rc;
  const FusedArgs a{raw, gt, y, partial, params, pstride, H, W, 0, 0, 0, 0, clip_hi, slot};
  switch (mode) {
    case 0: return dispatch<MODE_FWD>(a, d, N, dm_kind, st, rows_per_frame);
    case 1: return dispatch<MODE_STEP>(a, d, N, dm_kind, st, rows_per_frame);
    case 3: return dispatch<MODE_STEP_L1>(a, d, N, dm_kind, st, rows_per_frame);
    default: return dispatch<MODE_BWD>(a, d, N, dm_kind, st, rows_per_frame);
  }
}

}  // namespace risp
