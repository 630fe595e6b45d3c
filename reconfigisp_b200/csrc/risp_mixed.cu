// DARTS mixed-op (super_prune_fifteen_demos_four_bayer_two.py:185-212) and the loss.
//
//   probs = softmax(alpha); post = probs * [probs >= thr*max] / sum(.).detach()          (alpha_prune_*)
//   y     = sum_k post_k * candidate_k(x)                                                  (mixed_fwd)
//   bwd   : dx, d post_k = <dy, candidate_k(x)>, per-candidate parameter gradients         (mixed_bwd)
//
// The reference evaluates every candidate as its own module call and then runs 2K element-wise
// launches (`* prob`, `y + ...`), i.e. ~84 B/px per candidate.  Here the classical candidates
// (gamma / grayworld-apply / skip / wb-manual / wb-quadratic / gtm) are evaluated in registers from a
// single read of x, the materialised CNN candidates are read once each, and y is written once:
// 12 + 12*K_ext + 12 B/px forward, 24 + 12*K_ext + 12 B/px backward.  All K dot products and all
// parameter gradients come out of the same backward pass (register accumulators -> warp shuffle ->
// per-block partial -> deterministic finaliser).  No .item() syncs: weights are read on the device.
#include "risp_common.cuh"
#include "risp_stage.cuh"

namespace risp {

constexpr int kT = 256;
constexpr int kMixSlots = RISP_NSLOT + RISP_MAX_BRANCHES;   // 56 chain slots + 16 branch dot products

struct MixDesc {
  int K_cls, K_ext;
  int op[RISP_MAX_STAGES];
  int off[RISP_MAX_STAGES];
  int iarg[RISP_MAX_STAGES];
  const float* ext[RISP_MAX_BRANCHES];
  float* dext[RISP_MAX_BRANCHES];     // backward: where w_e * dy goes (the upstream gradient of candidate e), or null
};

template <int VEC> struct V3;
template <> struct V3<4> {
  float v[3][4];
  __device__ __forceinline__ void load(const float* p, long long HW, long long i, int C) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      if (c < C) { float4 t = ld_stream4(p + c * HW + 4 * i); v[c][0] = t.x; v[c][1] = t.y; v[c][2] = t.z; v[c][3] = t.w; }
      else { v[c][0] = v[c][1] = v[c][2] = v[c][3] = 0.f; }
    }
  }
  __device__ __forceinline__ void store(float* p, long long HW, long long i, int C) const {
#pragma unroll
    for (int c = 0; c < 3; ++c)
      if (c < C) st_stream4(p + c * HW + 4 * i, make_float4(v[c][0], v[c][1], v[c][2], v[c][3]));
  }
};
template <> struct V3<1> {
  float v[3][1];
  __device__ __forceinline__ void load(const float* p, long long HW, long long i, int C) {
#pragma unroll
    for (int c = 0; c < 3; ++c) v[c][0] = (c < C) ? p[c * HW + i] : 0.f;
  }
  __device__ __forceinline__ void store(float* p, long long HW, long long i, int C) const {
#pragma unroll
    for (int c = 0; c < 3; ++c)
      if (c < C) p[c * HW + i] = v[c][0];
  }
};

template <int VEC> struct MixNpx { static constexpr int value = (VEC == 4) ? 4 : 2; };

// Compile-time list of the classical candidates (like the chain kernels' Sig<>): with SIG != 0 the op of candidate j is a
// constant, so the interpreter's switch folds away and only that op's code and accumulators remain.  SIG == 0: generic.
// The supernet's sRGB step (super_prune_fifteen_demos_four_bayer_two.py:101-171): gamma, grayworld-apply, skip, wbmanual,
// wbquadratic, gtmmanual.
#define RISP_MIX_SIG_SRGB ::risp::make_sig(RISP_OP_GAMMA, RISP_OP_GAIN_CLIP, RISP_OP_SKIP, RISP_OP_GAIN, RISP_OP_POLY10, RISP_OP_GTM)
template <unsigned SIG>
struct MixSig {
  using SG = Sig<SIG>;
  static constexpr bool generic = (SIG == 0);
  __device__ __forceinline__ static bool live(const MixDesc& d, int j) { return generic ? (j < d.K_cls) : (j < SG::S); }
  __device__ __forceinline__ static int op(const MixDesc& d, int j) { return generic ? d.op[j] : SG::op_c(j); }
  __device__ __forceinline__ static int iarg(const MixDesc& d, int j) { return generic ? d.iarg[j] : 4; }
};

// 128-bit streaming load under a predicate (zeros when off): no branch, so the loads of a whole batch of candidate
// outputs are in flight together instead of one dependent round trip per candidate
__device__ __forceinline__ float4 ld_stream4_if(const float* p, bool on) {
  float4 v;
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.s32 q, %5, 0;\n\tmov.f32 %0, 0f00000000;\n\tmov.f32 %1, 0f00000000;\n\t"
               "mov.f32 %2, 0f00000000;\n\tmov.f32 %3, 0f00000000;\n\t"
               "@q ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];\n\t}"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "r"((int)on));
  return v;
}
constexpr int kExtBatch = 3;     // materialised candidates loaded together (3 planes x 128 bit each = 36 registers)
constexpr int kExtBatchFwd = 4;  // measured: 1 CTA/SM with 4 candidates in flight beats 2 CTAs with 2 (0.58 vs 0.44 of HBM peak)

// load / store one pixel group of a C-plane image (C = 1 or 3; missing planes read as 0)
template <int VEC>
__device__ __forceinline__ void mix_load(Px<MixNpx<VEC>::value>& px, const float* __restrict__ p, long long HW, long long i,
                                         int C) {
  V3<VEC> t;
  if (VEC == 4) {
    t.load(p, HW, i, C);
#pragma unroll
    for (int k = 0; k < 4; ++k) { px.b[k] = t.v[0][k]; px.g[k] = t.v[1][k]; px.r[k] = t.v[2][k]; }
  } else {
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const long long e = 2 * i + k;
      const bool ok = e < HW;
      px.b[k] = ok ? p[e] : 0.f;
      px.g[k] = (ok && C > 1) ? p[HW + e] : 0.f;
      px.r[k] = (ok && C > 2) ? p[2 * HW + e] : 0.f;
    }
  }
}
template <int VEC>
__device__ __forceinline__ void mix_store(const Px<MixNpx<VEC>::value>& px, float* __restrict__ p, long long HW, long long i,
                                          int C) {
  if (VEC == 4) {
    st_stream4(p + 4 * i, make_float4(px.b[0], px.b[1], px.b[2], px.b[3]));
    if (C > 1) st_stream4(p + HW + 4 * i, make_float4(px.g[0], px.g[1], px.g[2], px.g[3]));
    if (C > 2) st_stream4(p + 2 * HW + 4 * i, make_float4(px.r[0], px.r[1], px.r[2], px.r[3]));
  } else {
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const long long e = 2 * i + k;
      if (e < HW) {
        p[e] = px.b[k];
        if (C > 1) p[HW + e] = px.g[k];
        if (C > 2) p[2 * HW + e] = px.r[k];
      }
    }
  }
}

template <int VEC, unsigned SIG>
__global__ void __launch_bounds__(kT, 1)
mixed_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, long long HW, int C, MixDesc d,
                 const float* __restrict__ params, int pstride, const float* __restrict__ w) {
  constexpr int NPX = MixNpx<VEC>::value;
  const int n = blockIdx.y;
  const float* __restrict__ prow = params + (long long)n * pstride;
  const long long img = (long long)n * C * HW;
  float wk[RISP_MAX_STAGES], wext[RISP_MAX_BRANCHES];
#pragma unroll
  for (int k = 0; k < RISP_MAX_STAGES; ++k) wk[k] = (k < d.K_cls) ? w[k] : 0.f;
#pragma unroll
  for (int k = 0; k < RISP_MAX_BRANCHES; ++k) wext[k] = (k < d.K_ext) ? w[d.K_cls + k] : 0.f;
  const long long nvec = (VEC == 4) ? HW / 4 : (HW + 1) / 2;
  for (long long i = (long long)blockIdx.x * kT + threadIdx.x; i < nvec; i += (long long)gridDim.x * kT) {
    Px<NPX> X, Y;
    mix_load<VEC>(X, x + img, HW, i, C);
    // the first batch of materialised candidates is requested BEFORE the classical candidates are evaluated, so its round trip
    // hides behind their arithmetic (the loads are `asm volatile`: they stay where they are written)
    float4 E[kExtBatchFwd][3];
    auto issue_batch = [&](int e0) {
#pragma unroll
      for (int u = 0; u < kExtBatchFwd; ++u) {
        const int e = e0 + u;
        const bool live = (e < RISP_MAX_BRANCHES) && (e < d.K_ext) && !(wext[e < RISP_MAX_BRANCHES ? e : 0] < 1e-9f);
        const float* p = d.ext[e < RISP_MAX_BRANCHES ? e : 0] + img + 4 * i;
#pragma unroll
        for (int c = 0; c < 3; ++c) E[u][c] = ld_stream4_if(p + c * HW, live && c < C);
      }
    };
    if (VEC == 4 && d.K_ext > 0) issue_batch(0);
#pragma unroll
    for (int k = 0; k < NPX; ++k) { Y.b[k] = 0.f; Y.g[k] = 0.f; Y.r[k] = 0.f; }
#pragma unroll
    for (int j = 0; j < RISP_MAX_STAGES; ++j) {
      if (MixSig<SIG>::live(d, j) && !(wk[j] < 1e-9f)) {
        Px<NPX> t = X;
        stage_fwd(MixSig<SIG>::op(d, j), MixSig<SIG>::iarg(d, j), prow + d.off[j], t);
#pragma unroll
        for (int k = 0; k < NPX; ++k) {
          Y.b[k] = fmaf(wk[j], t.b[k], Y.b[k]); Y.g[k] = fmaf(wk[j], t.g[k], Y.g[k]); Y.r[k] = fmaf(wk[j], t.r[k], Y.r[k]);
        }
      }
    }
    if (VEC == 4) {
#pragma unroll
      for (int e0 = 0; e0 < RISP_MAX_BRANCHES; e0 += kExtBatchFwd) {
        if (e0 < d.K_ext) {                                   // uniform
          if (e0 > 0) issue_batch(e0);
#pragma unroll
          for (int u = 0; u < kExtBatchFwd; ++u) {
            const int e = e0 + u;
            const float we = (e < RISP_MAX_BRANCHES && e < d.K_ext && !(wext[e < RISP_MAX_BRANCHES ? e : 0] < 1e-9f)) ? wext[e < RISP_MAX_BRANCHES ? e : 0] : 0.f;
            Y.b[0] = fmaf(we, E[u][0].x, Y.b[0]); Y.b[1] = fmaf(we, E[u][0].y, Y.b[1]); Y.b[2] = fmaf(we, E[u][0].z, Y.b[2]); Y.b[3] = fmaf(we, E[u][0].w, Y.b[3]);
            Y.g[0] = fmaf(we, E[u][1].x, Y.g[0]); Y.g[1] = fmaf(we, E[u][1].y, Y.g[1]); Y.g[2] = fmaf(we, E[u][1].z, Y.g[2]); Y.g[3] = fmaf(we, E[u][1].w, Y.g[3]);
            Y.r[0] = fmaf(we, E[u][2].x, Y.r[0]); Y.r[1] = fmaf(we, E[u][2].y, Y.r[1]); Y.r[2] = fmaf(we, E[u][2].z, Y.r[2]); Y.r[3] = fmaf(we, E[u][2].w, Y.r[3]);
          }
        }
      }
    } else {
#pragma unroll
      for (int e = 0; e < RISP_MAX_BRANCHES; ++e) {
        if (e < d.K_ext) {
          const float we = wext[e];
          if (!(we < 1e-9f)) {
            Px<NPX> E;
            mix_load<VEC>(E, d.ext[e] + img, HW, i, C);
#pragma unroll
            for (int k = 0; k < NPX; ++k) {
              Y.b[k] = fmaf(we, E.b[k], Y.b[k]); Y.g[k] = fmaf(we, E.g[k], Y.g[k]); Y.r[k] = fmaf(we, E.r[k], Y.r[k]);
            }
          }
        }
      }
    }
    mix_store<VEC>(Y, y + img, HW, i, C);
  }
}

template <int VEC, bool BIG, unsigned SIG>
__global__ void __launch_bounds__(kT, 1)
mixed_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dx,
                 float* __restrict__ partial, long long HW, int C, MixDesc d, const float* __restrict__ params,
                 int pstride, const float* __restrict__ w) {
  constexpr int NPX = MixNpx<VEC>::value;
  const int n = blockIdx.y;
  const float* __restrict__ prow = params + (long long)n * pstride;
  const long long img = (long long)n * C * HW;
  // classical branches j (static index) and materialised branches e (static index) keep separate weights / dot products;
  // the branch number K_cls + e only appears when the partial row is written
  float wk[RISP_MAX_STAGES], dot[RISP_MAX_STAGES], wext[RISP_MAX_BRANCHES], dote[RISP_MAX_BRANCHES];
#pragma unroll
  for (int k = 0; k < RISP_MAX_STAGES; ++k) { wk[k] = (k < d.K_cls) ? w[k] : 0.f; dot[k] = 0.f; }
#pragma unroll
  for (int k = 0; k < RISP_MAX_BRANCHES; ++k) { wext[k] = (k < d.K_ext) ? w[d.K_cls + k] : 0.f; dote[k] = 0.f; }
  float accS[RISP_MAX_STAGES][RISP_SMALL_ACC];
  float2 accB[RISP_BIG_ACC];
#pragma unroll
  for (int s = 0; s < RISP_MAX_STAGES; ++s)
#pragma unroll
    for (int j = 0; j < RISP_SMALL_ACC; ++j) accS[s][j] = 0.f;
#pragma unroll
  for (int k = 0; k < RISP_BIG_ACC; ++k) accB[k] = make_float2(0.f, 0.f);

  const long long nvec = (VEC == 4) ? HW / 4 : (HW + 1) / 2;
  for (long long i = (long long)blockIdx.x * kT + threadIdx.x; i < nvec; i += (long long)gridDim.x * kT) {
    Px<NPX> X, G, DX;
    mix_load<VEC>(X, x + img, HW, i, C);
    mix_load<VEC>(G, dy + img, HW, i, C);
    float4 E[kExtBatch][3];
    auto issue_batch = [&](int e0) {            // first batch before the classical candidates: its latency hides behind them
#pragma unroll
      for (int u = 0; u < kExtBatch; ++u) {
        const int e = (e0 + u < RISP_MAX_BRANCHES) ? e0 + u : 0;
        const bool live = (e0 + u < RISP_MAX_BRANCHES) && (e < d.K_ext) && !(wext[e] < 1e-9f);
        const float* p = d.ext[e] + img + 4 * i;
#pragma unroll
        for (int c = 0; c < 3; ++c) E[u][c] = ld_stream4_if(p + c * HW, live && c < C);
      }
    };
    if (VEC == 4 && d.K_ext > 0) issue_batch(0);
#pragma unroll
    for (int k = 0; k < NPX; ++k) { DX.b[k] = 0.f; DX.g[k] = 0.f; DX.r[k] = 0.f; }
#pragma unroll
    for (int j = 0; j < RISP_MAX_STAGES; ++j) {
      if (MixSig<SIG>::live(d, j) && !(wk[j] < 1e-9f)) {
        Px<NPX> t = X;
        stage_fwd(MixSig<SIG>::op(d, j), MixSig<SIG>::iarg(d, j), prow + d.off[j], t);
        float a = 0.f;
#pragma unroll
        for (int k = 0; k < NPX; ++k) a = fmaf(G.b[k], t.b[k], fmaf(G.g[k], t.g[k], fmaf(G.r[k], t.r[k], a)));
        dot[j] += a;
        Px<NPX> dd = G;
        stage_bwd<NPX, BIG>(MixSig<SIG>::op(d, j), MixSig<SIG>::iarg(d, j), prow + d.off[j], X, t, dd, accS[j], accB);
#pragma unroll
        for (int k = 0; k < NPX; ++k) {
          DX.b[k] = fmaf(wk[j], dd.b[k], DX.b[k]); DX.g[k] = fmaf(wk[j], dd.g[k], DX.g[k]); DX.r[k] = fmaf(wk[j], dd.r[k], DX.r[k]);
        }
      }
    }
    if (VEC == 4) {
#pragma unroll
      for (int e0 = 0; e0 < RISP_MAX_BRANCHES; e0 += kExtBatch) {
        if (e0 < d.K_ext) {                                   // uniform
          if (e0 > 0) issue_batch(e0);
#pragma unroll
          for (int u = 0; u < kExtBatch; ++u) {
            if (e0 + u < RISP_MAX_BRANCHES) {
              float a = 0.f;
              a = fmaf(G.b[0], E[u][0].x, fmaf(G.b[1], E[u][0].y, fmaf(G.b[2], E[u][0].z, fmaf(G.b[3], E[u][0].w, a))));
              a = fmaf(G.g[0], E[u][1].x, fmaf(G.g[1], E[u][1].y, fmaf(G.g[2], E[u][1].z, fmaf(G.g[3], E[u][1].w, a))));
              a = fmaf(G.r[0], E[u][2].x, fmaf(G.r[1], E[u][2].y, fmaf(G.r[2], E[u][2].z, fmaf(G.r[3], E[u][2].w, a))));
              dote[e0 + u] += a;                               // skipped branches loaded zeros
              float* de = d.dext[e0 + u];
              if (de != nullptr && e0 + u < d.K_ext) {         // uniform: d ext_e = w_e * dy, written from the registers
                const float we = wext[e0 + u];
                float* q = de + img + 4 * i;
                st_stream4(q, make_float4(we * G.b[0], we * G.b[1], we * G.b[2], we * G.b[3]));
                if (C > 1) st_stream4(q + HW, make_float4(we * G.g[0], we * G.g[1], we * G.g[2], we * G.g[3]));
                if (C > 2) st_stream4(q + 2 * HW, make_float4(we * G.r[0], we * G.r[1], we * G.r[2], we * G.r[3]));
              }
            }
          }
        }
      }
    } else {
#pragma unroll
      for (int e = 0; e < RISP_MAX_BRANCHES; ++e) {
        if (e < d.K_ext && !(wext[e] < 1e-9f)) {
          Px<NPX> E;
          mix_load<VEC>(E, d.ext[e] + img, HW, i, C);
          float a = 0.f;
#pragma unroll
          for (int k = 0; k < NPX; ++k) a = fmaf(G.b[k], E.b[k], fmaf(G.g[k], E.g[k], fmaf(G.r[k], E.r[k], a)));
          dote[e] += a;
        }
        if (e < d.K_ext && d.dext[e] != nullptr) {
          Px<NPX> DE;
#pragma unroll
          for (int k = 0; k < NPX; ++k) { DE.b[k] = wext[e] * G.b[k]; DE.g[k] = wext[e] * G.g[k]; DE.r[k] = wext[e] * G.r[k]; }
          mix_store<VEC>(DE, d.dext[e] + img, HW, i, C);
        }
      }
    }
    if (dx) mix_store<VEC>(DX, dx + img, HW, i, C);
  }

  // parameter gradients carry the branch weight (d/dp of w_j * f_j)
  float bigw = 0.f;
#pragma unroll
  for (int j = 0; j < RISP_MAX_STAGES; ++j) {
    if (MixSig<SIG>::live(d, j)) {
#pragma unroll
      for (int q = 0; q < RISP_SMALL_ACC; ++q) accS[j][q] *= wk[j];
      if (op_is_big(MixSig<SIG>::op(d, j))) bigw = wk[j];
    }
  }
  __shared__ float red[kT / 32][kMixSlots];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int s = 0; s < RISP_MAX_STAGES; ++s)
#pragma unroll
    for (int j = 0; j < RISP_SMALL_ACC; ++j) {
      float v = warp_sum(accS[s][j]);
      if (lane == 0) red[wid][s * RISP_SMALL_ACC + j] = v;
    }
#pragma unroll
  for (int k = 0; k < RISP_BIG_ACC; ++k) {
    float v0 = BIG ? warp_sum(accB[k].x * bigw) : 0.f, v1 = BIG ? warp_sum(accB[k].y * bigw) : 0.f;
    if (lane == 0) { red[wid][RISP_SLOT_BIG + 2 * k] = v0; red[wid][RISP_SLOT_BIG + 2 * k + 1] = v1; }
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < RISP_MAX_BRANCHES; ++k) red[wid][RISP_NSLOT + k] = 0.f;
  }
  __syncwarp();
#pragma unroll
  for (int k = 0; k < RISP_MAX_STAGES; ++k) {
    float v = warp_sum(dot[k]);
    if (lane == 0 && k < d.K_cls) red[wid][RISP_NSLOT + k] = v;
  }
#pragma unroll
  for (int k = 0; k < RISP_MAX_BRANCHES; ++k) {
    float v = warp_sum(dote[k]);
    if (lane == 0 && k < d.K_ext) red[wid][RISP_NSLOT + d.K_cls + k] = v;
  }
  if (lane == 0) { red[wid][RISP_SLOT_LOSS] = 0.f; red[wid][RISP_SLOT_LOSS + 1] = 0.f; }
  __syncthreads();
  float* out = partial + ((long long)n * gridDim.x + blockIdx.x) * kMixSlots;
  for (int slot = threadIdx.x; slot < kMixSlots; slot += kT) {
    float v = 0.f;
    for (int ww = 0; ww < kT / 32; ++ww) v += red[ww][slot];
    out[slot] = v;
  }
}

// signature of the classical candidate list (0: generic kernel)
static unsigned mix_signature(const MixDesc& d, int C) {
  if (C != 3 || d.K_cls < 1 || d.K_cls > 6) return 0;
  unsigned sig = 0;
  for (int j = 0; j < d.K_cls; ++j) {
    if (d.op[j] == RISP_OP_GTM && d.iarg[j] != 4) return 0;
    sig |= (unsigned)(d.op[j] + 1) << (4 * j);
  }
  return sig;
}

static int mix_blocks(int N, long long HW) {
  long long nvec = (HW % 4 == 0) ? HW / 4 : (HW + 1) / 2;
  long long g = cdiv(nvec, kT);
  long long cap = (long long)sm_count() * 4 / (N > 0 ? N : 1);
  if (cap < 8) cap = 8;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

static int make_mix(MixDesc* d, const char* who, const int* ops, const int* off, const int* iarg, int K_cls,
                    const float* const* ext, int K_ext, int C, int* P_needed) {
  RISP_REQUIRE(K_cls >= 0 && K_cls <= RISP_MAX_STAGES, RISP_E_INVALID, "%s: K_cls %d not in [0,%d]", who, K_cls, RISP_MAX_STAGES);
  RISP_REQUIRE(K_ext >= 0 && K_cls + K_ext <= RISP_MAX_BRANCHES && K_cls + K_ext > 0, RISP_E_INVALID,
               "%s: %d+%d branches not in [1,%d]", who, K_cls, K_ext, RISP_MAX_BRANCHES);
  ChainDesc c;
  int rc = make_chain(&c, ops, off, iarg, K_cls, P_needed);   // same validation rules (<= one big op)
  if (rc != RISP_OK) return rc;
  memset(d, 0, sizeof(*d));
  d->K_cls = K_cls; d->K_ext = K_ext;
  for (int j = 0; j < K_cls; ++j) {
    RISP_REQUIRE(C == 3 || ops[j] == RISP_OP_SKIP, RISP_E_INVALID, "%s: single-plane images only take SKIP branches", who);
    d->op[j] = ops[j]; d->off[j] = off[j]; d->iarg[j] = iarg[j];
  }
  for (int e = 0; e < K_ext; ++e) {
    RISP_REQUIRE(ext && ext[e], RISP_E_INVALID, "%s: null candidate output %d", who, e);
    d->ext[e] = ext[e];
  }
  return RISP_OK;
}

// ---- alpha softmax / prune (K <= 32, one warp) ------------------------------------------------------
__global__ void alpha_prune_fwd_kernel(const float* __restrict__ alpha, float* __restrict__ post,
                                       int* __restrict__ n_pruned, int K, float thr) {
  const int lane = threadIdx.x;
  float a = lane < K ? alpha[lane] : -INFINITY;
  float m = warp_max(a);
  float e = lane < K ? expf(a - m) : 0.f;
  float p = e / warp_sum(e);
  float pmax = warp_max(p);
  bool pruned = (lane < K) && (p < thr * pmax);
  float kept = (lane < K && !pruned) ? p : 0.f;
  float s = warp_sum(kept);
  unsigned np = __popc(__ballot_sync(0xffffffffu, pruned));
  if (lane < K) post[lane] = kept / s;
  if (lane == 0 && n_pruned) *n_pruned = (int)np;
}

__global__ void alpha_prune_bwd_kernel(const float* __restrict__ alpha, const float* __restrict__ dpost,
                                       float* __restrict__ dalpha, int K, float thr) {
  const int lane = threadIdx.x;
  float a = lane < K ? alpha[lane] : -INFINITY;
  float m = warp_max(a);
  float e = lane < K ? expf(a - m) : 0.f;
  float p = e / warp_sum(e);
  float pmax = warp_max(p);
  bool keep = (lane < K) && !(p < thr * pmax);
  float s = warp_sum(keep ? p : 0.f);
  // post_k = keep_k * p_k / s  with s and keep detached  ->  dp_k = keep_k * dpost_k / s ; then softmax bwd
  float dp = keep ? dpost[lane] / s : 0.f;
  float inner = warp_sum(dp * p);
  if (lane < K) dalpha[lane] = p * (dp - inner);
}

// ---- loss -----------------------------------------------------------------------------------------
template <int L1>
__global__ void __launch_bounds__(kT)
loss_fwd_kernel(const float* __restrict__ y, const float* __restrict__ gt, float* __restrict__ partial,
                long long numel, int vec) {
  float acc = 0.f;
  if (vec) {
    for (long long i = (long long)blockIdx.x * kT + threadIdx.x; i < numel / 4; i += (long long)gridDim.x * kT) {
      float4 a = ld_stream4(y + 4 * i), b = ld_stream4(gt + 4 * i);
      float d0 = a.x - b.x, d1 = a.y - b.y, d2 = a.z - b.z, d3 = a.w - b.w;
      acc += L1 ? (fabsf(d0) + fabsf(d1)) + (fabsf(d2) + fabsf(d3)) : fmaf(d0, d0, d1 * d1) + fmaf(d2, d2, d3 * d3);
    }
  } else {
    for (long long i = (long long)blockIdx.x * kT + threadIdx.x; i < numel; i += (long long)gridDim.x * kT) {
      float dd = y[i] - gt[i];
      acc += L1 ? fabsf(dd) : dd * dd;
    }
  }
  __shared__ float red[kT / 32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  acc = warp_sum(acc);
  if (lane == 0) red[wid] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kT / 32; ++w) acc += red[w];
    partial[blockIdx.x] = acc;
  }
}

__global__ void loss_final_kernel(const float* __restrict__ partial, float* __restrict__ out, int B, float scale) {
  float acc = 0.f;
  for (int b = threadIdx.x; b < B; b += 32) acc += partial[b];
  acc = warp_sum(acc);
  if (threadIdx.x == 0) out[0] = acc * scale;
}

template <int L1>
__global__ void __launch_bounds__(kT)
loss_bwd_kernel(const float* __restrict__ y, const float* __restrict__ gt, const float* __restrict__ gscale,
                float* __restrict__ dy, long long numel, float inv_numel, int vec) {
  const float s = gscale[0] * inv_numel * (L1 ? 1.f : 2.f);
  if (vec) {
    for (long long i = (long long)blockIdx.x * kT + threadIdx.x; i < numel / 4; i += (long long)gridDim.x * kT) {
      float4 a = ld_stream4(y + 4 * i), b = ld_stream4(gt + 4 * i);
      float d[4] = {a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) d[k] = L1 ? (d[k] > 0.f ? s : (d[k] < 0.f ? -s : 0.f)) : d[k] * s;
      st_stream4(dy + 4 * i, make_float4(d[0], d[1], d[2], d[3]));
    }
  } else {
    for (long long i = (long long)blockIdx.x * kT + threadIdx.x; i < numel; i += (long long)gridDim.x * kT) {
      float dd = y[i] - gt[i];
      dy[i] = L1 ? (dd > 0.f ? s : (dd < 0.f ? -s : 0.f)) : dd * s;
    }
  }
}

static int loss_blocks(long long numel) {
  long long g = cdiv(numel, (long long)kT * 16);
  long long cap = (long long)sm_count() * 8;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace risp

using namespace risp;

extern "C" int risp_alpha_prune_fwd(const float* alpha, float* post, int* n_pruned, int K, float threshold,
                                    risp_stream_t stream) {
  RISP_REQUIRE(alpha && post && K >= 1 && K <= 32, RISP_E_INVALID, "risp_alpha_prune_fwd: K %d not in [1,32]", K);
  alpha_prune_fwd_kernel<<<1, 32, 0, as_stream(stream)>>>(alpha, post, n_pruned, K, threshold);
  return check_launch("alpha_prune_fwd_kernel");
}

extern "C" int risp_alpha_prune_bwd(const float* alpha, const float* dpost, float* dalpha, int K, float threshold,
                                    risp_stream_t stream) {
  RISP_REQUIRE(alpha && dpost && dalpha && K >= 1 && K <= 32, RISP_E_INVALID, "risp_alpha_prune_bwd: K %d not in [1,32]", K);
  alpha_prune_bwd_kernel<<<1, 32, 0, as_stream(stream)>>>(alpha, dpost, dalpha, K, threshold);
  return check_launch("alpha_prune_bwd_kernel");
}

static int mixed_common_checks(const char* who, const void* x, int N, long long HW, int C) {
  RISP_REQUIRE(x && N > 0 && HW > 0 && N <= 65535, RISP_E_INVALID, "%s: bad tensor arguments", who);
  RISP_REQUIRE(C == 1 || C == 3, RISP_E_INVALID, "%s: C must be 1 (Bayer) or 3 (BGR)", who);
  return RISP_OK;
}

// C is folded into the ABI through HW: callers pass the plane size; images with one plane use
// risp_mixed_*1 entry points below.
static int mixed_fwd_impl(const float* x, float* y, int N, long long HW, int C, const int* cls_ops, const int* cls_off,
                          const int* cls_iarg, int K_cls, const float* params, int param_stride,
                          const float* const* ext, int K_ext, const float* w, risp_stream_t stream) {
  int rc = mixed_common_checks("risp_mixed_fwd", x, N, HW, C);
  if (rc != RISP_OK) return rc;
  RISP_REQUIRE(y && w, RISP_E_INVALID, "risp_mixed_fwd: null y / w");
  MixDesc d;
  int P = 0;
  rc = make_mix(&d, "risp_mixed_fwd", cls_ops, cls_off, cls_iarg, K_cls, ext, K_ext, C, &P);
  if (rc != RISP_OK) return rc;
  RISP_REQUIRE(P == 0 || params, RISP_E_INVALID, "risp_mixed_fwd: params is null");
  bool vec = (HW % 4 == 0) && aligned16(x) && aligned16(y);
  for (int e = 0; e < K_ext; ++e) vec = vec && aligned16(ext[e]);
  dim3 grid(mix_blocks(N, HW), N);
  cudaStream_t st = as_stream(stream);
  if (vec && mix_signature(d, C) == RISP_MIX_SIG_SRGB) mixed_fwd_kernel<4, RISP_MIX_SIG_SRGB><<<grid, kT, 0, st>>>(x, y, HW, C, d, params, param_stride, w);
  else if (vec) mixed_fwd_kernel<4, 0><<<grid, kT, 0, st>>>(x, y, HW, C, d, params, param_stride, w);
  else mixed_fwd_kernel<1, 0><<<grid, kT, 0, st>>>(x, y, HW, C, d, params, param_stride, w);
  return check_launch("mixed_fwd_kernel");
}

static int mixed_bwd_impl(const float* x, const float* dy, float* dx, float* dw, float* dparams, int N, long long HW,
                          int C, const int* cls_ops, const int* cls_off, const int* cls_iarg, int K_cls,
                          const float* params, int param_stride, int P, const float* const* ext, int K_ext,
                          const float* w, void* workspace, size_t workspace_bytes, risp_stream_t stream, float* const* dext = nullptr) {
  int rc = mixed_common_checks("risp_mixed_bwd", x, N, HW, C);
  if (rc != RISP_OK) return rc;
  RISP_REQUIRE(dy && dw && w, RISP_E_INVALID, "risp_mixed_bwd: null dy / dw / w");
  MixDesc d;
  int Pn = 0;
  rc = make_mix(&d, "risp_mixed_bwd", cls_ops, cls_off, cls_iarg, K_cls, ext, K_ext, C, &Pn);
  if (rc != RISP_OK) return rc;
  bool big = false;
  for (int j = 0; j < K_cls; ++j) {
    RISP_REQUIRE(op_has_bwd(cls_ops[j]), RISP_E_UNSUPPORTED, "risp_mixed_bwd: op %d is forward-only", cls_ops[j]);
    big = big || op_is_big(cls_ops[j]);
  }
  RISP_REQUIRE(Pn <= P && (Pn == 0 || (params && dparams)), RISP_E_INVALID, "risp_mixed_bwd: parameter arguments");
  RISP_REQUIRE(param_stride == 0 || param_stride >= P, RISP_E_INVALID, "risp_mixed_bwd: param_stride");
  const int K = K_cls + K_ext;
  size_t need = risp_mixed_bwd_workspace(N, HW, P, K);
  RISP_REQUIRE(workspace && workspace_bytes >= need, RISP_E_WORKSPACE, "risp_mixed_bwd: workspace %zu < %zu", workspace_bytes, need);
  bool vec = (HW % 4 == 0) && aligned16(x) && aligned16(dy) && (!dx || aligned16(dx));
  for (int e = 0; e < K_ext; ++e) {
    vec = vec && aligned16(ext[e]);
    d.dext[e] = dext ? dext[e] : nullptr;
    vec = vec && (!d.dext[e] || aligned16(d.dext[e]));
  }
  const int B = mix_blocks(N, HW);
  dim3 grid(B, N);
  cudaStream_t st = as_stream(stream);
  float* partial = static_cast<float*>(workspace);
#define RISP_MIXB(V, BG, SG) mixed_bwd_kernel<V, BG, SG><<<grid, kT, 0, st>>>(x, dy, dx, partial, HW, C, d, params, param_stride, w)
  if (vec && mix_signature(d, C) == RISP_MIX_SIG_SRGB) RISP_MIXB(4, true, RISP_MIX_SIG_SRGB);
  else if (vec) { if (big) RISP_MIXB(4, true, 0); else RISP_MIXB(4, false, 0); }
  else          { if (big) RISP_MIXB(1, true, 0); else RISP_MIXB(1, false, 0); }
#undef RISP_MIXB
  rc = check_launch("mixed_bwd_kernel");
  if (rc != RISP_OK) return rc;
  // dw[k] = sum over the batch and blocks of the dot products
  short dst[RISP_MAX_BRANCHES], slot[RISP_MAX_BRANCHES];
  for (int k = 0; k < K; ++k) { dst[k] = (short)k; slot[k] = (short)(RISP_NSLOT + k); }
  rc = finalize_partials(partial, dw, N, B, kMixSlots, K, dst, slot, K, 1.f, true, st);
  if (rc != RISP_OK || P == 0) return rc;
  bool shared_row = (param_stride == 0);
  if (cudaMemsetAsync(dparams, 0, sizeof(float) * (size_t)P * (shared_row ? 1 : N), st) != cudaSuccess) {
    set_error("risp_mixed_bwd: memset failed");
    return RISP_E_CUDA;
  }
  ChainDesc c;
  memset(&c, 0, sizeof(c));
  c.S = K_cls;
  for (int j = 0; j < K_cls; ++j) { c.op[j] = cls_ops[j]; c.off[j] = cls_off[j]; c.iarg[j] = cls_iarg[j]; }
  SlotList m;
  chain_slot_list(c, &m);
  return finalize_partials(partial, dparams, N, B, kMixSlots, P, m.dst, m.slot, m.n, 1.f, shared_row, st);
}

extern "C" int risp_mixed_fwd(const float* x, float* y, int N, long long HW, const int* cls_ops, const int* cls_off,
                              const int* cls_iarg, int K_cls, const float* params, int param_stride,
                              const float* const* ext, int K_ext, const float* w, risp_stream_t stream) {
  return mixed_fwd_impl(x, y, N, HW, 3, cls_ops, cls_off, cls_iarg, K_cls, params, param_stride, ext, K_ext, w, stream);
}

extern "C" size_t risp_mixed_bwd_workspace(int N, long long HW, int P, int K) {
  (void)P; (void)K;
  if (N <= 0 || HW <= 0) return 0;
  return (size_t)N * mix_blocks(N, HW) * kMixSlots * sizeof(float);
}

extern "C" int risp_mixed_bwd(const float* x, const float* dy, float* dx, float* dw, float* dparams, int N,
                              long long HW, const int* cls_ops, const int* cls_off, const int* cls_iarg, int K_cls,
                              const float* params, int param_stride, int P, const float* const* ext, int K_ext,
                              const float* w, void* workspace, size_t workspace_bytes, risp_stream_t stream) {
  return mixed_bwd_impl(x, dy, dx, dw, dparams, N, HW, 3, cls_ops, cls_off, cls_iarg, K_cls, params, param_stride, P,
                        ext, K_ext, w, workspace, workspace_bytes, stream);
}

extern "C" int risp_mixed_bwd_dext(const float* x, const float* dy, float* dx, float* dw, float* dparams, float* const* dext,
                                   int N, long long HW, const int* cls_ops, const int* cls_off, const int* cls_iarg, int K_cls,
                                   const float* params, int param_stride, int P, const float* const* ext, int K_ext,
                                   const float* w, void* workspace, size_t workspace_bytes, risp_stream_t stream) {
  return mixed_bwd_impl(x, dy, dx, dw, dparams, N, HW, 3, cls_ops, cls_off, cls_iarg, K_cls, params, param_stride, P,
                        ext, K_ext, w, workspace, workspace_bytes, stream, dext);
}

// single-plane (Bayer-domain) variants: candidates are Skip and materialised tensors
extern "C" int risp_mixed1_fwd(const float* x, float* y, int N, long long HW, int n_skip, const float* const* ext,
                               int K_ext, const float* w, risp_stream_t stream) {
  int ops[RISP_MAX_STAGES] = {0}, off[RISP_MAX_STAGES] = {0}, ia[RISP_MAX_STAGES] = {0};
  RISP_REQUIRE(n_skip >= 0 && n_skip <= RISP_MAX_STAGES, RISP_E_INVALID, "risp_mixed1_fwd: n_skip");
  return mixed_fwd_impl(x, y, N, HW, 1, ops, off, ia, n_skip, nullptr, 0, ext, K_ext, w, stream);
}

extern "C" int risp_mixed1_bwd(const float* x, const float* dy, float* dx, float* dw, int N, long long HW, int n_skip,
                               const float* const* ext, int K_ext, const float* w, void* workspace,
                               size_t workspace_bytes, risp_stream_t stream) {
  int ops[RISP_MAX_STAGES] = {0}, off[RISP_MAX_STAGES] = {0}, ia[RISP_MAX_STAGES] = {0};
  RISP_REQUIRE(n_skip >= 0 && n_skip <= RISP_MAX_STAGES, RISP_E_INVALID, "risp_mixed1_bwd: n_skip");
  return mixed_bwd_impl(x, dy, dx, dw, nullptr, N, HW, 1, ops, off, ia, n_skip, nullptr, 0, 0, ext, K_ext, w, workspace,
                        workspace_bytes, stream);
}

extern "C" size_t risp_loss_workspace(long long numel) { return numel > 0 ? (size_t)loss_blocks(numel) * sizeof(float) : 0; }

extern "C" int risp_loss_fwd(const float* y, const float* gt, float* loss_out, long long numel, int l1, void* workspace,
                             size_t workspace_bytes, risp_stream_t stream) {
  RISP_REQUIRE(y && gt && loss_out && numel > 0, RISP_E_INVALID, "risp_loss_fwd: bad arguments");
  RISP_REQUIRE(workspace && workspace_bytes >= risp_loss_workspace(numel), RISP_E_WORKSPACE, "risp_loss_fwd: workspace too small");
  cudaStream_t st = as_stream(stream);
  int B = loss_blocks(numel);
  int vec = (numel % 4 == 0) && aligned16(y) && aligned16(gt);
  float* partial = static_cast<float*>(workspace);
  if (l1) loss_fwd_kernel<1><<<B, kT, 0, st>>>(y, gt, partial, numel, vec);
  else loss_fwd_kernel<0><<<B, kT, 0, st>>>(y, gt, partial, numel, vec);
  loss_final_kernel<<<1, 32, 0, st>>>(partial, loss_out, B, (float)(1.0 / (double)numel));
  return check_launch("loss_fwd");
}

extern "C" int risp_loss_bwd(const float* y, const float* gt, const float* gscale, float* dy, long long numel, int l1,
                             risp_stream_t stream) {
  RISP_REQUIRE(y && gt && gscale && dy && numel > 0, RISP_E_INVALID, "risp_loss_bwd: bad arguments");
  cudaStream_t st = as_stream(stream);
  int B = loss_blocks(numel);
  int vec = (numel % 4 == 0) && aligned16(y) && aligned16(gt) && aligned16(dy);
  float inv = (float)(1.0 / (double)numel);
  if (l1) loss_bwd_kernel<1><<<B, kT, 0, st>>>(y, gt, gscale, dy, numel, inv, vec);
  else loss_bwd_kernel<0><<<B, kT, 0, st>>>(y, gt, gscale, dy, numel, inv, vec);
  return check_launch("loss_bwd_kernel");
}
