// Packed-fp32 stage arithmetic of the fused raw -> BGR pipeline kernels (risp_fused.cu).
//
// Everything here works on a PAIR of neighbouring pixels held as float2 per channel, so a multiply / add /
// fma of the chain can be one Blackwell packed instruction (FFMA2 / FMUL2 / FADD2: two pixels per issue
// slot); the sites where two scalar instructions are cheaper are listed under "cheapest fp32 form per site".
// Stage parameters are NOT fetched per pixel: a tiny preparation kernel writes the chain's derived
// coefficients into a __constant__ block once per launch and the kernels read them through the
// constant bank -> uniform registers (`FFMA2 R, R.F32x2, UR.F32, R`: the scalar is broadcast to both
// halves by the instruction, so coefficients cost neither vector registers nor splat moves).
//
// Algebraic stage fusion: a diagonal gain directly in front of the 3x10 polynomial (wbmanual ->
// wbquadratic, the head of the all-classical pipeline 11_13_01_14) is folded into the polynomial's
// coefficients, q'[c][i] = q[c][i] * gmon_i(g) with gmon = [gb^2, gg^2, gr^2, gb gg, gb gr, gg gr, gb, gg,
// gr, 1].  The per-pixel work then only accumulates S[c][i] = sum e_c phi_i(x0); both parameter gradients
// are linear in S and are formed once per warp in the epilogue:
//     d/dq[c][i] = gmon_i S[c][i] ,   d/dg_k = sum_{c,i} q[c][i] (d gmon_i / d g_k) S[c][i]
// (Euler's identity for the monomials; no division, exact for g = 0 as well).
//
// Reference semantics: tools_origin.py:48-73 (gamma), :200-225 (wb manual), :313-359 (WbQuadratic),
// :409-440 (GtmManual); un-shipped kernels as defined in oracle/SPEC.md.
#pragma once
#include "risp_common.cuh"
#include "risp_stage.cuh"

namespace risp {
namespace fused {

// ---- effective chain (after folding), shared by the kernels (compile time) and the host / prep kernel ----------
enum { FOP_POLYG = 12 };   // GAIN folded into POLY10; other effective ops reuse enum risp_op

__host__ __device__ constexpr int fop_csize(int op) {   // floats of the stage's block in the constant row (even)
  return (op == RISP_OP_POLY10 || op == FOP_POLYG) ? 40 : (op == RISP_OP_GAMMA) ? 2 : (op == RISP_OP_GAIN) ? 4
         : (op == RISP_OP_GTM) ? 16 : 0;
}
__host__ __device__ constexpr int fop_nacc(int op) {    // float2 accumulators of the stage
  return (op == RISP_OP_POLY10 || op == FOP_POLYG) ? 30 : (op == RISP_OP_GAMMA) ? 1 : (op == RISP_OP_GAIN) ? 3
         : (op == RISP_OP_GTM) ? 4 : 0;
}
__host__ __device__ constexpr bool fop_supported(int op) {
  return op == RISP_OP_GAMMA || op == RISP_OP_GAIN || op == RISP_OP_POLY10 || op == RISP_OP_GTM || op == RISP_OP_SKIP;
}
// output of the stage is guaranteed to lie in [0,1]
__host__ __device__ constexpr bool fop_out01(int op) { return op != RISP_OP_GAIN && op != RISP_OP_SKIP; }

struct EffChain {
  int n;
  int op[RISP_MAX_STAGES];
  int src[RISP_MAX_STAGES];    // index of the stage in the ORIGINAL chain (for POLYG: the polynomial; the gain is src-1)
  int coff[RISP_MAX_STAGES];   // offset of the stage's block in the constant row
  int aoff[RISP_MAX_STAGES];   // offset of the stage's accumulators
  int nacc, ncst;
  bool ok;                     // every op is one the packed path implements
};

__host__ __device__ constexpr EffChain eff_from_ops(const int* ops, const int* iarg, int S) {
  EffChain e{};
  e.ok = (S >= 1 && S <= RISP_MAX_STAGES);
  int s = 0;
  while (s < S && e.ok) {
    int op = ops[s], src = s;
    if (!fop_supported(op) || (op == RISP_OP_GTM && iarg[s] != 4)) { e.ok = false; break; }
    if (op == RISP_OP_GAIN && s + 1 < S && ops[s + 1] == RISP_OP_POLY10) { op = FOP_POLYG; src = s + 1; s += 2; }
    else s += 1;
    e.op[e.n] = op; e.src[e.n] = src; e.coff[e.n] = e.ncst; e.aoff[e.n] = e.nacc;
    e.ncst += fop_csize(op); e.nacc += fop_nacc(op);
    e.n++;
  }
  // the tone curve is implemented for inputs known to lie in [0,1] (it always follows gamma / polynomial in the
  // shipped pipelines); anything else stays on the interpreter kernel
  for (int k = 0; k < e.n; ++k)
    if (e.op[k] == RISP_OP_GTM && (k == 0 || !fop_out01(e.op[k - 1]))) e.ok = false;
  return e;
}

template <unsigned SIG>
constexpr EffChain eff_of_sig() {
  int ops[RISP_MAX_STAGES] = {}, iarg[RISP_MAX_STAGES] = {};
  for (int s = 0; s < Sig<SIG>::count(); ++s) { ops[s] = Sig<SIG>::op_c(s); iarg[s] = 4; }
  return eff_from_ops(ops, iarg, Sig<SIG>::count());
}
template <unsigned SIG>
struct Eff { static constexpr EffChain e = eff_of_sig<SIG>(); };

constexpr int kCRowFloats = 64;   // one parameter row of derived constants (max over signatures: 40+2+4+16 = 62)
constexpr int kCRows = 8;         // rows per slot: per-image parameter rows up to N = 8, else the interpreter kernel runs
constexpr int kCSlots = 16;       // one slot per stream that uses the fused path (stream order makes reuse safe)

#ifdef __CUDACC__
// ---- packed helpers ---------------------------------------------------------------------------------------------
struct P2 { float2 b, g, r; };   // two neighbouring pixels

__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 mul2s(float2 a, float s) { return __fmul2_rn(a, make_float2(s, s)); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 add2s(float2 a, float s) { return __fadd2_rn(a, make_float2(s, s)); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 fma2s(float s, float2 b, float2 c) { return __ffma2_rn(make_float2(s, s), b, c); }
__device__ __forceinline__ float2 fma2ss(float s, float2 b, float c) { return __ffma2_rn(make_float2(s, s), b, make_float2(c, c)); }
__device__ __forceinline__ float2 sat2(float2 a) { return make_float2(__saturatef(a.x), __saturatef(a.y)); }
__device__ __forceinline__ float2 sel2(bool px, bool py, float2 a) { return make_float2(px ? a.x : 0.f, py ? a.y : 0.f); }
__device__ __forceinline__ float2 zero2() { return make_float2(0.f, 0.f); }

// ---- cheapest fp32 form per site of the backward-carrying kernels -------------------------------------------------
// A packed FFMA2 holds the FMA pipe for two cycles, and with vector register pairs as operands it costs more than the two
// scalar FFMA it replaces (profiles/r3_fma_rates.txt, cycles per warp instruction: FFMA2 R,R,R 4.3 against FFMA R,R,R 1.6;
// FFMA2 with a uniform coefficient pair 2.9 against FFMA with a coefficient 0.9-1.1).  So the sites below use scalar
// instructions in the backward-carrying kernels of chains with the 3x10 polynomial (the FMA-bound ones; template flag SC
// where a helper also serves other chains); each -DRISP_FUSED_PACKED_* switch restores the packed form of one site
// (per-site step times on the B200: profiles/r3_ablation.txt -- every site is faster scalar).  The gamma -> tone curve
// step is memory-bound and keeps the packed forms: with them scalar it took 0.1600 instead of 0.1555 ms per 48 MP.
//   * folded accumulators: both pixels of a pair go into ONE sum, acc.x = fma(u.y, v.y, fma(u.x, v.x, acc.x)); acc.y stays
//     the constant 0 (no register), and the epilogue's acc.x + acc.y reduces it unchanged -- the summation order is still
//     fixed, gradients stay bit-reproducible run to run.  Half the accumulator registers: the 37-parameter step kernel
//     fits 168 registers, three one-warp CTAs per SM sub-partition instead of two.
#ifndef RISP_FUSED_PACKED_POLY_FWD
constexpr bool kScalarPolyFwd = true;    // polynomial rows of the channel-major step: FFMA R,UR,R
#else
constexpr bool kScalarPolyFwd = false;
#endif
#ifndef RISP_FUSED_PACKED_S_ACC
constexpr bool kFoldS = true;            // polynomial gradient sums S[c][i] += e_c phi_i
#else
constexpr bool kFoldS = false;
#endif
#ifndef RISP_FUSED_PACKED_GTM_ACC
constexpr bool kFoldGtm = true;          // tone-curve hinge sums A_k
#else
constexpr bool kFoldGtm = false;
#endif
#ifndef RISP_FUSED_PACKED_GAMMA_ACC
constexpr bool kFoldGamma = true;        // gamma exponent sum
#else
constexpr bool kFoldGamma = false;
#endif
#ifndef RISP_FUSED_PACKED_LOSS
constexpr bool kScalarLoss = true;       // loss residual y - t and its sum
#else
constexpr bool kScalarLoss = false;
#endif
template <bool FOLD>
__device__ __forceinline__ void acc_fma(float2& acc, float2 u, float2 v) {     // acc += u * v
  if constexpr (FOLD) acc.x = fmaf(u.y, v.y, fmaf(u.x, v.x, acc.x));
  else acc = fma2(u, v, acc);
}
template <bool FOLD>
__device__ __forceinline__ void acc_add(float2& acc, float2 u) {               // acc += u
  if constexpr (FOLD) acc.x = (acc.x + u.x) + u.y;
  else acc = add2(acc, u);
}

// ---- stage state kept from the forward sweep for the backward sweep --------------------------------------------
struct GammaSaved { P2 x, l2, y; };
struct PolySaved { float2 phi[9]; P2 u, y; };     // phi = b2 g2 r2 bg br gr b g r  (coefficient order of WbQuadratic)
struct GainSaved { P2 x; };
struct GtmSaved { P2 x; float2 hd[3][3]; P2 m; };  // hd[c][k] = x_c - x_{k+1};  m = final-clamp mask (slow path only)

// ---- gamma: y = clamp(x, eps, 1)^gm ------------------------------------------------------------------------------
// RFORM (the stage's input gradient is needed): y = xc * r with r = xc^(gm-1) = ex2((gm-1) lg2 xc).  The backward sweep then
// has d y / d x = gm r without the reciprocal of the plain form (t / x): 2 MUFU per pixel and channel instead of 3.  Opt-in
// (-DRISP_FUSED_RFORM): on the B200 the step kernel got 2 % SLOWER with it (0.294 -> 0.300 ms per 48 MP).
template <bool IN01, bool RFORM = false>
__device__ __forceinline__ float2 gamma_fwd2(float2 x, float gm, float2& l2, float gm1 = 0.f, float2* r = nullptr) {
  float2 xc;
  xc.x = IN01 ? fmaxf(x.x, RISP_GAMMA_EPS) : fminf(fmaxf(x.x, RISP_GAMMA_EPS), 1.f);
  xc.y = IN01 ? fmaxf(x.y, RISP_GAMMA_EPS) : fminf(fmaxf(x.y, RISP_GAMMA_EPS), 1.f);
  l2 = make_float2(lg2_ftz(xc.x), lg2_ftz(xc.y));
  if constexpr (RFORM) {
    const float2 t = mul2s(l2, gm1);
    *r = make_float2(ex2_ftz(t.x), ex2_ftz(t.y));
    return mul2(*r, xc);
  } else {
    const float2 t = mul2s(l2, gm);
    return make_float2(ex2_ftz(t.x), ex2_ftz(t.y));
  }
}
template <bool IN01>
__device__ __forceinline__ P2 gamma_fwd(const P2& x, float gm, GammaSaved& sv) {
  P2 y;
  y.b = gamma_fwd2<IN01>(x.b, gm, sv.l2.b); y.g = gamma_fwd2<IN01>(x.g, gm, sv.l2.g); y.r = gamma_fwd2<IN01>(x.r, gm, sv.l2.r);
  sv.x = x; sv.y = y;
  return y;
}
// d <- dL/dx (WITHOUT the factor gm when DEFER: the caller multiplies the upstream accumulators once at the end);
// acc += d*y*lg2(xc)  (ln 2 applied in the epilogue).  rcp(x) may be inf/NaN where the mask is 0: selected away.
// NOMASK: the caller applies the clamp mask itself (merged with the mask of the stage in front), so v is returned as is.
template <bool IN01, bool NEED_DX, bool DEFER, bool NOMASK = false, bool RFORM = false, bool SC = true>
__device__ __forceinline__ float2 gamma_bwd2(float2 x, float2 y, float2 l2, float2 d, float gm, float2& acc, float2 r = float2()) {
  const float2 t = mul2(d, y);
  acc_fma<kFoldGamma && SC>(acc, t, l2);
  if (!NEED_DX) return zero2();
  float2 v = RFORM ? mul2(d, r) : mul2(t, make_float2(rcp_ftz(x.x), rcp_ftz(x.y)));
  if (!DEFER) v = mul2s(v, gm);
  if (NOMASK) return v;
  const bool mx = IN01 ? (x.x >= RISP_GAMMA_EPS) : (x.x >= RISP_GAMMA_EPS && x.x <= 1.f);
  const bool my = IN01 ? (x.y >= RISP_GAMMA_EPS) : (x.y >= RISP_GAMMA_EPS && x.y <= 1.f);
  return sel2(mx, my, v);
}
template <bool IN01, bool NEED_DX, bool DEFER>
__device__ __forceinline__ P2 gamma_bwd(const GammaSaved& sv, const P2& d, float gm, float2& acc) {
  P2 o;
  o.b = gamma_bwd2<IN01, NEED_DX, DEFER>(sv.x.b, sv.y.b, sv.l2.b, d.b, gm, acc);
  o.g = gamma_bwd2<IN01, NEED_DX, DEFER>(sv.x.g, sv.y.g, sv.l2.g, d.g, gm, acc);
  o.r = gamma_bwd2<IN01, NEED_DX, DEFER>(sv.x.r, sv.y.r, sv.l2.r, d.r, gm, acc);
  return o;
}

// ---- diagonal gain ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ P2 gain_fwd(const P2& x, const float* g, GainSaved& sv) {
  sv.x = x;
  P2 y;
  y.b = mul2s(x.b, g[0]); y.g = mul2s(x.g, g[1]); y.r = mul2s(x.r, g[2]);
  return y;
}
template <bool NEED_DX>
__device__ __forceinline__ P2 gain_bwd(const GainSaved& sv, const P2& d, const float* g, float2* acc) {
  acc[0] = fma2(d.b, sv.x.b, acc[0]); acc[1] = fma2(d.g, sv.x.g, acc[1]); acc[2] = fma2(d.r, sv.x.r, acc[2]);
  P2 o;
  if (NEED_DX) { o.b = mul2s(d.b, g[0]); o.g = mul2s(d.g, g[1]); o.r = mul2s(d.r, g[2]); }
  else { o.b = zero2(); o.g = zero2(); o.r = zero2(); }
  return o;
}

// ---- 3x10 polynomial: u_c = sum_i q[c][i] phi_i, y = clamp(u, 0, 1) ----------------------------------------------------
// constant block: q[3][10] at +0, 2*q[c][0..2] at +30 (for the input gradient of the squares)
__device__ __forceinline__ P2 poly_fwd(const P2& x, const float* q, PolySaved& sv) {
  sv.phi[0] = mul2(x.b, x.b); sv.phi[1] = mul2(x.g, x.g); sv.phi[2] = mul2(x.r, x.r);
  sv.phi[3] = mul2(x.b, x.g); sv.phi[4] = mul2(x.b, x.r); sv.phi[5] = mul2(x.g, x.r);
  sv.phi[6] = x.b; sv.phi[7] = x.g; sv.phi[8] = x.r;
  float2 u[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float2 t = fma2ss(q[c * 10], sv.phi[0], q[c * 10 + 9]);
#pragma unroll
    for (int i = 1; i < 9; ++i) t = fma2s(q[c * 10 + i], sv.phi[i], t);
    u[c] = t;
  }
  sv.u.b = u[0]; sv.u.g = u[1]; sv.u.r = u[2];
  sv.y.b = sat2(u[0]); sv.y.g = sat2(u[1]); sv.y.r = sat2(u[2]);
  return sv.y;
}
// torch.clamp's backward mask is inclusive: u in [0,1]  <=>  sat(u) == u
template <bool NEED_DX>
__device__ __forceinline__ P2 poly_bwd(const PolySaved& sv, const P2& d, const float* q, float2* acc) {
  float2 e[3];
  e[0] = sel2(sv.u.b.x == sv.y.b.x, sv.u.b.y == sv.y.b.y, d.b);
  e[1] = sel2(sv.u.g.x == sv.y.g.x, sv.u.g.y == sv.y.g.y, d.g);
  e[2] = sel2(sv.u.r.x == sv.y.r.x, sv.u.r.y == sv.y.r.y, d.r);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
#pragma unroll
    for (int i = 0; i < 9; ++i) acc_fma<kFoldS>(acc[c * 10 + i], e[c], sv.phi[i]);
    acc_add<kFoldS>(acc[c * 10 + 9], e[c]);
  }
  P2 o;
  if (NEED_DX) {
    float2 dphi[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      // squares use the doubled coefficients so that d(b^2) = b * (2 q) needs no extra multiply
      const float q0 = (i < 3) ? q[30 + i] : q[i], q1 = (i < 3) ? q[33 + i] : q[10 + i], q2 = (i < 3) ? q[36 + i] : q[20 + i];
      dphi[i] = fma2s(q2, e[2], fma2s(q1, e[1], mul2s(e[0], q0)));
    }
    const float2 b = sv.phi[6], g = sv.phi[7], r = sv.phi[8];
    o.b = fma2(b, dphi[0], fma2(g, dphi[3], fma2(r, dphi[4], dphi[6])));
    o.g = fma2(g, dphi[1], fma2(b, dphi[3], fma2(r, dphi[5], dphi[7])));
    o.r = fma2(r, dphi[2], fma2(b, dphi[4], fma2(g, dphi[5], dphi[8])));
  } else { o.b = zero2(); o.g = zero2(); o.r = zero2(); }
  return o;
}

// ---- 4-segment tone curve, input in [0,1] ------------------------------------------------------------------------
// Reference: tools_origin.py:429-435, out = (x - x_k) * slope_k + y_k on the half-open segment [x_k, x_k+1), x_k = k/4;
// x == 1 lies in no segment: the pass-through pixel (out = 1, slope 1, no knot gradient).
// constant block: s0, ds1, ds2, ds3, (1 - s3), slow flag, -, -, a_0..a_3, s_0..s_3   (a_k = y_k - x_k s_k)
//
// Table form (default): the segment of a pixel is looked up instead of being rebuilt from three hinges and four step
// masks.  FFMA.RZ(x, 4, 2^20) leaves floor(4x) in bits 3..5 of the sum (ulp 1/8), LOP3 turns that into the address of an
// 8-byte entry (a_k, s_k) of a 64-byte table in shared memory (entry 4: x == 1 -> pass-through; entry 7: NaN -> NaN),
// one LDS.64 fetches it:  out = s_k x + a_k,  d out / d x = s_k.  3 + 1 instructions per pixel and channel instead of
// 1.5 FADD2 + 3 FMNMX + 2 FFMA2 (forward) and 4 FSET + 2 FFMA2 (slope).  The knot gradients still come from the hinge sums
// A_0 = sum d x, A_k = sum d max(x - x_k, 0), the hinge being ONE saturating add (x - x_k < 1: the upper clamp never acts).
// The inference kernels keep the hinge form: they are bound by the memory system, and the dependent LDS in the middle of
// every pixel's chain costs them 4 % (measured); the backward-carrying kernels are bound by instruction issue.
#ifndef RISP_FUSED_NO_GTM_TABLE
constexpr bool kGtmTable = true;
#else
constexpr bool kGtmTable = false;
#endif
constexpr int kGtmTableBytes = 64;
__device__ __forceinline__ float2 gtm_lookup(float x, uint32_t tbl) {     // tbl: 64-byte aligned shared address
  const uint32_t bits = __float_as_uint(__fmaf_rz(x, 4.f, 1048576.f));
  const uint32_t addr = (bits & 0x38u) | tbl;
  float2 v;
  asm("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
  return v;
}
// one lane fills the table of a tone-curve stage from its constant block
__device__ __forceinline__ void gtm_table_fill(uint32_t tbl, const float* c) {
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float a = (k < 4) ? c[8 + k] : 0.f, s = (k < 4) ? c[12 + k] : 1.f;
    asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(tbl + 8u * k), "f"(a), "f"(s) : "memory");
  }
}
template <bool TABLE>
__device__ __forceinline__ float2 gtm_hinge(float2 x, float2 hd, float xk) {
  if constexpr (TABLE) return make_float2(__saturatef(x.x - xk), __saturatef(x.y - xk));
  else return make_float2(fmaxf(hd.x, 0.f), fmaxf(hd.y, 0.f));
}
// sv: state for the backward sweep -- table form: sv[0] = slope of the pixel's segment; hinge form: sv[k] = x - x_{k+1}
template <bool TABLE>
__device__ __forceinline__ float2 gtm_fwd2(float2 x, const float* c, float2 (&sv)[3], bool slow, float2& mask, uint32_t tbl) {
 if constexpr (TABLE) {
  const float2 e0 = gtm_lookup(x.x, tbl), e1 = gtm_lookup(x.y, tbl);
  sv[0] = make_float2(e0.y, e1.y);
  float2 y;
  if (!slow) {
    y.x = __saturatef(fmaf(e0.y, x.x, e0.x)); y.y = __saturatef(fmaf(e1.y, x.y, e1.x));
  } else {     // some knot outside [0,1]: the final clamp (:438) can be active, keep its mask
    const float2 f = make_float2(fmaf(e0.y, x.x, e0.x), fmaf(e1.y, x.y, e1.x));
    y = sat2(f);
    mask = make_float2((f.x == y.x || x.x >= 1.f) ? 1.f : 0.f, (f.y == y.y || x.y >= 1.f) ? 1.f : 0.f);
  }
 return y;
 } else {
  float2 (&hd)[3] = sv;
  hd[0] = add2s(x, -0.25f); hd[1] = add2s(x, -0.5f); hd[2] = add2s(x, -0.75f);
  float2 f = mul2s(x, c[0]);
  // hinge as ONE saturating add (x - x_k < 1): -DRISP_FUSED_FWD_MAXHINGE restores the packed add + FMNMX form
#ifndef RISP_FUSED_FWD_MAXHINGE
  constexpr bool SATH = true;
#else
  constexpr bool SATH = false;
#endif
  f = fma2s(c[1], gtm_hinge<SATH>(x, hd[0], 0.25f), f);
  f = fma2s(c[2], gtm_hinge<SATH>(x, hd[1], 0.5f), f);
  const float2 h3 = gtm_hinge<SATH>(x, hd[2], 0.75f);
  float2 y;
  if (!slow) {
    y.x = __saturatef(fmaf(c[3], h3.x, f.x)); y.y = __saturatef(fmaf(c[3], h3.y, f.y));
  } else {     // some knot outside [0,1]: the final clamp (:438) can be active, keep its mask
    f = fma2s(c[3], h3, f);
    y = sat2(f);
    mask = make_float2((f.x == y.x || x.x >= 1.f) ? 1.f : 0.f, (f.y == y.y || x.y >= 1.f) ? 1.f : 0.f);
  }
  return y;
 }
}
template <bool TABLE>
__device__ __forceinline__ P2 gtm_fwd(const P2& x, const float* c, GtmSaved& sv, bool slow, uint32_t tbl) {
  sv.x = x;
  P2 y;
  y.b = gtm_fwd2<TABLE>(x.b, c, sv.hd[0], slow, sv.m.b, tbl); y.g = gtm_fwd2<TABLE>(x.g, c, sv.hd[1], slow, sv.m.g, tbl);
  y.r = gtm_fwd2<TABLE>(x.r, c, sv.hd[2], slow, sv.m.r, tbl);
  return y;
}
// accumulates A_0 = sum d x, A_k = sum d max(x - x_k, 0); the knot gradients are the second differences
// 4 (A_{j-1} - 2 A_j + A_{j+1}) (hat basis = second difference of hinges; A_4 = 0 on [0,1]), formed in the epilogue.
template <bool NEED_DX, bool SC = true>
__device__ __forceinline__ float2 gtm_bwd2(float2 x, const float2 (&sv)[3], float2 d, const float* c, float2* acc) {
  acc_fma<kFoldGtm && SC>(acc[0], d, x);
 if constexpr (kGtmTable) {
#pragma unroll
  for (int k = 0; k < 3; ++k) acc_fma<kFoldGtm && SC>(acc[k + 1], d, gtm_hinge<true>(x, x, 0.25f * (float)(k + 1)));
  if (!NEED_DX) return zero2();
  return mul2(d, sv[0]);
 } else {
  const float2 (&hd)[3] = sv;
  float2 slope = make_float2(c[0], c[0]);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float2 st = make_float2(hd[k].x >= 0.f ? 1.f : 0.f, hd[k].y >= 0.f ? 1.f : 0.f);
    acc_fma<kFoldGtm && SC>(acc[k + 1], d, gtm_hinge<false>(x, hd[k], 0.f));
    if (NEED_DX) slope = fma2s(c[k + 1], st, slope);
  }
  if (!NEED_DX) return zero2();
  slope = fma2s(c[4], make_float2(x.x >= 1.f ? 1.f : 0.f, x.y >= 1.f ? 1.f : 0.f), slope);   // x == 1: slope -> 1
  return mul2(d, slope);
 }
}
template <bool NEED_DX>
__device__ __forceinline__ P2 gtm_bwd(const GtmSaved& sv, const P2& d0, const float* c, float2* acc, bool slow) {
  P2 d = d0;
  if (slow) { d.b = mul2(d.b, sv.m.b); d.g = mul2(d.g, sv.m.g); d.r = mul2(d.r, sv.m.r); }
  P2 o;
  o.b = gtm_bwd2<NEED_DX>(sv.x.b, sv.hd[0], d.b, c, acc); o.g = gtm_bwd2<NEED_DX>(sv.x.g, sv.hd[1], d.g, c, acc);
  o.r = gtm_bwd2<NEED_DX>(sv.x.r, sv.hd[2], d.r, c, acc);
  return o;
}
#endif  // __CUDACC__

}  // namespace fused
}  // namespace risp
