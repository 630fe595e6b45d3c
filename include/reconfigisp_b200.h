/*
 * reconfigisp_b200 -- C ABI of the B200 (sm_100a) ISP hot path.
 *
 * The reference (yuke93/ReconfigISP) is pure Python; the arithmetic of its classical ISP
 * stages lives behind the plugin call  Kernel().run(img, option, params_dict)  of five
 * un-shipped modules (codes/models/modules/tools_origin.py:13-17) and in a handful of
 * in-repo torch expressions.  This header is what an FFI binding for that path binds:
 * plain pointers and sizes, no torch types.  Every entry point
 *   - takes DEVICE pointers (fp32, NCHW planar, contiguous) unless the name ends in _host,
 *   - never allocates: outputs and workspaces are caller-owned (query *_workspace()),
 *   - enqueues on the given cudaStream_t (passed as void*), never synchronises,
 *   - returns RISP_OK or a negative error code and never throws; risp_last_error() has text.
 *
 * Image conventions (SURVEY.md §8a): Bayer = (N,1,H,W) RGGB, R=(0,0) G1=(0,1) G2=(1,0) B=(1,1)
 * (srcnn_demosaic_arch.py:39-42); colour = (N,3,H,W) in B,G,R plane order (tools_origin.py:328-331).
 */
#ifndef RECONFIGISP_B200_H
#define RECONFIGISP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RISP_ABI_VERSION 1

typedef void* risp_stream_t; /* cudaStream_t */

enum risp_status {
  RISP_OK = 0,
  RISP_E_INVALID = -1,     /* bad argument (maps to the reference's assert / ValueError) */
  RISP_E_ALIGN = -2,       /* pointer / extent not aligned as the entry point documents */
  RISP_E_CUDA = -3,        /* a CUDA runtime call failed */
  RISP_E_UNSUPPORTED = -4, /* op has no such direction (maps to NotImplementedError) */
  RISP_E_WORKSPACE = -5    /* workspace too small */
};

int risp_abi_version(void);
const char* risp_last_error(void);
int risp_sm_count(void);
/* number of kernels this library has launched (or recorded into a CUDA graph being captured) so far in this process;
 * bench.py reports launches per step from it */
long long risp_launch_count(void);

/* ---------------------------------------------------------------------------------------
 * Per-pixel stage chain on BGR planes.
 * One launch applies S <= RISP_MAX_STAGES per-pixel stages back to back in registers.
 * With S == 1 it is the drop-in for one plugin call; longer chains are stage fusion for
 * fixed pipelines (isp_universal.py:210-232 runs them as separate full-image passes).
 *
 * Stage parameters are KERNEL-level values (the [0,1]->range mappings of the wrappers,
 * e.g. gain = p*5 tools_origin.py:214, P = p*10-5 :326, stay in the host language):
 * ------------------------------------------------------------------------------------- */
#define RISP_MAX_STAGES 6

enum risp_op {
  RISP_OP_SKIP = 0,      /* Skip                      tools_origin.py:256-262            P=0  */
  RISP_OP_GAMMA = 1,     /* gamma 'manual'            :62-69   y=clamp(x,1e-8,1)^g       P=1  */
  RISP_OP_GAIN = 2,      /* whitebalance 'manual'     :214-221 y_c=x_c*g_c               P=3  */
  RISP_OP_GAIN_CLIP = 3, /* grayworld/whiteworld apply :35-41  y_c=clamp(x_c*g_c,0,1)    P=3  */
  RISP_OP_POLY10 = 4,    /* WbQuadratic               :326-357 y_c=clamp(sum_k P[c][k]phi_k) P=30 */
  RISP_OP_GTM = 5,       /* GtmManual(n_seg=iarg)     :425-438 piecewise-linear curve    P=iarg-1 */
  RISP_OP_CCM = 6,       /* 3x3 colour matrix (north_star extension), clamp [0,1]        P=9  */
  RISP_OP_REINHARD = 7,  /* globaltonemapping 'reinhard' :535  P=(a/Lavg, 1/w^2), fwd only    */
  RISP_OP_CRYSIS = 8,    /* 'crysisengine'            :574     P=(1/lum_adapted), fwd only    */
  RISP_OP_FILMIC = 9,    /* 'filmic'                  :615     P=(exposure, 1/f(w)), fwd only */
  RISP_OP_COUNT = 10
};

/* Chain description, all HOST arrays of length S:
 *   ops[s]       enum risp_op
 *   param_off[s] offset of the stage's first parameter inside one parameter row
 *   iarg[s]      integer argument (n_seg for RISP_OP_GTM, else 0)
 * params: DEVICE, row n at params + n*param_stride; param_stride == 0 shares row 0 across
 * the batch (the reference repeats one vector N times, super_prune...:208-209). */
int risp_chain_fwd(const float* x, float* y, int N, long long HW, const int* ops, const int* param_off,
                   const int* iarg, int S, const float* params, int param_stride, float in_scale,
                   float out_scale, risp_stream_t stream);

/* Kernel-level parameter row of a fixed pipeline from its trainable logits, table[i] = a[i]*sigmoid(logits[i]) + b[i] (the
 * wrappers' range mappings: gain = p*5 tools_origin.py:214, P = p*10-5 :326, gamma / knots = p), and the way back,
 * dlogits[i] = dtable[i]*a[i]*s*(1-s).  All DEVICE arrays of length P. */
int risp_param_table_fwd(const float* logits, const float* a, const float* b, float* table, int P, risp_stream_t stream);
int risp_param_table_bwd(const float* logits, const float* a, const float* dtable, float* dlogits, int P, risp_stream_t stream);

/* Backward of the chain: dx (nullable) and dparams.  dparams is (N,P) when param_stride==P and
 * (1,P) when param_stride==0; it is fully overwritten.  Deterministic (no float atomics).
 * Returns RISP_E_UNSUPPORTED if the chain holds a forward-only op. */
size_t risp_chain_bwd_workspace(int N, long long HW, int P);
int risp_chain_bwd(const float* x, const float* dy, float* dx, float* dparams, int N, long long HW,
                   const int* ops, const int* param_off, const int* iarg, int S, const float* params,
                   int param_stride, int P, void* workspace, size_t workspace_bytes, risp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Bayer-domain ops (bit-exact index work): RGGB pack / unpack and pixel shuffle
 * (srcnn_demosaic_arch.py:39-43, path_14l_bayer_arch.py:71-75, nn.PixelShuffle(2) :48).
 * ------------------------------------------------------------------------------------- */
int risp_pack_rggb(const float* raw, float* packed, int N, int H, int W, risp_stream_t stream);
int risp_unpack_rggb(const float* packed, float* raw, int N, int H, int W, risp_stream_t stream);
/* (N, 4*C, H/2, W/2) <-> (N, C, H, W), channel c*4 + dy*2 + dx  (PixelShuffle(2) and its adjoint) */
int risp_pixel_shuffle2(const float* in, float* out, int N, int C, int H, int W, risp_stream_t stream);
int risp_pixel_unshuffle2(const float* in, float* out, int N, int C, int H, int W, risp_stream_t stream);

/* Demosaic (demosaic.Demosaic().run, tools_origin.py:278-284,462-473,496-507). */
enum risp_demosaic { RISP_DM_NEAREST = 0, RISP_DM_BILINEAR = 1, RISP_DM_MALVAR = 2 };
/* y = clamp_hi? : MALVAR clips to [0, clip_hi] (8-bit output range of the wrapper). H, W even, W%4==0 */
int risp_demosaic_fwd(const float* raw, float* bgr, int N, int H, int W, int kind, float clip_hi,
                      risp_stream_t stream);
/* adjoint: draw = J^T dbgr (for MALVAR the clip mask is recomputed from raw) */
int risp_demosaic_bwd(const float* raw, const float* dbgr, float* draw, int N, int H, int W, int kind,
                      float clip_hi, risp_stream_t stream);

/* Bayer black-level + per-CFA-site gain (north_star extension; black level as in
 * data/preprocessing/generate_rggb2bgr_imgs_SID_Sony.py:50):
 *   y = clamp((max(x - bl, 0) / (1 - bl)) * gain[site], 0, 1);  params row = (bl, gR, gG1, gG2, gB) */
int risp_bayer_blc_wb_fwd(const float* raw, float* out, int N, int H, int W, const float* params,
                          int param_stride, risp_stream_t stream);
size_t risp_bayer_blc_wb_bwd_workspace(int N, int H, int W);
int risp_bayer_blc_wb_bwd(const float* raw, const float* dout, float* draw, float* dparams, int N, int H,
                          int W, const float* params, int param_stride, void* workspace,
                          size_t workspace_bytes, risp_stream_t stream);

/* Device-side input codec (SURVEY.md §8f-4): unsigned 8/16-bit codes -> fp32 code/denom, exactly the
 * host-side normalisation of the reference loaders (x/1023. s7isp_rggb2bgr_dataset.py:123, x/16383.
 * sid_sony_ratio_rggb2bgr_dataset.py:133, gt/255. :134) but after the PCIe hop (5 instead of 16 B/px). */
int risp_decode_codes(const void* src, float* dst, long long n, int bytes_per_code, float denom,
                      risp_stream_t stream);
/* The loader's random crop fused with the decode (sid_sony_ratio_rggb2bgr_dataset.py:109-136: even-aligned crop of the
 * full frame, then /16383): src (planes, H, W) codes on the device, dst (planes, h, w) fp32 = src[:, y0:y0+h, x0:x0+w]/denom.
 * y0, x0 must be even for a Bayer plane (CFA phase); checked when require_even != 0. */
int risp_crop_decode(const void* src, float* dst, int planes, int H, int W, int y0, int x0, int h, int w,
                     int bytes_per_code, float denom, int require_even, risp_stream_t stream);
/* Batched crop + decode from a frame store in HBM: a whole training batch in one launch, the same kernel and division as
 * risp_crop_decode (bit-identical to it and to risp_decode_codes).
 *   raw_store: (F,H,W) unsigned codes of raw_bytes_per_code (1 or 2) bytes.  gt_store: (G,3,H,W) uint8 BGR planes.
 *   pos: DEVICE int32 [B][4] = (raw frame, gt frame, y0, x0), 16-byte aligned; y0 and x0 must be even (CFA phase).
 *   img_out: (B,1,h,w) fp32 = code / white_level.  gt_out: (B,3,h,w) fp32 = code / 255, nullable (then gt_store and G
 *   are not used).
 *   status: DEVICE int32[1]; set to non-zero when a record names a frame outside the store, is odd, or puts the crop
 *   outside the frame.  That record is skipped (its outputs are left as they were); nothing outside the stores is read.
 *   Nothing here reads status or waits for the device: the caller checks it when it chooses to.
 * B * 4 (B without gt_out) must not exceed 65535. */
int risp_sample_crops(const void* raw_store, int raw_bytes_per_code, int F, const unsigned char* gt_store, int G, int H,
                      int W, const int* pos, int B, int h, int w, float white_level, float* img_out, float* gt_out,
                      int* status, risp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Fused fixed pipeline (isp_universal.py:210-232 / origin_universal.py:143-161 as ONE pass):
 *   raw --[blc/wb]--> demosaic(kind) --> per-pixel chain --> y        (16 B/px algorithmic)
 * and the proxy-tuning step (isp_model.py:128-142) without materialising y:
 *   loss = mean((y - gt)^2) ; dparams = d loss / d params              (32 B/px fwd+bwd)
 * ------------------------------------------------------------------------------------- */
int risp_pipeline_fwd(const float* raw, float* y, int N, int H, int W, int dm_kind, float dm_clip_hi,
                      const int* ops, const int* param_off, const int* iarg, int S, const float* params,
                      int param_stride, risp_stream_t stream);
size_t risp_pipeline_step_workspace(int N, int H, int W, int P);
/* loss_out: DEVICE float[1] (sum over all elements / (N*3*H*W)); dparams as in risp_chain_bwd;
 * y_out nullable (written when the caller wants the image as well). */
int risp_pipeline_mse_step(const float* raw, const float* gt, float* y_out, float* loss_out, float* dparams,
                           int N, int H, int W, int dm_kind, float dm_clip_hi, const int* ops,
                           const int* param_off, const int* iarg, int S, const float* params,
                           int param_stride, int P, void* workspace, size_t workspace_bytes,
                           risp_stream_t stream);

/* Same single pass with nn.L1Loss (isp_model.py:44-49: pixel_criterion 'l1'): loss = mean |y - gt|.  Pre-instantiated chain
 * signatures only (RISP_E_UNSUPPORTED otherwise: run demosaic + chain + risp_loss_* instead). */
int risp_pipeline_l1_step(const float* raw, const float* gt, float* y_out, float* loss_out, float* dparams,
                          int N, int H, int W, int dm_kind, float dm_clip_hi, const int* ops,
                          const int* param_off, const int* iarg, int S, const float* params,
                          int param_stride, int P, void* workspace, size_t workspace_bytes,
                          risp_stream_t stream);

/* risp_pipeline_mse_step / risp_pipeline_l1_step on N crops of h x w out of the frame stores of risp_sample_crops, read as
 * codes (5 B/px with a 16-bit raw instead of the 16 B/px of a decoded batch).  Image n is the crop at (pos[n].z, pos[n].w) of
 * raw frame pos[n].x, decoded in registers as code / white_level with the sampler's correctly rounded division, against the
 * same crop of GT frame pos[n].y, decoded as code / 255.  loss_out and dparams are those of risp_pipeline_mse_step /
 * risp_pipeline_l1_step on the batch risp_sample_crops decodes from the same records, bit for bit, with the same dispatch
 * (RISP_FUSED=0 included); no image is written.
 *   Stores: raw (F,H,W) of raw_bytes_per_code (1 or 2) byte codes, gt (G,3,H,W) 8-bit planar, as risp_pipeline_eval_store.
 *   pos: DEVICE int32 [N][4] = (raw frame, GT frame, y0, x0), 16-byte aligned.  A record whose frames lie outside a store,
 *   whose origin is odd or whose crop leaves the frame (the rule of risp_sample_crops) sets *status (DEVICE int32) and adds
 *   nothing to the loss or to any gradient (the normaliser stays N*3*h*w); nothing outside the stores is read.
 *   Geometry: W % 16 == 0 (the stores are read through tensor maps, rows of a 16-byte multiple), 16-byte aligned stores and
 *   pos, w % 4 == 0 and h even; RISP_E_UNSUPPORTED otherwise.  Workspace: risp_pipeline_step_workspace(N, h, w, P). */
int risp_pipeline_mse_step_store(const void* raw_store, int raw_bytes_per_code, int F, const unsigned char* gt_store, int G,
                                 int H, int W, const int* pos, int N, float white_level, int* status, int h, int w,
                                 float* loss_out, float* dparams, int dm_kind, float dm_clip_hi, const int* ops,
                                 const int* param_off, const int* iarg, int S, const float* params, int param_stride, int P,
                                 void* workspace, size_t workspace_bytes, risp_stream_t stream);
int risp_pipeline_l1_step_store(const void* raw_store, int raw_bytes_per_code, int F, const unsigned char* gt_store, int G,
                                int H, int W, const int* pos, int N, float white_level, int* status, int h, int w,
                                float* loss_out, float* dparams, int dm_kind, float dm_clip_hi, const int* ops,
                                const int* param_off, const int* iarg, int S, const float* params, int param_stride, int P,
                                void* workspace, size_t workspace_bytes, risp_stream_t stream);

/* Backward of risp_pipeline_fwd for an upstream gradient dy (N,3,H,W): recomputes the forward from
 * raw in registers (nothing was saved) and reduces d/dparams; 16 B/px.  No gradient w.r.t. raw: the
 * containers never need one (candidate-net weights are frozen, SURVEY.md §3.2).  Workspace as above. */
int risp_pipeline_bwd(const float* raw, const float* dy, float* dparams, int N, int H, int W, int dm_kind,
                      float dm_clip_hi, const int* ops, const int* param_off, const int* iarg, int S,
                      const float* params, int param_stride, int P, void* workspace, size_t workspace_bytes,
                      risp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Evaluation metric of the reference (test.py, test_split.py: tensor2bgr -> psnr per image).  Both images are quantised as
 * tensor2bgr does, q(v) = trunc(clip(fl32(v*255), 0, 255)) (NaN -> 0, the codes of risp_to_u8_hwc), and
 *   sse_out[n] = sum_{c,h,w} (q(y) - q(gt))^2        DEVICE long long[N], exact
 * PSNR_n = 20 log10(255 / sqrt(sse_n / (C*H*W))) is formed on the host (inf when sse_n == 0).
 * ------------------------------------------------------------------------------------- */
/* any fp32 (N,C,H,W) pair, any H and W; one read of each */
int risp_sse_u8(const float* y, const float* gt, long long* sse_out, int N, int C, int H, int W, risp_stream_t stream);
/* The same sum for y = risp_pipeline_fwd(raw, ...) without writing y (16 B/px: raw + gt).  Same arguments and the same
 * dispatch as risp_pipeline_fwd, so the codes are that entry point's codes.  u8_out (nullable, 4-byte aligned) receives the
 * 8-bit image as (N,H,W,3) BGR bytes, the image test.py writes with cv2.imwrite. */
size_t risp_pipeline_eval_workspace(int N, int H, int W);
int risp_pipeline_eval(const float* raw, const float* gt, unsigned char* u8_out, long long* sse_out, int N, int H, int W,
                       int dm_kind, float dm_clip_hi, const int* ops, const int* param_off, const int* iarg, int S,
                       const float* params, int param_stride, void* workspace, size_t workspace_bytes,
                       risp_stream_t stream);
/* risp_pipeline_eval on whole frames of the stores of risp_sample_crops, read as codes (5 B/px with a 16-bit raw): image n
 * is raw frame pos[n].x, decoded in registers as code / white_level with the sampler's correctly rounded division, against
 * the 8-bit planar GT frame pos[n].y, whose codes are compared as they are (a stored code is its own tensor2bgr code).
 * sse_out and u8_out are risp_pipeline_eval's on the batch risp_sample_crops decodes from the same whole-frame records,
 * bit for bit, with the same dispatch (RISP_FUSED=0 included).
 *   pos: DEVICE int32 [N][4] = (raw frame, GT frame, 0, 0), 16-byte aligned.  A record that names a frame outside a store
 *   or a non-zero origin sets *status (DEVICE int32) and adds nothing (its sse_out is 0); nothing outside the stores is read.
 *   H even, W % 4 == 0.  The packed kernels read the stores through tensor maps: where they take the chain, W must be a
 *   multiple of 16 (16-byte rows), else RISP_E_UNSUPPORTED.  Workspace: risp_pipeline_eval_workspace(N, H, W). */
int risp_pipeline_eval_store(const void* raw_store, int raw_bytes_per_code, int F, const unsigned char* gt_store, int G,
                             int H, int W, const int* pos, int N, float white_level, int* status, unsigned char* u8_out,
                             long long* sse_out, int dm_kind, float dm_clip_hi, const int* ops, const int* param_off,
                             const int* iarg, int S, const float* params, int param_stride, void* workspace,
                             size_t workspace_bytes, risp_stream_t stream);

/* Per-image SSIM of the same 8-bit codes (skimage 0.16 compare_ssim(a, b, multichannel=True) with its defaults: uniform 7x7
 * window, sample covariance, K1 = 0.01, K2 = 0.03, data_range 255, a border of 3 pixels cropped).  For every channel and
 * interior pixel (h in [3, H-3), w in [3, W-3)) the 7x7 integer sums Sa, Sb, Saa, Sbb, Sab of the codes give
 *   P1 = 2 Sa Sb, Q1 = Sa^2 + Sb^2, P2 = 2 (49 Sab - Sa Sb), Q2 = 49 (Saa + Sbb) - Sa^2 - Sb^2     exact in int32
 *   S  = (P1 + c1)(P2 + c2) / ((Q1 + c1)(Q2 + c2)),  c1 = 49^2 (0.01*255)^2,  c2 = 49*48 (0.03*255)^2    fp32, rounded
 *   ssim_sum_out[n] = sum_{c,h,w} rint(S * 2^32)         DEVICE long long[N], exact: the same bits on any grid
 * SSIM_n = ssim_sum_out[n] / (2^32 C (H-6)(W-6)) is formed on the host.  Identical images give exactly 1 per pixel, and
 * swapping the operands gives the same bits.  y is fp32 (N,C,H,W) or the 8-bit (N,H,W,C) image of risp_to_u8_hwc /
 * risp_pipeline_eval; gt is fp32 (N,C,H,W).  H, W >= 7 and C (H-6)(W-6) < 2^31.  One read of each operand. */
enum risp_image_layout { RISP_IMG_F32_NCHW = 0, RISP_IMG_U8_NHWC = 1 };
int risp_ssim_u8(const void* y, int y_layout, const float* gt, long long* ssim_sum_out, int N, int C, int H, int W,
                 risp_stream_t stream);
/* The same sums against GT frames of a store: image n of y (C = 3) against the 8-bit planar frame pos[n].y of gt_store
 * (G,3,H,W), whose codes enter as they are -- bit-identical to risp_ssim_u8 with the decoded fp32 GT.  pos: DEVICE int32
 * [N][4] records of risp_pipeline_eval_store; a record whose GT frame lies outside the store or whose origin is not
 * (0, 0) sets *status and adds nothing (its sum is 0). */
int risp_ssim_u8_store(const void* y, int y_layout, const unsigned char* gt_store, int G, const int* pos, int* status,
                       long long* ssim_sum_out, int N, int H, int W, risp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Per-image statistics (grayworld tools_origin.py:35-41, SRCNNRes global features
 * srcnn_res_arch.py:36-40, whiteworld :655-662, conditional-module histogram :120-129).
 * ------------------------------------------------------------------------------------- */
size_t risp_plane_stats_workspace(int planes, long long HW);
/* out: (planes, 3) = min, mean, max of every plane */
int risp_plane_stats(const float* x, float* out, int planes, long long HW, void* workspace,
                     size_t workspace_bytes, risp_stream_t stream);
/* idx: (planes, 2) int32 = row-major position of the FIRST minimum / maximum of every plane -- the pixel that
 * torch.min(x, dim=3) -> torch.min(.., dim=2) (srcnn_res_arch.py:36-40) routes its gradient to; stats from risp_plane_stats */
int risp_plane_argfirst(const float* x, const float* stats, int* idx, int planes, long long HW, risp_stream_t stream);
/* dx (planes, HW) = backward of [min, mean, max]: g (planes, 3) upstream gradients, idx from risp_plane_argfirst */
int risp_plane_stats_bwd(const float* g, const int* idx, float* dx, int planes, long long HW, risp_stream_t stream);
/* out: (N,) mean over pixels of log(1e-6 + lum(scale*x)) for BGR images (reinhard) */
int risp_loglum_mean(const float* x, float* out, int N, long long HW, float scale, void* workspace,
                     size_t workspace_bytes, risp_stream_t stream);
/* torch.histc(plane, bins, 0, 1) per plane; out (planes, bins) float counts */
int risp_histc01(const float* x, float* out, int planes, long long HW, int bins, risp_stream_t stream);
/* exact k-th largest value per plane (radix select); k: DEVICE int64 (planes,), 1-based.
 * workspace >= risp_kth_largest_workspace(planes) */
size_t risp_kth_largest_workspace(int planes);
int risp_kth_largest(const float* x, const long long* k, float* out, int planes, long long HW,
                     void* workspace, size_t workspace_bytes, risp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Stencil stages on BGR images (spatialnoisereduction.run tools_origin.py:696-710,742-751;
 * guided filter / sharpening are north_star extensions).  Shared-memory halo tiles.
 * ------------------------------------------------------------------------------------- */
/* window/sigma_color/sigma_space: DEVICE per-image arrays (window: int32, odd, <= 15) */
/* spatialnoisereduction.run(img, 'fastnlm', {block_size, search_block: IntTensor(N,), decay_factor: Tensor(N,)})
 * (tools_origin.py:785-797): non-local means as defined in oracle/SPEC.md -- s x s search window, b x b patches compared
 * jointly over the 3 channels, w = exp(-mean_sq_diff / h^2), reflect-101 borders.  max_halo >= max_n(b/2 + s/2), <= 16. */
int risp_fastnlm_fwd(const float* x, float* y, int N, int H, int W, const int* block_size, const int* search_block,
                     const float* decay_factor, int max_halo, risp_stream_t stream);

/* max_window: HOST upper bound of window[] (sizes the halo tile); larger device values are clamped */
int risp_bilateral_fwd(const float* x, float* y, int N, int H, int W, const int* window,
                       const float* sigma_color, const float* sigma_space, int max_window,
                       risp_stream_t stream);
int risp_median_fwd(const float* x, float* y, int N, int H, int W, int size, risp_stream_t stream);
int risp_guided_fwd(const float* x, float* y, int N, int H, int W, int radius, float eps, void* workspace,
                    size_t workspace_bytes, risp_stream_t stream);
size_t risp_guided_workspace(int N, int H, int W);
/* unsharp mask, 5x5 binomial: y = clamp(x + amount[n]*(x - blur(x)), 0, 1) */
int risp_sharpen_fwd(const float* x, float* y, int N, int H, int W, const float* amount,
                     risp_stream_t stream);
size_t risp_sharpen_bwd_workspace(int N, int H, int W);
int risp_sharpen_bwd(const float* x, const float* dy, float* dx, float* damount, int N, int H, int W,
                     const float* amount, void* workspace, size_t workspace_bytes, risp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * DARTS mixed-op (super_prune_fifteen_demos_four_bayer_two.py:185-212).
 * ------------------------------------------------------------------------------------- */
#define RISP_MAX_BRANCHES 16
/* softmax(alpha) -> prune (< thr*max -> 0, mask from detached probs) -> / sum.detach()
 * post: (K,) DEVICE; n_pruned: DEVICE int32[1].  All on device: no .item() sync (:193). */
int risp_alpha_prune_fwd(const float* alpha, float* post, int* n_pruned, int K, float threshold,
                         risp_stream_t stream);
int risp_alpha_prune_bwd(const float* alpha, const float* dpost, float* dalpha, int K, float threshold,
                         risp_stream_t stream);

/* y = sum_j w[j]*f_j(x; params) + sum_i w[K_cls+i]*ext_i   on (N,3,HW) images.
 *   cls_ops/cls_off/cls_iarg: K_cls classical single-stage branches evaluated in registers from x
 *   ext: HOST array of K_ext DEVICE pointers to materialised candidate outputs (the CNN candidates)
 *   w: DEVICE (K_cls+K_ext,) post-prune weights; a weight < 1e-9 skips the branch (:197) */
int risp_mixed_fwd(const float* x, float* y, int N, long long HW, const int* cls_ops, const int* cls_off,
                   const int* cls_iarg, int K_cls, const float* params, int param_stride,
                   const float* const* ext, int K_ext, const float* w, risp_stream_t stream);
size_t risp_mixed_bwd_workspace(int N, long long HW, int P, int K);
/* dx (nullable): sum_j w_j J_j^T dy ; dw (K,): <dy, branch output> ; dparams as risp_chain_bwd
 * (already scaled by w_j).  d ext_i = w_i * dy is left to the consumer (pass dy and w_i on). */
int risp_mixed_bwd(const float* x, const float* dy, float* dx, float* dw, float* dparams, int N,
                   long long HW, const int* cls_ops, const int* cls_off, const int* cls_iarg, int K_cls,
                   const float* params, int param_stride, int P, const float* const* ext, int K_ext,
                   const float* w, void* workspace, size_t workspace_bytes, risp_stream_t stream);

/* Same, and the upstream gradients of the materialised candidates leave the same pass: dext is a HOST array of K_ext DEVICE
 * pointers (entries may be NULL); dext[i] receives w[K_cls+i] * dy (N,3,HW).  Saves one 24 B/px kernel per CNN candidate. */
int risp_mixed_bwd_dext(const float* x, const float* dy, float* dx, float* dw, float* dparams, float* const* dext, int N,
                        long long HW, const int* cls_ops, const int* cls_off, const int* cls_iarg, int K_cls,
                        const float* params, int param_stride, int P, const float* const* ext, int K_ext,
                        const float* w, void* workspace, size_t workspace_bytes, risp_stream_t stream);

/* Single-plane (Bayer-domain) mixed-op: n_skip Skip candidates + K_ext materialised candidates
 * (the Bayer step: PathRestore14lBayer + Skip, super_prune...:57-74). */
int risp_mixed1_fwd(const float* x, float* y, int N, long long HW, int n_skip, const float* const* ext,
                    int K_ext, const float* w, risp_stream_t stream);
int risp_mixed1_bwd(const float* x, const float* dy, float* dx, float* dw, int N, long long HW, int n_skip,
                    const float* const* ext, int K_ext, const float* w, void* workspace,
                    size_t workspace_bytes, risp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Loss (nn.MSELoss / nn.L1Loss, darts_model.py:60-65).  loss_out DEVICE float[1].
 * ------------------------------------------------------------------------------------- */
size_t risp_loss_workspace(long long numel);
int risp_loss_fwd(const float* y, const float* gt, float* loss_out, long long numel, int l1, void* workspace,
                  size_t workspace_bytes, risp_stream_t stream);
/* dy = gscale[0] * d mean-loss / dy ;  gscale DEVICE float[1] (upstream gradient) */
int risp_loss_bwd(const float* y, const float* gt, const float* gscale, float* dy, long long numel, int l1,
                  risp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Patch split / merge (utils/util_path_restore.py:47-134) on device, NCHW.
 * ------------------------------------------------------------------------------------- */
/* tiles (T,C,h,w) from one frame (C,H,W); origins ys (ny), xs (nx) HOST int arrays, T = ny*nx */
int risp_whole2patch(const float* frame, float* tiles, int C, int H, int W, int h, int w, const int* ys,
                     int ny, const int* xs, int nx, risp_stream_t stream);
/* frame = sum_t tile_t * mask / count_map, ramp mask (i+1)/(e+1), eh=(h-sh)/2, ew=(w-sw)/2;
 * gather form (no atomics, deterministic).  clip01 != 0 also applies clip(.,0,1) (test_split.py:107) */
int risp_patch2whole(const float* tiles, float* frame, int C, int H, int W, int h, int w, int sh, int sw,
                     const int* ys, int ny, const int* xs, int nx, int clip01, risp_stream_t stream);

/* Same blend with the result also (or only: frame may be NULL) as 8-bit HWC -- `(np.clip(merged, 0, 1) * 255.).astype(np.uint8)`
 * of test_split.py:107 fused into the blend, so the D2H copy of a 12 MP result is 36 MB instead of 144 MB. */
int risp_patch2whole_u8(const float* tiles, float* frame, unsigned char* frame_u8, int C, int H, int W, int h, int w, int sh,
                        int sw, const int* ys, int ny, const int* xs, int nx, risp_stream_t stream);
/* tensor2bgr (utils/util.py:118-135) on the device: (C,H,W) fp32 -> (H,W,C) uint8 = trunc(clip(x*255, 0, 255)) */
int risp_to_u8_hwc(const float* x, unsigned char* out, int C, int H, int W, risp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Dense convolution for the CNN candidates (srcnn_res_arch.py:15-24, srcnn_demosaic_arch.py:14-25,
 * path_14l_bayer_arch.py:6-57, path_14l_bgr_arch.py): NCHW fp32, stride 1, "same" zero padding,
 * K in {1,3,5,9}, exact fp32 accumulation, with the fusions those architectures need.
 *   y = [mask_out > 0] * ( act_out( conv(act_in([mask_in > 0] * x), W) + bias ) + res' )
 * flags: RELU_IN (the leading in-place ReLU of ResidualBlock, path_14l_bayer_arch.py:9-21), RELU_OUT,
 * ADD_RES, RES_RELU (res' = relu(res): the relu-skip quirk).  The masks serve the backward pass.
 * Weights are passed in the prepared layout (Cin, K*K, CoutPad); transpose_flip != 0 prepares the
 * operator of the data gradient (dx = conv(dy, W^T flipped)) from the same nn.Conv2d weight.
 * ------------------------------------------------------------------------------------- */
enum risp_conv_flags { RISP_CONV_RELU_IN = 1, RISP_CONV_RELU_OUT = 2, RISP_CONV_ADD_RES = 4, RISP_CONV_RES_RELU = 8 };
size_t risp_conv2d_prepared_weight_floats(int Cin, int Cout, int K, int transpose_flip);
int risp_conv2d_prepare_weights(const float* weight, float* wk, int Cin, int Cout, int K, int transpose_flip,
                                risp_stream_t stream);
int risp_conv2d_fwd(const float* x, const float* mask_in, const float* wk, const float* bias, const float* res,
                    const float* mask_out, float* y, int N, int Cin, int Cout, int H, int W, int K, int flags,
                    risp_stream_t stream);

/* Weight gradient of the same convolution (proxy fine-tuning, darts_ft_model.py:206-246):
 *   dW[co][ci][ky][kx] = sum dy'[n][co][y][x] * x'[n][ci][y+ky-P][x+kx-P],  dy' = dy*[mask_dy > 0], x' = relu?(x)
 * dweight has the nn.Conv2d layout (Cout,Cin,K,K).  Deterministic (per-block partials + fixed-order finaliser). */
size_t risp_conv2d_bwd_weight_workspace(int Cin, int Cout, int K);
int risp_conv2d_bwd_weight(const float* x, const float* dy, const float* mask_dy, float* dweight, int N, int Cin,
                           int Cout, int H, int W, int K, int relu_in, void* workspace, size_t workspace_bytes,
                           risp_stream_t stream);

/* Tensor-core path of the same convolution: implicit GEMM on tcgen05 (kind::tf32, TMEM accumulators) with a
 * 3-term hi/lo split so the result stays fp32-accurate (<= ~1e-6 relative), on CHANNEL-BLOCKED activations
 * (N, H, C4/4, W, 4) where C4 = channels padded to a multiple of 4 (risp_conv_tc_padded_channels).
 * risp_to_blocked / risp_from_blocked convert from / to planar NCHW.  Same flags and mask semantics as
 * risp_conv2d_fwd; the output goes to the blocked tensor y_blk (required) and, if y_planar is not NULL, is also copied to
 * that planar NCHW tensor. */
int risp_conv_tc_supported(int Cin, int Cout, int K);
int risp_conv_tc_padded_channels(int C);
size_t risp_conv_tc_weight_floats(int Cin, int Cout, int K, int transpose_flip);
int risp_conv_tc_prepare_weights(const float* weight, float* out, int Cin, int Cout, int K, int transpose_flip,
                                 risp_stream_t stream);
int risp_to_blocked(const float* planar, float* blocked, int N, int C, int CG, int H, int W, risp_stream_t stream);
int risp_from_blocked(const float* blocked, float* planar, int N, int C, int CG, int H, int W, risp_stream_t stream);
int risp_conv_tc_fwd(const float* x_blk, const float* mask_in_blk, const float* wprep, const float* bias,
                     const float* res_blk, const float* mask_out_blk, float* y_blk, float* y_planar, int N, int Cin,
                     int Cout, int H, int W, int K, int flags, risp_stream_t stream);
/* The same with a position-dependent bias: bias_tab (N, K*K, pad16(Cout)) is indexed by the border class of the output
 * pixel (class = min(y, PAD) from the top, K-1 - min(H-1-y, PAD) from the bottom, likewise in x; needs H, W >= K-1).
 * This is how SRCNNRes' spatially constant input channels (per-image min/mean/max and parameters broadcast over the
 * frame, srcnn_res_arch.py:36-48) are folded out of its first convolution: their contribution is a per-image bias that
 * only differs where the zero padding cuts taps off.  risp_blocked_class_sums is the backward of that table: the sums
 * of a blocked gradient (masked by [mask > 0] if given) over the pixels of every class, out (N, K, K, CP). */
int risp_conv_tc_fwd_tab(const float* x_blk, const float* mask_in_blk, const float* wprep, const float* bias,
                         const float* bias_tab, const float* res_blk, const float* mask_out_blk, float* y_blk,
                         float* y_planar, int N, int Cin, int Cout, int H, int W, int K, int flags, risp_stream_t stream);
/* the table itself: tab (N, J) = b (J) + feat (N, F) x S (F, J) with J = K*K*pad16(Cout), F <= 32; and d feat = d tab x S^T */
int risp_bias_table_fwd(const float* feat, const float* S, const float* b, float* tab, int N, int F, int J, risp_stream_t stream);
int risp_bias_table_bwd(const float* dtab, const float* S, float* dfeat, int N, int F, int J, risp_stream_t stream);
/* Grouped launches for a BANK of networks with identical layer shapes (the eight SRCNNRes proxies of a supernet step,
 * super_prune_fifteen_demos_four_bayer_two.py:101-171): G <= 8 groups x N_per_group images in ONE launch.  The output,
 * masks and bias table have G*N_per_group images; group g uses the prepared weights at wprep + slots[g]*w_group_floats,
 * the bias at bias + slots[g]*bias_group_floats, S / b of the table at slot slots[g]; with x_shared / res_shared the
 * input / residual have N_per_group images that every group reads.  slots: HOST array of G ints. */
int risp_conv_tc_fwd_grouped(const float* x_blk, const float* mask_in_blk, const float* wprep, const float* bias,
                             const float* bias_tab, const float* res_blk, const float* mask_out_blk, float* y_blk,
                             float* y_planar, int G, int N_per_group, const int* slots, long long w_group_floats,
                             int bias_group_floats, int x_shared, int res_shared, int Cin, int Cout, int H, int W,
                             int K, int flags, risp_stream_t stream);
int risp_bias_table_fwd_grouped(const float* feat, const float* S, const float* b, float* tab, int G, int N_per_group,
                                const int* slots, int F, int J, risp_stream_t stream);
int risp_bias_table_bwd_grouped(const float* dtab, const float* S, float* dfeat, int G, int N_per_group, const int* slots,
                                int F, int J, risp_stream_t stream);
size_t risp_blocked_class_sums_workspace(int N, int C, int H, int K);
int risp_blocked_class_sums(const float* g_blk, const float* mask_blk, float* out, int N, int C, int CP, int H, int W, int K,
                            void* workspace, size_t workspace_bytes, risp_stream_t stream);

/* Diagnostic: cycles to issue / complete `iters` tcgen05 tf32 MMAs (M=128, N=NP, K=8) from one thread with the
 * operand layout of risp_conv_tc_fwd.  out: DEVICE long long[2] = {issue cycles, total cycles}. */
/* Diagnostic: per-phase clock64 timeline of one CTA of the last tensor-core convolution (builds with -DRISP_TC_TRACE only;
 * zeros otherwise).  out_host: HOST long long[16]. */
int risp_debug_tc_trace(long long* out_host);
/* Tuning knob: selects an alternative tile configuration of risp_conv_tc_fwd where one is compiled in (0 = default). */
int risp_debug_tc_variant(int variant);
int risp_debug_mma_rate(long long* out, int NP, int iters, int n_acc, int split3, int a_pw, risp_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Gradient exchange over NVLink peer memory (the all-reduce of module-parameter and architecture-weight gradients:
 * DDP in darts_model.py:31,173; 37 .. 216 floats per backward pass).  Every rank allocates a small buffer with
 * risp_p2p_alloc, the 64-byte IPC handles are exchanged by the host (any transport), peers map them with
 * risp_p2p_open, and risp_p2p_allreduce_mean averages a vector in place: peer stores + epoch flags + a rank-ordered sum
 * in one single-CTA kernel (bit-identical on every rank, CUDA-graph capturable, bounded wait).
 * ------------------------------------------------------------------------------------- */
size_t risp_p2p_buffer_bytes(int world, int cap);
int risp_p2p_alloc(size_t bytes, void** ptr, unsigned char* handle64);
int risp_p2p_open(const unsigned char* handle64, void** peer_ptr);
int risp_p2p_close(void* peer_ptr);
int risp_p2p_free(void* ptr);
int risp_p2p_timeouts(const void* buffer, int world, int cap, unsigned* out_host);
int risp_p2p_allreduce_mean(float* data, int n, void* const* bases, int rank, int world, int cap, int timeout_ms,
                            risp_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RECONFIGISP_B200_H */
