"""CPU oracle for the ReconfigISP hot path  --  TEST INFRASTRUCTURE, NOT PRODUCT.

This file is a plain torch-on-CPU restatement of the arithmetic on the path
`BASELINE.json: north_star` names (the differentiable ISP module stack + the DARTS
mixed-op).  Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s
`cpu_baseline` / `--impl reference` legs may import it, and only as the checker /
the timed CPU baseline.  The product (`reconfigisp_b200/`) never imports it.

Pinning status (SURVEY.md §8c):
  * PINNED against the reference's own code (golden vectors in `tests/golden/`,
    produced by `oracle/gen_golden.py` which imports `/root/reference`):
      wb_quadratic, gtm_manual, skip, fc_params (conditional modules), srcnn_res,
      srcnn_demosaic, path14l_bayer, path14l_bgr, mixed_op (softmax/prune/weighted
      sum), darts hessian formula, whole2patch / patch2whole / create_patch_mask,
      pack_rggb.
  * PARITY UNPINNED (arithmetic lives in the un-shipped `/DATA/ISP_Kernels`,
    `tools_origin.py:8-17`; the definitions below are OUR choices, written down in
    `oracle/SPEC.md`, consistent with every in-repo anchor):
      gamma_manual, wb_manual (the multiply), wb_grayworld, wb_whiteworld,
      demosaic_{nearest,bilinear,laplacian}, tone_{reinhard,crysis,filmic},
      denoise_{bilateral,median}.
  * EXTENSIONS with no reference counterpart (north_star stages; parity to this
    oracle only): black_level, bayer_wb, ccm, guided_filter, sharpen.

Conventions: images fp32 (or fp64 when called with doubles) NCHW; Bayer (N,1,H,W)
RGGB with R=(0,0) G1=(0,1) G2=(1,0) B=(1,1) (`srcnn_demosaic_arch.py:39-42`);
colour (N,3,H,W) in BGR order (`tools_origin.py:328-331`).
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

GAMMA_EPS = 1e-8
DIV_EPS = 1e-6
TONE_PARAM_MIN = 1e-3


# ----------------------------------------------------------------------------------
# Bayer indexing (bit-exact rows)
# ----------------------------------------------------------------------------------
def bayer_masks(H, W, device='cpu'):
    """Boolean masks (R, G1, G2, B), each (H, W).  `srcnn_demosaic_arch.py:39-42`."""
    yy = torch.arange(H, device=device).view(H, 1)
    xx = torch.arange(W, device=device).view(1, W)
    ev_y, ev_x = (yy % 2 == 0), (xx % 2 == 0)
    return ev_y & ev_x, ev_y & ~ev_x, ~ev_y & ev_x, ~ev_y & ~ev_x


def mosaic_bgr(img_bgr):
    """(N,3,H,W) BGR -> (N,1,H,W) RGGB mosaic (sampling; used for synthetic data)."""
    N, _, H, W = img_bgr.shape
    mR, mG1, mG2, mB = bayer_masks(H, W, img_bgr.device)
    b, g, r = img_bgr[:, 0], img_bgr[:, 1], img_bgr[:, 2]
    raw = r * mR + g * (mG1 | mG2) + b * mB
    return raw.unsqueeze(1)


def pack_rggb(x):
    """(N,1,H,W) -> (N,4,H/2,W/2) [R,G1,G2,B].  `path_14l_bayer_arch.py:71-75`."""
    return torch.cat([x[:, :, 0::2, 0::2], x[:, :, 0::2, 1::2],
                      x[:, :, 1::2, 0::2], x[:, :, 1::2, 1::2]], dim=1)


def unpack_rggb(x4):
    """Inverse of pack_rggb == nn.PixelShuffle(2) on 4 channels (`path_14l_bayer_arch.py:48`)."""
    return F.pixel_shuffle(x4, 2)


# ----------------------------------------------------------------------------------
# Per-pixel sRGB ops
# ----------------------------------------------------------------------------------
def gamma_manual(x, gamma):
    """UNPINNED (`tools_origin.py:62-69`).  y = clamp(x, eps, 1) ** gamma, gamma (N,1)."""
    g = gamma.view(-1, 1, 1, 1)
    return torch.clamp(x, GAMMA_EPS, 1.0) ** g


def wb_manual(x, gain):
    """UNPINNED multiply (`tools_origin.py:214-221`).  y_c = x_c * gain_c, gain (N,3) in [0,5]."""
    return x * gain.view(gain.shape[0], 3, 1, 1)


def wb_grayworld(x):
    """UNPINNED (`tools_origin.py:22,35-41`).  gain_c = mean(all)/mean_c; clip [0,1]."""
    m = x.mean(dim=(2, 3))                      # (N,3)
    g = m.mean(dim=1, keepdim=True) / torch.clamp(m, min=DIV_EPS)
    return torch.clamp(x * g.view(-1, 3, 1, 1), 0.0, 1.0)


def wb_quadratic(x, params):
    """PINNED.  `tools_origin.py:313-359`: P = (p*10-5).view(N,3,10);
    out_c = clamp(sum_k P[c,k]*phi_k), phi = [b2,g2,r2,bg,br,gr,b,g,r,1]."""
    P = (params * 10 - 5).view(-1, 3, 10)
    b, g, r = x[:, 0], x[:, 1], x[:, 2]
    phi = torch.stack([b * b, g * g, r * r, b * g, b * r, g * r, b, g, r, torch.ones_like(b)], dim=1)
    out = torch.einsum('nck,nkhw->nchw', P, phi)
    return torch.clamp(out, 0.0, 1.0)


def ccm(x, m):
    """EXTENSION.  3x3 colour-correction matrix (N,9) row-major over BGR, clip [0,1]."""
    M = m.view(-1, 3, 3)
    return torch.clamp(torch.einsum('ncd,ndhw->nchw', M, x), 0.0, 1.0)


def gtm_manual(x, params, n_seg=4):
    """PINNED.  `tools_origin.py:409-440`: knots of batch element 0 only, half-open
    segment tests, pixels outside [0,1) pass through, final clamp."""
    pts = params[0]
    out = x.clone()
    bound = torch.linspace(0, 1, steps=n_seg + 1, dtype=torch.float32).to(x.dtype)
    for k in range(n_seg):
        sx, ex = bound[k], bound[k + 1]
        sy = pts[k - 1] if k > 0 else 0.
        ey = pts[k] if k < n_seg - 1 else 1.
        slope = (ey - sy) / (ex - sx)
        out = torch.where((x >= sx) & (x < ex), (x - sx) * slope + sy, out)
    return torch.clamp(out, 0.0, 1.0)


def gain_clip(x, gain):
    """EXTENSION.  y_c = clamp(x_c * gain_c, 0, 1), gain (N,3)."""
    return torch.clamp(wb_manual(x, gain), 0.0, 1.0)


def pixel_chain(x, stages, p):
    """A fused per-pixel chain (the stage list of `ops.Chain`) with KERNEL-level parameter rows p (N,P) or (1,P), packed
    in stage order: gain / gain_clip (3 gains), poly10 (the 30 coefficients P[c][k] themselves, not the [0,1] logits of
    wb_quadratic), gamma (1), (gtm, n) (n-1 knots, each image's own row: no batch-element-0 quirk), ccm (9), skip (0).
    Runs in the dtype of x; the tests call it in float64 on the kernels' fp32 inputs."""
    N = x.shape[0]
    p = p.expand(N, -1)
    o = 0
    for s in stages:
        name, iarg = (s, 0) if isinstance(s, str) else s
        if name == 'gain':
            x = wb_manual(x, p[:, o:o + 3]); o += 3
        elif name == 'gain_clip':
            x = gain_clip(x, p[:, o:o + 3]); o += 3
        elif name == 'poly10':
            x = wb_quadratic(x, (p[:, o:o + 30] + 5) / 10); o += 30
        elif name == 'gamma':
            x = gamma_manual(x, p[:, o:o + 1]); o += 1
        elif name == 'gtm':
            x = torch.cat([gtm_manual(x[i:i + 1], p[i:i + 1, o:o + iarg - 1], iarg) for i in range(N)]); o += iarg - 1
        elif name == 'ccm':
            x = ccm(x, p[:, o:o + 9]); o += 9
        elif name != 'skip':
            raise ValueError('pixel_chain: no reference for stage %r' % name)
    assert o == p.shape[1], (o, p.shape)
    return x


def _lum(x):
    return 0.114 * x[:, 0] + 0.587 * x[:, 1] + 0.299 * x[:, 2]


def tone_reinhard(x255, white_point, middle_grey):
    """UNPINNED (`tools_origin.py:535-546`), data in [0,255], params (N,) raw in [0,1].
    v = a/Lavg * x01;  y = v (1 + v/w^2) / (1 + v);  Lavg = exp(mean(log(1e-6 + lum)))."""
    x = x255 / 255.0
    lavg = torch.exp(torch.log(_lum(x) + 1e-6).mean(dim=(1, 2)))          # (N,)
    a = torch.clamp(torch.as_tensor(middle_grey, dtype=x.dtype), min=TONE_PARAM_MIN)
    w = torch.clamp(torch.as_tensor(white_point, dtype=x.dtype), min=TONE_PARAM_MIN)
    s = (a / lavg).view(-1, 1, 1, 1)
    v = s * x
    y = v * (1 + v / (w * w).view(-1, 1, 1, 1)) / (1 + v)
    return torch.clamp(y, 0.0, 1.0) * 255.0


def tone_crysis(x255, lum_adapted):
    """UNPINNED (`tools_origin.py:574-584`).  y = 1 - exp(-x01 / l)."""
    x = x255 / 255.0
    l = torch.clamp(torch.as_tensor(lum_adapted, dtype=x.dtype), min=TONE_PARAM_MIN).view(-1, 1, 1, 1)
    return torch.clamp(1 - torch.exp(-x / l), 0.0, 1.0) * 255.0


def _hable(v):
    A, B, C, D, E, Fc = 0.15, 0.50, 0.10, 0.20, 0.02, 0.30
    return (v * (A * v + C * B) + D * E) / (v * (A * v + B) + D * Fc) - E / Fc


def tone_filmic(x255, white_point, exposure_bias):
    """UNPINNED (`tools_origin.py:613-626`).  Hable curve: y = f(e*x01) / f(w)."""
    x = x255 / 255.0
    w = torch.clamp(torch.as_tensor(white_point, dtype=x.dtype), min=TONE_PARAM_MIN).view(-1, 1, 1, 1)
    e = torch.as_tensor(exposure_bias, dtype=x.dtype).view(-1, 1, 1, 1)
    y = _hable(e * x) / _hable(w)
    return torch.clamp(y, 0.0, 1.0) * 255.0


def kth_largest_per_plane(x, k):
    """(N,C,H,W), k (N,) int -> (N,C) k-th largest value of every plane (1-based)."""
    N, C = x.shape[:2]
    flat = x.reshape(N, C, -1)
    srt = torch.sort(flat, dim=2, descending=True).values
    idx = (torch.as_tensor(k).view(N, 1, 1) - 1).expand(N, C, 1)
    return torch.gather(srt, 2, idx).squeeze(2)


def whiteworld_rank(ratio, hw):
    """k = clamp(ceil(ratio * H*W), 1, H*W) computed in float32 like the product does."""
    r = np.asarray(ratio, dtype=np.float32).reshape(-1)
    k = np.ceil(r.astype(np.float32) * np.float32(hw)).astype(np.int64)
    return np.clip(k, 1, hw)


def wb_whiteworld(x255, white_point_ratio):
    """UNPINNED (`tools_origin.py:655-662`).  Per channel: t_c = k-th largest value,
    k = ceil(ratio*HW); y = clip(x * 255 / max(t_c, eps), 0, 255)."""
    N, C, H, W = x255.shape
    k = torch.from_numpy(whiteworld_rank(white_point_ratio, H * W))
    t = kth_largest_per_plane(x255, k)                                      # (N,3)
    g = 255.0 / torch.clamp(t, min=DIV_EPS * 255.0)
    return torch.clamp(x255 * g.view(N, C, 1, 1), 0.0, 255.0)


# ----------------------------------------------------------------------------------
# Demosaic  (UNPINNED; `tools_origin.py:278-284,462-473,496-507`)
# ----------------------------------------------------------------------------------
def demosaic_nearest(raw):
    """(N,1,H,W) -> (N,3,H,W) BGR.  R,B replicated over the 2x2 cell, G from the same row."""
    p = pack_rggb(raw)                                                      # R,G1,G2,B
    up = lambda t: t.repeat_interleave(2, dim=2).repeat_interleave(2, dim=3)
    r, b = up(p[:, 0:1]), up(p[:, 3:4])
    g_top = p[:, 1:2].repeat_interleave(2, dim=3)                           # (N,1,H/2,W)
    g_bot = p[:, 2:3].repeat_interleave(2, dim=3)
    g = torch.stack([g_top, g_bot], dim=3).reshape(raw.shape)
    return torch.cat([b, g, r], dim=1)


def demosaic_bilinear(raw):
    """Standard bilinear CFA interpolation, reflect-101 borders."""
    N, _, H, W = raw.shape
    kg = torch.tensor([[0, 1, 0], [1, 4, 1], [0, 1, 0]], dtype=torch.float64) / 4
    kc = torch.tensor([[1, 2, 1], [2, 4, 2], [1, 2, 1]], dtype=torch.float64) / 4
    # reflect-101 padding preserves the CFA phase, so pad first then mask; the padded
    # image's origin is (-1,-1), so the R/B phases swap in the padded frame
    pad = F.pad(raw, (1, 1, 1, 1), mode='reflect')
    pR, pG1, pG2, pB = bayer_masks(H + 2, W + 2, raw.device)
    mR_p, mG_p, mB_p = pB, (pG1 | pG2), pR
    conv = lambda m, k: F.conv2d(pad * m.to(raw.dtype), k.to(raw.dtype).view(1, 1, 3, 3))
    r, g, b = conv(mR_p, kc), conv(mG_p, kg), conv(mB_p, kc)
    return torch.cat([b, g, r], dim=1)


# Malvar-He-Cutler 5x5 kernels (x8)
_MHC_G_AT_RB = [[0, 0, -1, 0, 0], [0, 0, 2, 0, 0], [-1, 2, 4, 2, -1], [0, 0, 2, 0, 0], [0, 0, -1, 0, 0]]
_MHC_C_ROW = [[0, 0, .5, 0, 0], [0, -1, 0, -1, 0], [-1, 4, 5, 4, -1], [0, -1, 0, -1, 0], [0, 0, .5, 0, 0]]
_MHC_C_DIAG = [[0, 0, -1.5, 0, 0], [0, 2, 0, 2, 0], [-1.5, 0, 6, 0, -1.5], [0, 2, 0, 2, 0], [0, 0, -1.5, 0, 0]]


def demosaic_laplacian(raw, vmax=1.0):
    """Malvar-He-Cutler gradient-corrected linear interpolation, reflect-101 borders,
    result clipped to [0, vmax] (8-bit output range of the wrapper)."""
    N, _, H, W = raw.shape
    dt = raw.dtype
    mR, mG1, mG2, mB = [m.to(dt) for m in bayer_masks(H, W, raw.device)]
    pad = F.pad(raw, (2, 2, 2, 2), mode='reflect')
    k = lambda a: (torch.tensor(a, dtype=torch.float64) / 8).to(dt).view(1, 1, 5, 5)
    f_g = F.conv2d(pad, k(_MHC_G_AT_RB))
    f_row = F.conv2d(pad, k(_MHC_C_ROW))                         # colour neighbours left/right
    f_col = F.conv2d(pad, k(_MHC_C_ROW).transpose(2, 3))         # colour neighbours up/down
    f_diag = F.conv2d(pad, k(_MHC_C_DIAG))
    g = raw * (mG1 + mG2) + f_g * (mR + mB)
    r = raw * mR + f_row * mG1 + f_col * mG2 + f_diag * mB
    b = raw * mB + f_col * mG1 + f_row * mG2 + f_diag * mR
    return torch.clamp(torch.cat([b, g, r], dim=1), 0.0, vmax)


# ----------------------------------------------------------------------------------
# Denoise (UNPINNED; OpenCV semantics, `tools_origin.py:696-710,742-751`)
# ----------------------------------------------------------------------------------
def denoise_bilateral(x, window, sigma_color, sigma_space):
    """(N,3,H,W) any range; window (N,) odd ints, sigmas (N,).  L1 colour distance over
    the 3 channels, circular support r<=window/2, exact exp, reflect-101 borders."""
    N, C, H, W = x.shape
    out = torch.empty_like(x)
    for n in range(N):
        d = int(window[n])
        rad = d // 2
        sc, ss = float(sigma_color[n]), float(sigma_space[n])
        xp = F.pad(x[n:n + 1], (rad,) * 4, mode='reflect')[0]
        num = torch.zeros_like(x[n])
        den = torch.zeros_like(x[n, 0])
        for dy in range(-rad, rad + 1):
            for dx in range(-rad, rad + 1):
                r2 = dy * dy + dx * dx
                if math.sqrt(r2) > rad:
                    continue
                nb = xp[:, rad + dy: rad + dy + H, rad + dx: rad + dx + W]
                dist = (nb - x[n]).abs().sum(dim=0)
                w = torch.exp(-(dist * dist) / (2 * sc * sc)) * math.exp(-r2 / (2 * ss * ss))
                num += w * nb
                den += w
        out[n] = num / den
    return out


def denoise_fastnlm(x, block_size, search_block, decay):
    """UNPINNED (`tools_origin.py:785-797`; definition in SPEC.md).  (N,3,H,W) any range; per-image odd block /
    search sizes, decay h on the data's scale.  Classic non-local means: weights exp(-d2/h^2) with d2 the mean
    squared difference of the b x b patches over the 3 channels; reflect-101 borders."""
    N, C, H, W = x.shape
    out = torch.empty_like(x)
    for n in range(N):
        rb, rs = int(block_size[n]) // 2, int(search_block[n]) // 2
        h = float(decay[n])
        R = rb + rs
        xp = F.pad(x[n:n + 1], (R,) * 4, mode='reflect') if R > 0 else x[n:n + 1]
        num = torch.zeros_like(x[n]); den = torch.zeros_like(x[n, 0])
        ctr = xp[:, :, rs: rs + H + 2 * rb, rs: rs + W + 2 * rb]
        for dy in range(-rs, rs + 1):
            for dx in range(-rs, rs + 1):
                sh = xp[:, :, rs + dy: rs + dy + H + 2 * rb, rs + dx: rs + dx + W + 2 * rb]
                d2 = F.avg_pool2d(((ctr - sh) ** 2).sum(dim=1, keepdim=True), 2 * rb + 1, stride=1)[0, 0] / 3.0
                w = torch.exp(-d2 / (h * h))
                num += w * xp[0, :, R + dy: R + dy + H, R + dx: R + dx + W]
                den += w
        out[n] = num / den
    return out


def denoise_median(x, size):
    """Per-channel k x k median, replicate borders (cv2.medianBlur semantics)."""
    rad = size // 2
    xp = F.pad(x, (rad,) * 4, mode='replicate')
    win = xp.unfold(2, size, 1).unfold(3, size, 1).reshape(*x.shape, size * size)
    return win.sort(dim=-1).values[..., (size * size) // 2]


def median_size_from_param(p0):
    """`tools_origin.py:744`: k = 2*int(p[0]*7)+3 in {3..15} (17 at p==1)."""
    return 2 * int(np.float32(p0) * 7) + 3


def bilateral_window_from_param(p):
    """`tools_origin.py:698` quirk: (p.int()*7)*2+3 -> 3 for p in [0,1), 17 at p==1."""
    return (torch.as_tensor(p).int() * 7) * 2 + 3


# ----------------------------------------------------------------------------------
# Extensions (north_star stages without a reference counterpart)
# ----------------------------------------------------------------------------------
def black_level(raw, bl):
    """`generate_rggb2bgr_imgs_SID_Sony.py:50`: max(x - bl, 0) / (1 - bl), bl (N,1)."""
    b = bl.view(-1, 1, 1, 1)
    return torch.clamp(raw - b, min=0.0) / (1 - b)


def bayer_wb(raw, gains):
    """Per-CFA-site gains (N,4) ordered [R,G1,G2,B]; clip [0,1]."""
    N, _, H, W = raw.shape
    ms = bayer_masks(H, W, raw.device)
    g = sum(m.to(raw.dtype) * gains[:, i].view(N, 1, 1) for i, m in enumerate(ms))
    return torch.clamp(raw * g.unsqueeze(1), 0.0, 1.0)


def _box(x, r):
    C = x.shape[1]
    k = torch.ones(C, 1, 2 * r + 1, 2 * r + 1, dtype=x.dtype) / float((2 * r + 1) ** 2)
    return F.conv2d(F.pad(x, (r,) * 4, mode='reflect'), k, groups=C)


def guided_filter(x, radius, eps):
    """Self-guided filter (He et al.), per channel, box radius r, reflect-101 borders."""
    mean = _box(x, radius)
    var = _box(x * x, radius) - mean * mean
    a = var / (var + eps)
    b = mean - a * mean
    return _box(a, radius) * x + _box(b, radius)


_GAUSS5 = np.outer([1, 4, 6, 4, 1], [1, 4, 6, 4, 1]) / 256.0


def sharpen(x, amount):
    """Unsharp mask with a 5x5 binomial blur: y = clip(x + amount*(x - blur(x)), 0, 1), amount (N,1)."""
    C = x.shape[1]
    k = torch.tensor(_GAUSS5, dtype=x.dtype).view(1, 1, 5, 5).repeat(C, 1, 1, 1)
    blur = F.conv2d(F.pad(x, (2,) * 4, mode='reflect'), k, groups=C)
    return torch.clamp(x + amount.view(-1, 1, 1, 1) * (x - blur), 0.0, 1.0)


# ----------------------------------------------------------------------------------
# Conditional modules (`tools_origin.py:109-163`)
# ----------------------------------------------------------------------------------
def histc_planes(x, bins):
    """(N,3,H,W) -> (N, 3*bins); torch.histc(min=0,max=1) per plane (`tools_origin.py:120-129`)."""
    N, C = x.shape[:2]
    return torch.stack([torch.cat([torch.histc(x[n, c].detach().float(), bins=bins, min=0, max=1)
                                   for c in range(C)]) for n in range(N)])


def fc_params(hist, flat, in_out_channels):
    """PINNED.  `tools_origin.py:131-161`: weights are `.view(in,out)` slices, ReLU between
    layers, + global params, sigmoid."""
    idx, feat = 0, hist
    L = len(in_out_channels) - 1
    for i in range(L):
        ci, co = in_out_channels[i], in_out_channels[i + 1]
        Wm = flat[idx: idx + ci * co].view(ci, co); idx += ci * co
        bv = flat[idx: idx + co]; idx += co
        feat = feat @ Wm + bv
        if i != L - 1:
            feat = torch.relu(feat)
    # quirk kept from the reference (`tools_origin.py:158`): a single element is read
    glob = flat[idx]
    return torch.sigmoid(glob + feat)


# ----------------------------------------------------------------------------------
# CNN candidates (architectures in-repo, weights supplied by caller as state dicts)
# ----------------------------------------------------------------------------------
def srcnn_res(x, params, sd):
    """PINNED.  `srcnn_res_arch.py:27-53`.  sd keys: srcnn.{0,2,4}.{weight,bias}."""
    N, _, H, W = x.shape
    fmin = x.amin(dim=(2, 3)); fmax = x.amax(dim=(2, 3)); fmean = x.mean(dim=3).mean(dim=2)
    feat = torch.cat([fmin, fmean, fmax, params], dim=1).view(N, -1, 1, 1).expand(-1, -1, H, W)
    h = torch.cat([x, feat], dim=1)
    h = torch.relu(F.conv2d(h, sd['srcnn.0.weight'], sd['srcnn.0.bias'], padding=4))
    h = torch.relu(F.conv2d(h, sd['srcnn.2.weight'], sd['srcnn.2.bias'], padding=2))
    h = F.conv2d(h, sd['srcnn.4.weight'], sd['srcnn.4.bias'], padding=2)
    return x + h


def srcnn_demosaic(raw, sd):
    """PINNED.  `srcnn_demosaic_arch.py:27-55` with param_channel == 0."""
    h = pack_rggb(raw)
    h = torch.relu(F.conv2d(h, sd['srcnn.0.weight'], sd['srcnn.0.bias'], padding=4))
    h = torch.relu(F.conv2d(h, sd['srcnn.2.weight'], sd['srcnn.2.bias']))
    h = F.conv2d(h, sd['srcnn.4.weight'], sd['srcnn.4.bias'], padding=2)
    return F.pixel_shuffle(h, 2)


SRCNN_DEMOSAIC_SHAPES = (('srcnn.0.weight', (64, 4, 9, 9)), ('srcnn.0.bias', (64,)),
                         ('srcnn.2.weight', (32, 64, 1, 1)), ('srcnn.2.bias', (32,)),
                         ('srcnn.4.weight', (12, 32, 5, 5)), ('srcnn.4.bias', (12,)))


def demosaicnet_standin_state(seed=4):
    """DemosaicNet (`tools_origin.py:289-310`) is an external network whose weights are not
    shipped.  Stand-in: SRCNNDemosaic architecture, weights N(0,1)*0.05 from a fixed seed."""
    g = torch.Generator().manual_seed(seed)
    return {k: torch.randn(shp, generator=g) * 0.05 for k, shp in SRCNN_DEMOSAIC_SHAPES}


def _path14l_trunk(h, sd, pre):
    h = F.conv2d(h, sd[pre + '0.weight'], sd[pre + '0.bias'], padding=1)
    for i in range(6):
        # quirk: the block starts with an in-place ReLU, so the skip is relu(h)
        # (`path_14l_bayer_arch.py:9-21`)
        s = torch.relu(h)
        t = F.conv2d(s, sd[pre + '1.%d.basic.1.weight' % i], sd[pre + '1.%d.basic.1.bias' % i], padding=1)
        t = F.conv2d(torch.relu(t), sd[pre + '1.%d.basic.3.weight' % i], sd[pre + '1.%d.basic.3.bias' % i], padding=1)
        h = t + s
    return F.conv2d(torch.relu(h), sd[pre + '3.weight'], sd[pre + '3.bias'], padding=1)


def path14l_bayer(raw, sd):
    """PINNED.  `path_14l_bayer_arch.py:59-88` (no global residual)."""
    return F.pixel_shuffle(_path14l_trunk(pack_rggb(raw), sd, 'path_restore_14l.'), 2)


def path14l_bgr(x, sd):
    """PINNED.  `path_14l_bgr_arch.py:56-86` (BGR->RGB, trunk, RGB->BGR)."""
    return _path14l_trunk(x.flip(1), sd, 'path_restore_14l.').flip(1)


# ----------------------------------------------------------------------------------
# Mixed-op (`super_prune_fifteen_demos_four_bayer_two.py:185-212`)
# ----------------------------------------------------------------------------------
def prune_probs(alpha, threshold):
    """PINNED.  Returns (post_probs [differentiable], n_pruned)."""
    probs = torch.softmax(alpha, dim=0)
    det = probs.detach()
    keep = ~(det < threshold * det.max())
    post = probs * keep.to(probs.dtype)
    post = post / post.sum().detach()
    return post, int((~keep).sum())


def mixed_op(outs, alpha, threshold):
    """PINNED.  y = sum_k out_k * post_k, skipping post_k < 1e-9."""
    post, _ = prune_probs(alpha, threshold)
    y = 0
    for o, p in zip(outs, post):
        if p < 1e-9:
            continue
        y = y + o * p
    return y


def darts_hessian(dalpha_pos, dalpha_neg, eps):
    """PINNED quirk.  `darts_model.py:323`: (pos - neg) / 2. * eps."""
    return [(p - n) / 2. * eps for p, n in zip(dalpha_pos, dalpha_neg)]


# ----------------------------------------------------------------------------------
# Patch split / merge (`utils/util_path_restore.py:47-134`), numpy HWC like the reference
# ----------------------------------------------------------------------------------
def create_patch_mask(size, edge):
    h, w = size
    eh, ew = edge
    # the reference computes 1.*(i+1)/(e+1) in float64 then stores float32
    def ramp64(n, e):
        v = np.ones(n, dtype=np.float32)
        for i in range(e):
            v[i] = 1. * (i + 1) / (e + 1)
            v[-1 - i] = 1. * (i + 1) / (e + 1)
        return v
    return np.minimum(ramp64(h, eh)[:, None], ramp64(w, ew)[None, :]).astype(np.float32)


def patch_origins(L, l, s):
    """`util_path_restore.py:88-89`."""
    return list(range(0, L - l, s)) + [L - l]


def whole2patch(img, size, stride):
    h, w = size
    sh, sw = stride
    H, W, C = img.shape
    mask = create_patch_mask((h, w), ((h - sh) // 2, (w - sw) // 2))
    count = np.zeros((H, W), dtype=np.float32)
    patches, pos = [], []
    for y in patch_origins(H, h, sh):
        for x in patch_origins(W, w, sw):
            pos.append([y, x])
            count[y:y + h, x:x + w] += mask
            patches.append(img[y:y + h, x:x + w, :])
    return np.asarray(patches), np.asarray(pos), count


def patch2whole(patches, positions, count_map, stride):
    H, W = count_map.shape
    h, w, C = patches.shape[1:4]
    sh, sw = stride
    mask = create_patch_mask((h, w), ((h - sh) // 2, (w - sw) // 2))[:, :, None]
    image = np.zeros((H, W, C), dtype=np.float32)
    for p, (y, x) in zip(patches, positions):
        image[y:y + h, x:x + w, :] += p * mask
    return image / count_map[:, :, None]


def mse(a, b):
    return ((a - b) ** 2).mean()
