"""torch.autograd wrappers over the C ABI (include/reconfigisp_b200.h).

PyTorch is plumbing here: it owns device memory, streams and the autograd tape; every
arithmetic step on an image happens in the hand-written sm_100a kernels.  All ops take
CUDA fp32 NCHW tensors and raise on anything else (no CPU / eager fallback).
"""
import torch

from . import _lib as L

OP = {k[len('RISP_OP_'):].lower(): v for k, v in L.ENUMS.items() if k.startswith('RISP_OP_') and k != 'RISP_OP_COUNT'}
DM = {'nearest': L.ENUMS['RISP_DM_NEAREST'], 'bilinear': L.ENUMS['RISP_DM_BILINEAR'], 'malvar': L.ENUMS['RISP_DM_MALVAR'],
      'laplacian': L.ENUMS['RISP_DM_MALVAR']}
MAX_STAGES = L.ENUMS['RISP_MAX_STAGES']
_NPARAM = {'skip': 0, 'gamma': 1, 'gain': 3, 'gain_clip': 3, 'poly10': 30, 'ccm': 9, 'reinhard': 2, 'crysis': 1,
           'filmic': 2}
FWD_ONLY = ('reinhard', 'crysis', 'filmic')
BIG = ('poly10', 'ccm')


def n_params(op, iarg=0):
    return iarg - 1 if op == 'gtm' else _NPARAM[op]


def _img(t, C=None):
    if torch.is_tensor(t) and not t.is_cuda:
        raise RuntimeError('reconfigisp_b200 ops run on CUDA tensors only (no CPU fallback); got a %s tensor' % t.device)
    if not (torch.is_tensor(t) and t.is_cuda and t.dtype == torch.float32 and t.dim() == 4):
        raise ValueError('expected a CUDA fp32 NCHW tensor, got %s' % (type(t).__name__ if not torch.is_tensor(t)
                                                                      else (t.device, t.dtype, tuple(t.shape)),))
    if C is not None and t.shape[1] != C:
        raise ValueError('expected %d channels, got %d' % (C, t.shape[1]))
    return t.contiguous()


class Chain:
    """A fused sequence of per-pixel stages: [(op_name, iarg)], parameters packed row-wise."""

    def __init__(self, stages):
        stages = [(s, 0) if isinstance(s, str) else tuple(s) for s in stages]
        self.names = [s for s, _ in stages]
        self.iargs = [i for _, i in stages]
        self.counts = [n_params(s, i) for s, i in stages]
        self.offsets, off = [], 0
        for c in self.counts:
            self.offsets.append(off)
            off += c
        self.P = off
        self.S = len(stages)
        if self.S > MAX_STAGES:
            raise ValueError('a fused chain holds at most %d stages' % MAX_STAGES)
        if sum(n in BIG for n in self.names) > 1:
            raise ValueError('at most one poly10/ccm stage per fused chain')
        self.differentiable = not any(n in FWD_ONLY for n in self.names)
        self._ops = L.iarr([OP[n] for n in self.names])
        self._off = L.iarr(self.offsets)
        self._iarg = L.iarr(self.iargs)

    def desc(self):
        return self._ops, self._off, self._iarg, self.S


_FUSED_SIGNATURES = (('gain', 'poly10', 'gamma', 'gtm'), ('gamma', 'poly10', 'gain'), ('gamma', 'poly10'), ('gamma', 'gtm'))


def fused_chain_supported(chain):
    """True when the packed single-pass kernels (csrc/risp_fused.cu) are instantiated for this chain: the sRGB tails of the
    shipped pipelines (11_13_01_14, 01_13_11, 01_13, 01_14; 4-segment tone curve)."""
    return tuple(chain.names) in _FUSED_SIGNATURES and all(i == 4 for n, i in zip(chain.names, chain.iargs) if n == 'gtm')


def _param_table(params, N, P):
    """(N,P) or (1,P)/(P,) -> contiguous table and the ABI row stride (0 = shared row)."""
    if P == 0:
        return None, 0
    if params.dim() == 1:
        params = params.view(1, -1)
    assert params.shape[1] == P, 'chain needs %d parameters per row, got %d' % (P, params.shape[1])
    assert params.shape[0] in (1, N), 'parameter rows must be 1 or the batch size'
    params = params.contiguous().float()
    return params, (0 if params.shape[0] == 1 else P)


class _ChainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, params, chain, in_scale, out_scale):
        x = _img(x, 3)
        N, _, H, W = x.shape
        tab, stride = _param_table(params, N, chain.P) if chain.P else (None, 0)
        y = torch.empty_like(x)
        L.call('risp_chain_fwd', L.ptr(x), L.ptr(y), N, H * W, *chain.desc(), L.ptr(tab), stride,
               float(in_scale), float(out_scale), L.stream())
        ctx.chain, ctx.stride, ctx.scales = chain, stride, (in_scale, out_scale)
        ctx.pshape = None if params is None else params.shape
        ctx.save_for_backward(x, tab)
        return y

    @staticmethod
    def backward(ctx, dy):
        chain = ctx.chain
        if not chain.differentiable:
            raise NotImplementedError('chain %s holds a forward-only (Origin*) stage' % chain.names)
        if ctx.scales != (1.0, 1.0):
            raise NotImplementedError('backward of a scaled chain is not provided')
        x, tab = ctx.saved_tensors
        N, _, H, W = x.shape
        dy = _img(dy, 3)
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        P = chain.P
        dpar = torch.empty((1 if ctx.stride == 0 else N, P), device=x.device, dtype=torch.float32) if P else None
        ws = L.workspace(L.size('risp_chain_bwd_workspace', N, H * W, P), x.device)
        L.call('risp_chain_bwd', L.ptr(x), L.ptr(dy), L.ptr(dx), L.ptr(dpar), N, H * W, *chain.desc(), L.ptr(tab),
               ctx.stride, P, L.ptr(ws), ws.numel() * 4, L.stream())
        if dpar is not None:
            dpar = dpar.view(ctx.pshape)
        return dx, dpar, None, None, None


def chain_apply(x, chain, params=None, in_scale=1.0, out_scale=1.0):
    """y = stages(x).  params: (N,P) | (1,P) | (P,) kernel-level parameters (or None when P == 0)."""
    if chain.S == 0 or all(n == 'skip' for n in chain.names):
        if in_scale == 1.0 and out_scale == 1.0:
            return x
    return _ChainFn.apply(x, params, chain, float(in_scale), float(out_scale))


_SINGLE = {}


def _single(op, iarg=0):
    key = (op, iarg)
    if key not in _SINGLE:
        _SINGLE[key] = Chain([(op, iarg)])
    return _SINGLE[key]


def gamma(x, g): return chain_apply(x, _single('gamma'), g)
def gain(x, g): return chain_apply(x, _single('gain'), g)
def gain_clip(x, g): return chain_apply(x, _single('gain_clip'), g)
def poly10(x, coef): return chain_apply(x, _single('poly10'), coef)
def ccm(x, m): return chain_apply(x, _single('ccm'), m)
def gtm(x, knots, n_seg=4): return chain_apply(x, _single('gtm', n_seg), knots)


# ---- statistics ---------------------------------------------------------------------------------
def plane_stats(x):
    """(N,C,H,W) -> (N,C,3) [min, mean, max] per plane (no autograd)."""
    x = _img(x)
    N, C, H, W = x.shape
    out = torch.empty((N, C, 3), device=x.device, dtype=torch.float32)
    ws = L.workspace(L.size('risp_plane_stats_workspace', N * C, H * W), x.device)
    L.call('risp_plane_stats', L.ptr(x), L.ptr(out), N * C, H * W, L.ptr(ws), ws.numel() * 4, L.stream())
    return out


class _PlaneStats3Fn(torch.autograd.Function):
    """(N,C,H,W) -> (N, 3C) = [min_c | mean_c | max_c] per image, the global features of SRCNNRes (srcnn_res_arch.py:36-40).
    Backward: the mean spreads evenly; min / max send their gradient to the FIRST pixel (row-major) that attains them -- what
    `torch.min(x, dim=3)` followed by `torch.min(.., dim=2)` does on the CPU reference."""

    @staticmethod
    def forward(ctx, x):
        x = _img(x)
        N, C, H, W = x.shape
        st = plane_stats(x)                                            # (N,C,3)
        idx = torch.empty((N * C, 2), device=x.device, dtype=torch.int32)
        L.call('risp_plane_argfirst', L.ptr(x), L.ptr(st), L.ptr(idx), N * C, H * W, L.stream())
        ctx.save_for_backward(idx)
        ctx.shape = (N, C, H, W)
        return st.permute(0, 2, 1).reshape(N, 3 * C)

    @staticmethod
    def backward(ctx, g):
        idx, = ctx.saved_tensors
        N, C, H, W = ctx.shape
        gp = g.reshape(N, 3, C).permute(0, 2, 1).contiguous()          # (N,C,3) like the statistics
        dx = torch.empty((N, C, H, W), device=g.device, dtype=torch.float32)
        L.call('risp_plane_stats_bwd', L.ptr(gp), L.ptr(idx), L.ptr(dx), N * C, H * W, L.stream())
        return dx


def plane_stats3(x):
    return _PlaneStats3Fn.apply(x)


def loglum_mean(x, scale=1.0):
    x = _img(x, 3)
    N, _, H, W = x.shape
    out = torch.empty((N,), device=x.device, dtype=torch.float32)
    ws = L.workspace(L.size('risp_plane_stats_workspace', N, H * W), x.device)
    L.call('risp_loglum_mean', L.ptr(x), L.ptr(out), N, H * W, float(scale), L.ptr(ws), ws.numel() * 4, L.stream())
    return out


def histc01(x, bins):
    """torch.histc(plane, bins, 0, 1) for every plane, on the device: (N,C,H,W) -> (N, C*bins)."""
    x = _img(x)
    N, C, H, W = x.shape
    out = torch.empty((N, C * bins), device=x.device, dtype=torch.float32)
    L.call('risp_histc01', L.ptr(x.detach()), L.ptr(out), N * C, H * W, int(bins), L.stream())
    return out


def kth_largest(x, k):
    """Exact k-th largest value of every plane; k: int64 tensor (N,) or (N,C), 1-based."""
    x = _img(x)
    N, C, H, W = x.shape
    k = k.to(device=x.device, dtype=torch.int64)
    k = (k.view(N, 1).expand(N, C) if k.numel() == N else k.view(N, C)).contiguous()
    out = torch.empty((N, C), device=x.device, dtype=torch.float32)
    ws = L.workspace(L.size('risp_kth_largest_workspace', N * C), x.device)
    L.call('risp_kth_largest', L.ptr(x), L.ptr(k), L.ptr(out), N * C, H * W, L.ptr(ws), ws.numel() * 4, L.stream())
    return out


class _GrayworldFn(torch.autograd.Function):
    """y = clamp(x * g, 0, 1), g_c = mean(all)/mean_c  (oracle/SPEC.md; tools_origin.py:22-45).
    Backward = one chain backward (dx_local, dg) + the rank-1 term through the means."""

    @staticmethod
    def forward(ctx, x):
        x = _img(x, 3)
        m = plane_stats(x)[..., 1]                                   # (N,3)
        mc = torch.clamp(m, min=1e-6)
        g = (m.mean(dim=1, keepdim=True) / mc).contiguous()
        y = _ChainFn.apply(x, g, _single('gain_clip'), 1.0, 1.0)
        ctx.save_for_backward(x, g, m)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, g, m = ctx.saved_tensors
        N, _, H, W = x.shape
        dy = _img(dy, 3)
        ch = _single('gain_clip')
        dx = torch.empty_like(x)
        dg = torch.empty((N, 3), device=x.device, dtype=torch.float32)
        ws = L.workspace(L.size('risp_chain_bwd_workspace', N, H * W, 3), x.device)
        L.call('risp_chain_bwd', L.ptr(x), L.ptr(dy), L.ptr(dx), L.ptr(dg), N, H * W, *ch.desc(), L.ptr(g), 3, 3,
               L.ptr(ws), ws.numel() * 4, L.stream())
        # g_c = mbar / max(m_c, eps), mbar = mean_c m_c  ->  dL/dm_j = sum_c dg_c/(3 mc_c) - dg_j mbar/mc_j^2 [m_j >= eps]
        mc = torch.clamp(m, min=1e-6)
        mbar = m.mean(dim=1, keepdim=True)
        dm = (dg / mc).sum(dim=1, keepdim=True) / 3.0 - dg * mbar / (mc * mc) * (m >= 1e-6).float()
        # rank-1 term: every pixel of plane j receives dm_j / (H*W); applied with one more chain pass
        dx = _add_plane_constant(dx, dm / float(H * W))
        return dx


def _add_plane_constant(x, c):
    """x[n,ch] += c[n,ch] in place (tiny torch op on a (N,3,1,1) broadcast -> one elementwise kernel)."""
    return x.add_(c.view(c.shape[0], c.shape[1], 1, 1))


def grayworld(x):
    return _GrayworldFn.apply(x)


# ---- tone operators (forward-only Origin* stages) ---------------------------------------------------
def _hable(v):
    A, B, C, D, E, F = 0.15, 0.50, 0.10, 0.20, 0.02, 0.30
    return (v * (A * v + C * B) + D * E) / (v * (A * v + B) + D * F) - E / F


def tone_reinhard(x, white_point, middle_grey, data_scale=1.0):
    """x in [0, data_scale]; params (N,) device tensors in [0,1]  (tools_origin.py:513-550)."""
    x = _img(x.detach(), 3)
    lavg = torch.exp(loglum_mean(x, 1.0 / data_scale))
    a = torch.clamp(middle_grey.float(), min=1e-3)
    w = torch.clamp(white_point.float(), min=1e-3)
    p = torch.stack([a / lavg, 1.0 / (w * w)], dim=1)
    return chain_apply(x, _single('reinhard'), p, 1.0 / data_scale, data_scale)


def tone_crysis(x, lum_adapted, data_scale=1.0):
    p = (1.0 / torch.clamp(lum_adapted.float(), min=1e-3)).view(-1, 1)
    return chain_apply(_img(x.detach(), 3), _single('crysis'), p, 1.0 / data_scale, data_scale)


def tone_filmic(x, white_point, exposure_bias, data_scale=1.0):
    w = torch.clamp(white_point.float(), min=1e-3)
    p = torch.stack([exposure_bias.float(), 1.0 / _hable(w)], dim=1)
    return chain_apply(_img(x.detach(), 3), _single('filmic'), p, 1.0 / data_scale, data_scale)


def whiteworld(x, ratio, data_scale=1.0):
    """k = ceil(ratio*HW)-th largest value per plane maps to white (oracle/SPEC.md)."""
    x = _img(x.detach(), 3)
    N, _, H, W = x.shape
    hw = float(H * W)
    k = torch.clamp(torch.ceil(ratio.float().view(N) * hw), 1, hw).to(torch.int64)
    t = kth_largest(x, k)
    g = 1.0 / torch.clamp(t / data_scale, min=1e-6)
    return chain_apply(x, _single('gain_clip'), g, 1.0 / data_scale, data_scale)


# ---- Bayer ----------------------------------------------------------------------------------------
class _ShuffleFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, up):
        x = _img(x)
        N, C, H, W = x.shape
        ctx.up = up
        if up:
            assert C % 4 == 0
            out = torch.empty((N, C // 4, H * 2, W * 2), device=x.device, dtype=torch.float32)
            L.call('risp_pixel_shuffle2', L.ptr(x), L.ptr(out), N, C // 4, H * 2, W * 2, L.stream())
        else:
            out = torch.empty((N, C * 4, H // 2, W // 2), device=x.device, dtype=torch.float32)
            L.call('risp_pixel_unshuffle2', L.ptr(x), L.ptr(out), N, C, H, W, L.stream())
        return out

    @staticmethod
    def backward(ctx, d):
        return _ShuffleFn.apply(d, not ctx.up), None


def pixel_shuffle2(x): return _ShuffleFn.apply(x, True)
def pixel_unshuffle2(x): return _ShuffleFn.apply(x, False)
def pack_rggb(raw): return _ShuffleFn.apply(_img(raw, 1), False)
def unpack_rggb(p): return _ShuffleFn.apply(_img(p, 4), True)


class _DemosaicFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, raw, kind, clip_hi):
        raw = _img(raw, 1)
        N, _, H, W = raw.shape
        out = torch.empty((N, 3, H, W), device=raw.device, dtype=torch.float32)
        L.call('risp_demosaic_fwd', L.ptr(raw), L.ptr(out), N, H, W, DM[kind], float(clip_hi), L.stream())
        ctx.kind, ctx.clip_hi = kind, clip_hi
        ctx.save_for_backward(raw)
        return out

    @staticmethod
    def backward(ctx, d):
        raw, = ctx.saved_tensors
        N, _, H, W = raw.shape
        d = _img(d, 3)
        draw = torch.empty_like(raw)
        L.call('risp_demosaic_bwd', L.ptr(raw), L.ptr(d), L.ptr(draw), N, H, W, DM[ctx.kind], float(ctx.clip_hi), L.stream())
        return draw, None, None


def demosaic(raw, kind, clip_hi=1.0):
    return _DemosaicFn.apply(raw, kind, clip_hi)


class _BlcWbFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, raw, params):
        raw = _img(raw, 1)
        N, _, H, W = raw.shape
        tab, stride = _param_table(params, N, 5)
        out = torch.empty_like(raw)
        L.call('risp_bayer_blc_wb_fwd', L.ptr(raw), L.ptr(out), N, H, W, L.ptr(tab), stride, L.stream())
        ctx.stride, ctx.pshape = stride, params.shape
        ctx.save_for_backward(raw, tab)
        return out

    @staticmethod
    def backward(ctx, d):
        raw, tab = ctx.saved_tensors
        N, _, H, W = raw.shape
        d = _img(d, 1)
        draw = torch.empty_like(raw) if ctx.needs_input_grad[0] else None
        dpar = torch.empty((1 if ctx.stride == 0 else N, 5), device=raw.device, dtype=torch.float32)
        ws = L.workspace(L.size('risp_bayer_blc_wb_bwd_workspace', N, H, W), raw.device)
        L.call('risp_bayer_blc_wb_bwd', L.ptr(raw), L.ptr(d), L.ptr(draw), L.ptr(dpar), N, H, W, L.ptr(tab), ctx.stride,
               L.ptr(ws), ws.numel() * 4, L.stream())
        return draw, dpar.view(ctx.pshape)


def bayer_blc_wb(raw, params):
    """params (N,5)|(1,5): black level, gains [R,G1,G2,B]."""
    return _BlcWbFn.apply(raw, params)


def decode_codes(codes, denom, out=None):
    """uint8 / uint16 (or int16) codes on the device -> fp32 codes/denom (the loaders' /255., /1023., /16383.)."""
    if not codes.is_cuda:
        raise RuntimeError('decode_codes runs on CUDA tensors only')
    codes = codes.contiguous()
    nbytes = codes.element_size()
    assert nbytes in (1, 2) and not codes.dtype.is_floating_point
    if out is None:
        out = torch.empty(codes.shape, device=codes.device, dtype=torch.float32)
    assert out.shape == codes.shape and out.dtype == torch.float32 and out.is_contiguous()
    L.call('risp_decode_codes', L.ptr(codes), L.ptr(out), codes.numel(), nbytes, float(denom), L.stream())
    return out


def crop_decode(codes, y0, x0, h, w, denom, bayer=True):
    """The loader's random crop + normalisation on the device (sid_sony_ratio_rggb2bgr_dataset.py:109-136): `codes`
    (planes,H,W) or (N,C,H,W) uint8 / uint16 full frames already in HBM -> fp32 crop / denom.  A Bayer crop must start on an
    even row and column (the reference aligns it the same way, s7isp_rggb2bgr_test_dataset.py:106-113)."""
    if not codes.is_cuda:
        raise RuntimeError('crop_decode runs on CUDA tensors only')
    codes = codes.contiguous()
    H, W = codes.shape[-2:]
    planes = codes.numel() // (H * W)
    out = torch.empty(tuple(codes.shape[:-2]) + (h, w), device=codes.device, dtype=torch.float32)
    L.call('risp_crop_decode', L.ptr(codes), L.ptr(out), planes, H, W, int(y0), int(x0), int(h), int(w), codes.element_size(),
           float(denom), int(bool(bayer)), L.stream())
    return out


def sample_crops(raw_store, gt_store, pos, h, w, white_level, status, img_out=None, gt_out=None):
    """A batch of crops out of frame stores in HBM in one launch (`risp_sample_crops`, the kernel of `crop_decode`).
    raw_store (F,H,W) uint8 / int16 codes (int16 holds the bit pattern of unsigned 16-bit codes), gt_store (G,3,H,W) uint8 BGR
    or None, pos (B,4) int32 CUDA records (raw frame, gt frame, y0, x0) with even origins, status (1,) int32 CUDA.
    -> img (B,1,h,w) = code / white_level and gt (B,3,h,w) = code / 255 (None without gt_store), fp32, written into
    img_out / gt_out when given.  A bad record sets status and is skipped; nothing here reads status or waits for the device."""
    F, H, W = raw_store.shape
    if raw_store.dtype not in (torch.uint8, torch.int16):
        raise ValueError('sample_crops: raw codes must be uint8 or int16, got %s' % raw_store.dtype)
    if gt_store is not None and (gt_store.dtype != torch.uint8 or tuple(gt_store.shape[1:]) != (3, H, W)):
        raise ValueError('sample_crops: gt_store must be uint8 (G,3,%d,%d), got %s %s' % (H, W, gt_store.dtype, tuple(gt_store.shape)))
    if pos.dtype != torch.int32 or pos.dim() != 2 or pos.shape[1] != 4:
        raise ValueError('sample_crops: pos must be int32 (B,4), got %s %s' % (pos.dtype, tuple(pos.shape)))
    if status.dtype != torch.int32 or status.numel() < 1:
        raise ValueError('sample_crops: status must be an int32 tensor')
    B = pos.shape[0]
    dev = raw_store.device
    if img_out is None:
        img_out = torch.empty((B, 1, h, w), device=dev, dtype=torch.float32)
    if gt_store is None:
        gt_out = None
    elif gt_out is None:
        gt_out = torch.empty((B, 3, h, w), device=dev, dtype=torch.float32)
    if tuple(img_out.shape) != (B, 1, h, w) or img_out.dtype != torch.float32 or \
            (gt_out is not None and (tuple(gt_out.shape) != (B, 3, h, w) or gt_out.dtype != torch.float32)):
        raise ValueError('sample_crops: outputs must be fp32 (%d,1,%d,%d) and (%d,3,%d,%d)' % (B, h, w, B, h, w))
    G = 0 if gt_store is None else gt_store.shape[0]
    L.call('risp_sample_crops', L.ptr(raw_store), raw_store.element_size(), F, L.ptr(gt_store), G, H, W, L.ptr(pos), B, int(h),
           int(w), float(white_level), L.ptr(img_out), L.ptr(gt_out), L.ptr(status), L.stream())
    return img_out, gt_out


def to_u8_hwc(x):
    """`utils.util.tensor2bgr(tensor)` on the device: (C,H,W) or (1,C,H,W) fp32 -> (H,W,C) uint8 = trunc(clip(x*255, 0, 255))."""
    x = (x[0] if x.dim() == 4 else x).detach().contiguous()
    C, H, W = x.shape
    out = torch.empty((H, W, C), device=x.device, dtype=torch.uint8)
    L.call('risp_to_u8_hwc', L.ptr(x), L.ptr(out), C, H, W, L.stream())
    return out


# ---- stencils ---------------------------------------------------------------------------------------
def bilateral(x, window, sigma_color, sigma_space, max_window=None):
    x = _img(x.detach(), 3)
    N, _, H, W = x.shape
    window = window.to(device=x.device, dtype=torch.int32).contiguous()
    if max_window is None:
        max_window = int(window.max().item())        # the only host sync; callers that know the bound pass it
    y = torch.empty_like(x)
    L.call('risp_bilateral_fwd', L.ptr(x), L.ptr(y), N, H, W, L.ptr(window), L.ptr(sigma_color.float().contiguous()),
           L.ptr(sigma_space.float().contiguous()), int(max_window), L.stream())
    return y


def fastnlm(x, block_size, search_block, decay_factor, max_halo=None):
    """Non-local means (oracle/SPEC.md); per-image odd block / search sizes and decay h."""
    x = _img(x.detach(), 3)
    N, _, H, W = x.shape
    block_size = block_size.to(device=x.device, dtype=torch.int32).contiguous()
    search_block = search_block.to(device=x.device, dtype=torch.int32).contiguous()
    if max_halo is None:
        max_halo = int((block_size // 2 + search_block // 2).max().item())
    y = torch.empty_like(x)
    L.call('risp_fastnlm_fwd', L.ptr(x), L.ptr(y), N, H, W, L.ptr(block_size), L.ptr(search_block),
           L.ptr(decay_factor.to(x.device).float().contiguous()), int(max_halo), L.stream())
    return y


def median(x, size):
    x = _img(x.detach(), 3)
    N, _, H, W = x.shape
    y = torch.empty_like(x)
    L.call('risp_median_fwd', L.ptr(x), L.ptr(y), N, H, W, int(size), L.stream())
    return y


def guided_filter(x, radius, eps):
    x = _img(x.detach(), 3)
    N, _, H, W = x.shape
    y = torch.empty_like(x)
    ws = L.workspace(L.size('risp_guided_workspace', N, H, W), x.device)
    L.call('risp_guided_fwd', L.ptr(x), L.ptr(y), N, H, W, int(radius), float(eps), L.ptr(ws), ws.numel() * 4, L.stream())
    return y


class _SharpenFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, amount):
        x = _img(x, 3)
        N, _, H, W = x.shape
        a = amount.float().reshape(N).contiguous()
        y = torch.empty_like(x)
        L.call('risp_sharpen_fwd', L.ptr(x), L.ptr(y), N, H, W, L.ptr(a), L.stream())
        ctx.ashape = amount.shape
        ctx.save_for_backward(x, a)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, a = ctx.saved_tensors
        N, _, H, W = x.shape
        dy = _img(dy, 3)
        dx = torch.empty_like(x)
        da = torch.empty((N,), device=x.device, dtype=torch.float32)
        ws = L.workspace(L.size('risp_sharpen_bwd_workspace', N, H, W), x.device)
        L.call('risp_sharpen_bwd', L.ptr(x), L.ptr(dy), L.ptr(dx), L.ptr(da), N, H, W, L.ptr(a), L.ptr(ws),
               ws.numel() * 4, L.stream())
        return dx, da.view(ctx.ashape)


def sharpen(x, amount):
    return _SharpenFn.apply(x, amount)


# ---- loss -------------------------------------------------------------------------------------------
class _LossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y, gt, l1):
        y, gt = y.contiguous(), gt.contiguous()
        assert y.is_cuda and gt.is_cuda and y.shape == gt.shape
        out = torch.empty((1,), device=y.device, dtype=torch.float32)
        ws = L.workspace(L.size('risp_loss_workspace', y.numel()), y.device)
        L.call('risp_loss_fwd', L.ptr(y), L.ptr(gt), L.ptr(out), y.numel(), int(l1), L.ptr(ws), ws.numel() * 4, L.stream())
        ctx.l1 = l1
        ctx.save_for_backward(y, gt)
        return out.view(())

    @staticmethod
    def backward(ctx, g):
        y, gt = ctx.saved_tensors
        dy = torch.empty_like(y)
        gs = g.reshape(1).float().contiguous()
        L.call('risp_loss_bwd', L.ptr(y), L.ptr(gt), L.ptr(gs), L.ptr(dy), y.numel(), int(ctx.l1), L.stream())
        return dy, None, None


def mse_loss(y, gt): return _LossFn.apply(y, gt, False)
def l1_loss(y, gt): return _LossFn.apply(y, gt, True)


# ---- DARTS mixed-op ----------------------------------------------------------------------------------
class _AlphaPruneFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, alpha, threshold, n_pruned_out):
        a = alpha.detach().float().contiguous()
        post = torch.empty_like(a)
        L.call('risp_alpha_prune_fwd', L.ptr(a), L.ptr(post), L.ptr(n_pruned_out), a.numel(), float(threshold), L.stream())
        ctx.threshold = threshold
        ctx.save_for_backward(a)
        return post

    @staticmethod
    def backward(ctx, dpost):
        a, = ctx.saved_tensors
        da = torch.empty_like(a)
        L.call('risp_alpha_prune_bwd', L.ptr(a), L.ptr(dpost.contiguous()), L.ptr(da), a.numel(), float(ctx.threshold), L.stream())
        return da, None, None


def alpha_prune(alpha, threshold, n_pruned_out=None):
    """softmax -> online prune -> renormalise (super_prune...:185-193), all on the device."""
    return _AlphaPruneFn.apply(alpha, threshold, n_pruned_out)


class _MixedFn(torch.autograd.Function):
    """y = sum_j w_j f_j(x; params) + sum_i w_{K_cls+i} ext_i."""

    @staticmethod
    def forward(ctx, x, params, w, chain, n_ext, *ext):
        C = x.shape[1]
        x = _img(x, C)
        N, _, H, W = x.shape
        ext = [_img(e, C) for e in ext]
        w = w.float().contiguous()
        y = torch.empty_like(x)
        if C == 3:
            tab, stride = _param_table(params, N, chain.P) if chain.P else (None, 0)
            L.call('risp_mixed_fwd', L.ptr(x), L.ptr(y), N, H * W, *chain.desc(), L.ptr(tab), stride,
                   L.parr(ext), len(ext), L.ptr(w), L.stream())
        else:
            tab, stride = None, 0
            L.call('risp_mixed1_fwd', L.ptr(x), L.ptr(y), N, H * W, chain.S, L.parr(ext), len(ext), L.ptr(w), L.stream())
        ctx.chain, ctx.stride, ctx.C = chain, stride, C
        ctx.pshape = None if params is None else params.shape
        ctx.save_for_backward(x, tab, w, *ext)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, tab, w, *ext = ctx.saved_tensors
        chain, C = ctx.chain, ctx.C
        N, _, H, W = x.shape
        dy = _img(dy, C)
        K = chain.S + len(ext)
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        dw = torch.empty((K,), device=x.device, dtype=torch.float32)
        P = chain.P
        dpar = torch.empty((1 if ctx.stride == 0 else N, P), device=x.device, dtype=torch.float32) if P else None
        ws = L.workspace(L.size('risp_mixed_bwd_workspace', N, H * W, P, K), x.device)
        dext = None
        if C == 3:
            # d ext_i = w_i * dy leaves the same pass (written from the registers that hold dy)
            dext = [torch.empty_like(dy) if ctx.needs_input_grad[5 + i] else None for i in range(len(ext))]
            L.call('risp_mixed_bwd_dext', L.ptr(x), L.ptr(dy), L.ptr(dx), L.ptr(dw), L.ptr(dpar), L.parr_opt(dext), N, H * W,
                   *chain.desc(), L.ptr(tab), ctx.stride, P, L.parr(ext), len(ext), L.ptr(w), L.ptr(ws), ws.numel() * 4, L.stream())
        else:
            L.call('risp_mixed1_bwd', L.ptr(x), L.ptr(dy), L.ptr(dx), L.ptr(dw), N, H * W, chain.S, L.parr(ext),
                   len(ext), L.ptr(w), L.ptr(ws), ws.numel() * 4, L.stream())
        if dpar is not None:
            dpar = dpar.view(ctx.pshape)
        # d ext_i = w_i * dy : a skipped branch (w < 1e-9) gets no gradient, like the reference's `continue`
        if dext is None:
            dext = [scale_by_device(dy, w, chain.S + i) if ctx.needs_input_grad[5 + i] else None for i in range(len(ext))]
        return (dx, dpar, dw, None, None, *dext)


def scale_by_device(t, w, idx):
    """t * w[idx] with w on the device (no host sync)."""
    if t.shape[1] == 3:
        return chain_apply(t, _single('gain'), w[idx].expand(3).reshape(1, 3))
    return t * w[idx]


def mixed_op(x, chain, params, w, ext=()):
    """chain: `Chain` of the classical candidates (each one stage, evaluated from x in registers);
    ext: materialised candidate outputs; w: (K_cls+K_ext,) post-prune weights on the device."""
    return _MixedFn.apply(x, params, w, chain, len(ext), *ext)


# ---- fused fixed pipeline ------------------------------------------------------------------------------
def pipeline_fwd(raw, dm_kind, chain, params=None, clip_hi=1.0):
    raw = _img(raw.detach(), 1)
    N, _, H, W = raw.shape
    tab, stride = _param_table(params.detach(), N, chain.P) if chain.P else (None, 0)
    y = torch.empty((N, 3, H, W), device=raw.device, dtype=torch.float32)
    L.call('risp_pipeline_fwd', L.ptr(raw), L.ptr(y), N, H, W, DM[dm_kind], float(clip_hi), *chain.desc(), L.ptr(tab),
           stride, L.stream())
    return y


def sse_u8(y, gt):
    """Per-image sum of squared differences of the 8-bit codes tensor2bgr makes of y and gt (utils/util.py:118-135:
    trunc(clip(x*255, 0, 255))) -> int64 (N,) CUDA tensor, exact.  y, gt: fp32 (N,C,H,W) or (C,H,W), any H and W.
    Nothing waits for the device: `metrics.psnr_from_sse` turns the sums into PSNR."""
    y, gt = y.detach(), gt.detach()
    if y.dim() == 3:
        y, gt = y.unsqueeze(0), gt.unsqueeze(0)
    y, gt = _img(y), _img(gt)
    if y.shape != gt.shape:
        raise ValueError('sse_u8: shapes differ, %s and %s' % (tuple(y.shape), tuple(gt.shape)))
    N, C, H, W = y.shape
    sse = torch.zeros((N,), device=y.device, dtype=torch.int64)
    if y.numel() == 0:
        return sse
    L.call('risp_sse_u8', L.ptr(y), L.ptr(gt), L.ptr(sse), N, C, H, W, L.stream())
    return sse


def ssim_u8(y, gt):
    """Per-image SSIM of the 8-bit images of y and gt (skimage `compare_ssim(a, b, multichannel=True)` on the tensor2bgr
    codes: uniform 7x7 window, border of 3 cropped) as exact int64 (N,) CUDA sums of rint(S * 2^32) over the C (H-6)(W-6)
    interior values; `metrics.ssim_from_sums` turns them into SSIM.  Nothing waits for the device.
    y: fp32 (N,C,H,W) / (C,H,W), or the uint8 (N,H,W,C) / (H,W,C) image of `to_u8_hwc`, `pipeline_eval(u8=True)` or
    `patch2whole_u8`; gt: fp32 (N,C,H,W) / (C,H,W).  H and W must be at least 7."""
    y, gt = y.detach(), gt.detach()
    if gt.dim() == 3:
        gt = gt.unsqueeze(0)
    if y.dim() == 3:
        y = y.unsqueeze(0)
    gt = _img(gt)
    N, C, H, W = gt.shape
    if y.dtype == torch.uint8:
        if not y.is_cuda:
            raise RuntimeError('reconfigisp_b200 ops run on CUDA tensors only (no CPU fallback); got a %s tensor' % y.device)
        if tuple(y.shape) != (N, H, W, C):
            raise ValueError('ssim_u8: the 8-bit y must be (N,H,W,C) = %s, got %s' % ((N, H, W, C), tuple(y.shape)))
        y, layout = y.contiguous(), L.ENUMS['RISP_IMG_U8_NHWC']
    else:
        y, layout = _img(y), L.ENUMS['RISP_IMG_F32_NCHW']
        if y.shape != gt.shape:
            raise ValueError('ssim_u8: shapes differ, %s and %s' % (tuple(y.shape), tuple(gt.shape)))
    if H < 7 or W < 7:
        raise ValueError('ssim_u8: the 7x7 window needs H and W >= 7, got %d x %d' % (H, W))
    out = torch.empty((N,), device=gt.device, dtype=torch.int64)
    if N == 0:
        return out
    L.call('risp_ssim_u8', L.ptr(y), layout, L.ptr(gt), L.ptr(out), N, C, H, W, L.stream())
    return out


def pipeline_eval(raw, gt, dm_kind, chain, params=None, clip_hi=1.0, u8=False):
    """Evaluate the fused pipeline against gt without writing its image: -> (sse, u8_or_None).  sse is `sse_u8` of
    `pipeline_fwd(raw, dm_kind, chain, params, clip_hi)` and gt, int64 (N,); with u8=True the 8-bit image of the output
    comes along as (N,H,W,3) BGR uint8 (`to_u8_hwc` of each image).  16 B/px: raw and gt are read once."""
    raw, gt = _img(raw.detach(), 1), _img(gt.detach(), 3)
    N, _, H, W = raw.shape
    if gt.shape != (N, 3, H, W):
        raise ValueError('pipeline_eval: gt must be (%d,3,%d,%d), got %s' % (N, H, W, tuple(gt.shape)))
    tab, stride = _param_table(params.detach(), N, chain.P) if chain.P else (None, 0)
    sse = torch.empty((N,), device=raw.device, dtype=torch.int64)
    out8 = torch.empty((N, H, W, 3), device=raw.device, dtype=torch.uint8) if u8 else None
    ws = L.workspace(L.size('risp_pipeline_eval_workspace', N, H, W), raw.device)
    L.call('risp_pipeline_eval', L.ptr(raw), L.ptr(gt), L.ptr(out8), L.ptr(sse), N, H, W, DM[dm_kind], float(clip_hi),
           *chain.desc(), L.ptr(tab), stride, L.ptr(ws), ws.numel() * 4, L.stream())
    return sse, out8


def _store_args(raw_store, gt_store, pos, status, who):
    if raw_store.dtype not in (torch.uint8, torch.int16) or raw_store.dim() != 3:
        raise ValueError('%s: raw codes must be uint8 or int16 (F,H,W), got %s %s' % (who, raw_store.dtype, tuple(raw_store.shape)))
    F, H, W = raw_store.shape
    if gt_store.dtype != torch.uint8 or tuple(gt_store.shape[1:]) != (3, H, W):
        raise ValueError('%s: gt_store must be uint8 (G,3,%d,%d), got %s %s' % (who, H, W, gt_store.dtype, tuple(gt_store.shape)))
    if pos.dtype != torch.int32 or pos.dim() != 2 or pos.shape[1] != 4:
        raise ValueError('%s: pos must be int32 (N,4), got %s %s' % (who, pos.dtype, tuple(pos.shape)))
    if status.dtype != torch.int32 or status.numel() < 1:
        raise ValueError('%s: status must be an int32 tensor' % who)
    return F, H, W


def pipeline_eval_store(raw_store, gt_store, pos, white_level, status, dm_kind, chain, params=None, clip_hi=1.0, u8=False,
                        sse_out=None, u8_out=None):
    """`pipeline_eval` on whole frames of the stores of `sample_crops`, read as codes (`risp_pipeline_eval_store`):
    image n is raw frame pos[n,0] / white_level against GT frame pos[n,1], pos (N,4) int32 CUDA records (raw frame, GT
    frame, 0, 0).  -> (sse, u8_or_None), the values `pipeline_eval` gives on the batch `sample_crops` decodes from the same
    records, written into sse_out / u8_out when given.  A bad record sets status (its sse is 0); nothing waits for the device."""
    F, H, W = _store_args(raw_store, gt_store, pos, status, 'pipeline_eval_store')
    N = pos.shape[0]
    tab, stride = _param_table(params.detach(), N, chain.P) if chain.P else (None, 0)
    sse = torch.empty((N,), device=raw_store.device, dtype=torch.int64) if sse_out is None else sse_out
    out8 = None
    if u8:
        out8 = torch.empty((N, H, W, 3), device=raw_store.device, dtype=torch.uint8) if u8_out is None else u8_out
    if tuple(sse.shape) != (N,) or sse.dtype != torch.int64 or (out8 is not None and (tuple(out8.shape) != (N, H, W, 3) or out8.dtype != torch.uint8)):
        raise ValueError('pipeline_eval_store: outputs must be int64 (%d,) and uint8 (%d,%d,%d,3)' % (N, N, H, W))
    ws = L.workspace(L.size('risp_pipeline_eval_workspace', N, H, W), raw_store.device)
    L.call('risp_pipeline_eval_store', L.ptr(raw_store), raw_store.element_size(), F, L.ptr(gt_store), gt_store.shape[0], H, W,
           L.ptr(pos), N, float(white_level), L.ptr(status), L.ptr(out8), L.ptr(sse), DM[dm_kind], float(clip_hi),
           *chain.desc(), L.ptr(tab), stride, L.ptr(ws), ws.numel() * 4, L.stream())
    return sse, out8


def ssim_u8_store(y, gt_store, pos, status, out=None):
    """`ssim_u8` of y against GT frames of a store (`risp_ssim_u8_store`): image n against frame pos[n,1] of gt_store (G,3,H,W)
    uint8, the same bits as `ssim_u8` with the decoded fp32 GT.  y: the uint8 (N,H,W,3) image of `pipeline_eval_store` or
    fp32 (N,3,H,W).  -> int64 (N,) CUDA sums (into out when given).  A bad record sets status (its sum is 0)."""
    y = y.detach()
    if pos.dtype != torch.int32 or pos.dim() != 2 or pos.shape[1] != 4:
        raise ValueError('ssim_u8_store: pos must be int32 (N,4), got %s %s' % (pos.dtype, tuple(pos.shape)))
    if status.dtype != torch.int32 or status.numel() < 1:
        raise ValueError('ssim_u8_store: status must be an int32 tensor')
    N = pos.shape[0]
    G, _, H, W = gt_store.shape
    if gt_store.dtype != torch.uint8 or gt_store.shape[1] != 3:
        raise ValueError('ssim_u8_store: gt_store must be uint8 (G,3,H,W), got %s %s' % (gt_store.dtype, tuple(gt_store.shape)))
    if y.dtype == torch.uint8:
        if tuple(y.shape) != (N, H, W, 3):
            raise ValueError('ssim_u8_store: the 8-bit y must be (N,H,W,3) = %s, got %s' % ((N, H, W, 3), tuple(y.shape)))
        layout = L.ENUMS['RISP_IMG_U8_NHWC']
    else:
        y, layout = _img(y, 3), L.ENUMS['RISP_IMG_F32_NCHW']
        if tuple(y.shape) != (N, 3, H, W):
            raise ValueError('ssim_u8_store: y must be (%d,3,%d,%d), got %s' % (N, H, W, tuple(y.shape)))
    if H < 7 or W < 7:
        raise ValueError('ssim_u8_store: the 7x7 window needs H and W >= 7, got %d x %d' % (H, W))
    out = torch.empty((N,), device=gt_store.device, dtype=torch.int64) if out is None else out
    L.call('risp_ssim_u8_store', L.ptr(y), layout, L.ptr(gt_store), G, L.ptr(pos), L.ptr(status), L.ptr(out), N, H, W, L.stream())
    return out


class PipelineStep:
    """Pre-allocated state for repeated proxy-tuning steps on frames of one geometry."""

    def __init__(self, N, H, W, dm_kind, chain, device, clip_hi=1.0, shared_row=True, l1=False):
        self.N, self.H, self.W, self.dm, self.chain, self.clip_hi = N, H, W, DM[dm_kind], chain, float(clip_hi)
        self.entry = 'risp_pipeline_l1_step' if l1 else 'risp_pipeline_mse_step'    # nn.L1Loss / nn.MSELoss (isp_model.py:44-49)
        self.stride = 0 if shared_row else chain.P
        self.loss = torch.empty((1,), device=device, dtype=torch.float32)
        self.dparams = torch.empty((1 if shared_row else N, max(1, chain.P)), device=device, dtype=torch.float32)
        self.ws = L.workspace(L.size('risp_pipeline_step_workspace', N, H, W, chain.P), device)

    def __call__(self, raw, gt, params, y_out=None):
        """-> (loss (1,), dparams).  raw (N,1,H,W), gt (N,3,H,W), params (1|N, P) kernel-level."""
        L.call(self.entry, L.ptr(raw), L.ptr(gt), L.ptr(y_out), L.ptr(self.loss), L.ptr(self.dparams),
               self.N, self.H, self.W, self.dm, self.clip_hi, *self.chain.desc(), L.ptr(params), self.stride,
               self.chain.P, L.ptr(self.ws), self.ws.numel() * 4, L.stream())
        return self.loss, self.dparams

    def store(self, raw_store, gt_store, pos, white_level, status, params):
        """The same step on the N crops of H x W that the records pos (N,4) int32 CUDA name in the frame stores of
        `sample_crops`, read as codes (`risp_pipeline_*_step_store`) -> (loss (1,), dparams), bitwise the values `__call__`
        gives on `sample_crops(raw_store, gt_store, pos, H, W, white_level, ...)`.  A bad record sets status and adds nothing
        (the normaliser stays N*3*H*W).  Needs frames with W % 16 == 0 (NotImplementedError otherwise)."""
        F, FH, FW = _store_args(raw_store, gt_store, pos, status, 'PipelineStep.store')
        if pos.shape[0] != self.N:
            raise ValueError('PipelineStep.store: %d records for a step of %d images' % (pos.shape[0], self.N))
        L.call(self.entry + '_store', L.ptr(raw_store), raw_store.element_size(), F, L.ptr(gt_store), gt_store.shape[0], FH, FW,
               L.ptr(pos), self.N, float(white_level), L.ptr(status), self.H, self.W, L.ptr(self.loss), L.ptr(self.dparams),
               self.dm, self.clip_hi, *self.chain.desc(), L.ptr(params), self.stride, self.chain.P, L.ptr(self.ws),
               self.ws.numel() * 4, L.stream())
        return self.loss, self.dparams


class _PipelineMseFn(torch.autograd.Function):
    """loss = mse(pipeline(raw; params), gt) with d loss / d params from the same single pass."""

    @staticmethod
    def forward(ctx, params, raw, gt, dm_kind, chain, clip_hi, l1=False):
        raw, gt = _img(raw, 1), _img(gt, 3)
        N, _, H, W = raw.shape
        tab, stride = _param_table(params, N, chain.P)
        step = PipelineStep(N, H, W, dm_kind, chain, raw.device, clip_hi, shared_row=(stride == 0), l1=l1)
        loss, dpar = step(raw, gt, tab)
        ctx.pshape = params.shape
        ctx.save_for_backward(dpar)
        return loss.view(())

    @staticmethod
    def backward(ctx, g):
        dpar, = ctx.saved_tensors
        return (dpar * g).view(ctx.pshape), None, None, None, None, None, None


def pipeline_mse(params, raw, gt, dm_kind, chain, clip_hi=1.0):
    return _PipelineMseFn.apply(params, raw, gt, dm_kind, chain, clip_hi, False)


def pipeline_l1(params, raw, gt, dm_kind, chain, clip_hi=1.0):
    """mean |pipeline(raw; params) - gt| with d loss / d params from the same single pass (pre-instantiated chains)."""
    return _PipelineMseFn.apply(params, raw, gt, dm_kind, chain, clip_hi, True)


# ---- patches ----------------------------------------------------------------------------------------
def patch_origins(L_, l, s):
    """util_path_restore.py:88-89."""
    return list(range(0, L_ - l, s)) + [L_ - l]


def whole2patch(frame, size, stride):
    """frame (C,H,W) or (1,C,H,W) CUDA -> tiles (T,C,h,w), positions [(y,x)]."""
    f = frame[0] if frame.dim() == 4 else frame
    f = f.contiguous()
    C, H, W = f.shape
    h, w = size
    sh, sw = stride
    assert sh <= h <= H and sw <= w <= W and C >= 1
    ys, xs = patch_origins(H, h, sh), patch_origins(W, w, sw)
    tiles = torch.empty((len(ys) * len(xs), C, h, w), device=f.device, dtype=torch.float32)
    L.call('risp_whole2patch', L.ptr(f), L.ptr(tiles), C, H, W, h, w, L.iarr(ys), len(ys), L.iarr(xs), len(xs), L.stream())
    return tiles, [(y, x) for y in ys for x in xs]


def patch2whole_u8(tiles, frame_hw, stride, want_float=False):
    """Blend + `(np.clip(merged, 0, 1) * 255.).astype(np.uint8)` (test_split.py:104-108) in one kernel -> (H,W,C) uint8
    [, (C,H,W) fp32 clipped]."""
    tiles = tiles.contiguous()
    T, C, h, w = tiles.shape
    H, W = frame_hw
    sh, sw = stride
    ys, xs = patch_origins(H, h, sh), patch_origins(W, w, sw)
    assert T == len(ys) * len(xs)
    out8 = torch.empty((H, W, C), device=tiles.device, dtype=torch.uint8)
    outf = torch.empty((C, H, W), device=tiles.device, dtype=torch.float32) if want_float else None
    L.call('risp_patch2whole_u8', L.ptr(tiles), L.ptr(outf), L.ptr(out8), C, H, W, h, w, sh, sw, L.iarr(ys), len(ys), L.iarr(xs),
           len(xs), L.stream())
    return (out8, outf) if want_float else out8


def patch2whole(tiles, frame_hw, stride, clip01=False):
    tiles = tiles.contiguous()
    T, C, h, w = tiles.shape
    H, W = frame_hw
    sh, sw = stride
    ys, xs = patch_origins(H, h, sh), patch_origins(W, w, sw)
    assert T == len(ys) * len(xs)
    out = torch.empty((C, H, W), device=tiles.device, dtype=torch.float32)
    L.call('risp_patch2whole', L.ptr(tiles), L.ptr(out), C, H, W, h, w, sh, sw, L.iarr(ys), len(ys), L.iarr(xs), len(xs),
           int(bool(clip01)), L.stream())
    return out


# ---- dense convolution of the CNN candidates -------------------------------------------------------------
CONV_RELU_IN, CONV_RELU_OUT, CONV_ADD_RES, CONV_RES_RELU = (L.ENUMS['RISP_CONV_RELU_IN'], L.ENUMS['RISP_CONV_RELU_OUT'],
                                                           L.ENUMS['RISP_CONV_ADD_RES'], L.ENUMS['RISP_CONV_RES_RELU'])
def invalidate_weight_cache(module_or_tensor):
    """Drop the prepared (kernel-layout) copies of convolution weights.  The caches are keyed by the tensor's version counter,
    which in-place updates through `weight.data` (old-style checkpoint loaders, EMA code) do NOT bump: call this after such
    an update -- `load_state_dict`, optimizers and every ordinary in-place op are tracked and need nothing."""
    tensors = [module_or_tensor] if isinstance(module_or_tensor, torch.Tensor) else list(module_or_tensor.parameters())
    for t in tensors:
        for attr in ('_risp_wk', '_risp_wtc'):
            if hasattr(t, attr):
                delattr(t, attr)
    if not isinstance(module_or_tensor, torch.Tensor):
        for m in module_or_tensor.modules():
            m.__dict__.pop('_risp_derived', None)


def _prepared_weights(weight, transpose_flip):
    """(Cout,Cin,K,K) -> kernel layout.  Cached ON the weight tensor object (so the cache dies with it; a
    pointer-keyed cache would alias once the allocator reuses the address) and keyed by its version counter."""
    cache = getattr(weight, '_risp_wk', None)
    key = (bool(transpose_flip), weight._version, weight.data_ptr())
    if cache is None or key not in cache:
        Cout, Cin, K, _ = weight.shape
        n = L.size('risp_conv2d_prepared_weight_floats', Cin, Cout, K, int(transpose_flip))
        wk = torch.empty((n,), device=weight.device, dtype=torch.float32)
        L.call('risp_conv2d_prepare_weights', L.ptr(weight.detach().contiguous()), L.ptr(wk), Cin, Cout, K, int(transpose_flip), L.stream())
        if cache is None or any(k[1:] != key[1:] for k in cache):
            cache = {}          # the weight was updated in place (fine-tuning): drop the stale layouts
        cache[key] = wk
        try:
            weight._risp_wk = cache
        except Exception:
            pass
    return cache[key]


def _conv_raw(x, mask_in, wk, bias, res, mask_out, Cout, K, flags):
    N, Cin, H, W = x.shape
    y = torch.empty((N, Cout, H, W), device=x.device, dtype=torch.float32)
    L.call('risp_conv2d_fwd', L.ptr(x), L.ptr(mask_in), L.ptr(wk), L.ptr(bias), L.ptr(res), L.ptr(mask_out), L.ptr(y),
           N, Cin, Cout, H, W, K, int(flags), L.stream())
    return y


class _ConvFn(torch.autograd.Function):
    """y = relu_out?(conv(relu_in?(x), W) + b) + relu?(res).  Backward: data gradients only -- the candidate
    networks are frozen constants on this path (SURVEY.md §3.2)."""

    @staticmethod
    def forward(ctx, x, res, weight, bias, relu_in, relu_out, res_relu):
        x = _img(x)
        Cout, Cin, K, _ = weight.shape
        assert x.shape[1] == Cin, 'conv2d: %d input channels, weight expects %d' % (x.shape[1], Cin)
        assert not (relu_out and res is not None), 'output ReLU and residual never co-occur in the candidate nets'
        flags = (CONV_RELU_IN if relu_in else 0) | (CONV_RELU_OUT if relu_out else 0)
        if res is not None:
            res = _img(res, Cout)
            flags |= CONV_ADD_RES | (CONV_RES_RELU if res_relu else 0)
        b = None if bias is None else bias.detach().float().contiguous()
        y = _conv_raw(x, None, _prepared_weights(weight, False), b, res, None, Cout, K, flags)
        ctx.cfg = (relu_in, relu_out, res_relu, Cin, K)
        x_full = x if (weight.requires_grad or (bias is not None and bias.requires_grad)) else None
        ctx.save_for_backward(x if relu_in else None, y if relu_out else None, res if (res is not None and res_relu) else None, weight, x_full)
        ctx.has_res = res is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x, y, res, weight, x_full = ctx.saved_tensors
        relu_in, relu_out, res_relu, Cin, K = ctx.cfg
        dy = dy.contiguous()
        dx = dres = None
        if ctx.needs_input_grad[0]:
            # dx = [x > 0]? * conv(dy * [y > 0]?, W^T flipped)
            dx = _conv_raw(dy, y if relu_out else None, _prepared_weights(weight, True), None, None, x if relu_in else None,
                           Cin, K, 0)
        if ctx.has_res and ctx.needs_input_grad[1]:
            dres = dy if not res_relu else dy * (res > 0).to(dy.dtype)
        dw = db = None
        if ctx.needs_input_grad[2] or ctx.needs_input_grad[3]:
            dw, db = conv_weight_grads(x_full, dy, y if relu_out else None, weight.shape, relu_in,
                                       ctx.needs_input_grad[2], ctx.needs_input_grad[3])
        return dx, dres, dw, db, None, None, None


def conv_weight_grads(x, dy, y_mask, wshape, relu_in, want_w=True, want_b=True):
    """dW (nn.Conv2d layout) and db of y = conv(relu?(x), W) + b for an upstream gradient dy (masked by [y_mask > 0])."""
    Cout, Cin, K, _ = wshape
    N, _, H, W = x.shape
    dw = db = None
    if want_w:
        dw = torch.empty(tuple(wshape), device=x.device, dtype=torch.float32)
        ws = L.workspace(L.size('risp_conv2d_bwd_weight_workspace', Cin, Cout, K), x.device)
        L.call('risp_conv2d_bwd_weight', L.ptr(x.contiguous()), L.ptr(dy.contiguous()), L.ptr(y_mask), L.ptr(dw), N, Cin, Cout, H, W, K,
               int(bool(relu_in)), L.ptr(ws), ws.numel() * 4, L.stream())
    if want_b:
        # db[co] = sum dy': a per-plane reduction (own kernel) + a (N,Cout) -> (Cout,) sum
        dyb = dy if y_mask is None else chain_apply_mask(dy, y_mask)
        db = plane_stats(dyb)[..., 1].sum(dim=0) * float(H * W)
    return dw, db


def chain_apply_mask(t, mask):
    """t * [mask > 0] (tiny helper for the bias gradient; elementwise torch op on the fine-tune path only)."""
    return t * (mask > 0).to(t.dtype)


def conv2d(x, weight, bias=None, relu_in=False, relu_out=False, residual=None, residual_relu=False):
    return _ConvFn.apply(x, residual, weight, bias, relu_in, relu_out, residual_relu)


# ---- tensor-core convolution on channel-blocked activations (csrc/risp_conv_tc.cu) ------------------------
def tc_groups(C):
    """number of 4-channel groups of the blocked layout = risp_conv_tc_padded_channels(C) / 4 (restated: launch-path hot spot)."""
    return (C + 3) // 4


class _ToBlockedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x = _img(x)
        N, C, H, W = x.shape
        CG = tc_groups(C)
        out = torch.empty((N, H, CG, W, 4), device=x.device, dtype=torch.float32)
        L.call('risp_to_blocked', L.ptr(x), L.ptr(out), N, C, CG, H, W, L.stream())
        ctx.C = C
        return out

    @staticmethod
    def backward(ctx, d):
        return _FromBlockedFn.apply(d.contiguous(), ctx.C)


class _FromBlockedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xb, C):
        xb = xb.contiguous()
        N, H, CG, W, _ = xb.shape
        out = torch.empty((N, C, H, W), device=xb.device, dtype=torch.float32)
        L.call('risp_from_blocked', L.ptr(xb), L.ptr(out), N, C, CG, H, W, L.stream())
        return out

    @staticmethod
    def backward(ctx, d):
        return _ToBlockedFn.apply(d.contiguous()), None


def to_blocked(x): return _ToBlockedFn.apply(x)
def from_blocked(xb, C): return _FromBlockedFn.apply(xb, C)


def _tc_weights(weight, transpose_flip):
    cache = getattr(weight, '_risp_wtc', None)
    key = (bool(transpose_flip), weight._version, weight.data_ptr())
    if cache is None or key not in cache:
        Cout, Cin, K, _ = weight.shape
        n = L.size('risp_conv_tc_weight_floats', Cin, Cout, K, int(transpose_flip))
        wk = torch.empty((n,), device=weight.device, dtype=torch.float32)
        L.call('risp_conv_tc_prepare_weights', L.ptr(weight.detach().contiguous()), L.ptr(wk), Cin, Cout, K, int(transpose_flip), L.stream())
        torch.cuda.current_stream().synchronize()       # prepared once, then read from whichever stream the candidate runs on
        if cache is None or any(k[1:] != key[1:] for k in cache):
            cache = {}
        cache[key] = wk
        try:
            weight._risp_wtc = cache
        except Exception:
            pass
    return cache[key]


def _conv_tc_raw(xb, mask_in, wk, bias, resb, mask_out, Cin, Cout, K, flags, bias_tab=None):
    N, H, _, W, _ = xb.shape
    yb = torch.empty((N, H, tc_groups(Cout), W, 4), device=xb.device, dtype=torch.float32)
    L.call('risp_conv_tc_fwd_tab', L.ptr(xb), L.ptr(mask_in), L.ptr(wk), L.ptr(bias), L.ptr(bias_tab), L.ptr(resb), L.ptr(mask_out),
           L.ptr(yb), None, N, Cin, Cout, H, W, K, int(flags), L.stream())
    return yb


def blocked_class_sums(gb, mask_b, C, K):
    """(N,H,CG,W,4) blocked gradient -> (N, K*K, pad16(C)) sums over the K x K border classes of the pixels (the backward of a
    position-class bias table, see risp_conv_tc_fwd_tab)."""
    N, H, _, W, _ = gb.shape
    CP = (C + 15) // 16 * 16
    out = torch.empty((N, K * K, CP), device=gb.device, dtype=torch.float32)
    ws = L.workspace(L.size('risp_blocked_class_sums_workspace', N, C, H, K), gb.device)
    L.call('risp_blocked_class_sums', L.ptr(gb), L.ptr(mask_b), L.ptr(out), N, C, CP, H, W, K, L.ptr(ws), ws.numel() * 4, L.stream())
    return out


class _ConvTcFn(torch.autograd.Function):
    """Blocked-layout convolution on the tensor cores; same contract as `_ConvFn` (data gradients only)."""

    @staticmethod
    def forward(ctx, xb, resb, weight, bias, relu_in, relu_out, res_relu, bias_tab=None):
        xb = xb.contiguous()
        Cout, Cin, K, _ = weight.shape
        assert xb.shape[2] == tc_groups(Cin), 'blocked input has %d groups, weight expects %d' % (xb.shape[2], tc_groups(Cin))
        assert not (relu_out and resb is not None)
        flags = (CONV_RELU_IN if relu_in else 0) | (CONV_RELU_OUT if relu_out else 0)
        if resb is not None:
            resb = resb.contiguous()
            flags |= CONV_ADD_RES | (CONV_RES_RELU if res_relu else 0)
        b = None if bias is None else bias.detach().float().contiguous()
        if bias_tab is not None:
            assert bias is None and tuple(bias_tab.shape) == (xb.shape[0], K * K * ((Cout + 15) // 16 * 16)), 'bias table: (N, K*K*pad16(Cout))'
            bias_tab = bias_tab.detach().contiguous()
        yb = _conv_tc_raw(xb, None, _tc_weights(weight, False), b, resb, None, Cin, Cout, K, flags, bias_tab)
        ctx.cfg = (relu_in, relu_out, res_relu, Cin, Cout, K)
        ctx.has_tab = bias_tab is not None
        xb_full = xb if (weight.requires_grad or (bias is not None and bias.requires_grad)) else None
        ctx.save_for_backward(xb if relu_in else None, yb if relu_out else None, resb if (resb is not None and res_relu) else None, weight, xb_full)
        ctx.has_res = resb is not None
        return yb

    @staticmethod
    def backward(ctx, dyb):
        xb, yb, resb, weight, xb_full = ctx.saved_tensors
        relu_in, relu_out, res_relu, Cin, Cout, K = ctx.cfg
        dyb = dyb.contiguous()
        dxb = dres = None
        if ctx.needs_input_grad[0]:
            dxb = _conv_tc_raw(dyb, yb if relu_out else None, _tc_weights(weight, True), None, None, xb if relu_in else None,
                               Cout, Cin, K, 0)
        if ctx.has_res and ctx.needs_input_grad[1]:
            dres = dyb if not res_relu else dyb * (resb > 0).to(dyb.dtype)
        dw = db = None
        if ctx.needs_input_grad[2] or ctx.needs_input_grad[3]:
            # fine-tuning path only: the weight-gradient kernel works on planar tensors
            xp = _FromBlockedFn.apply(xb_full, Cin)
            dyp = _FromBlockedFn.apply(dyb, Cout)
            yp = _FromBlockedFn.apply(yb, Cout) if relu_out else None
            dw, db = conv_weight_grads(xp, dyp, yp, weight.shape, relu_in, ctx.needs_input_grad[2], ctx.needs_input_grad[3])
        dtab = None
        if ctx.has_tab and ctx.needs_input_grad[7]:
            dtab = blocked_class_sums(dyb, yb if relu_out else None, Cout, K).view(dyb.shape[0], -1)
        return dxb, dres, dw, db, None, None, None, dtab


class _BiasTableFn(torch.autograd.Function):
    """tab (N, J) = b_rep (J,) + feat (N, F) @ S (F, J) with S a constant; two small kernels of this library (cuBLAS picks an
    ~85 us gemv for the 4 x 5184 x 14 backward shape)."""

    @staticmethod
    def forward(ctx, feat, S, b_rep):
        feat = feat.contiguous().float()
        N, F = feat.shape
        J = S.shape[1]
        tab = torch.empty((N, J), device=feat.device, dtype=torch.float32)
        L.call('risp_bias_table_fwd', L.ptr(feat), L.ptr(S), L.ptr(b_rep), L.ptr(tab), N, F, J, L.stream())
        ctx.save_for_backward(S)
        return tab

    @staticmethod
    def backward(ctx, dtab):
        S, = ctx.saved_tensors
        dtab = dtab.contiguous()
        N, J = dtab.shape
        F = S.shape[0]
        dfeat = torch.empty((N, F), device=dtab.device, dtype=torch.float32)
        L.call('risp_bias_table_bwd', L.ptr(dtab), L.ptr(S), L.ptr(dfeat), N, F, J, L.stream())
        return dfeat, None, None


def bias_table(feat, S, b_rep):
    return _BiasTableFn.apply(feat, S, b_rep)


class _ResBlockTcFn(torch.autograd.Function):
    """ResidualBlock of the Path-Restore trunks (path_14l_bayer_arch.py:6-21) with frozen weights, blocked in / out:
        t = relu(conv1(relu(x)));  y = conv2(t) + relu(x)          (the in-place leading ReLU makes the skip relu(x))
    Backward in two launches, no elementwise glue:  dt = conv2^T(dy);  dx = [x > 0] * (conv1^T(dt * [t > 0]) + dy)
    -- the skip gradient rides in the data-gradient convolution's residual slot and both ReLU masks are applied while
    staging / in the epilogue."""

    @staticmethod
    def forward(ctx, xb, w1, b1, w2, b2):
        xb = xb.contiguous()
        C = w1.shape[0]
        K = w1.shape[2]
        b1 = None if b1 is None else b1.detach().float().contiguous()
        b2 = None if b2 is None else b2.detach().float().contiguous()
        t = _conv_tc_raw(xb, None, _tc_weights(w1, False), b1, None, None, C, C, K, CONV_RELU_IN | CONV_RELU_OUT)
        y = _conv_tc_raw(t, None, _tc_weights(w2, False), b2, xb, None, C, C, K, CONV_ADD_RES | CONV_RES_RELU)
        ctx.save_for_backward(xb, t, w1, w2)
        return y

    @staticmethod
    def backward(ctx, dy):
        xb, t, w1, w2 = ctx.saved_tensors
        dy = dy.contiguous()
        C, K = w1.shape[0], w1.shape[2]
        dt = _conv_tc_raw(dy, None, _tc_weights(w2, True), None, None, None, C, C, K, 0)
        dx = _conv_tc_raw(dt, t, _tc_weights(w1, True), None, dy, xb, C, C, K, CONV_ADD_RES)
        return dx, None, None, None, None


def resblock_tc(xb, w1, b1, w2, b2):
    return _ResBlockTcFn.apply(xb, w1, b1, w2, b2)


# ---- a bank of SRCNNRes proxies evaluated together (grouped launches) ---------------------------------------------------------
def _gconv(xb, mask_in, W, bias, bias_stride, tab, resb, G, N, slots, x_shared, res_shared, Cin, Cout, K, flags):
    """one grouped tensor-core convolution: G*N output images; W (n_slots, floats) prepared weights of every bank member"""
    H, Wd = xb.shape[1], xb.shape[3]
    yb = torch.empty((G * N, H, tc_groups(Cout), Wd, 4), device=xb.device, dtype=torch.float32)
    L.call('risp_conv_tc_fwd_grouped', L.ptr(xb), L.ptr(mask_in), L.ptr(W), L.ptr(bias), L.ptr(tab), L.ptr(resb), None, L.ptr(yb), None,
           G, N, slots, W.shape[1], int(bias_stride), int(x_shared), int(res_shared), Cin, Cout, H, Wd, K, int(flags), L.stream())
    return yb


class _SRCNNResBankFn(torch.autograd.Function):
    """y_g = SRCNNRes_g(x, p_g) for the G active members of a bank (same x, different weights and parameters):
    (N,3,H,W), (1, sum P_g) -> (G*N, 3, H, W).  Every layer is ONE grouped launch (the members have identical layer shapes
    once the constant channels are folded into the bias table), forward and backward; the statistics, the blocked copy of
    x and the gradient paths into x (data gradient of the first layer, residual, min/mean/max routing) are shared.
    At the reference's 4 x 256^2 batch a single member's layer is 1.7-3.5 waves of CTAs; eight together are 14-28."""

    @staticmethod
    def forward(ctx, x, par_cat, bank, active):
        x = _img(x, 3)
        N, _, H, Wd = x.shape
        G = len(active)
        slots = L.iarr(active)
        dev = x.device
        xb = torch.empty((N, H, 1, Wd, 4), device=dev, dtype=torch.float32)
        L.call('risp_to_blocked', L.ptr(x), L.ptr(xb), N, 3, 1, H, Wd, L.stream())
        st = plane_stats(x)                                             # (N,3,3) [min, mean, max] per plane
        idx = torch.empty((N * 3, 2), device=dev, dtype=torch.int32)
        L.call('risp_plane_argfirst', L.ptr(x), L.ptr(st), L.ptr(idx), N * 3, H * Wd, L.stream())
        st9 = st.permute(0, 2, 1).reshape(N, 9)
        Pmax, F, J = bank['Pmax'], bank['F'], bank['J']
        pidx = bank['par_index'](tuple(active), dev)                      # where every active parameter lands in (G, Pmax)
        par_pad = torch.zeros((G * Pmax,), device=dev, dtype=torch.float32).index_copy_(0, pidx, par_cat.detach().reshape(-1).float())
        feat = torch.cat([st9.unsqueeze(0).expand(G, N, 9), par_pad.view(G, 1, Pmax).expand(G, N, Pmax)], dim=2).contiguous()
        tab = torch.empty((G * N, J), device=dev, dtype=torch.float32)
        L.call('risp_bias_table_fwd_grouped', L.ptr(feat), L.ptr(bank['S']), L.ptr(bank['BR']), L.ptr(tab), G, N, slots, F, J, L.stream())
        h1 = _gconv(xb, None, bank['W1'], None, 0, tab, None, G, N, slots, 1, 0, 3, 64, 9, CONV_RELU_OUT)
        h2 = _gconv(h1, None, bank['W2'], bank['B2'], 32, None, None, G, N, slots, 0, 0, 64, 32, 5, CONV_RELU_OUT)
        yb = _gconv(h2, None, bank['W3'], bank['B3'], 3, None, xb, G, N, slots, 0, 1, 32, 3, 5, CONV_ADD_RES)
        y = torch.empty((G * N, 3, H, Wd), device=dev, dtype=torch.float32)
        L.call('risp_from_blocked', L.ptr(yb), L.ptr(y), G * N, 3, 1, H, Wd, L.stream())
        ctx.save_for_backward(h1, h2, idx, pidx)
        ctx.bank, ctx.active, ctx.shape = bank, list(active), (N, H, Wd)
        return y

    @staticmethod
    def backward(ctx, dy):
        h1, h2, idx, pidx = ctx.saved_tensors
        bank, active = ctx.bank, ctx.active
        N, H, Wd = ctx.shape
        G = len(active)
        slots = L.iarr(active)
        dev = dy.device
        dy = dy.contiguous()
        dyb = torch.empty((G * N, H, 1, Wd, 4), device=dev, dtype=torch.float32)
        L.call('risp_to_blocked', L.ptr(dy), L.ptr(dyb), G * N, 3, 1, H, Wd, L.stream())
        dh2 = _gconv(dyb, None, bank['W3T'], None, 0, None, None, G, N, slots, 0, 0, 3, 32, 5, 0)
        dh1 = _gconv(dh2, h2, bank['W2T'], None, 0, None, None, G, N, slots, 0, 0, 32, 64, 5, 0)
        dxg = _gconv(dh1, h1, bank['W1T'], None, 0, None, None, G, N, slots, 0, 0, 64, 3, 9, 0)
        Pmax, F, J = bank['Pmax'], bank['F'], bank['J']
        dtab = blocked_class_sums(dh1, h1, 64, 9).view(G * N, J)
        dfeat = torch.empty((G * N, F), device=dev, dtype=torch.float32)
        L.call('risp_bias_table_bwd_grouped', L.ptr(dtab), L.ptr(bank['S']), L.ptr(dfeat), G, N, slots, F, J, L.stream())
        dfeat = dfeat.view(G, N, F)
        dpar = dfeat[:, :, 9:].sum(dim=1).reshape(-1).index_select(0, pidx).view(1, -1) if ctx.needs_input_grad[1] else None
        dx = None
        if ctx.needs_input_grad[0]:
            dst = dfeat[:, :, :9].sum(dim=0)                                         # (N, 9) = d [min | mean | max]
            gp = dst.reshape(N, 3, 3).permute(0, 2, 1).contiguous()                  # (N, C, 3) like the statistics
            dx = torch.empty((N, 3, H, Wd), device=dev, dtype=torch.float32)
            L.call('risp_plane_stats_bwd', L.ptr(gp), L.ptr(idx), L.ptr(dx), N * 3, H * Wd, L.stream())
            # first-layer data gradients + the residual path of every member, summed over the bank
            dxb = (dxg + dyb).view(G, N, H, 1, Wd, 4).sum(dim=0)
            dxp = torch.empty((N, 3, H, Wd), device=dev, dtype=torch.float32)
            L.call('risp_from_blocked', L.ptr(dxb), L.ptr(dxp), N, 3, 1, H, Wd, L.stream())
            dx += dxp
        return dx, dpar, None, None


def srcnn_res_bank(x, par_cat, bank, active):
    return _SRCNNResBankFn.apply(x, par_cat, bank, active)


def conv2d_tc(xb, weight, bias=None, relu_in=False, relu_out=False, residual=None, residual_relu=False, bias_tab=None):
    """Blocked in, blocked out.  bias_tab (N, K*K*pad16(Cout)): differentiable position-class bias (instead of `bias`)."""
    return _ConvTcFn.apply(xb, residual, weight, bias, relu_in, relu_out, residual_relu, bias_tab)
