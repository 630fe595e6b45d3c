"""Narrow items of the fused step and evaluation kernels: when a frame's last strip is 1..64 columns wide, the warp marches
it as 128/nw lane groups on as many row pairs (csrc/risp_fused.cu).  Checked on remnants of 4..124 columns, frames
narrower than one strip and heights that are not multiples of 8:
* the step against the float64 oracle, with the tolerances of tests/test_fused_gpu.py, and the L1 step against this
  library's op-by-op path;
* the step's output image bit for bit against the same pixels computed by a full-width strip (the frame widened to a whole
  strip: the pixels away from the right border do not depend on the width), and every result bit-reproducible;
* the evaluation mode: exactly the sums and the 8-bit image of the inference kernel, which has no narrow items."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import isp_oracle as O   # noqa: E402  (the checker)

IDENT = [0.0] * 30
IDENT[6] = IDENT[17] = IDENT[28] = 1.0
SIGS = {'A': (['gain', 'poly10', 'gamma', ('gtm', 4)], [1.1, 0.9, 1.2] + IDENT + [0.55, 0.2, 0.5, 0.8]),
        'D': (['gamma', ('gtm', 4)], [0.55, 0.2, 0.5, 0.8])}
DM = {'bilinear': O.demosaic_bilinear, 'malvar': lambda r: O.demosaic_laplacian(r, 1.0)}
# W % 128 in {4, 28, 32, 36, 60, 64, 68, 124} and frames narrower than a strip; H % 8 != 0
WIDTHS = [132, 156, 288, 164, 188, 192, 196, 252, 32, 64, 100]
SHAPES = [(1 if i % 2 else 4, 54 if i % 2 else 38, w) for i, w in enumerate(WIDTHS)]


@pytest.fixture(scope='module')
def ops():
    import reconfigisp_b200.ops as ops
    return ops


def oracle_chain(x, st, p):
    N, o = x.shape[0], 0
    for s in st:
        name = s if isinstance(s, str) else s[0]
        if name == 'gain':
            x = O.wb_manual(x, p[:, o:o + 3]); o += 3
        elif name == 'poly10':
            x = O.wb_quadratic(x, (p[:, o:o + 30] + 5) / 10); o += 30
        elif name == 'gamma':
            x = O.gamma_manual(x, p[:, o:o + 1]); o += 1
        elif name == 'gtm':
            x = torch.cat([O.gtm_manual(x[i:i + 1], p[i:i + 1, o:o + 3], 4) for i in range(N)]); o += 3
    return x


def relclose(a, b, rtol=2e-3, atol=1e-6):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    lim = atol + rtol * float(b.abs().max())
    assert float((a - b).abs().max()) <= lim, (float((a - b).abs().max()), lim)


def inputs(N, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    raw = torch.rand(N, 1, H, W, generator=g) * 1.05
    gt = torch.rand(N, 3, H, W, generator=g)
    return raw, gt, g


def step(ops, raw, gt, kind, st, p):
    """-> y, loss, dparams of one fused MSE step (y written by the kernel)."""
    N, _, H, W = raw.shape
    y = torch.empty(N, 3, H, W, device='cuda')
    loss, dp = ops.PipelineStep(N, H, W, kind, ops.Chain(st), 'cuda')(raw, gt, p, y)
    return y, loss.clone(), dp.clone()


@pytest.mark.parametrize('kind', sorted(DM))
@pytest.mark.parametrize('sig', sorted(SIGS))
@pytest.mark.parametrize('shape', SHAPES)
def test_narrow_step_vs_oracle(ops, kind, sig, shape):
    N, H, W = shape
    raw, gt, g = inputs(N, H, W, W * 7 + H + len(kind + sig))
    st, vals = SIGS[sig]
    params = torch.tensor([vals]) + 0.02 * torch.randn(1, len(vals), generator=g)
    po = params.double().requires_grad_()
    yo = oracle_chain(DM[kind](raw.double()), st, po.expand(N, -1))
    lo = O.mse(yo, gt.double())
    dpo, = torch.autograd.grad(lo, po)
    y, _, _ = step(ops, raw.cuda(), gt.cuda(), kind, st, params.cuda())
    assert float((y.cpu().double() - yo.detach()).abs().max()) <= 1e-4
    pg = params.cuda().requires_grad_()
    lg = ops.pipeline_mse(pg, raw.cuda(), gt.cuda(), kind, ops.Chain(st))
    dpg, = torch.autograd.grad(lg, pg)
    assert abs(float(lg.detach()) - float(lo.detach())) <= 1e-5 * max(1.0, float(lo.detach()))
    relclose(dpg, dpo)
    # per-image parameter rows
    if N > 1:
        pN = params.repeat(N, 1) * (1 + 0.01 * torch.arange(N).view(N, 1))
        poN = pN.double().requires_grad_()
        doN, = torch.autograd.grad(O.mse(oracle_chain(DM[kind](raw.double()), st, poN), gt.double()), poN)
        pgN = pN.cuda().requires_grad_()
        dgN, = torch.autograd.grad(ops.pipeline_mse(pgN, raw.cuda(), gt.cuda(), kind, ops.Chain(st)), pgN)
        relclose(dgN, doN)


@pytest.mark.parametrize('shape', [(4, 38, 164), (1, 54, 32), (2, 1030, 1060)])
def test_narrow_l1_step_equals_op_by_op_path(ops, shape):
    N, H, W = shape
    raw, gt, g = inputs(N, H, W, 11 + W)
    raw, gt = raw.cuda(), gt.cuda()
    st, vals = SIGS['A']
    chain = ops.Chain(st)
    p1 = (torch.tensor([vals]) + 0.02 * torch.randn(1, len(vals), generator=g)).cuda().requires_grad_()
    d1, = torch.autograd.grad(ops.pipeline_l1(p1, raw, gt, 'bilinear', chain), p1)
    p2 = p1.detach().clone().requires_grad_()
    l2 = ops.l1_loss(ops.chain_apply(ops.demosaic(raw, 'bilinear'), chain, p2), gt)
    d2, = torch.autograd.grad(l2, p2)
    relclose(d1, d2, rtol=1e-3)


@pytest.mark.parametrize('kind', sorted(DM))
@pytest.mark.parametrize('shape', [(4, 38, 132), (1, 54, 32), (4, 1030, 1060), (4, 3000, 4000)])
def test_narrow_step_pixels_equal_full_strip(ops, kind, shape):
    """Narrow and full-width items compute each pixel with the same arithmetic: bit-identical images.  Loss, gradients
    and image are bit-reproducible (each CTA's item list and summation order are static)."""
    N, H, W = shape
    Ww = W - W % 128 + 128                  # the same frame widened to whole strips: no narrow item
    raw_w, gt_w, g = inputs(N, H, Ww, W + H)
    raw_w, gt_w = raw_w.cuda(), gt_w.cuda()
    raw, gt = raw_w[..., :W].contiguous(), gt_w[..., :W].contiguous()
    for sig, (st, vals) in SIGS.items():
        p = (torch.tensor([vals]) + 0.02 * torch.randn(1, len(vals), generator=g)).cuda()
        y0, l0, d0 = step(ops, raw, gt, kind, st, p)
        y1, l1, d1 = step(ops, raw, gt, kind, st, p)
        assert torch.equal(y0, y1) and torch.equal(l0, l1) and torch.equal(d0, d1), sig
        yw, _, _ = step(ops, raw_w, gt_w, kind, st, p)
        # columns W-2, W-1 read the reflected border
        assert torch.equal(y0[..., :W - 2], yw[..., :W - 2]), sig
        del y0, y1, yw


@pytest.mark.parametrize('kind', sorted(DM))
@pytest.mark.parametrize('shape', SHAPES[:8] + [(4, 1030, 1060)])
def test_narrow_eval_equals_inference(ops, kind, shape):
    N, H, W = shape
    raw, gt, g = inputs(N, H, W, 3 * W + H)
    raw, gt = raw.cuda(), gt.cuda()
    st, vals = SIGS['A']
    chain = ops.Chain(st)
    p = (torch.tensor([vals]) + 0.02 * torch.randn(1, len(vals), generator=g)).cuda()
    y = ops.pipeline_fwd(raw, kind, chain, p)
    sse, u8 = ops.pipeline_eval(raw, gt, kind, chain, p, u8=True)
    assert torch.equal(sse, ops.sse_u8(y, gt)), (sse.tolist(), ops.sse_u8(y, gt).tolist())
    for n in range(N):
        assert torch.equal(u8[n], ops.to_u8_hwc(y[n]))
