"""GPU checks of the evaluation metric (tensor2bgr -> per-image PSNR of test.py / test_split.py):

* `ops.sse_u8` against the numpy restatement (oracle/metrics_oracle.py) on edge values, ragged widths and a 12 MP worst case;
* the evaluation mode of the pipeline kernels (`ops.pipeline_eval`): packed signatures, demosaic only and interpreter chains
  give exactly `sse_u8(pipeline_fwd(...), gt)` and the 8-bit image of `to_u8_hwc`, byte for byte, also under RISP_FUSED=0
  and with 2-row items (both read once per process: child processes);
* `_Universal.evaluate` and `IspModel.evaluate` against the metric of the forward, and the CPU oracle pipeline within the
  tolerance of the fp32 forward."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
pytestmark = pytest.mark.gpu

from oracle import isp_oracle as O             # noqa: E402  (the checkers)
from oracle import metrics_oracle as M         # noqa: E402

IDENT = [0.0] * 30
IDENT[6] = IDENT[17] = IDENT[28] = 1.0
SIGS = {
    'A': ['gain', 'poly10', 'gamma', ('gtm', 4)],
    'B': ['gamma', 'poly10', 'gain'],
    'C': ['gamma', 'poly10'],
    'D': ['gamma', ('gtm', 4)],
    'skip': [],                                  # demosaic only
}
GENERIC = {                                      # chains without a packed signature: the interpreter kernel
    's7isp': ['filmic', 'gamma', 'poly10'],      # OriginUniversal ..._Demosaic_01_sRGB_04_01_13 (nearest -> filmic -> gamma -> poly)
    'gtm5': ['gamma', ('gtm', 5), 'gain_clip'],
    'ccm': ['gain', 'ccm', 'gamma'],
    'crysis': ['crysis', ('gtm', 4)],
}
KINDS = ['nearest', 'bilinear', 'malvar']
SHAPES = [(2, 12, 132), (1, 6, 8), (3, 50, 520)]   # partial last strip, the smallest frame, several strips


def stage_params(st, g, knots=(0.2, 0.5, 0.8)):
    vals = []
    for s in st:
        name, iarg = (s, 0) if isinstance(s, str) else s
        if name in ('gain', 'gain_clip'):
            vals += [1.1, 0.9, 1.2]
        elif name == 'poly10':
            vals += (torch.tensor(IDENT) + torch.randn(30, generator=g) * 0.03).tolist()
        elif name == 'gamma':
            vals += [0.55]
        elif name == 'gtm':
            vals += list(knots) if iarg == 4 else torch.linspace(0.1, 0.9, iarg - 1).tolist()
        elif name == 'ccm':
            vals += [0.9, 0.05, 0.05, 0.1, 0.8, 0.1, 0.0, 0.1, 0.9]
        elif name == 'filmic':
            vals += [2.0, 1.3]
        elif name == 'crysis':
            vals += [1.7]
    return torch.tensor([vals])


def inputs(N, H, W, seed):
    """raw with exact 0 / 1 samples, GT over [-0.1, 1.1] with exact k/255 codes, their fp32 neighbours and a NaN."""
    g = torch.Generator().manual_seed(seed)
    raw = torch.rand(N, 1, H, W, generator=g) * 1.05
    raw.view(-1)[:3] = torch.tensor([0., 1., 0.5])
    gt = torch.rand(N, 3, H, W, generator=g) * 1.2 - 0.1
    k = torch.randint(0, 256, (N, 3, H, W), generator=g).float() / 255.
    pick = torch.rand(N, 3, H, W, generator=g)
    gt = torch.where(pick < 0.3, k, gt)
    gt = torch.where((pick >= 0.3) & (pick < 0.4), torch.nextafter(k, torch.tensor(-1.0)), gt)
    gt.view(-1)[5] = float('nan')
    return raw, gt, g


@pytest.fixture(scope='module')
def ops():
    import reconfigisp_b200.ops as ops
    return ops


def check_eval(ops, raw, gt, kind, chain, params):
    """pipeline_eval == sse_u8(pipeline_fwd) exactly, and its 8-bit image == to_u8_hwc of every output image."""
    raw, gt = raw.cuda(), gt.cuda()
    p = None if params is None else params.cuda()
    y = ops.pipeline_fwd(raw, kind, chain, p)
    ref = ops.sse_u8(y, gt)
    sse, u8 = ops.pipeline_eval(raw, gt, kind, chain, p, u8=True)
    sse2, none = ops.pipeline_eval(raw, gt, kind, chain, p)
    assert none is None and sse.dtype == torch.int64 and u8.shape == (raw.shape[0], raw.shape[2], raw.shape[3], 3)
    assert torch.equal(sse, ref), (sse.tolist(), ref.tolist())
    assert torch.equal(sse2, ref)
    for n in range(raw.shape[0]):
        assert torch.equal(u8[n], ops.to_u8_hwc(y[n]))
    return sse.cpu()


# ---- standalone metric --------------------------------------------------------------------------------------------
def test_sse_u8_equals_numpy_on_edge_values(ops):
    g = torch.Generator().manual_seed(11)
    for (N, C, H, W) in [(3, 3, 17, 37), (2, 3, 8, 1000), (1, 1, 5, 3), (2, 4, 9, 130)]:     # ragged W, odd sizes
        k = torch.randint(0, 256, (N, C, H, W), generator=g).float() / 255.
        y = torch.rand(N, C, H, W, generator=g) * 1.4 - 0.2
        pick = torch.rand(N, C, H, W, generator=g)
        y = torch.where(pick < 0.25, k, y)
        y = torch.where((pick >= 0.25) & (pick < 0.35), torch.nextafter(k, torch.tensor(2.0)), y)
        y = torch.where((pick >= 0.35) & (pick < 0.45), torch.nextafter(k, torch.tensor(-1.0)), y)
        y.view(-1)[:4] = torch.tensor([float('nan'), float('inf'), -float('inf'), 1.0])
        gt = torch.rand(N, C, H, W, generator=g) * 1.2 - 0.1
        gt.view(-1)[7] = float('nan')
        ref = M.sse_u8(y.numpy(), gt.numpy())
        got = ops.sse_u8(y.cuda(), gt.cuda())
        assert got.dtype == torch.int64 and got.is_cuda
        assert np.array_equal(got.cpu().numpy(), ref), (got.tolist(), ref)
        # the 3-D form, and images that start off a 16-byte boundary (views into the batch): scalar head
        yc, gc = y.cuda(), gt.cuda()
        assert int(ops.sse_u8(yc[-1], gc[-1])[0]) == int(ref[-1])
        if N > 1:
            assert np.array_equal(ops.sse_u8(yc[1:], gc[1:]).cpu().numpy(), ref[1:])      # offset views: scalar head
    from reconfigisp_b200 import metrics
    assert np.array_equal(metrics.psnr(y.cuda(), gt.cuda()), M.psnr(y.numpy(), gt.numpy()))


def test_sse_u8_12mp_worst_case_exceeds_32_bits(ops):
    H, W = 3000, 4000
    y = torch.ones(1, 3, H, W, device='cuda')
    gt = torch.zeros(1, 3, H, W, device='cuda')
    assert int(ops.sse_u8(y, gt)[0]) == 3 * H * W * 65025
    raw = torch.ones(1, 1, H, W, device='cuda')
    sse, _ = ops.pipeline_eval(raw, gt, 'nearest', ops.Chain([]))         # demosaic of a white frame is white
    assert int(sse[0]) == 3 * H * W * 65025


# ---- evaluation mode of the pipeline kernels ---------------------------------------------------------------------------
@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('sig', sorted(SIGS))
def test_fused_eval_equals_forward_metric(ops, kind, sig):
    st = SIGS[sig]
    chain = ops.Chain(st)
    assert sig == 'skip' or ops.fused_chain_supported(chain)
    for (N, H, W) in SHAPES:
        raw, gt, g = inputs(N, H, W, sum(map(ord, kind + sig)) + H * W)
        params = stage_params(st, g) if chain.P else None
        check_eval(ops, raw, gt, kind, chain, params)
        if chain.P:
            rows = params.repeat(N, 1) * (1 + 0.01 * torch.arange(N).view(N, 1))    # per-image parameter rows
            check_eval(ops, raw, gt, kind, chain, rows)
    if 'gtm' in [s if isinstance(s, str) else s[0] for s in st]:
        raw, gt, g = inputs(2, 20, 136, 5)
        for knots in ((-0.2, 0.5, 1.3), (0.6, 0.3, 0.9)):                          # out-of-[0,1] knots: final clamp
            check_eval(ops, raw, gt, kind, chain, stage_params(st, g, knots))


@pytest.mark.parametrize('name', sorted(GENERIC))
def test_generic_eval_equals_forward_metric(ops, name):
    st = GENERIC[name]
    chain = ops.Chain(st)
    assert not ops.fused_chain_supported(chain)
    for kind in KINDS:
        for (N, H, W) in SHAPES:
            raw, gt, g = inputs(N, H, W, sum(map(ord, kind + name)) + H * W)
            params = stage_params(st, g)
            check_eval(ops, raw, gt, kind, chain, params)
            check_eval(ops, raw, gt, kind, chain, params.repeat(N, 1) * (1 + 0.01 * torch.arange(N).view(N, 1)))


def child_cases(out):
    """Run in a child process: every packed signature and two interpreter chains, checked there; the sums go to an npz."""
    import reconfigisp_b200.ops as ops
    res = {}
    for name, st in list(SIGS.items()) + [('s7isp', GENERIC['s7isp']), ('gtm5', GENERIC['gtm5'])]:
        chain = ops.Chain(st)
        for kind in KINDS:
            raw, gt, g = inputs(2, 260, 1000, sum(map(ord, kind + name)))
            params = stage_params(st, g) if chain.P else None
            res['%s_%s' % (name, kind)] = check_eval(ops, raw, gt, kind, chain, params).numpy()
    np.savez(out, **res)


def run_child(env_update, out):
    env = dict(os.environ)
    env.pop('RISP_FUSED', None)
    env.pop('RISP_FUSED_STEP_ROWS', None)
    env.update(env_update)
    cmd = [sys.executable] + (['-s'] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    return np.load(out)


def test_eval_under_interpreter_only_and_with_two_row_items(tmp_path):
    """RISP_FUSED=0: every chain takes the interpreter kernels, eval and forward alike (checked in the child).
    RISP_FUSED_STEP_ROWS=2: many 2-row items per CTA; the sums are integers, so they equal the default geometry's."""
    ref = run_child({}, tmp_path / 'default.npz')
    interp = run_child({'RISP_FUSED': '0'}, tmp_path / 'interp.npz')
    rows2 = run_child({'RISP_FUSED_STEP_ROWS': '2'}, tmp_path / 'rows2.npz')
    for k in ref.files:
        assert np.array_equal(rows2[k], ref[k]), k
        assert interp[k].shape == ref[k].shape


# ---- containers and the tuning driver ------------------------------------------------------------------------------
def _nets():
    from reconfigisp_b200.modules.isp_universal import IspUniversal
    from reconfigisp_b200.modules.origin_universal import OriginUniversal
    return [
        ('packed', lambda f: OriginUniversal('/x/', 'Bayer_02_Demosaic_02_sRGB_11_13_01_14', weight_seed=10, fuse=f), 'head'),
        ('packed_isp', lambda f: IspUniversal('/x/', (None,) * 6, 'Bayer_02_Demosaic_01_sRGB_11_13_01_14', weight_seed=10,
                                              fuse=f), 'head'),
        ('s7isp', lambda f: OriginUniversal('/x/', 'Bayer_02_Demosaic_01_sRGB_04_01_13', weight_seed=10, fuse=f), 'head'),
        ('cnn_last', lambda f: IspUniversal('/x/', (None,) * 4, 'Bayer_02_Demosaic_01_sRGB_11_12', weight_seed=10, fuse=f),
         'module'),
    ]


@pytest.mark.parametrize('fuse', [True, False])
def test_container_evaluate_equals_metric_of_forward(fuse):
    from reconfigisp_b200 import metrics, ops
    from reconfigisp_b200.synthetic import synthetic_frames
    raw, gt = synthetic_frames(2, 48, 136, seed=3)
    raw, gt = raw.cuda(), gt.cuda()
    for name, make, last in _nets():
        net = make(fuse).cuda()
        if fuse:
            segs = [s for s in net._make_plan() if not (s[0] == 'chain' and not s[2])]
            assert segs[-1][0] == last, (name, segs)
        with torch.no_grad():
            y = net(raw)
        inter = net.intermediate_results
        before = [p.detach().clone() for p in net.all_params]
        sse, u8 = net.evaluate(raw, gt, u8=True)
        assert net.intermediate_results is inter
        assert all(torch.equal(a, p.detach()) for a, p in zip(before, net.all_params))
        assert torch.equal(sse, ops.sse_u8(y, gt)), name
        assert np.array_equal(metrics.psnr_from_sse(sse, 3 * 48 * 136), metrics.psnr(y, gt))
        for n in range(2):
            assert torch.equal(u8[n], ops.to_u8_hwc(y[n])), name
        assert net.evaluate(raw, gt)[1] is None


def _model(seed_arch='Bayer_02_Demosaic_02_sRGB_11_13_01_14'):
    from reconfigisp_b200.tuning import IspModel
    opt = {'model': 'isp', 'is_train': True,
           'network_G': {'which_model_G': 'OriginUniversal', 'architecture': seed_arch, 'weight_seed': 10},
           'train': {'lr_G': 1e-2, 'beta1': 0.9, 'beta2': 0.99, 'pixel_criterion': 'l2', 'lr_scheme': 'MultiStepLR',
                     'lr_steps': [100], 'lr_gamma': 0.5}}
    return IspModel(opt)


def test_ispmodel_evaluate_codes_feed_and_training_untouched():
    from reconfigisp_b200 import metrics, ops
    g = torch.Generator().manual_seed(8)
    N, H, W = 2, 64, 136
    raw = torch.randint(0, 1024, (N, 1, H, W), generator=g, dtype=torch.int32).to(torch.int16)     # uint16-style codes
    gt = torch.randint(0, 256, (N, 3, H, W), generator=g, dtype=torch.int32).to(torch.uint8)
    a, b = _model(), _model()
    for m in (a, b):
        m.feed_data((raw, gt))
        for _ in range(3):
            m.optimize_parameters()
    # evaluate() on a (host uint16 / uint8 codes, decoded on the device) == the metric of test()[0]
    grad = a._flat_grad.clone()
    params = [p.detach().clone() for p in a.netG.trainable_parameters]
    sse, u8 = a.evaluate(u8=True)
    y, _ = a.test()
    assert torch.equal(sse, ops.sse_u8(y, a.gt))
    assert np.array_equal(metrics.psnr_from_sse(sse, 3 * H * W), metrics.psnr(y, a.gt))
    assert torch.equal(u8[1], ops.to_u8_hwc(y[1]))
    assert torch.equal(a._flat_grad, grad)
    assert all(torch.equal(p0, p.detach()) for p0, p in zip(params, a.netG.trainable_parameters))
    # the GT codes come back unchanged: q(c/255) == c
    assert torch.equal(torch.stack([ops.to_u8_hwc(a.gt[n]) for n in range(N)]).cpu(), gt.permute(0, 2, 3, 1))
    # a second host batch (the other buffer set), evaluated, then the next step: identical to the model that did not evaluate
    raw2 = torch.randint(0, 1024, (N, 1, H, W), generator=g, dtype=torch.int32).to(torch.int16)
    for m in (a, b):
        m.feed_data((raw2, gt))
    a.evaluate()
    for m in (a, b):
        m.optimize_parameters()
    assert torch.equal(a.l_pix, b.l_pix)
    for pa, pb in zip(a.netG.trainable_parameters, b.netG.trainable_parameters):
        assert torch.equal(pa.detach(), pb.detach())


def test_eval_against_cpu_oracle(ops):
    """Catches a wrong forward (not only a self-consistent one): PSNR within 0.01 dB of the fp64 oracle pipeline and the
    numpy metric; at most 0.1 % of the codes differ, none by more than 1 (the 1e-4 forward tolerance can flip a truncation)."""
    N, H, W = 2, 48, 264
    g = torch.Generator().manual_seed(12)
    raw = torch.rand(N, 1, H, W, generator=g)
    gt = torch.randint(0, 256, (N, 3, H, W), generator=g).float() / 255.
    st = SIGS['A']
    chain = ops.Chain(st)
    p = stage_params(st, g)
    x = O.demosaic_bilinear(raw.double())
    x = O.wb_manual(x, p[:, 0:3].double().expand(N, 3))
    x = O.wb_quadratic(x, ((p[:, 3:33].double() + 5) / 10).expand(N, 30))
    x = O.gamma_manual(x, p[:, 33:34].double().expand(N, 1))
    yo = torch.cat([O.gtm_manual(x[i:i + 1], p[:, 34:37].double(), 4) for i in range(N)]).float().numpy()
    sse, u8 = ops.pipeline_eval(raw.cuda(), gt.cuda(), 'bilinear', chain, p.cuda(), u8=True)
    from reconfigisp_b200.metrics import psnr_from_sse
    got = psnr_from_sse(sse, 3 * H * W)
    ref = M.psnr(yo, gt.numpy())
    assert np.abs(got - ref).max() <= 0.01, (got, ref)
    codes = np.stack([M.tensor2bgr(yo[n]) for n in range(N)]).astype(int)
    diff = np.abs(u8.cpu().numpy().astype(int) - codes)
    assert diff.max() <= 1 and (diff > 0).mean() <= 1e-3, (diff.max(), (diff > 0).mean())


if __name__ == '__main__':
    child_cases(sys.argv[1])
