"""GPU checks of the per-image 8-bit SSIM (`ops.ssim_u8`, `metrics.ssim`, `evaluate(..., ssim=True)`):

* against the numpy oracle (oracle/ssim_oracle.py) within 1e-6 per image, on edge values, the smallest frame, ragged widths,
  several strips, a flat region with +-1-code noise and a 12 MP pair;
* exact properties of the integer sums: identical operands give C (H-6)(W-6) 2^32, swapped operands the same sums, and the
  fp32 NCHW operand, its 8-bit NHWC image, an image alone, inside a batch and as an offset view all give the same bits;
* the containers' and the tuning driver's `evaluate(ssim=True)`, the tiled path, and capture in a CUDA graph."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
pytestmark = pytest.mark.gpu

from oracle import ssim_oracle as SO           # noqa: E402

SHAPES = [(3, 3, 17, 37), (2, 3, 7, 7), (1, 1, 9, 1000), (2, 4, 9, 130), (3, 3, 50, 520)]
TOL = 1e-6


@pytest.fixture(scope='module')
def ops():
    import reconfigisp_b200.ops as ops
    return ops


def edge_pair(N, C, H, W, seed):
    """y over [-0.2, 1.2] with exact k/255 codes, their fp32 neighbours, NaN and +-inf; gt over [-0.1, 1.1] with a NaN
    (the generator of the PSNR tests)."""
    g = torch.Generator().manual_seed(seed)
    k = torch.randint(0, 256, (N, C, H, W), generator=g).float() / 255.
    y = torch.rand(N, C, H, W, generator=g) * 1.4 - 0.2
    pick = torch.rand(N, C, H, W, generator=g)
    y = torch.where(pick < 0.25, k, y)
    y = torch.where((pick >= 0.25) & (pick < 0.35), torch.nextafter(k, torch.tensor(2.0)), y)
    y = torch.where((pick >= 0.35) & (pick < 0.45), torch.nextafter(k, torch.tensor(-1.0)), y)
    y.view(-1)[:4] = torch.tensor([float('nan'), float('inf'), -float('inf'), 1.0])
    gt = torch.rand(N, C, H, W, generator=g) * 1.2 - 0.1
    gt = torch.where(pick < 0.5, (y + (torch.rand(N, C, H, W, generator=g) - 0.5) * 0.05).nan_to_num(0.3), gt)
    gt.view(-1)[7] = float('nan')
    return y, gt


def u8_of(ops, y):
    return torch.stack([ops.to_u8_hwc(y[n]) for n in range(y.shape[0])])


def misaligned(t):
    """A copy of t that starts 1 element past an allocation (off every vector boundary): the scalar load path."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


def check_against_oracle(ops, y, gt):
    from reconfigisp_b200 import metrics
    N, C, H, W = gt.shape
    sums = ops.ssim_u8(y.cuda(), gt.cuda())
    assert sums.dtype == torch.int64 and sums.is_cuda and sums.shape == (N,)
    got = metrics.ssim_from_sums(sums, C, H, W)
    ref = SO.ssim(y.numpy(), gt.numpy())
    assert np.abs(got - ref).max() <= TOL, (got, ref)
    return sums


def test_ssim_u8_equals_oracle_on_edge_values(ops):
    for i, (N, C, H, W) in enumerate(SHAPES):
        y, gt = edge_pair(N, C, H, W, 30 + i)
        sums = check_against_oracle(ops, y, gt)
        yc, gc = y.cuda(), gt.cuda()
        # the 3-D form, each image alone, the tail of the batch as an offset view, and unaligned copies (scalar loads)
        for n in range(N):
            assert torch.equal(ops.ssim_u8(yc[n], gc[n]), sums[n:n + 1]), (N, C, H, W, n)
        if N > 1:
            assert torch.equal(ops.ssim_u8(yc[1:], gc[1:]), sums[1:])
        assert torch.equal(ops.ssim_u8(misaligned(yc), misaligned(gc)), sums)
        assert torch.equal(ops.ssim_u8(misaligned(yc), gc), sums)
        # the 8-bit NHWC operand: the same codes, so the same bits (vector and scalar byte paths)
        u8 = u8_of(ops, yc)
        assert torch.equal(ops.ssim_u8(u8, gc), sums), (N, C, H, W)
        assert torch.equal(ops.ssim_u8(misaligned(u8), gc), sums)
        assert torch.equal(ops.ssim_u8(u8[-1], gc[-1]), sums[-1:])
        # swapped operands
        assert torch.equal(ops.ssim_u8(gc, yc), sums)


def test_flat_region_with_one_code_noise(ops):
    """Constant code 200 against itself plus +-1-code noise: S is close to its cancellation point there, and moments
    formed in fp32 miss the oracle by about 1e-5."""
    g = torch.Generator().manual_seed(5)
    for (N, C, H, W) in [(2, 3, 64, 200), (1, 3, 300, 1004)]:
        codes = torch.full((N, C, H, W), 200.)
        y = codes / 255.
        gt = (codes + torch.randint(-1, 2, (N, C, H, W), generator=g).float()) / 255.
        check_against_oracle(ops, y, gt)
        check_against_oracle(ops, gt, y)


def test_identical_operands_give_exactly_one_and_swaps_are_symmetric(ops):
    from reconfigisp_b200 import metrics
    for i, (N, C, H, W) in enumerate(SHAPES):
        y, gt = edge_pair(N, C, H, W, 60 + i)
        yc, gc = y.cuda(), gt.cuda()
        full = C * (H - 6) * (W - 6) * 2 ** 32
        for t in (yc, gc):
            assert ops.ssim_u8(t, t).tolist() == [full] * N
            assert ops.ssim_u8(u8_of(ops, t), t).tolist() == [full] * N
        assert metrics.ssim(yc, yc).tolist() == [1.0] * N
        assert torch.equal(ops.ssim_u8(yc, gc), ops.ssim_u8(gc, yc))


def test_batch_position_does_not_change_the_sums(ops):
    """The row chunking follows N, so an image alone, inside a larger batch and at any position is scored on another
    grid: integer sums, the same bits."""
    y, gt = edge_pair(9, 3, 203, 1000, 77)
    yc, gc = y.cuda(), gt.cuda()
    full = ops.ssim_u8(yc, gc)
    for n in (0, 4, 8):
        assert torch.equal(ops.ssim_u8(yc[n], gc[n]), full[n:n + 1])
    perm = torch.tensor([8, 3, 0, 5, 1, 7, 2, 6, 4])
    assert torch.equal(ops.ssim_u8(yc[perm], gc[perm]), full[perm.cuda()])
    assert torch.equal(ops.ssim_u8(yc[2:7], gc[2:7]), full[2:7])


def test_pipeline_eval_image_scores_like_the_forward(ops):
    """The (N,H,W,3) image of pipeline_eval(u8=True) is to_u8_hwc of the forward, so its SSIM is the forward's, bit for bit."""
    g = torch.Generator().manual_seed(3)
    N, H, W = 3, 50, 520
    raw = torch.rand(N, 1, H, W, generator=g).cuda()
    gt = torch.rand(N, 3, H, W, generator=g).cuda()
    chain = ops.Chain(['gamma', ('gtm', 4)])
    p = torch.tensor([[0.55, 0.2, 0.5, 0.8]]).cuda()
    y = ops.pipeline_fwd(raw, 'bilinear', chain, p)
    _, u8 = ops.pipeline_eval(raw, gt, 'bilinear', chain, p, u8=True)
    assert u8.shape == (N, H, W, 3)
    assert torch.equal(ops.ssim_u8(u8, gt), ops.ssim_u8(y, gt))


def test_12mp_pair_against_oracle_and_repeatable(ops):
    H, W = 3000, 4000
    g = torch.Generator().manual_seed(12)
    gt = torch.rand(1, 3, H, W, generator=g)
    y = (gt + (torch.rand(1, 3, H, W, generator=g) - 0.5) * 0.1).clamp(-0.05, 1.05)
    sums = check_against_oracle(ops, y, gt)
    yc, gc = y.cuda(), gt.cuda()
    assert torch.equal(ops.ssim_u8(yc, gc), sums)
    assert torch.equal(ops.ssim_u8(u8_of(ops, yc), gc), sums)


# ---- containers, the tuning driver, the tiled path ----------------------------------------------------------------
NETS = {'A': 'Bayer_02_Demosaic_02_sRGB_11_13_01_14',        # bilinear, gain, 3x10 polynomial, gamma, tone curve
        'D': 'Bayer_02_Demosaic_02_sRGB_01_14'}              # bilinear, gamma, tone curve


@pytest.mark.parametrize('name', sorted(NETS))
def test_container_evaluate_with_ssim(name):
    from reconfigisp_b200 import ops
    from reconfigisp_b200.modules.origin_universal import OriginUniversal
    from reconfigisp_b200.synthetic import synthetic_frames
    raw, gt = synthetic_frames(2, 48, 136, seed=3)
    raw, gt = raw.cuda(), gt.cuda()
    net = OriginUniversal('/x/', NETS[name], weight_seed=10, fuse=True).cuda()
    ref_net = OriginUniversal('/x/', NETS[name], weight_seed=10, fuse=False).cuda()
    segs = [s for s in net._make_plan() if not (s[0] == 'chain' and not s[2])]
    assert segs[-1][0] == 'head', segs                      # the evaluation mode of the pipeline kernels
    with torch.no_grad():
        y = net(raw)
        y_seq = ref_net(raw)
    inter = net.intermediate_results
    before = [p.detach().clone() for p in net.all_params]
    plain = net.evaluate(raw, gt)
    assert len(plain) == 2 and plain[1] is None and torch.equal(plain[0], ops.sse_u8(y, gt))
    sse, none, sums = net.evaluate(raw, gt, ssim=True)
    assert none is None
    sse8, u8, sums8 = net.evaluate(raw, gt, u8=True, ssim=True)
    assert torch.equal(sse, plain[0]) and torch.equal(sse8, plain[0])
    ref = ops.ssim_u8(y, gt)
    assert torch.equal(sums, ref) and torch.equal(sums8, ref), name
    assert torch.equal(u8, u8_of(ops, y))
    assert net.intermediate_results is inter
    assert all(torch.equal(a, p.detach()) for a, p in zip(before, net.all_params))
    # the unfused net: the forward and then ssim_u8 on it
    s2 = ref_net.evaluate(raw, gt, ssim=True)
    assert len(s2) == 3 and s2[1] is None and torch.equal(s2[2], ops.ssim_u8(y_seq, gt))
    if torch.equal(y, y_seq):
        assert torch.equal(s2[2], sums)
    from reconfigisp_b200 import metrics
    assert np.abs(metrics.ssim_from_sums(s2[2], 3, 48, 136) - metrics.ssim_from_sums(sums, 3, 48, 136)).max() <= 1e-4


def test_ispmodel_evaluate_with_ssim_leaves_training_alone():
    from reconfigisp_b200 import ops
    from reconfigisp_b200.tuning import IspModel

    def model():
        opt = {'model': 'isp', 'is_train': True,
               'network_G': {'which_model_G': 'OriginUniversal', 'architecture': NETS['A'], 'weight_seed': 10},
               'train': {'lr_G': 1e-2, 'beta1': 0.9, 'beta2': 0.99, 'pixel_criterion': 'l2', 'lr_scheme': 'MultiStepLR',
                         'lr_steps': [100], 'lr_gamma': 0.5}}
        return IspModel(opt)

    g = torch.Generator().manual_seed(8)
    N, H, W = 2, 64, 136
    raw = torch.randint(0, 1024, (N, 1, H, W), generator=g, dtype=torch.int32).to(torch.int16)
    gt = torch.randint(0, 256, (N, 3, H, W), generator=g, dtype=torch.int32).to(torch.uint8)
    a, b = model(), model()
    for m in (a, b):
        m.feed_data((raw, gt))
        for _ in range(3):
            m.optimize_parameters()
    grad = a._flat_grad.clone()
    params = [p.detach().clone() for p in a.netG.trainable_parameters]
    sse, none, sums = a.evaluate(ssim=True)
    y, _ = a.test()
    assert none is None
    assert torch.equal(sse, ops.sse_u8(y, a.gt))
    assert torch.equal(sums, ops.ssim_u8(y, a.gt))
    assert torch.equal(a._flat_grad, grad)
    assert all(torch.equal(p0, p.detach()) for p0, p in zip(params, a.netG.trainable_parameters))
    raw2 = torch.randint(0, 1024, (N, 1, H, W), generator=g, dtype=torch.int32).to(torch.int16)
    for m in (a, b):
        m.feed_data((raw2, gt))
    a.evaluate(u8=True, ssim=True)
    for m in (a, b):
        m.optimize_parameters()
    assert torch.equal(a.l_pix, b.l_pix)
    for pa, pb in zip(a.netG.trainable_parameters, b.netG.trainable_parameters):
        assert torch.equal(pa.detach(), pb.detach())


def test_tiled_path_uint8_equals_clipped_float(ops):
    from reconfigisp_b200 import metrics
    from reconfigisp_b200.patch import split_inference
    g = torch.Generator().manual_seed(4)
    H, W, ps, st = 200, 264, 64, 56
    raw = torch.rand(1, 1, H, W, generator=g).cuda()
    gt = torch.rand(3, H, W, generator=g).cuda()
    chain = ops.Chain(['gain', 'gamma'])
    p = torch.tensor([[1.3, 1.0, 0.8, 0.5]]).cuda()
    fn = lambda t: ops.pipeline_fwd(t, 'bilinear', chain, p)            # noqa: E731  gain > 1: values above 1 to clip
    img8 = split_inference(fn, raw, ps, st, uint8=True)
    imgf = split_inference(fn, raw, ps, st, clip01=True)
    assert img8.shape == (H, W, 3) and img8.dtype == torch.uint8
    a, b = metrics.ssim(img8, gt), metrics.ssim(imgf, gt)
    assert a.shape == (1,) and np.array_equal(a, b)
    assert np.abs(a - SO.ssim(imgf[None].cpu().numpy(), gt[None].cpu().numpy())).max() <= TOL


def test_ssim_u8_replays_in_a_cuda_graph(ops):
    y, gt = edge_pair(2, 3, 130, 520, 9)
    yc, gc = y.cuda(), gt.cuda()
    u8 = u8_of(ops, yc)
    ref = ops.ssim_u8(yc, gc)
    ref8 = ops.ssim_u8(u8, gc)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                       # warm-up on the capture stream
        ops.ssim_u8(yc, gc)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = ops.ssim_u8(yc, gc)
        out8 = ops.ssim_u8(u8, gc)
    for _ in range(3):
        out.fill_(-1)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, ref) and torch.equal(out8, ref8)


def test_bad_shapes_raise(ops):
    y = torch.rand(1, 3, 6, 20, device='cuda')
    with pytest.raises(ValueError):
        ops.ssim_u8(y, y)
    y = torch.rand(1, 3, 20, 6, device='cuda')
    with pytest.raises(ValueError):
        ops.ssim_u8(y, y)
    a, b = torch.rand(1, 3, 20, 20, device='cuda'), torch.rand(1, 3, 20, 21, device='cuda')
    with pytest.raises(ValueError):
        ops.ssim_u8(a, b)
    with pytest.raises(ValueError):
        ops.ssim_u8(u8_of(ops, a).permute(0, 3, 1, 2), a)               # an NCHW byte image is not the layout
