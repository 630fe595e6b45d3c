"""CUDA-event times of the per-image 8-bit SSIM on 4 x 12 MP frames (576 MB of fp32 output + GT, well above L2):

  1. ops.ssim_u8 with an fp32 NCHW output (24 B/px read) and with its 8-bit NHWC image (15 B/px read)
  2. net.evaluate() against net.evaluate(ssim=True) on chains A and D (fused head: the SSIM reads the evaluation mode's
     8-bit image)
  3. the same SSIM composed from torch ops on the same GPU: codes, then float64 avg_pool2d of the five moments
  4. one frame through the host: D2H of the fp32 output and GT + the numpy oracle (host clock, for scale)

Prints the GPU's name, power limit and maximum SM clock, then one line per variant: ms per 48 MP and the algorithmic bytes
over the time against the measured HBM peak.

    python scripts/time_ssim.py [launches=30] [repeats=3]
"""
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402
from oracle import ssim_oracle as SO  # noqa: E402
from oracle.metrics_oracle import tensor2bgr  # noqa: E402
from reconfigisp_b200 import metrics, ops  # noqa: E402
from reconfigisp_b200.modules.origin_universal import OriginUniversal  # noqa: E402
from reconfigisp_b200.synthetic import synthetic_frames  # noqa: E402

N, H, W = 4, 3000, 4000
HBM_PEAK = 6532e9          # B/s, the measured peak DESIGN.md §7 uses
NETS = {'A 11_13_01_14 bilinear': 'Bayer_02_Demosaic_02_sRGB_11_13_01_14',
        'D 01_14 bilinear': 'Bayer_02_Demosaic_02_sRGB_01_14'}


def gpu_info():
    q = 'name,power.limit,clocks.max.sm'
    r = subprocess.run(['nvidia-smi', '--query-gpu=' + q, '--format=csv,noheader'], capture_output=True, text=True)
    return r.stdout.strip() or torch.cuda.get_device_name()


def event_ms(fn, launches, repeats):
    for _ in range(5):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        e0.record()
        for _ in range(launches):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1) / launches)
    return statistics.median(ms), ms


def torch_ssim(y, gt):
    """The definition composed from torch ops: tensor2bgr codes, float64 7x7 means of the five moments (avg_pool2d without
    padding gives the interior pixels only), skimage's formula, the mean per image."""
    def codes(v):
        return torch.nan_to_num(v * 255, nan=0.0).clamp(0, 255).trunc().double()
    a, b = codes(y), codes(gt)
    box = lambda t: F.avg_pool2d(t, 7, stride=1)                       # noqa: E731
    ua, ub = box(a), box(b)
    va, vb, vab = box(a * a) - ua * ua, box(b * b) - ub * ub, box(a * b) - ua * ub
    cn = 49.0 / 48.0
    c1, c2 = (0.01 * 255) ** 2, (0.03 * 255) ** 2
    s = (2 * ua * ub + c1) * (2 * cn * vab + c2) / ((ua * ua + ub * ub + c1) * (cn * (va + vb) + c2))
    return s.mean(dim=(1, 2, 3))


def line(label, med, ms, bpp):
    bw = '' if bpp is None else '   %2d B/px / time = %.3f of peak' % (bpp, bpp * N * H * W / (med * 1e-3) / HBM_PEAK)
    print('  %-36s %8.4f ms per %.0f MP%s   (repeats: %s)' % (label, med, N * H * W / 1e6, bw,
                                                             ' '.join('%.4f' % x for x in ms)))


def main():
    launches = int(sys.argv[1]) if len(sys.argv) > 1 else 30
    repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    print('gpu:', gpu_info())
    raw, gt = synthetic_frames(N, H, W, seed=10)
    raw, gt = raw.cuda(), gt.cuda()
    print('frames: %d x %dx%d (%.0f MP), launches %d x repeats %d; HBM peak %.0f GB/s' % (N, H, W, N * H * W / 1e6, launches,
                                                                                       repeats, HBM_PEAK / 1e9))
    chain = ops.Chain(['gamma', ('gtm', 4)])
    p = torch.tensor([[0.5, 0.25, 0.5, 0.75]], device='cuda')
    y = ops.pipeline_fwd(raw, 'bilinear', chain, p)
    _, u8 = ops.pipeline_eval(raw, gt, 'bilinear', chain, p, u8=True)
    ref = ops.ssim_u8(y, gt)
    assert torch.equal(ops.ssim_u8(u8, gt), ref)
    val = metrics.ssim_from_sums(ref, 3, H, W)
    tv = torch_ssim(y, gt).cpu().numpy()
    print('\n[ssim_u8, output of chain D]  SSIM: %s   torch float64 composition: %s   max diff %.2e'
          % (' '.join('%.6f' % v for v in val), ' '.join('%.6f' % v for v in tv), np.abs(val - tv).max()))
    for label, fn, bpp, n in [('ssim_u8 fp32 / fp32', lambda: ops.ssim_u8(y, gt), 24, launches),
                              ('ssim_u8 u8 NHWC / fp32', lambda: ops.ssim_u8(u8, gt), 15, launches),
                              ('torch float64 avg_pool2d composition', lambda: torch_ssim(y, gt), 24, 3)]:
        med, ms = event_ms(fn, n, repeats)
        line(label, med, ms, bpp)

    for name, arch in NETS.items():
        net = OriginUniversal('/x/', arch, weight_seed=10, fuse=True).cuda()
        sse, _, sums = net.evaluate(raw, gt, ssim=True)
        assert torch.equal(sse, net.evaluate(raw, gt)[0])
        print('\n[evaluate, chain %s]  PSNR %s  SSIM %s' % (name, ' '.join('%.3f' % v for v in metrics.psnr_from_sse(sse, 3 * H * W)),
                                                          ' '.join('%.6f' % v for v in metrics.ssim_from_sums(sums, 3, H, W))))
        for label, fn in [('evaluate()', lambda: net.evaluate(raw, gt)),
                          ('evaluate(ssim=True)', lambda: net.evaluate(raw, gt, ssim=True))]:
            med, ms = event_ms(fn, launches, repeats)
            line(label, med, ms, None)

    ts = []
    for _ in range(2):
        torch.cuda.synchronize()
        t = time.perf_counter()
        yh, gh = y[0].cpu().numpy(), gt[0].cpu().numpy()
        v = SO.calculate_ssim(tensor2bgr(yh), tensor2bgr(gh))
        ts.append((time.perf_counter() - t) * 1e3)
    assert abs(v - val[0]) <= 1e-6, (v, val[0])
    print('\n  %-36s %8.1f ms per 12 MP frame (host clock; x%d for 48 MP)' % ('host: D2H + numpy oracle (1 frame)', min(ts), N))


if __name__ == '__main__':
    main()
