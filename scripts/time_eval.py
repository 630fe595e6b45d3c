"""CUDA-event times of evaluating a pipeline on 4 x 12 MP synthetic frames (768 MB of raw + GT, well above L2), against
what scoring the same output took before the evaluation mode existed:

  1. ops.pipeline_eval, without and with the 8-bit image (16 B/px read; + 3 B/px written with it)
  2. ops.pipeline_fwd alone (16 B/px: raw read, fp32 image written)
  3. the device composition: pipeline_fwd + to_u8_hwc of output and GT (per image) + the squared differences in torch
  4. one frame through the host: D2H of the fp32 output and GT + numpy tensor2bgr / PSNR (host clock, for scale)

Chains: signature A (Bayer_02_Demosaic_02_sRGB_11_13_01_14, bilinear), signature D (sRGB_01_14, bilinear), and the S7ISP
chain (nearest -> filmic -> gamma -> polynomial) on the interpreter kernel.  Prints the GPU's name, power limit and
maximum SM clock, then one line per variant: ms per 48 MP and 16 B/px over the time against the measured HBM peak.

    python scripts/time_eval.py [launches=50] [repeats=3]
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
from reconfigisp_b200 import metrics, ops  # noqa: E402
from reconfigisp_b200.synthetic import synthetic_frames  # noqa: E402

N, H, W = 4, 3000, 4000
HBM_PEAK = 6532e9          # B/s, the measured peak DESIGN.md §7 uses
IDENT = [0.0] * 30
IDENT[6] = IDENT[17] = IDENT[28] = 1.0
CHAINS = {
    'A 11_13_01_14 bilinear': ('bilinear', ['gain', 'poly10', 'gamma', ('gtm', 4)], [1.05, 1.0, 0.95] + IDENT + [0.5, 0.25, 0.5, 0.75]),
    'D 01_14 bilinear': ('bilinear', ['gamma', ('gtm', 4)], [0.5, 0.25, 0.5, 0.75]),
    'S7ISP 04_01_13 nearest (interpreter)': ('nearest', ['filmic', 'gamma', 'poly10'], [2.0, 1.3, 0.5] + IDENT),
}


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


def main():
    launches = int(sys.argv[1]) if len(sys.argv) > 1 else 50
    repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    print('gpu:', gpu_info())
    raw, gt = synthetic_frames(N, H, W, seed=10)
    raw, gt = raw.cuda(), gt.cuda()
    mp = N * H * W / 1e6
    print('frames: %d x %dx%d (%.0f MP), launches %d x repeats %d; HBM peak %.0f GB/s' % (N, H, W, mp, launches, repeats,
                                                                                       HBM_PEAK / 1e9))
    for name, (kind, st, vals) in CHAINS.items():
        chain = ops.Chain(st)
        p = torch.tensor([vals], device='cuda')
        y = ops.pipeline_fwd(raw, kind, chain, p)
        ref = ops.sse_u8(y, gt)
        assert torch.equal(ops.pipeline_eval(raw, gt, kind, chain, p)[0], ref)

        def compose():
            yy = ops.pipeline_fwd(raw, kind, chain, p)
            out = []
            for n in range(N):
                a, b = ops.to_u8_hwc(yy[n]), ops.to_u8_hwc(gt[n])
                out.append(((a.int() - b.int()) ** 2).sum(dtype=torch.int64))
            return torch.stack(out)
        assert torch.equal(compose(), ref)
        rows = [('pipeline_eval', lambda: ops.pipeline_eval(raw, gt, kind, chain, p)),
                ('pipeline_eval + u8', lambda: ops.pipeline_eval(raw, gt, kind, chain, p, u8=True)),
                ('pipeline_fwd alone', lambda: ops.pipeline_fwd(raw, kind, chain, p)),
                ('fwd + to_u8_hwc x2 + torch SSE', compose)]
        print('\n[%s]  PSNR of frame 0: %.4f dB' % (name, metrics.psnr_from_sse(ref, 3 * H * W)[0]))
        for label, fn in rows:
            med, ms = event_ms(fn, launches, repeats)
            print('  %-32s %8.4f ms per %.0f MP   16 B/px / time = %.3f of peak   (repeats: %s)'
                  % (label, med, mp, 16 * N * H * W / (med * 1e-3) / HBM_PEAK, ' '.join('%.4f' % x for x in ms)))
        # one frame through the host
        ts = []
        for _ in range(3):
            torch.cuda.synchronize()
            t = time.perf_counter()
            yh, gh = y[0].cpu().numpy(), gt[0].cpu().numpy()
            a = np.clip(np.transpose(yh, (1, 2, 0)) * np.float32(255), 0, 255).astype(np.uint8)
            b = np.clip(np.transpose(gh, (1, 2, 0)) * np.float32(255), 0, 255).astype(np.uint8)
            mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
            ts.append((time.perf_counter() - t) * 1e3)
            assert abs(mse * 3 * H * W - float(ref[0])) <= 1e-9 * float(ref[0]) + 1
        print('  %-32s %8.1f ms per 12 MP frame (host clock; x%d for 48 MP)' % ('host: D2H + numpy (1 frame)', min(ts), N))


if __name__ == '__main__':
    main()
