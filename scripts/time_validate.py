"""Time validation on the HBM-resident dataset: whole frames scored straight from the frame store's codes against the
composition it replaces, on one GPU.

    python scripts/time_validate.py [--reps 3] [--parent DIR --bench-rounds 3]

A store of 16 synthetic 12 MP frames (16-bit raw codes, 8-bit GT codes) is validated in batches of 4 frames (48 MP) with
chain A (bilinear), chain D (Malvar) and an interpreter chain (filmic, gamma, poly10; bilinear).  Per chain, ms per 48 MP:
  (a) store:        `ops.pipeline_eval_store` -- reads 2 B raw + 3 B GT codes per pixel (5 B/px);
  (b) composition:  `ops.sample_crops` of the whole frames into an fp32 batch (2 + 3 read, 16 written) + `ops.pipeline_eval`
                    (16 read): 37 B/px;
  (c) each with SSIM: (a) + the 8-bit image written (3 B/px) and `ops.ssim_u8_store` (3 + 3 read): 14 B/px;
                    (b) + the 8-bit image (3) and `ops.ssim_u8` against the fp32 GT (3 + 12): 55 B/px.
Achieved bandwidth is those bytes over CUDA-event time.  The store (16 x 12 MP x 5 B = 960 MB) is larger than L2, and a
timed pass walks all 16 frames.  Every timed window is checked: the store path's sums equal the composition's.
--parent DIR: also run `bench.py --no-cpu` alternately in this tree and in DIR (a checkout of another commit, built), to
show that the step kernels did not move."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import H, W, peaks  # noqa: E402
from reconfigisp_b200 import ops  # noqa: E402
from reconfigisp_b200.data import DeviceDataset  # noqa: E402
from reconfigisp_b200.synthetic import synthetic_frames  # noqa: E402

DATASHEET_HBM_GBS = 7700.0
IDENT = [0.0] * 30
IDENT[6] = IDENT[17] = IDENT[28] = 1.0
CHAINS = {
    'A (bilinear)': ('bilinear', ['gain', 'poly10', 'gamma', ('gtm', 4)], [1.1, 0.9, 1.2] + IDENT + [0.55, 0.2, 0.5, 0.8]),
    'D (malvar)': ('malvar', ['gamma', ('gtm', 4)], [0.55, 0.2, 0.5, 0.8]),
    'interpreter (bilinear)': ('bilinear', ['filmic', 'gamma', 'poly10'], [2.0, 1.3, 0.55] + IDENT),
}
BPX = {'store': 5, 'composition': 37, 'store+ssim': 14, 'composition+ssim': 55}


def timed(fn, n, warmup, reps):
    for _ in range(warmup):
        fn()
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / n)
    return out


def card():
    q = subprocess.run(['nvidia-smi', '-i', str(torch.cuda.current_device()), '--query-gpu=name,power.limit,clocks.max.sm',
                        '--format=csv,noheader'], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def bench_ab(parent, rounds):
    cmd = [sys.executable, 'bench.py', '--gpus', '1', '--no-cpu']
    res = {'this': [], 'parent': []}
    for r in range(rounds):
        for name, cwd in (('this', ROOT), ('parent', parent)) if r % 2 == 0 else (('parent', parent), ('this', ROOT)):
            env = dict(os.environ)
            env.pop('RISP_LIB_PATH', None)
            p = subprocess.run(cmd, cwd=cwd, env=env, capture_output=True, text=True, timeout=1800)
            line = [ln for ln in p.stdout.splitlines() if ln.startswith('{')]
            if p.returncode != 0 or not line:
                raise SystemExit('bench.py failed in %s:\n%s' % (cwd, p.stderr[-3000:]))
            v = json.loads(line[-1])
            res[name].append(v)
            print('  bench %-6s round %d: %s' % (name, r, line[-1][:300]), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--frames', type=int, default=16)
    ap.add_argument('--batch', type=int, default=4)
    ap.add_argument('--passes', type=int, default=10, help='passes over the whole store per timed window')
    ap.add_argument('--parent', help='a built checkout of the commit to compare bench.py against')
    ap.add_argument('--bench-rounds', type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('time_validate.py measures on a GPU; none found')
    print('card (name, power limit, max SM clock):', card())
    hbm_peak, _, peak_src = peaks()
    raws, gts = [], []
    for k in range(0, args.frames, 4):
        r, g = synthetic_frames(min(4, args.frames - k), H, W, seed=10 + k)
        raws += list(torch.round(r * 1023).to(torch.int16)[:, 0])
        gts += list(torch.round(g * 255).to(torch.uint8))
    ds = DeviceDataset(raws, gts, 1023., 16)
    del raws, gts
    dev = torch.device('cuda')
    recs, _ = ds.plan_.frames('all')
    B = args.batch
    pos = [torch.from_numpy(recs[i:i + B]).to(dev) for i in range(0, len(recs), B)]
    img = torch.empty((B, 1, H, W), device=dev)
    gt = torch.empty((B, 3, H, W), device=dev)
    u8 = torch.empty((B, H, W, 3), device=dev, dtype=torch.uint8)
    sse = torch.empty((len(pos), B), device=dev, dtype=torch.int64)
    ss = torch.empty((len(pos), B), device=dev, dtype=torch.int64)
    px = B * H * W
    print('store: %d frames of %dx%d, %.0f MB of codes; batches of %d frames (%.0f MP)' % (
        len(recs), H, W, (ds.raw_store.numel() * 2 + ds.gt_store.numel()) / 1e6, B, px / 1e6))
    for cname, (dm, st, vals) in CHAINS.items():
        chain = ops.Chain(st)
        params = torch.tensor([vals], device=dev)

        def store(with_ssim):
            for k, p in enumerate(pos):
                ops.pipeline_eval_store(ds.raw_store, ds.gt_store, p, 1023., ds.status, dm, chain, params, u8=with_ssim,
                                        sse_out=sse[k], u8_out=u8 if with_ssim else None)
                if with_ssim:
                    ops.ssim_u8_store(u8, ds.gt_store, p, ds.status, out=ss[k])

        def composition(with_ssim):
            for k, p in enumerate(pos):
                ops.sample_crops(ds.raw_store, ds.gt_store, p, H, W, 1023., ds.status, img, gt)
                s, y8 = ops.pipeline_eval(img, gt, dm, chain, params, u8=with_ssim)
                sse[k].copy_(s)
                if with_ssim:
                    ss[k].copy_(ops.ssim_u8(y8, gt))
        results = {}
        for name, fn, with_ssim in (('store', store, False), ('composition', composition, False),
                                    ('store+ssim', store, True), ('composition+ssim', composition, True)):
            ms = timed(lambda: fn(with_ssim), args.passes, 1, args.reps)
            results[name] = (sse.clone(), ss.clone() if with_ssim else None)
            per = [m / len(pos) for m in ms]                 # ms per batch of B frames
            mid = sorted(per)[len(per) // 2]
            gbs = BPX[name] * px / (mid / 1e3) / 1e9
            print('%-24s %-18s %.4f ms per %.0f MP (%.4f-%.4f)  %2d B/px  %5.0f GB/s = %.3f of the 7.7 TB/s data sheet, '
                  '%.3f of %.0f GB/s (%s)' % (cname, name, mid, px / 1e6, min(per), max(per), BPX[name], gbs,
                                               gbs / DATASHEET_HBM_GBS, gbs / hbm_peak, hbm_peak, peak_src), flush=True)
        assert torch.equal(results['store'][0], results['composition'][0]), cname
        assert torch.equal(results['store+ssim'][0], results['composition+ssim'][0]), cname
        assert torch.equal(results['store+ssim'][1], results['composition+ssim'][1]), cname
        ds.check()
    if args.parent:
        del ds
        torch.cuda.empty_cache()
        print('bench.py --no-cpu, this tree vs %s, alternating:' % args.parent)
        res = bench_ab(args.parent, args.bench_rounds)
        for name, vals in res.items():
            print('  %-6s values: %s' % (name, [v.get('value') for v in vals]))


if __name__ == '__main__':
    main()
