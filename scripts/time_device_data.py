"""Time training from a dataset resident in HBM (`data.DeviceDataset`) against the pinned-host codes path, on one GPU.

    python scripts/time_device_data.py [--reps 3]

Prints the card and its power limit, then per workload the ms per step of
  (a) the step on resident fp32 data (`bench.py`'s `value` loop),
  (b) `DeviceDataset.sample` + step, with and without reading the loss every step,
  (c) `feed_data` of pinned host int16 raw + uint8 GT codes + step + loss read (`bench.py`'s `e2e` loop),
for the bench's tuning workload (4 x 12 MP whole-frame crops, store of 16 synthetic frames) and the reference's tuning
shape (8 x 224^2 crops from the same 12 MP frames), and the sampler kernel alone: 21 B per output pixel (2 B raw code +
3 B GT codes read, 16 B fp32 written) over CUDA-event time.  Each figure is timed `--reps` times (min / max shown)."""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import H, W, opt_tuning, peaks  # noqa: E402
from reconfigisp_b200 import ops  # noqa: E402
from reconfigisp_b200.data import DeviceDataset  # noqa: E402
from reconfigisp_b200.synthetic import synthetic_frames  # noqa: E402
from reconfigisp_b200.tuning import IspModel  # noqa: E402

DATASHEET_HBM_GBS = 7700.0
BYTES_PER_PX = 2 + 3 + 16


def timed(fn, n, warmup, reps):
    """ms per call of fn over n calls, after `warmup` calls, `reps` times; synchronised around each window."""
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


def fmt(ms):
    return '%.4f ms (%.4f-%.4f)' % (sorted(ms)[len(ms) // 2], min(ms), max(ms))


def card():
    q = subprocess.run(['nvidia-smi', '-i', str(torch.cuda.current_device()), '--query-gpu=name,power.limit,clocks.max.sm',
                        '--format=csv,noheader'], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def workload(ds, raws, gts, B, crop, reps, steps):
    """(a), (b), (c) for B crops of `crop` per step; -> dict of ms lists."""
    dev = torch.device('cuda')
    h, w = crop
    res = {}
    # (a) resident fp32 data: decoded once from the store's first frames
    model = IspModel(opt_tuning())
    img0, gt0 = ds.sample(B, 'all')
    model.feed_data((img0.clone(), gt0.clone()))
    res['a_resident'] = timed(model.optimize_parameters, steps, 5, reps)

    # (b) sample + step (the model reads the sampler's persistent buffers in place: the captured step keeps replaying)
    def step_b():
        model.feed_data(ds.sample(B, 'all'))
        model.optimize_parameters()

    def step_b_item():
        step_b()
        return float(model.log_dict['loss'].item())
    res['b_sample_step'] = timed(step_b, steps, 5, reps)
    res['b_sample_step_loss_read'] = timed(step_b_item, steps, 5, reps)

    # (c) pinned host codes, double-buffered feed, loss read every step (bench.py's e2e loop)
    rec = ds.plan('all', 0, B)
    fr = ds.plan_.raw_frames[rec[:, 0]]
    raw_c = torch.stack([raws[f][:, y:y + h, x:x + w] for f, y, x in zip(fr, rec[:, 2], rec[:, 3])]).pin_memory()
    gt_c = torch.stack([gts[f][:, y:y + h, x:x + w] for f, y, x in zip(fr, rec[:, 2], rec[:, 3])]).pin_memory()
    model.feed_data((raw_c, gt_c))

    def step_c():
        model.optimize_parameters()
        model.feed_data((raw_c, gt_c))
        return float(model.log_dict['loss'].item())
    res['c_host_codes'] = timed(step_c, min(steps, 40), 4, reps)

    # the crops the sampler makes equal the host path's decode of the same codes
    img, gt = ds.sample(B, 'all')
    rec = ds.plan('all', ds.steps['all'] - 1, B)
    fr = ds.plan_.raw_frames[rec[:, 0]]
    ref = torch.stack([raws[f][:, y:y + h, x:x + w] for f, y, x in zip(fr, rec[:, 2], rec[:, 3])]).to(dev)
    assert torch.equal(img, ops.decode_codes(ref.contiguous(), 1023.)), 'sampled crops differ from the decoded codes'

    # the sampler kernel alone, records already on the device
    pos = torch.from_numpy(rec).to(dev)
    res['kernel'] = timed(lambda: ops.sample_crops(ds.raw_store, ds.gt_store, pos, h, w, 1023., ds.status, img, gt), 200, 10, reps)
    ds.check()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--frames', type=int, default=16)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('time_device_data.py measures on a GPU; none found')
    print('card:', card())
    hbm_peak, _, peak_src = peaks()
    raws, gts = [], []
    for k in range(0, args.frames, 4):                 # 16 x 12 MP in chunks: host fp32 of 4 frames at a time
        r, g = synthetic_frames(min(4, args.frames - k), H, W, seed=10 + k)
        raws += list(torch.round(r * 1023).to(torch.int16))
        gts += list(torch.round(g * 255).to(torch.uint8))
    for name, B, crop, steps in (('bench tuning workload: 4 x 12 MP whole frames', 4, (H, W), 100),
                                 ('reference tuning shape: 8 x 224^2 crops of 12 MP frames', 8, (224, 224), 400)):
        ds = DeviceDataset([f[0] for f in raws], gts, 1023., crop)
        res = workload(ds, raws, gts, B, crop, args.reps, steps)
        px = B * crop[0] * crop[1]
        print('\n%s (store: %d frames, %.0f MB of codes)' % (name, len(raws), (ds.raw_store.numel() * 2 + ds.gt_store.numel()) / 1e6))
        for key, ms in res.items():
            mid = sorted(ms)[len(ms) // 2]
            line = '  %-26s %s  %9.1f MP/s' % (key, fmt(ms), px / 1e6 / (mid / 1e3))
            if key == 'kernel':
                gbs = BYTES_PER_PX * px / (mid / 1e3) / 1e9
                line += '  %.0f GB/s = %.3f of the 7.7 TB/s data sheet, %.3f of %.0f GB/s (%s)' % (
                    gbs, gbs / DATASHEET_HBM_GBS, gbs / hbm_peak, hbm_peak, peak_src)
            print(line)
        del ds
        torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
