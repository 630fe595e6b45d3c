"""Time training from a dataset resident in HBM (`data.DeviceDataset`) against the pinned-host codes path, on one GPU.

    python scripts/time_device_data.py [--reps 3]

Prints the card and its power limit, then per workload the ms per step of
  (a) the step on resident fp32 data (`bench.py`'s `value` loop),
  (b) `DeviceDataset.sample` + step, with and without reading the loss every step,
  (d) `DeviceDataset.records` + the step reading the store's codes (MSE and L1 models),
  (c) `feed_data` of pinned host int16 raw + uint8 GT codes + step + loss read (`bench.py`'s `e2e` loop),
for the bench's tuning workload (4 x 12 MP whole-frame crops, store of 16 synthetic frames) and the reference's tuning
shape (8 x 224^2 crops from the same 12 MP frames); then the kernels alone, records already on the device: the sampler
(21 B per output pixel: 2 B raw code + 3 B GT codes read, 16 B fp32 written, over CUDA-event time) and the MSE / L1 step
(parameter table, step kernel, finaliser) on the decoded fp32 batch against the same step reading the store.  Each figure is
timed `--reps` times (min / max shown); the arms of a workload take turns within each repetition."""
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


def alternate(arms, n, warmup, reps):
    """timed() of every arm, the arms taking turns within each repetition -> {name: ms list}."""
    res = {k: [] for k in arms}
    for r in range(reps):
        for k, (fn, nk) in arms.items():
            res[k] += timed(fn, nk or n, warmup if r == 0 else 2, 1)
    return res


def workload(ds, raws, gts, B, crop, reps, steps):
    """(a), (b), (d), (c) and the kernels for B crops of `crop` per step; -> dict of ms lists."""
    dev = torch.device('cuda')
    h, w = crop
    # (a) resident fp32 data: decoded once from the store's first frames
    model = IspModel(opt_tuning())
    img0, gt0 = ds.sample(B, 'all')
    model.feed_data((img0.clone(), gt0.clone()))
    # (b) sample + step (the model reads the sampler's persistent buffers in place: the captured step keeps replaying)
    model_b = IspModel(opt_tuning())

    def step_b():
        model_b.feed_data(ds.sample(B, 'all'))
        model_b.optimize_parameters()

    def step_b_item():
        step_b()
        return float(model_b.log_dict['loss'].item())
    # (d) records + the step reading the store (the captured step reads the persistent record buffer)
    models_d = {loss: IspModel(dict(opt_tuning(), train=dict(opt_tuning()['train'], pixel_criterion=loss))) for loss in ('l2', 'l1')}

    def step_d(loss):
        def fn():
            models_d[loss].feed_data(ds.records(B, 'all'))
            models_d[loss].optimize_parameters()
        return fn
    res = alternate({'a_resident': (model.optimize_parameters, 0), 'b_sample_step': (step_b, 0),
                     'd_records_store_step_mse': (step_d('l2'), 0), 'd_records_store_step_l1': (step_d('l1'), 0),
                     'b_sample_step_loss_read': (step_b_item, 0)}, steps, 5, reps)
    assert all(m._store_step() is not None for m in models_d.values()), 'the store step did not run'

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

    # the kernels alone, records already on the device: the sampler, and each step on the decoded batch / on the store
    pos = torch.from_numpy(rec).to(dev)
    f = models_d['l2']._fast_plan()
    tab = f['table']
    kern = {'kernel': (lambda: ops.sample_crops(ds.raw_store, ds.gt_store, pos, h, w, 1023., ds.status, img, gt), 200)}
    for loss in ('l2', 'l1'):
        st = ops.PipelineStep(B, h, w, f['dm'], f['chain'], dev, l1=(loss == 'l1'))
        kern['step_%s_fp32' % loss] = ((lambda st=st: st(img, gt, tab)), 200)
        kern['step_%s_store' % loss] = ((lambda st=st: st.store(ds.raw_store, ds.gt_store, pos, 1023., ds.status, tab)), 200)
        a = [t.clone() for t in st(img, gt, tab)]
        b = [t.clone() for t in st.store(ds.raw_store, ds.gt_store, pos, 1023., ds.status, tab)]
        assert all(torch.equal(x, y) for x, y in zip(a, b)), 'the store step differs from the step on the decoded batch'
    res.update(alternate(kern, 200, 10, reps))
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
