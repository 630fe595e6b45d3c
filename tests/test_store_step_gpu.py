"""Tuning from the code store (B200): the step kernels reading crops of the frame stores (`ops.PipelineStep.store`) against
the composition they replace -- `sample_crops` of the same records followed by the step on the decoded batch -- bit for
bit on every dispatch path, and `IspModel` fed `DeviceDataset.records` against the same model fed `DeviceDataset.sample`."""
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

IDENT = [0.0] * 30
IDENT[6] = IDENT[17] = IDENT[28] = 1.0
SIGS = {
    'A': ['gain', 'poly10', 'gamma', ('gtm', 4)],
    'B': ['gamma', 'poly10', 'gain'],
    'C': ['gamma', 'poly10'],
    'D': ['gamma', ('gtm', 4)],
    'skip': [],                                  # demosaic only (no parameter: the interpreter kernel)
}
# no packed signature: the interpreter kernel, without and with a big (poly10 / ccm) stage
INTERPS = [['gain', ('gtm', 3)], ['gain', 'ccm', 'gamma']]
KINDS = ['nearest', 'bilinear', 'malvar']
# raw code dtype, largest code + 1, white level
RAWS = [(np.uint16, 1024, 1023.), (np.int16, 16384, 16383.), (np.uint8, 256, 255.)]
FH, FW = 40, 240                                 # frames: W % 16 == 0
CROPS = [(22, 128), (20, 160), (22, 192)]        # w % 128 = 0, 32, 64 (narrow items); h not a multiple of 4


def stage_params(st, g, rows=1):
    vals = []
    for s in st:
        name, iarg = (s, 0) if isinstance(s, str) else s
        if name == 'gain':
            vals += [1.1, 0.9, 1.2]
        elif name == 'poly10':
            vals += (torch.tensor(IDENT) + torch.randn(30, generator=g) * 0.03).tolist()
        elif name == 'gamma':
            vals += [0.55]
        elif name == 'gtm':
            vals += [0.2, 0.5, 0.8] if iarg in (0, 4) else [k / iarg for k in range(1, iarg)]
        elif name == 'ccm':
            vals += (torch.eye(3).reshape(-1) + torch.randn(9, generator=g) * 0.03).tolist()
    if not vals:
        return None
    t = torch.tensor([vals]).repeat(rows, 1)
    if rows > 1:                                 # per-image rows: small per-row perturbations
        t = t * (1 + 0.02 * torch.randn(t.shape, generator=g))
    return t


def make_store(F, H, W, dtype, hi, wl, seed, crop):
    from reconfigisp_b200.data import DeviceDataset
    rng = np.random.default_rng(seed)
    raws = rng.integers(0, hi, (F, 1, H, W)).astype(dtype)
    gts = rng.integers(0, 256, (F, 3, H, W)).astype(np.uint8)
    return DeviceDataset(raws, gts, wl, crop, seed=seed), raws, gts


def edge_records(F, H, W, h, w, u8):
    """Crops touching each frame edge and corner, interior crops with x0 % 4 == 2, and for 8-bit stores every even x0 % 16."""
    ys, xs = [0, H - h], [0, W - w]
    recs = [(y, x) for y in ys for x in xs]
    recs += [(2, 2), ((H - h) // 4 * 2, 6 if W - w >= 6 else 2)]
    if u8:
        recs += [(2 * (k % max(1, (H - h) // 2 + 1)), x) for k, x in enumerate(range(2, min(16, W - w + 1), 2))]
    return [(i % F, (i + 1) % F, y, x) for i, (y, x) in enumerate(recs)]


def check(ds, kind, st, recs, g, l1=False, shared=True):
    """store step == step on the decoded batch, bitwise; -> (loss, dparams)"""
    from reconfigisp_b200 import ops
    chain = ops.Chain(st)
    if l1 and not shared:
        recs = recs[:8]        # the L1 step takes per-image parameter rows for up to 8 images (on a decoded batch as well)
    N, h, w = len(recs), ds.h, ds.w
    pos = torch.tensor(recs, dtype=torch.int32).cuda()
    params = stage_params(st, g, 1 if shared else N)
    params = None if params is None else params.cuda()
    step = ops.PipelineStep(N, h, w, kind, chain, 'cuda', shared_row=shared, l1=l1)
    loss, dpar = [t.clone() for t in step.store(ds.raw_store, ds.gt_store, pos, ds.white_level, ds.status, params)]
    img, gt = ops.sample_crops(ds.raw_store, ds.gt_store, pos, h, w, ds.white_level, ds.status)
    ref_loss, ref_dpar = step(img, gt, params)
    assert torch.equal(loss, ref_loss), (kind, st, l1, loss.item(), ref_loss.item())
    assert torch.equal(dpar, ref_dpar), (kind, st, l1, (dpar - ref_dpar).abs().max().item())
    assert torch.isfinite(loss).all() and torch.isfinite(dpar).all()
    return loss, dpar


@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('sig', list(SIGS))
def test_store_step_equals_decoded_batch_on_packed_chains(kind, sig):
    """Every raw code type, every narrow-item width, MSE and L1, a shared row and per-image rows."""
    g = torch.Generator().manual_seed(sum(map(ord, kind + sig)))
    for i, (dtype, hi, wl) in enumerate(RAWS):
        h, w = CROPS[(i + KINDS.index(kind)) % 3]
        ds, _, _ = make_store(5, FH, FW, dtype, hi, wl, seed=i + 10 * KINDS.index(kind), crop=(h, w))
        recs = edge_records(5, FH, FW, h, w, dtype == np.uint8)
        for l1 in ((False, True) if sig != 'skip' else (False,)):
            for shared in (True, False):
                check(ds, kind, SIGS[sig], recs, g, l1=l1, shared=shared)
        ds.check()


def test_store_step_every_width_and_code_type_on_one_chain():
    g = torch.Generator().manual_seed(3)
    for dtype, hi, wl in RAWS:
        for h, w in CROPS:
            ds, _, _ = make_store(4, FH, FW, dtype, hi, wl, seed=w, crop=(h, w))
            recs = edge_records(4, FH, FW, h, w, dtype == np.uint8)
            check(ds, 'malvar', SIGS['A'], recs, g)
            check(ds, 'bilinear', SIGS['D'], recs, g, l1=True, shared=False)
            ds.check()


def test_store_step_interpreter_chain():
    g = torch.Generator().manual_seed(6)
    for i, (dtype, hi, wl) in enumerate(RAWS):
        h, w = CROPS[i]
        ds, _, _ = make_store(4, FH, FW, dtype, hi, wl, seed=20 + i, crop=(h, w))
        recs = edge_records(4, FH, FW, h, w, dtype == np.uint8)
        for kind in KINDS:
            for st in INTERPS:
                check(ds, kind, st, recs, g)
                check(ds, kind, st, recs, g, shared=False)
        ds.check()


def test_store_step_more_than_64_images():
    """N > 64: the one-warp-per-entry finaliser."""
    g = torch.Generator().manual_seed(7)
    ds, _, _ = make_store(6, FH, FW, np.uint16, 1024, 1023., seed=7, crop=(8, 32))
    rng = np.random.default_rng(7)
    recs = [(int(rng.integers(0, 6)), int(rng.integers(0, 6)), 2 * int(rng.integers(0, 17)), 2 * int(rng.integers(0, 105)))
            for _ in range(70)]
    for st in [SIGS['A']] + INTERPS:
        check(ds, 'bilinear', st, recs, g)
        check(ds, 'bilinear', st, recs, g, shared=False)
    check(ds, 'malvar', SIGS['B'], recs, g, l1=True)
    ds.check()


def test_out_of_crop_pixels_are_never_read():
    """Every pixel outside the crops holds the extreme codes (raw at its maximum, GT 255): the step still equals the decoded
    batch, which never sees them.  A masked lane or group that kept a non-zero target would break the equality."""
    from reconfigisp_b200.data import DeviceDataset
    g = torch.Generator().manual_seed(11)
    rng = np.random.default_rng(11)
    for dtype, hi, wl in RAWS:
        for h, w in CROPS:
            recs = edge_records(8, FH, FW, h, w, dtype == np.uint8)[:8]
            F = len(recs)
            raws = np.full((F, 1, FH, FW), np.iinfo(dtype).max, dtype=dtype)
            gts = np.full((F, 3, FH, FW), 255, dtype=np.uint8)
            recs = [(i, i, y, x) for i, (_, _, y, x) in enumerate(recs)]          # one crop per frame
            for i, _, y, x in recs:
                raws[i, :, y:y + h, x:x + w] = rng.integers(0, hi, (1, h, w))
                gts[i, :, y:y + h, x:x + w] = rng.integers(0, 256, (3, h, w))
            ds = DeviceDataset(raws, gts, wl, (h, w))
            for kind in KINDS:
                check(ds, kind, SIGS['A'], recs, g)
                check(ds, kind, SIGS['D'], recs, g, l1=True)
            check(ds, 'bilinear', INTERPS[1], recs, g)
            ds.check()


def test_bad_records_add_nothing_and_set_the_status():
    from reconfigisp_b200 import ops
    h, w = 22, 160
    ds, _, _ = make_store(3, FH, FW, np.uint16, 1024, 1023., seed=3, crop=(h, w))
    good = [(0, 1, 0, 0), (2, 2, FH - h, FW - w), (1, 0, 4, 2)]
    for st, l1 in ((SIGS['A'], False), (SIGS['D'], True), (INTERPS[0], False)):
        chain = ops.Chain(st)
        params = stage_params(st, torch.Generator().manual_seed(0)).cuda()
        ref = ops.PipelineStep(3, h, w, 'bilinear', chain, 'cuda', l1=l1)
        rl, rd = [t.clone() for t in ref.store(ds.raw_store, ds.gt_store, torch.tensor(good, dtype=torch.int32).cuda(),
                                               1023., ds.status, params)]
        ds.check()
        step = ops.PipelineStep(4, h, w, 'bilinear', chain, 'cuda', l1=l1)
        for bad in ((3, 0, 0, 0), (0, 3, 0, 0), (-1, 0, 0, 0), (0, 0, 1, 0), (0, 0, 0, 3), (0, 0, FH - h + 2, 0),
                    (0, 0, 0, FW - w + 2), (0, 0, -2, 0)):
            pos = torch.tensor(good[:1] + [bad] + good[1:], dtype=torch.int32).cuda()
            loss, dpar = step.store(ds.raw_store, ds.gt_store, pos, 1023., ds.status, params)
            assert torch.isfinite(loss).all() and torch.isfinite(dpar).all(), bad
            assert torch.allclose(loss, rl * 3 / 4, rtol=1e-5, atol=0), (bad, loss.item(), rl.item())
            assert torch.allclose(dpar, rd * 3 / 4, rtol=1e-4, atol=1e-7), bad
            with pytest.raises(RuntimeError):
                ds.check()
            assert int(ds.status.item()) == 0


def test_store_step_rejects_geometry_the_tensor_maps_cannot_describe():
    from reconfigisp_b200 import ops
    ds, _, _ = make_store(2, 16, 40, np.uint16, 1024, 1023., seed=1, crop=(8, 16))
    pos = torch.tensor([[0, 0, 0, 0]], dtype=torch.int32).cuda()
    chain = ops.Chain(SIGS['D'])
    params = stage_params(SIGS['D'], torch.Generator().manual_seed(0)).cuda()
    with pytest.raises(NotImplementedError):                         # frame W % 16 != 0
        ops.PipelineStep(1, 8, 16, 'bilinear', chain, 'cuda').store(ds.raw_store, ds.gt_store, pos, 1023., ds.status, params)
    ds, _, _ = make_store(2, 16, 48, np.uint16, 1024, 1023., seed=1, crop=(8, 18))
    with pytest.raises(NotImplementedError):                         # crop w % 4 != 0
        ops.PipelineStep(1, 8, 18, 'bilinear', chain, 'cuda').store(ds.raw_store, ds.gt_store, pos, 1023., ds.status, params)


def test_store_step_equals_decoded_batch_on_whole_12mp_frames():
    g = torch.Generator().manual_seed(12)
    ds, _, _ = make_store(3, 3000, 4000, np.uint16, 16384, 16383., seed=12, crop=(3000, 4000))
    recs = [(0, 1, 0, 0), (2, 0, 0, 0)]
    check(ds, 'bilinear', SIGS['A'], recs, g)
    check(ds, 'malvar', SIGS['D'], recs, g, l1=True)
    ds.check()


def child_cases(out):
    """In a child process (RISP_FUSED=0: every chain on the interpreter kernels): store step == decoded batch there."""
    from reconfigisp_b200 import ops
    g = torch.Generator().manual_seed(9)
    for i, (dtype, hi, wl) in enumerate(RAWS):
        h, w = CROPS[i]
        ds, _, _ = make_store(5, FH, FW, dtype, hi, wl, seed=30 + i, crop=(h, w))
        recs = edge_records(5, FH, FW, h, w, dtype == np.uint8)
        for kind in KINDS:
            for st in [SIGS['A'], SIGS['C'], SIGS['skip']] + INTERPS:
                check(ds, kind, st, recs, g)
            check(ds, kind, SIGS['B'], recs, g, shared=False)
        pos = torch.tensor(recs, dtype=torch.int32).cuda()
        step = ops.PipelineStep(len(recs), h, w, 'bilinear', ops.Chain(SIGS['D']), 'cuda', l1=True)
        try:                                     # L1 is a packed-kernel step: unsupported here, as on a decoded batch
            step.store(ds.raw_store, ds.gt_store, pos, wl, ds.status, stage_params(SIGS['D'], g).cuda())
            raise AssertionError('the L1 store step ran without the packed kernels')
        except NotImplementedError:
            pass
        ds.check()
    open(out, 'w').write('ok')


def test_store_step_under_interpreter_only(tmp_path):
    env = dict(os.environ)
    env.pop('RISP_FUSED_STEP_ROWS', None)
    env['RISP_FUSED'] = '0'
    out = tmp_path / 'ok.txt'
    cmd = [sys.executable] + (['-s'] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    assert out.read_text() == 'ok'


# ---- IspModel fed records ------------------------------------------------------------------------------------------
def _opt(arch='Bayer_02_Demosaic_02_sRGB_11_13_01_14', loss='l2', which='OriginUniversal', **kw):
    net = {'which_model_G': which, 'architecture': arch, 'weight_seed': 10}
    if which == 'IspUniversal':
        net['individual_module_paths'] = kw.pop('paths')
    opt = {'model': 'isp', 'is_train': True, 'network_G': net,
           'train': {'lr_G': 1e-3, 'beta1': 0.9, 'beta2': 0.99, 'pixel_criterion': loss, 'lr_scheme': 'MultiStepLR',
                     'lr_steps': [20000], 'lr_gamma': 0.5},
           'path': {'pretrain_model_G': None}}
    opt.update(kw)
    return opt


def _frames(F, H, W, seed=10):
    from reconfigisp_b200.synthetic import synthetic_frames
    raw_f, gt_f = synthetic_frames(F, H, W, seed=seed)
    return torch.round(raw_f * 1023).to(torch.int16), torch.round(gt_f * 255).to(torch.uint8)


def _train(opt, raws, gts, crop, feed, steps=7, B=8, store_step=None):
    from reconfigisp_b200.data import DeviceDataset
    from reconfigisp_b200.tuning import IspModel
    ds = DeviceDataset(raws, gts, 1023., crop, seed=3)
    m = IspModel(opt)
    out = []
    for s in range(steps):
        m.feed_data(getattr(ds, feed)(B, 'all'))
        if store_step is not None:
            assert (m._store_step() is not None) == store_step
        m.optimize_parameters()
        out.append((m.log_dict['loss'].item(), m._flat_grad.clone(),
                    torch.cat([p.detach().reshape(-1) for p in m.netG.trainable_parameters])))
    ds.check()
    return m, ds, out


def _same_runs(a, b):
    for s, ((l0, g0, p0), (l1, g1, p1)) in enumerate(zip(a, b)):
        assert l0 == l1 and torch.equal(g0, g1) and torch.equal(p0, p1), (s, l0, l1)


@pytest.mark.parametrize('loss', ['l2', 'l1'])
@pytest.mark.parametrize('graph', [True, False])
def test_isp_model_records_feed_trains_like_sample_feed(loss, graph):
    raws, gts = _frames(6, 96, 128)
    opt = _opt(loss=loss, cuda_graph=graph)
    m, _, rec = _train(opt, raws, gts, (64, 96), 'records', store_step=True)
    assert bool(m.__dict__.get('_graphs')) == graph
    _, _, ref = _train(opt, raws, gts, (64, 96), 'sample')
    _same_runs(rec, ref)


@pytest.mark.parametrize('case', ['cnn', 'frame_w_not_16'])
def test_isp_model_records_feed_falls_back_and_agrees(case):
    if case == 'cnn':
        raws, gts = _frames(6, 96, 128)
        opt = _opt('Bayer_02_Demosaic_01_sRGB_11_12', which='IspUniversal', paths=(None,) * 4)
        crop, steps, B = (32, 48), 4, 2
    else:
        raws, gts = _frames(6, 96, 136)                 # W % 16 == 8: the tensor maps cannot describe the stores
        opt, crop, steps, B = _opt(), (64, 96), 7, 8
    m, _, rec = _train(opt, raws, gts, crop, 'records', steps=steps, B=B, store_step=False)
    _, _, ref = _train(opt, raws, gts, crop, 'sample', steps=steps, B=B)
    _same_runs(rec, ref)


def test_output_test_and_evaluate_after_a_records_feed():
    from reconfigisp_b200.data import DeviceDataset
    from reconfigisp_b200.tuning import IspModel
    raws, gts = _frames(6, 96, 128)
    res = []
    for feed in ('records', 'sample'):
        ds = DeviceDataset(raws, gts, 1023., (64, 96), seed=3)
        m = IspModel(_opt())
        for _ in range(3):
            m.feed_data(getattr(ds, feed)(4, 'all'))
            m.optimize_parameters()
        out = m.output.clone()
        y, _ = m.test()
        ev = m.evaluate(u8=True, ssim=True)
        res.append((out, y.detach().clone(), [t.clone() for t in ev if t is not None]))
        ds.check()
    (o0, y0, e0), (o1, y1, e1) = res
    assert torch.equal(o0, o1) and torch.equal(y0, y1)
    assert all(torch.equal(a, b) for a, b in zip(e0, e1))


def test_records_feed_makes_no_host_sync_and_launches_no_sampler():
    from reconfigisp_b200.data import DeviceDataset
    from reconfigisp_b200.tuning import IspModel
    raws, gts = _frames(6, 96, 128)
    ds = DeviceDataset(raws, gts, 1023., (64, 96), seed=3)
    m = IspModel(_opt())
    for _ in range(6):                                   # eager steps, capture, replay
        m.feed_data(ds.records(8, 'all'))
        m.optimize_parameters()
    assert m.__dict__.get('_graphs')
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        for _ in range(3):
            m.feed_data(ds.records(8, 'all'))
            m.optimize_parameters()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            m.feed_data(ds.records(8, 'all'))
            m.optimize_parameters()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert any('fused_kernel' in n for n in names), sorted(set(names))
    assert not any('crop_decode_kernel' in n for n in names), sorted(set(names))
    ds.check()


WORKER = r'''
import os, sys, torch
sys.path.insert(0, os.environ['RISP_ROOT'])
import torch.distributed as dist
from reconfigisp_b200 import dist as D
from reconfigisp_b200.data import DeviceDataset
from reconfigisp_b200.synthetic import synthetic_frames
from reconfigisp_b200.tuning import IspModel
rank, world, local = D.init_from_env('nccl')
torch.cuda.set_device(local)
raw_f, gt_f = synthetic_frames(8, 96, 128, seed=10)
raws, gts = torch.round(raw_f * 1023).to(torch.int16), torch.round(gt_f * 255).to(torch.uint8)
opt = {'model': 'isp', 'is_train': True,
       'network_G': {'which_model_G': 'OriginUniversal', 'architecture': 'Bayer_02_Demosaic_02_sRGB_11_13_01_14', 'weight_seed': 10},
       'train': {'lr_G': 1e-3, 'beta1': 0.9, 'beta2': 0.99, 'pixel_criterion': 'l2', 'lr_scheme': 'MultiStepLR',
                 'lr_steps': [20000], 'lr_gamma': 0.5},
       'path': {'pretrain_model_G': None}}
runs = {}
for feed in ('records', 'sample'):
    ds = DeviceDataset(raws, gts, 1023., (64, 96), seed=3, rank=rank, world=world)
    m = IspModel(opt)
    out = []
    for s in range(7):
        m.feed_data(getattr(ds, feed)(4, 'all'))
        m.optimize_parameters()
        out.append((m.log_dict['loss'].item(), torch.cat([p.detach().reshape(-1) for p in m.netG.trainable_parameters]).cpu()))
    ds.check()
    runs[feed] = out
for (l0, p0), (l1, p1) in zip(runs['records'], runs['sample']):
    assert l0 == l1 and torch.equal(p0, p1), (rank, l0, l1)
dist.barrier()
if rank == 0:
    open(os.environ['RISP_OUT'], 'w').write('ok')
dist.destroy_process_group()
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs >= 2 GPUs')
def test_world_two_records_feed_trains_like_sample_feed(tmp_path):
    script = tmp_path / 'worker.py'
    script.write_text(WORKER)
    out = tmp_path / 'ok.txt'
    env = dict(os.environ, RISP_ROOT=ROOT, RISP_OUT=str(out))
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--standalone', '--nproc_per_node=2', str(script)]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert out.read_text() == 'ok'


if __name__ == '__main__':
    child_cases(sys.argv[1])
