"""Validation on the resident dataset (B200): the evaluation kernels reading the frame store's codes
(`ops.pipeline_eval_store`, `ops.ssim_u8_store`) against the composition they replace -- `sample_crops` of whole frames
followed by `pipeline_eval` / `ssim_u8` -- bit for bit on every dispatch path, and `DeviceDataset.evaluate` against a host
loop of `net.evaluate` over the same frames."""
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

from oracle import isp_oracle as O             # noqa: E402
from oracle import metrics_oracle as M         # noqa: E402
from oracle import ssim_oracle as SO           # noqa: E402

IDENT = [0.0] * 30
IDENT[6] = IDENT[17] = IDENT[28] = 1.0
SIGS = {
    'A': ['gain', 'poly10', 'gamma', ('gtm', 4)],
    'B': ['gamma', 'poly10', 'gain'],
    'C': ['gamma', 'poly10'],
    'D': ['gamma', ('gtm', 4)],
    'skip': [],                                  # demosaic only
}
INTERP = ['filmic', 'gamma', 'poly10']           # no packed signature: the interpreter kernel
KINDS = ['nearest', 'bilinear', 'malvar']
# raw code dtype, largest code + 1, white level
RAWS = [(np.uint16, 1024, 1023.), (np.int16, 16384, 16383.), (np.uint8, 256, 255.)]
WIDTHS = [256, 160, 192]                         # W % 128 = 0, 32, 64 (narrow items)


def stage_params(st, g):
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
            vals += [0.2, 0.5, 0.8]
        elif name == 'filmic':
            vals += [2.0, 1.3]
    return torch.tensor([vals]) if vals else None


def make_store(F, G, H, W, dtype, hi, wl, seed, hwc=False, pairs=None, crop=None):
    from reconfigisp_b200.data import DeviceDataset
    rng = np.random.default_rng(seed)
    raws = rng.integers(0, hi, (F, 1, H, W)).astype(dtype)
    raws.reshape(-1)[:3] = [0, hi - 1, hi // 2]
    gts = rng.integers(0, 256, (G, 3, H, W)).astype(np.uint8)
    g = np.ascontiguousarray(gts.transpose(0, 2, 3, 1)) if hwc else gts
    return DeviceDataset(raws, g, wl, crop or (H, W), pairs=pairs, seed=seed), raws, gts


def composition(ds, pos, kind, chain, params, ssim=False):
    """Today's way: decode whole frames with sample_crops, then pipeline_eval (and ssim_u8 of its image)."""
    from reconfigisp_b200 import ops
    img, gt = ops.sample_crops(ds.raw_store, ds.gt_store, pos, ds.H, ds.W, ds.white_level, ds.status)
    sse, u8 = ops.pipeline_eval(img, gt, kind, chain, params, u8=True)
    return sse, u8, (ops.ssim_u8(u8, gt) if ssim else None), gt


def check_store(ds, kind, st, g, batch=3, ssim=False):
    from reconfigisp_b200 import ops
    chain = ops.Chain(st)
    params = stage_params(st, g)
    params = None if params is None else params.cuda()
    recs, _ = ds.plan_.frames('all')
    pos_all = torch.from_numpy(recs).cuda()
    for i in range(0, len(recs), batch):                     # the last batch is short when batch does not divide the split
        pos = pos_all[i:i + batch]
        sse, u8 = ops.pipeline_eval_store(ds.raw_store, ds.gt_store, pos, ds.white_level, ds.status, kind, chain, params,
                                          u8=True)
        ref_sse, ref_u8, ref_ss, gt = composition(ds, pos, kind, chain, params, ssim)
        assert torch.equal(sse, ref_sse), (kind, st, sse.tolist(), ref_sse.tolist())
        assert torch.equal(u8, ref_u8), (kind, st)
        sse2, none = ops.pipeline_eval_store(ds.raw_store, ds.gt_store, pos, ds.white_level, ds.status, kind, chain, params)
        assert none is None and torch.equal(sse2, ref_sse)
        if ssim:
            assert torch.equal(ops.ssim_u8_store(u8, ds.gt_store, pos, ds.status), ref_ss)
            y = ops.pipeline_fwd(ops.sample_crops(ds.raw_store, None, pos, ds.H, ds.W, ds.white_level, ds.status)[0], kind,
                                 chain, params)
            assert torch.equal(ops.ssim_u8_store(y, ds.gt_store, pos, ds.status), ops.ssim_u8(y, gt))
    ds.check()


@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('sig', list(SIGS))
def test_store_eval_equals_composition_on_packed_chains(kind, sig):
    """Every raw code type at every narrow-item width; H = 38 is not a multiple of 8; 5 frames in batches of 3."""
    g = torch.Generator().manual_seed(sum(map(ord, kind + sig)))
    for i, (dtype, hi, wl) in enumerate(RAWS):
        W = WIDTHS[(i + KINDS.index(kind)) % 3]
        ds, _, _ = make_store(5, 5, 38, W, dtype, hi, wl, seed=i + 10 * KINDS.index(kind))
        check_store(ds, kind, SIGS[sig], g)


@pytest.mark.parametrize('dtype,hi,wl', RAWS)
def test_store_eval_hwc_gt_pairs_and_all_widths(dtype, hi, wl):
    pairs = [0, 0, 0, 1, 1, 2, 2]
    g = torch.Generator().manual_seed(5)
    for W in WIDTHS:
        ds, _, _ = make_store(7, 3, 46, W, dtype, hi, wl, seed=W, hwc=True, pairs=pairs)
        assert ds.gt_store.shape[0] == 3
        check_store(ds, 'bilinear', SIGS['A'], g, batch=4)
        check_store(ds, 'malvar', SIGS['D'], g, batch=2)


def test_store_eval_interpreter_chain_and_ssim():
    g = torch.Generator().manual_seed(6)
    for i, (dtype, hi, wl) in enumerate(RAWS):
        ds, _, _ = make_store(4, 4, 40, 96 + 16 * i, dtype, hi, wl, seed=20 + i)
        for kind in KINDS:
            check_store(ds, kind, INTERP, g, ssim=True)
        check_store(ds, 'bilinear', SIGS['B'], g, ssim=True)


def test_store_eval_rejects_widths_the_tensor_maps_cannot_describe():
    """The packed kernels read the stores through tensor maps (rows of 16-byte multiples); the interpreter does not."""
    from reconfigisp_b200 import ops
    ds, _, _ = make_store(2, 2, 16, 40, np.uint16, 1024, 1023., seed=1)
    pos = torch.from_numpy(ds.plan_.frames('all')[0]).cuda()
    with pytest.raises(NotImplementedError):
        ops.pipeline_eval_store(ds.raw_store, ds.gt_store, pos, 1023., ds.status, 'bilinear', ops.Chain(SIGS['D']),
                                stage_params(SIGS['D'], torch.Generator().manual_seed(0)).cuda())
    g = torch.Generator().manual_seed(2)
    check_store(ds, 'bilinear', INTERP, g)


def child_cases(out):
    """In a child process (RISP_FUSED=0: every chain on the interpreter kernels): store == composition, checked there."""
    g = torch.Generator().manual_seed(9)
    for i, (dtype, hi, wl) in enumerate(RAWS):
        ds, _, _ = make_store(5, 5, 38, WIDTHS[i], dtype, hi, wl, seed=30 + i)
        for kind in KINDS:
            for st in (SIGS['A'], SIGS['skip'], INTERP):
                check_store(ds, kind, st, g, ssim=True)
    open(out, 'w').write('ok')


def test_store_eval_under_interpreter_only(tmp_path):
    env = dict(os.environ)
    env.pop('RISP_FUSED_STEP_ROWS', None)
    env['RISP_FUSED'] = '0'
    out = tmp_path / 'ok.txt'
    cmd = [sys.executable] + (['-s'] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    assert out.read_text() == 'ok'


def test_store_metrics_match_the_oracles_on_a_small_frame():
    from reconfigisp_b200 import metrics, ops
    H, W = 24, 32
    ds, raws, gts = make_store(2, 2, H, W, np.uint16, 1024, 1023., seed=4)
    pos = torch.from_numpy(ds.plan_.frames('all')[0]).cuda()
    sse, u8 = ops.pipeline_eval_store(ds.raw_store, ds.gt_store, pos, 1023., ds.status, 'bilinear', ops.Chain([]), None,
                                      u8=True)
    ss = ops.ssim_u8_store(u8, ds.gt_store, pos, ds.status)
    y = u8.permute(0, 3, 1, 2).cpu().numpy().astype(np.float32) / np.float32(255.)     # its codes are its own tensor2bgr codes
    gt = gts.astype(np.float32) / np.float32(255.)
    assert sse.cpu().numpy().tolist() == M.sse_u8(y, gt).tolist()
    assert np.allclose(metrics.psnr_from_sse(sse, 3 * H * W), M.psnr(y, gt), rtol=0, atol=1e-9)
    assert np.allclose(metrics.ssim_from_sums(ss, 3, H, W), SO.ssim(y, gt), rtol=0, atol=1e-6)
    # the image itself: the fp64 oracle demosaic of code / 1023, codes within 1 (a truncation may flip)
    ref = O.demosaic_bilinear(torch.from_numpy(raws.astype(np.float64) / 1023.)).numpy()
    ref8 = np.stack([M.tensor2bgr(r) for r in ref]).astype(int)
    d = np.abs(ref8 - u8.cpu().numpy().astype(int))
    assert d.max() <= 1 and (d > 0).mean() < 1e-3
    ds.check()


def test_bad_records_set_the_status_and_check_raises():
    from reconfigisp_b200 import ops
    ds, _, _ = make_store(3, 3, 16, 32, np.uint16, 1024, 1023., seed=3)
    chain = ops.Chain(SIGS['D'])
    params = stage_params(SIGS['D'], torch.Generator().manual_seed(0)).cuda()
    for bad in ([3, 0, 0, 0], [0, 3, 0, 0], [-1, 0, 0, 0], [0, 0, 2, 0], [0, 0, 0, 4]):
        pos = torch.tensor([[1, 1, 0, 0], bad, [2, 2, 0, 0]], dtype=torch.int32).cuda()
        ref = composition(ds, pos[[0, 2]], 'bilinear', chain, params)[0]
        for interp in (False, True):
            st, pr = (INTERP, stage_params(INTERP, torch.Generator().manual_seed(0)).cuda()) if interp else (chain, params)
            c = ops.Chain(st) if interp else chain
            sse, _ = ops.pipeline_eval_store(ds.raw_store, ds.gt_store, pos, 1023., ds.status, 'bilinear', c, pr, u8=True)
            assert int(sse[1]) == 0, bad
            if not interp:
                assert sse[[0, 2]].tolist() == ref.tolist()
            with pytest.raises(RuntimeError):
                ds.check()
            assert int(ds.status.item()) == 0
        if bad[1] == 3 or bad[2] or bad[3]:
            y8 = torch.zeros((3, 16, 32, 3), dtype=torch.uint8, device='cuda')
            assert int(ops.ssim_u8_store(y8, ds.gt_store, pos, ds.status)[1]) == 0
            with pytest.raises(RuntimeError):
                ds.check()


# ---- DeviceDataset.evaluate ----------------------------------------------------------------------------------------
def _nets():
    from reconfigisp_b200.modules.isp_universal import IspUniversal
    from reconfigisp_b200.modules.origin_universal import OriginUniversal
    return [
        ('origin_head', lambda: OriginUniversal('/x/', 'Bayer_02_Demosaic_02_sRGB_11_13_01_14', weight_seed=10), True),
        ('isp_head', lambda: IspUniversal('/x/', (None,) * 6, 'Bayer_02_Demosaic_01_sRGB_11_13_01_14', weight_seed=10), True),
        ('grayworld', lambda: OriginUniversal('/x/', 'Bayer_02_Demosaic_02_sRGB_05_11_13_01', weight_seed=10), False),
        ('cnn', lambda: IspUniversal('/x/', (None,) * 4, 'Bayer_02_Demosaic_01_sRGB_11_12', weight_seed=10), False),
    ]


def host_loop(net, ds, split, raws, gts, ssim, batch):
    """The reference's validation: every frame of the split, whole, through net.evaluate, decoded on the host (batches of
    the same frames, so that a CNN stage sees the same batch shapes)."""
    lo, hi = ds.plan_.spans[split]
    out = []
    for f in range(lo, hi, batch):
        e = min(hi, f + batch)
        raw = torch.from_numpy(raws[f:e].astype(np.float32) / np.float32(ds.white_level)).cuda()
        gt = torch.from_numpy(gts[f:e].astype(np.float32) / np.float32(255.)).cuda()
        out.append(net.evaluate(raw, gt, ssim=ssim))
    return torch.cat([r[0] for r in out]), (torch.cat([r[2] for r in out]) if ssim else None)


@pytest.mark.parametrize('name', ['origin_head', 'isp_head', 'grayworld', 'cnn'])
def test_dataset_evaluate_equals_host_loop(name):
    make, store = {n: (m, s) for n, m, s in _nets()}[name]
    net = make().cuda()
    assert (net.store_eval_plan() is not None) == store
    H, W = 48, 160
    ds, raws, gts = make_store(7, 7, H, W, np.uint16, 1024, 1023., seed=8)
    before = [p.detach().clone() for p in net.all_params]
    for split, batch in (('val', 3), ('all', 4), ('train', 1)):
        frames, sse, ss = ds.evaluate(net, split, batch=batch, ssim=True)
        ref_sse, ref_ss = host_loop(net, ds, split, raws.view(np.uint16) if raws.dtype == np.int16 else raws, gts, True, batch)
        lo, hi = ds.plan_.spans[split]
        assert frames.tolist() == list(range(lo, hi))
        assert torch.equal(sse, ref_sse), (name, split, sse.tolist(), ref_sse.tolist())
        assert torch.equal(ss, ref_ss), (name, split)
        f2, sse2 = ds.evaluate(net, split, batch=batch)
        assert torch.equal(sse2, sse) and torch.equal(f2, frames)
    assert all(torch.equal(a, p.detach()) for a, p in zip(before, net.all_params))
    ds.check()


def test_evaluate_makes_no_host_sync():
    from reconfigisp_b200.modules.origin_universal import OriginUniversal
    net = OriginUniversal('/x/', 'Bayer_02_Demosaic_02_sRGB_11_13_01_14', weight_seed=10).cuda()
    ds, _, _ = make_store(6, 6, 32, 128, np.uint16, 1024, 1023., seed=2)
    ds.evaluate(net, 'val', batch=2, ssim=True)                   # first call: records uploaded, buffers made
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        for _ in range(3):
            res = ds.evaluate(net, 'val', batch=2, ssim=True)
            ds.evaluate(net, 'all', batch=4)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    from reconfigisp_b200 import metrics
    assert np.isfinite(metrics.psnr_from_sse(res[1], 3 * 32 * 128)).all()
    ds.check()


def test_evaluate_between_training_steps_changes_nothing():
    """A run that validates trains on the same batches, reaches graph replay and ends with the same parameters."""
    from reconfigisp_b200.data import DeviceDataset
    from reconfigisp_b200.synthetic import synthetic_frames
    from reconfigisp_b200.tuning import IspModel
    opt = {'model': 'isp', 'is_train': True,
           'network_G': {'which_model_G': 'OriginUniversal', 'architecture': 'Bayer_02_Demosaic_02_sRGB_11_13_01_14',
                         'weight_seed': 10},
           'train': {'lr_G': 1e-3, 'beta1': 0.9, 'beta2': 0.99, 'pixel_criterion': 'l2', 'lr_scheme': 'MultiStepLR',
                     'lr_steps': [20000], 'lr_gamma': 0.5},
           'path': {'pretrain_model_G': None}}
    raw_f, gt_f = synthetic_frames(6, 96, 128, seed=10)
    raws, gts = torch.round(raw_f * 1023).to(torch.int16), torch.round(gt_f * 255).to(torch.uint8)

    def run(validate):
        ds = DeviceDataset(raws, gts, 1023., (64, 96), seed=3)
        m = IspModel(opt)
        out = []
        for s in range(7):
            m.feed_data(ds.sample(3, 'all'))
            m.optimize_parameters()
            out.append((m.log_dict['loss'].item(), m._flat_grad.clone()))
            if validate and s % 2 == 0:
                ds.evaluate(m, 'val', batch=2, ssim=True)
                ds.evaluate(m.netG, 'all', batch=4)
        assert m.__dict__.get('_graphs'), 'the step never reached graph replay'
        assert ds.steps == {'train': 0, 'val': 0, 'all': 7}
        ds.check()
        return out, torch.cat([p.detach().reshape(-1) for p in m.netG.trainable_parameters])
    a, pa = run(True)
    b, pb = run(False)
    for s, ((l0, g0), (l1, g1)) in enumerate(zip(a, b)):
        assert l0 == l1 and torch.equal(g0, g1), s
    assert torch.equal(pa, pb)


def test_store_eval_equals_composition_at_12mp():
    ds, _, _ = make_store(4, 4, 3000, 4000, np.uint16, 16384, 16383., seed=12, crop=16)
    g = torch.Generator().manual_seed(12)
    for kind, sig in (('bilinear', 'A'), ('malvar', 'D')):
        check_store(ds, kind, SIGS[sig], g, batch=4, ssim=(sig == 'A'))


WORKER = r'''
import os, sys, torch, numpy as np
sys.path.insert(0, os.environ['RISP_ROOT'])
import torch.distributed as dist
from reconfigisp_b200 import dist as D
from reconfigisp_b200.data import DeviceDataset
from reconfigisp_b200.modules.origin_universal import OriginUniversal
from reconfigisp_b200.modules.isp_universal import IspUniversal
rank, world, local = D.init_from_env('nccl')
torch.cuda.set_device(local)
rng = np.random.default_rng(1)
raws = rng.integers(0, 1024, (9, 1, 48, 160)).astype(np.uint16)
gts = rng.integers(0, 256, (9, 3, 48, 160)).astype(np.uint8)
out = {}
for name, net in (('head', OriginUniversal('/x/', 'Bayer_02_Demosaic_02_sRGB_11_13_01_14', weight_seed=10)),
                  ('grayworld', OriginUniversal('/x/', 'Bayer_02_Demosaic_02_sRGB_05_11_13_01', weight_seed=10))):
    net = net.cuda()
    for w, r in ((1, 0), (world, rank)):
        ds = DeviceDataset(raws, gts, 1023., 16, rank=r, world=w)
        if w == 1 and rank != 0:
            continue
        for split in ('val', 'all'):
            res = ds.evaluate(net, split, batch=2, ssim=True)
            out['%s_%s_%d' % (name, split, w)] = torch.stack(res).cpu()
        ds.check()
allr = [None] * world
dist.all_gather_object(allr, {k: v for k, v in out.items() if k.endswith('_%d' % world)})
if rank == 0:
    for k, v in out.items():
        if k.endswith('_1'):
            for r in range(world):
                assert torch.equal(allr[r][k[:-2] + '_%d' % world], v), (k, r)
    open(os.environ['RISP_OUT'], 'w').write('ok')
dist.barrier(); dist.destroy_process_group()
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs >= 2 GPUs')
def test_world_two_evaluate_returns_the_world_one_tensors(tmp_path):
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
