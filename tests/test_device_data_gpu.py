"""The HBM-resident dataset on the device: `risp_sample_crops` bit-exact against numpy slicing and division, its check of
bad records, and the tuning / search models trained from `DeviceDataset.sample` against the same crops fed from the host."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _codes(F, H, W, dtype, hi, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, hi, (F, 1, H, W)).astype(dtype)


def _gts(G, H, W, seed):
    return np.random.default_rng(seed).integers(0, 256, (G, 3, H, W)).astype(np.uint8)


def _expected(ds, raws, gts, rec, white_level):
    """numpy: the records' crops of the host frames, / white_level and / 255 in fp32."""
    p = ds.plan_
    h, w = ds.h, ds.w
    img = np.stack([raws[p.raw_frames[r[0]], :, r[2]:r[2] + h, r[3]:r[3] + w] for r in rec])
    gt = np.stack([gts[p.gt_frames[r[1]], :, r[2]:r[2] + h, r[3]:r[3] + w] for r in rec])
    return img.astype(np.float32) / np.float32(white_level), gt.astype(np.float32) / np.float32(255.)


@pytest.mark.parametrize('dtype,hi,white_level', [(np.uint16, 65536, 16383.), (np.int16, 16384, 16383.), (np.uint8, 256, 255.),
                                                  (np.uint16, 1024, 1023.)])
@pytest.mark.parametrize('crop', [(24, 32), (22, 30), (10, 6)])
def test_sample_is_bit_exact_against_numpy(dtype, hi, white_level, crop):
    from reconfigisp_b200.data import DeviceDataset
    H, W, B = 40, 58, 5
    raws, gts = _codes(6, H, W, dtype, hi, 1), _gts(6, H, W, 2)
    ds = DeviceDataset(raws, gts, white_level, crop, seed=7)
    for step, split in enumerate(('train', 'val', 'all', 'train')):
        rec = ds.plan(split, ds.steps[split], B)
        img, gt = ds.sample(B, split)
        ei, eg = _expected(ds, raws.view(np.uint16) if dtype == np.int16 else raws, gts, rec, white_level)
        assert np.array_equal(img.cpu().numpy(), ei), (split, step)
        assert np.array_equal(gt.cpu().numpy(), eg), (split, step)
    ds.check()


def test_whole_frames_equal_decode_codes_and_hwc_gt():
    from reconfigisp_b200 import ops
    from reconfigisp_b200.data import DeviceDataset
    H, W = 48, 64
    raws, gts = _codes(4, H, W, np.uint16, 1024, 3), _gts(4, H, W, 4)
    ds = DeviceDataset(raws, np.ascontiguousarray(gts.transpose(0, 2, 3, 1)), 1023., (H, W))
    rec = ds.plan('all', 0, 4)
    img, gt = ds.sample(4, 'all')
    order = ds.plan_.raw_frames[rec[:, 0]]
    ref_img = ops.decode_codes(torch.from_numpy(raws[order].view(np.int16)).cuda(), 1023.)
    ref_gt = ops.decode_codes(torch.from_numpy(gts[order]).cuda(), 255.)
    assert torch.equal(img, ref_img) and torch.equal(gt, ref_gt)


def test_pairs_with_several_raws_per_gt_and_a_shard():
    from reconfigisp_b200.data import DeviceDataset
    H, W = 32, 44
    pairs = [0, 0, 0, 1, 1, 2, 2, 2, 2]
    raws, gts = _codes(9, H, W, np.uint16, 16384, 5), _gts(3, H, W, 6)
    for rank in range(2):
        ds = DeviceDataset([torch.from_numpy(f[0].astype(np.int16)) for f in raws], torch.from_numpy(gts), 16383., 12,
                           pairs=pairs, rank=rank, world=2)
        assert ds.raw_store.shape[0] == len(range(rank, 9, 2))
        for _ in range(4):
            rec = ds.plan('all', ds.steps['all'], 3)
            img, gt = ds.sample(3, 'all')
            ei, eg = _expected(ds, raws, gts, rec, 16383.)
            assert np.array_equal(img.cpu().numpy(), ei) and np.array_equal(gt.cpu().numpy(), eg)
            assert [pairs[f] for f in ds.plan_.raw_frames[rec[:, 0]]] == ds.plan_.gt_frames[rec[:, 1]].tolist()
        ds.check()


def test_one_record_equals_crop_decode():
    from reconfigisp_b200 import ops
    H, W, h, w = 60, 80, 32, 40
    raw = torch.from_numpy(_codes(3, H, W, np.int16, 16384, 7)[:, 0]).cuda()
    gt = torch.from_numpy(_gts(2, H, W, 8)).cuda()
    status = torch.zeros(1, dtype=torch.int32, device='cuda')
    pos = torch.tensor([[2, 1, 12, 34]], dtype=torch.int32, device='cuda')
    img, g = ops.sample_crops(raw, gt, pos, h, w, 16383., status)
    assert torch.equal(img[0], ops.crop_decode(raw[2:3], 12, 34, h, w, 16383.))
    assert torch.equal(g[0], ops.crop_decode(gt[1], 12, 34, h, w, 255., bayer=False))
    only, none = ops.sample_crops(raw, None, pos, h, w, 16383., status)
    assert none is None and torch.equal(only, img)
    assert int(status.item()) == 0


def test_bad_record_sets_status_and_is_skipped():
    """An odd origin whose crop is still inside the allocation: the record is skipped and flagged, the others are right."""
    from reconfigisp_b200 import ops
    H, W, h, w = 32, 40, 8, 12
    raws, gts = _codes(2, H, W, np.uint16, 1024, 9), _gts(2, H, W, 10)
    raw, gt = torch.from_numpy(raws[:, 0].view(np.int16)).cuda(), torch.from_numpy(gts).cuda()
    rec = np.array([[0, 1, 4, 6], [1, 0, 3, 6], [1, 1, 0, 28]], dtype=np.int32)
    pos = torch.from_numpy(rec).cuda()
    status = torch.zeros(1, dtype=torch.int32, device='cuda')
    img = torch.full((3, 1, h, w), float('nan'), device='cuda')
    g = torch.full((3, 3, h, w), float('nan'), device='cuda')
    ops.sample_crops(raw, gt, pos, h, w, 1023., status, img, g)
    assert int(status.item()) != 0
    for k in (0, 2):
        r = rec[k]
        assert np.array_equal(img[k].cpu().numpy(), raws[r[0], :, r[2]:r[2] + h, r[3]:r[3] + w].astype(np.float32) / np.float32(1023.))
        assert np.array_equal(g[k].cpu().numpy(), gts[r[1], :, r[2]:r[2] + h, r[3]:r[3] + w].astype(np.float32) / np.float32(255.))
    assert torch.isnan(img[1]).all() and torch.isnan(g[1]).all()


def test_sample_does_not_sync_and_returns_stable_buffers():
    from reconfigisp_b200.data import DeviceDataset
    raws, gts = _codes(4, 32, 48, np.uint16, 1024, 11), _gts(4, 32, 48, 12)
    ds = DeviceDataset(raws, gts, 1023., 16)
    first = [t.data_ptr() for t in ds.sample(3) + ds.sample(3, 'val')]
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        for _ in range(5):
            ptrs = [t.data_ptr() for t in ds.sample(3) + ds.sample(3, 'val')]
            assert ptrs == first
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert len(set(first)) == 4                      # train and val batches do not alias
    ds.check()


def _opt_tuning():
    return {'model': 'isp', 'is_train': True,
            'network_G': {'which_model_G': 'OriginUniversal', 'architecture': 'Bayer_02_Demosaic_02_sRGB_11_13_01_14', 'weight_seed': 10},
            'train': {'lr_G': 1e-3, 'beta1': 0.9, 'beta2': 0.99, 'pixel_criterion': 'l2', 'lr_scheme': 'MultiStepLR',
                      'lr_steps': [20000], 'lr_gamma': 0.5},
            'path': {'pretrain_model_G': None}}


def test_isp_model_trains_the_same_from_the_store_and_from_host_codes():
    """Past the eager steps into graph replay: losses, gradients and parameters bit-identical to the host-codes feed."""
    from reconfigisp_b200.data import DeviceDataset
    from reconfigisp_b200.synthetic import synthetic_frames
    from reconfigisp_b200.tuning import IspModel
    raw_f, gt_f = synthetic_frames(6, 96, 128, seed=10)
    raws = torch.round(raw_f * 1023).to(torch.int16)
    gts = torch.round(gt_f * 255).to(torch.uint8)
    B, crop, steps = 3, (64, 96), 7
    ds = DeviceDataset(raws, gts, 1023., crop, seed=3)
    recs = [ds.plan('all', s, B) for s in range(steps)]

    def run(feed):
        m = IspModel(_opt_tuning())
        out = []
        for s in range(steps):
            m.feed_data(feed(s))
            m.optimize_parameters()
            out.append((m.log_dict['loss'].item(), m._flat_grad.clone()))
        assert m.__dict__.get('_graphs'), 'the step never reached graph replay'
        return out, torch.cat([p.detach().reshape(-1) for p in m.netG.trainable_parameters])

    def host(s):
        r = recs[s]
        fr = ds.plan_.raw_frames[r[:, 0]]
        img = torch.stack([raws[f, :, y:y + crop[0], x:x + crop[1]] for f, y, x in zip(fr, r[:, 2], r[:, 3])])
        gt = torch.stack([gts[f, :, y:y + crop[0], x:x + crop[1]] for f, y, x in zip(fr, r[:, 2], r[:, 3])])
        return img.contiguous(), gt.contiguous()
    dev, p_dev = run(lambda s: ds.sample(B, 'all'))
    ref, p_ref = run(host)
    for s, ((l0, g0), (l1, g1)) in enumerate(zip(dev, ref)):
        assert l0 == l1 and torch.equal(g0, g1), s
    assert torch.equal(p_dev, p_ref)
    ds.check()


def test_darts_model_iteration_from_the_store_equals_host_feed():
    from reconfigisp_b200.data import DeviceDataset
    from reconfigisp_b200.search import DartsModel
    opt = {'model': 'darts', 'network_G': {'which_model_G': 'SuperPruneFifteenDemosFourBayerTwo', 'n_step': 3, 'n_modules': 15,
                                          'prune_threshold': 0.2, 'weight_seed': 10},
           'train': {'lr_G': 1e-3, 'momentum_G': 0.9, 'lr_meta': 1e-3, 'beta1': 0.9, 'beta2': 0.999, 'pixel_criterion': 'l2'}}
    H, W, B, S = 96, 112, 2, 48
    raws, gts = _codes(8, H, W, np.uint16, 1024, 13), _gts(8, H, W, 14)
    ds = DeviceDataset(raws, gts, 1023., S, seed=5)
    rt, rv = ds.plan('train', 0, B), ds.plan('val', 0, B)
    feeds = {'device': ds.sample(B) + ds.sample(B, 'val'),
             'host': tuple(torch.from_numpy(a) for a in _expected(ds, raws, gts, rt, 1023.) + _expected(ds, raws, gts, rv, 1023.))}
    res = {}
    for name, data in feeds.items():
        m = DartsModel(opt)
        m.feed_data(data)
        m.optimize_alphas()
        m.optimize_parameters()
        res[name] = [m.img, m.gt, m.val_img, m.val_gt, m.log_dict['loss'].detach().reshape(1), torch.as_tensor(m.val_loss).reshape(1).cuda()] + \
            [a.grad for a in m.netG.alphas] + [p.detach() for p in m.netG.trainable_parameters if p.numel()]
    for k, (a, b) in enumerate(zip(res['device'], res['host'])):
        assert torch.equal(a, b), k
    ds.check()
