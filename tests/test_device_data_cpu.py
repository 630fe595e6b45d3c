"""The host side of the HBM-resident dataset: the sampling plan and the input checks of `DeviceDataset` (no GPU)."""
import numpy as np
import pytest

from reconfigisp_b200.data import DeviceDataset, SamplingPlan


def _global(p, rec):
    """Records of a plan -> (global raw frame, global GT frame) pairs."""
    return p.raw_frames[rec[:, 0]], p.gt_frames[rec[:, 1]]


def test_plan_is_deterministic_for_seed_rank_world():
    a = SamplingPlan(20, np.arange(20), (64, 80), (16, 24), seed=3, rank=1, world=2)
    b = SamplingPlan(20, np.arange(20), (64, 80), (16, 24), seed=3, rank=1, world=2)
    for split in ('train', 'val', 'all'):
        for step in (0, 1, 7):
            ra, rb = a.plan(split, step, 6), b.plan(split, step, 6)
            assert ra.dtype == np.int32 and ra.shape == (6, 4)
            assert np.array_equal(ra, rb)
    # out-of-order queries give the same batches (a pure function of the step)
    assert np.array_equal(b.plan('train', 7, 6), a.plan('train', 7, 6))
    c = SamplingPlan(20, np.arange(20), (64, 80), (16, 24), seed=4, rank=1, world=2)
    assert not all(np.array_equal(a.plan('all', s, 6), c.plan('all', s, 6)) for s in range(3))


@pytest.mark.parametrize('B', [1, 3, 5, 7])
def test_each_epoch_visits_every_frame_of_the_shard_once(B):
    p = SamplingPlan(30, np.arange(30), (32, 32), (8, 8), seed=10, rank=2, world=3)
    for split in ('train', 'val', 'all'):
        n = len(p.shards[split])
        stream = np.concatenate([p.plan(split, s, B)[:, 0] for s in range(4 * n // B + 2)])
        for e in range(3):
            ep = stream[e * n:(e + 1) * n]
            assert sorted(ep.tolist()) == sorted(p.shards[split].tolist())
        assert not all(np.array_equal(stream[:n], stream[e * n:(e + 1) * n]) for e in (1, 2))   # epochs are reshuffled


def test_shards_are_disjoint_and_cover_the_dataset():
    F, world = 23, 4
    seen = []
    for r in range(world):
        p = SamplingPlan(F, np.arange(F), (16, 16), (4, 4), rank=r, world=world)
        assert all(f % world == r for f in p.raw_frames)
        frames = set()
        for s in range(40):
            raw, gt = _global(p, p.plan('all', s, 3))
            assert np.array_equal(raw, gt)
            frames |= set(raw.tolist())
        assert frames == set(p.raw_frames.tolist())
        seen.append(frames)
    assert set().union(*seen) == set(range(F)) and sum(len(s) for s in seen) == F


def test_train_and_val_halves_are_disjoint():
    F = 17
    for world in (1, 3):
        train, val = set(), set()
        for r in range(world):
            p = SamplingPlan(F, np.arange(F), (16, 16), (4, 4), rank=r, world=world)
            for s in range(30):
                train |= set(_global(p, p.plan('train', s, 2))[0].tolist())
                val |= set(_global(p, p.plan('val', s, 2))[0].tolist())
        assert train == set(range(F // 2)) and val == set(range(F // 2, F))


def test_pairs_map_raws_to_their_gt_frames():
    pairs = np.array([0, 0, 0, 1, 1, 2, 2, 2])
    for r in range(2):
        p = SamplingPlan(8, pairs, (16, 16), (4, 4), rank=r, world=2)
        assert set(p.gt_frames.tolist()) == set(pairs[p.raw_frames].tolist())
        for s in range(10):
            raw, gt = _global(p, p.plan('all', s, 3))
            assert np.array_equal(gt, pairs[raw])


def test_origins_are_even_in_range_and_cover_every_legal_position():
    H, W, h, w = 14, 20, 6, 8
    p = SamplingPlan(4, np.arange(4), (H, W), (h, w), seed=5)
    rec = np.concatenate([p.plan('all', s, 16) for s in range(200)])
    ys, xs = rec[:, 2], rec[:, 3]
    assert (ys % 2 == 0).all() and (xs % 2 == 0).all()
    assert ys.min() >= 0 and xs.min() >= 0 and (ys + h).max() <= H and (xs + w).max() <= W
    assert set(zip(ys.tolist(), xs.tolist())) == {(y, x) for y in range(0, H - h + 1, 2) for x in range(0, W - w + 1, 2)}
    whole = SamplingPlan(2, np.arange(2), (H, W), (H, W)).plan('all', 0, 4)
    assert (whole[:, 2:] == 0).all()


def test_plan_rejects_bad_splits_and_empty_shards():
    p = SamplingPlan(3, np.arange(3), (8, 8), (2, 2), rank=2, world=3)
    with pytest.raises(ValueError):
        p.plan('test', 0, 1)
    with pytest.raises(ValueError):
        p.plan('train', 0, 1)                 # frame 2 is in the val half: rank 2 holds no training frame
    with pytest.raises(ValueError):
        SamplingPlan(3, np.arange(3), (8, 8), (2, 2), rank=3, world=3)


def _frames(F=4, H=16, W=24, dtype=np.uint16):
    rng = np.random.default_rng(0)
    return rng.integers(0, 1000, (F, 1, H, W)).astype(dtype), rng.integers(0, 256, (F, 3, H, W)).astype(np.uint8)


@pytest.mark.parametrize('case', ['raw_dtype', 'gt_dtype', 'mixed_raw_dtypes', 'raw_sizes', 'gt_size', 'odd_frame', 'odd_crop',
                                  'crop_too_large', 'pairs_len', 'pairs_range', 'negative_int16', 'empty', 'white_level'])
def test_device_dataset_rejects_bad_inputs(case):
    raws, gts = _frames()
    kw = dict(white_level=1023., crop=8)
    if case == 'raw_dtype':
        raws = raws.astype(np.float32)
    elif case == 'gt_dtype':
        gts = gts.astype(np.uint16)
    elif case == 'mixed_raw_dtypes':
        raws = [raws[0, 0], raws[1, 0].astype(np.uint8)]
    elif case == 'raw_sizes':
        raws = [raws[0, 0], raws[1, 0, :, :22]]
    elif case == 'gt_size':
        gts = gts[:, :, :, :22]
    elif case == 'odd_frame':
        raws, gts = raws[:, :, :15], gts[:, :, :15]
    elif case == 'odd_crop':
        kw['crop'] = (8, 7)
    elif case == 'crop_too_large':
        kw['crop'] = (18, 8)
    elif case == 'pairs_len':
        kw['pairs'] = [0, 1, 2]
    elif case == 'pairs_range':
        kw['pairs'] = [0, 1, 2, 4]
    elif case == 'negative_int16':
        raws = raws.astype(np.int16)
        raws[2, 0, 3, 3] = -1
    elif case == 'empty':
        raws = []
    elif case == 'white_level':
        kw['white_level'] = 0.
    with pytest.raises(ValueError):
        DeviceDataset(raws, gts, **kw)


def test_sample_crops_is_declared_in_the_header():
    from reconfigisp_b200 import _lib
    ret, args = _lib.PROTOS['risp_sample_crops']
    assert [a for _, a in args] == ['raw_store', 'raw_bytes_per_code', 'F', 'gt_store', 'G', 'H', 'W', 'pos', 'B', 'h', 'w',
                                    'white_level', 'img_out', 'gt_out', 'status', 'stream']
