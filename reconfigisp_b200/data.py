"""Training data resident in HBM: a frame store of integer codes and batched crop sampling on the device.

The reference's loaders decode a full-frame PNG on the host for every sample, crop it there and ship fp32 over PCIe
(sid_sony_ratio_rggb2bgr_dataset.py:109-136, s7isp_rggb2bgr_dataset.py:123).  `DeviceDataset` uploads the frames once,
as codes (2 + 3 B per pixel for a 16-bit raw and its 8-bit GT), and fills each batch with one launch of
`risp_sample_crops`: the loader's even-aligned random crop and its division (`/white_level`, `/255`), bit-exact.  Only the
plan -- B records of 16 bytes -- crosses PCIe per batch.

    ds = DeviceDataset(raws, gts, white_level=1023., crop=224, rank=rank, world=world)
    model.feed_data(ds.sample(8, 'all'))                        # tuning (IspModel): every frame of the shard
    model.feed_data(ds.sample(4) + ds.sample(4, 'val'))         # search (DartsModel): DARTS train / validation halves

PNG decode stays on the host (cv2), once per frame, before the store is built.  The reference's dataset classes, file
layouts and augmentation are not reproduced.  The SID loader's exposure-ratio amplification (sid_sony_ratio_...) is not
applied either: its formula is not recorded in this repository, so a caller that needs it scales the codes beforehand.
"""
import numpy as np
import torch

from . import ops

SPLITS = ('train', 'val', 'all')


def _even_pair(v, what):
    h, w = (v, v) if np.isscalar(v) else tuple(v)
    h, w = int(h), int(w)
    if h <= 0 or w <= 0 or h % 2 or w % 2:
        raise ValueError('%s must be even and positive (the RGGB phase), got %dx%d' % (what, h, w))
    return h, w


class SamplingPlan:
    """Which frame and which crop every record of every batch reads; host only, reproducible from (seed, rank, world).

    Frames are split like the reference's samplers (data_sampler.py:69-150): 'train' is the first half of the frames and
    'val' the second half (the DARTS training and validation halves of DistIterTrainSampler / DistIterValSampler); 'all'
    is every frame.  Rank r of `world` owns the frames i = r (mod world), so shards are disjoint and cover the dataset.
    Each epoch of a split is a seeded permutation of the rank's frames of that split; batches are consecutive runs of
    that endless sequence.  Crop origins are uniform over the even positions of [0, H-h] x [0, W-w].

    Records hold LOCAL store indices: the store keeps the rank's raw frames `raw_frames` (global indices, ascending) and
    the GT frames they pair with, `gt_frames`."""

    def __init__(self, n_frames, pairs, frame_hw, crop_hw, seed=10, rank=0, world=1):
        self.H, self.W = frame_hw
        self.h, self.w = crop_hw
        self.seed, self.rank, self.world = int(seed), int(rank), int(world)
        if self.world < 1 or not 0 <= self.rank < self.world:
            raise ValueError('rank %d of world %d' % (rank, world))
        pairs = np.asarray(pairs, dtype=np.int64)
        self.raw_frames = np.arange(self.rank, n_frames, self.world)
        self.gt_frames = np.unique(pairs[self.raw_frames])
        self._raw_slot = {int(f): k for k, f in enumerate(self.raw_frames)}
        self._gt_of = np.searchsorted(self.gt_frames, pairs[self.raw_frames]).astype(np.int32)   # raw slot -> GT slot
        half = n_frames // 2
        spans = {'train': (0, half), 'val': (half, n_frames), 'all': (0, n_frames)}
        self.shards = {s: np.array([self._raw_slot[int(f)] for f in self.raw_frames if lo <= f < hi], dtype=np.int64)
                       for s, (lo, hi) in spans.items()}
        self._perm = {}

    def epoch(self, split, e):
        """Local raw slots of this rank's frames of `split` in the order epoch e visits them."""
        key = (split, e)
        if key not in self._perm:
            rng = np.random.Generator(np.random.PCG64([self.seed, self.rank, self.world, SPLITS.index(split), e]))
            if len(self._perm) > 4:
                self._perm.clear()
            self._perm[key] = self.shards[split][rng.permutation(len(self.shards[split]))]
        return self._perm[key]

    def plan(self, split, step, B):
        """Records of batch `step` of B crops from `split`: int32 (B,4) = (raw slot, GT slot, y0, x0)."""
        if split not in SPLITS:
            raise ValueError('split must be one of %s, got %r' % (SPLITS, split))
        n = len(self.shards[split])
        if n == 0:
            raise ValueError("rank %d of %d holds no frame of the '%s' split" % (self.rank, self.world, split))
        first = step * B
        slots = np.concatenate([self.epoch(split, e) for e in range(first // n, (first + B - 1) // n + 1)])
        slots = slots[first % n:first % n + B]
        rng = np.random.Generator(np.random.PCG64([self.seed, self.rank, self.world, SPLITS.index(split), 1 << 20, step]))
        out = np.empty((B, 4), dtype=np.int32)
        out[:, 0] = slots
        out[:, 1] = self._gt_of[slots]
        out[:, 2] = 2 * rng.integers(0, (self.H - self.h) // 2 + 1, B)
        out[:, 3] = 2 * rng.integers(0, (self.W - self.w) // 2 + 1, B)
        return out


def _frames(x):
    """A (F,C,...) array / tensor or a list of frames -> list of per-frame arrays (views, no copy)."""
    if isinstance(x, (list, tuple)):
        return list(x)
    return [x[i] for i in range(x.shape[0])]


def _host_codes(f):
    """One frame -> CPU tensor of the store's dtype (int16 holds unsigned 16-bit codes bit for bit), no copy where possible."""
    if isinstance(f, np.ndarray):
        if f.dtype == np.uint16:
            f = f.view(np.int16)
        return torch.from_numpy(np.ascontiguousarray(f))
    if f.dtype == torch.uint16:
        f = f.view(torch.int16)
    return f.contiguous()


class DeviceDataset:
    """A dataset resident in HBM and its batched crop sampler (module docstring).

    raws: integer code frames of one size -- uint16, int16 (non-negative) or uint8; (F,1,H,W) or a list of (H,W); numpy
          arrays or CPU tensors.
    gts:  uint8 BGR frames, planar (G,3,H,W) or cv2's (G,H,W,3) (transposed once, at load).
    white_level: raw divisor (1023., 16383., ...); the GT divisor is 255.
    crop: h or (h, w), even.  pairs: raw frame -> GT frame (default: the identity).
    seed, rank, world: the sampling plan (`SamplingPlan`); this rank uploads only its shard.

    `sample(B, split)` returns the same two device tensors on every call with the same (split, B): a CUDA-graph step that
    reads them keeps replaying, and the next `sample` of that key overwrites them in stream order."""

    def __init__(self, raws, gts, white_level, crop, pairs=None, seed=10, rank=0, world=1):
        raw_list, gt_list = _frames(raws), _frames(gts)
        if not raw_list or not gt_list:
            raise ValueError('DeviceDataset needs at least one raw and one GT frame')
        F, G = len(raw_list), len(gt_list)
        raw_dtypes = {str(f.dtype).replace('torch.', '') for f in raw_list}
        if len(raw_dtypes) != 1 or not raw_dtypes <= {'uint16', 'int16', 'uint8'}:
            raise ValueError('raw frames must be all uint16, all int16 or all uint8, got %s' % sorted(raw_dtypes))
        if {str(f.dtype).replace('torch.', '') for f in gt_list} != {'uint8'}:
            raise ValueError('GT frames must be uint8')
        shape = tuple(raw_list[0].shape)
        if len(shape) == 3 and shape[0] == 1:
            shape = shape[1:]
        if len(shape) != 2:
            raise ValueError('raw frames must be (F,1,H,W) or a list of (H,W), got a frame of shape %s' % (tuple(raw_list[0].shape),))
        H, W = shape
        if H % 2 or W % 2:
            raise ValueError('frames must have even H and W (the RGGB phase), got %dx%d' % (H, W))
        for f in raw_list:
            if tuple(f.shape) not in ((H, W), (1, H, W)):
                raise ValueError('raw frames differ in size: %s and %s' % ((H, W), tuple(f.shape)))
        hwc = tuple(gt_list[0].shape) == (H, W, 3) and tuple(gt_list[0].shape) != (3, H, W)
        want = (H, W, 3) if hwc else (3, H, W)
        for f in gt_list:
            if tuple(f.shape) != want:
                raise ValueError('GT frames must be (3,%d,%d) or (%d,%d,3) like the raws, got %s' % (H, W, H, W, tuple(f.shape)))
        if raw_dtypes == {'int16'}:
            for i, f in enumerate(raw_list):
                if int(f.min()) < 0:
                    raise ValueError('raw frame %d holds negative codes' % i)
        h, w = _even_pair(crop, 'crop')
        if h > H or w > W:
            raise ValueError('a %dx%d crop does not fit %dx%d frames' % (h, w, H, W))
        pairs = np.arange(F) if pairs is None else np.asarray(pairs)
        if pairs.shape != (F,) or pairs.dtype.kind not in 'iu' or (F and (pairs.min() < 0 or pairs.max() >= G)):
            raise ValueError('pairs must give each of the %d raw frames a GT frame in [0, %d)' % (F, G))
        if not float(white_level) > 0:
            raise ValueError('white_level must be positive, got %r' % (white_level,))
        self.H, self.W, self.h, self.w, self.white_level = H, W, h, w, float(white_level)
        self.plan_ = SamplingPlan(F, pairs, (H, W), (h, w), seed, rank, world)
        self._upload(raw_list, gt_list, hwc)
        self.steps = {s: 0 for s in SPLITS}
        self._bufs = {}

    def _upload(self, raw_list, gt_list, hwc):
        if not torch.cuda.is_available():
            raise RuntimeError('DeviceDataset needs a CUDA device (no CPU fallback)')
        self.device = torch.device('cuda', torch.cuda.current_device())      # the stream `sample` launches on
        p = self.plan_
        raw_bpc = 1 if str(raw_list[0].dtype).endswith('uint8') else 2
        need = len(p.raw_frames) * self.H * self.W * raw_bpc + len(p.gt_frames) * 3 * self.H * self.W
        free, _ = torch.cuda.mem_get_info(self.device)
        if need > free:
            raise MemoryError('the frame store needs %d bytes but %s has %d bytes free' % (need, self.device, free))
        dt = torch.uint8 if raw_bpc == 1 else torch.int16
        self.raw_store = torch.empty((len(p.raw_frames), self.H, self.W), device=self.device, dtype=dt)
        self.gt_store = torch.empty((len(p.gt_frames), 3, self.H, self.W), device=self.device, dtype=torch.uint8)
        for k, i in enumerate(p.raw_frames):                  # one frame at a time: host memory is never doubled
            self.raw_store[k].copy_(_host_codes(raw_list[i]).reshape(self.H, self.W))
        for k, i in enumerate(p.gt_frames):
            f = gt_list[i]
            if hwc:
                f = np.transpose(np.asarray(f), (2, 0, 1)) if isinstance(f, np.ndarray) else f.permute(2, 0, 1)
            self.gt_store[k].copy_(_host_codes(f))
        self.status = torch.zeros((1,), device=self.device, dtype=torch.int32)

    def plan(self, split, step, B):
        """Host records of batch `step` (int32 (B,4), `SamplingPlan.plan`)."""
        return self.plan_.plan(split, step, B)

    def sample(self, B, split='train'):
        """The next batch of `split` -> (img (B,1,h,w), gt (B,3,h,w)) fp32 device tensors, the same two on every call with
        this (split, B).  One copy of B*16 bytes and one launch on the current stream; nothing waits for the device."""
        plan = self.plan_.plan(split, self.steps[split], B)
        self.steps[split] += 1
        key = (split, B)
        bufs = self._bufs.get(key)
        if bufs is None:
            bufs = self._bufs[key] = (torch.empty((B, 4), device=self.device, dtype=torch.int32),
                                      torch.empty((B, 1, self.h, self.w), device=self.device, dtype=torch.float32),
                                      torch.empty((B, 3, self.h, self.w), device=self.device, dtype=torch.float32))
        pos, img, gt = bufs
        # pageable source: the driver stages the 16 B/record before returning, so the plan's array may go at once
        pos.copy_(torch.from_numpy(plan), non_blocking=True)
        ops.sample_crops(self.raw_store, self.gt_store, pos, self.h, self.w, self.white_level, self.status, img, gt)
        return img, gt

    def check(self):
        """Wait for the device and raise if any launch since the last check met a bad record (then clear the flag)."""
        bad = int(self.status.item())
        if bad:
            self.status.zero_()
            raise RuntimeError('risp_sample_crops skipped a record that was out of range or odd')
