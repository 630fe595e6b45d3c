"""Validation on the resident dataset, host side (no GPU): `SamplingPlan.frames` and the argument checks of the store
evaluation entry points, which run before any CUDA call."""
import ctypes

import numpy as np
import pytest

from reconfigisp_b200.data import SamplingPlan


@pytest.mark.parametrize('F,world', [(1, 1), (7, 1), (7, 2), (23, 4), (9, 3), (5, 8)])
def test_frames_cover_each_split_once_across_ranks_in_ascending_order(F, world):
    pairs = np.arange(F)
    plans = [SamplingPlan(F, pairs, (16, 16), (8, 8), rank=r, world=world) for r in range(world)]
    spans = {'train': range(0, F // 2), 'val': range(F // 2, F), 'all': range(F)}
    for split, span in spans.items():
        seen = []
        for p in plans:
            rec, ids = p.frames(split)
            assert rec.dtype == np.int32 and rec.shape == (len(ids), 4) and ids.dtype == np.int64
            assert (rec[:, 2:] == 0).all()                                   # whole frames
            assert np.array_equal(ids, np.sort(ids))                         # ascending global order
            assert np.array_equal(p.raw_frames[rec[:, 0]], ids)             # records name this rank's frames
            assert ((ids % world) == p.rank).all()
            seen += ids.tolist()
        assert sorted(seen) == list(span), split                             # every frame exactly once


def test_frames_honour_pairs():
    pairs = np.array([0, 0, 0, 1, 1, 2, 2, 2, 2])
    for world in (1, 2, 3):
        for r in range(world):
            p = SamplingPlan(9, pairs, (16, 16), (8, 8), rank=r, world=world)
            for split in ('train', 'val', 'all'):
                rec, ids = p.frames(split)
                assert np.array_equal(p.gt_frames[rec[:, 1]], pairs[ids])


def test_frames_reject_an_unknown_split():
    p = SamplingPlan(4, np.arange(4), (16, 16), (8, 8))
    with pytest.raises(ValueError):
        p.frames('test')


def _lib():
    from reconfigisp_b200 import _build, _lib as L
    lib = ctypes.CDLL(_build.LIB)
    lib.risp_last_error.restype = ctypes.c_char_p
    for name in ('risp_pipeline_eval_store', 'risp_ssim_u8_store'):
        fn = getattr(lib, name)
        fn.restype = ctypes.c_int
        fn.argtypes = [t for t, _ in L.PROTOS[name][1]]
    return lib, L


def test_store_entry_points_are_declared_in_the_header():
    from reconfigisp_b200 import _lib as L
    assert [a for _, a in L.PROTOS['risp_pipeline_eval_store'][1]] == [
        'raw_store', 'raw_bytes_per_code', 'F', 'gt_store', 'G', 'H', 'W', 'pos', 'N', 'white_level', 'status', 'u8_out',
        'sse_out', 'dm_kind', 'dm_clip_hi', 'ops', 'param_off', 'iarg', 'S', 'params', 'param_stride', 'workspace',
        'workspace_bytes', 'stream']
    assert [a for _, a in L.PROTOS['risp_ssim_u8_store'][1]] == [
        'y', 'y_layout', 'gt_store', 'G', 'pos', 'status', 'ssim_sum_out', 'N', 'H', 'W', 'stream']


def test_store_entry_points_reject_bad_arguments_without_a_gpu():
    """Null, negative and oversized arguments come back as error codes with the entry point's name, before any CUDA call."""
    lib, L = _lib()
    fake = ctypes.c_void_p(1 << 20)            # 16-byte aligned, never dereferenced: validation fails first
    odd = ctypes.c_void_p((1 << 20) + 4)
    ops_, off, iarg = L.iarr([L.ENUMS['RISP_OP_GAMMA']]), L.iarr([0]), L.iarr([0])

    def ev(raw=fake, bpc=2, F=2, gt=fake, G=2, H=16, W=16, pos=fake, N=2, wl=1023., status=fake, u8=None, sse=fake, dm=1,
           params=fake, work=fake, ws=1 << 20):
        return lib.risp_pipeline_eval_store(raw, bpc, F, gt, G, H, W, pos, N, wl, status, u8, sse, dm, 1.0, ops_, off, iarg,
                                            1, params, 0, work, ws, None)

    for kw in (dict(raw=None), dict(gt=None), dict(pos=None), dict(status=None), dict(sse=None), dict(bpc=4), dict(bpc=0),
               dict(F=0), dict(F=-3), dict(G=0), dict(N=0), dict(N=-1), dict(N=70000), dict(H=2), dict(W=-16), dict(wl=0.),
               dict(wl=-1.), dict(dm=7), dict(params=None), dict(work=None), dict(F=1 << 30, H=4000, W=4000),
               dict(G=1 << 30, H=4000, W=4000)):
        rc = ev(**kw)
        assert rc == L.RISP_E_INVALID, (kw, rc)
        assert b'risp_pipeline_eval_store' in lib.risp_last_error(), kw
    for kw in (dict(H=7), dict(W=18), dict(raw=odd), dict(gt=odd), dict(pos=odd), dict(u8=ctypes.c_void_p((1 << 20) + 1))):
        rc = ev(**kw)
        assert rc == L.RISP_E_ALIGN, (kw, rc)

    def ss(y=fake, layout=1, gt=fake, G=2, pos=fake, status=fake, out=fake, N=2, H=16, W=16):
        return lib.risp_ssim_u8_store(y, layout, gt, G, pos, status, out, N, H, W, None)

    for kw in (dict(y=None), dict(gt=None), dict(pos=None), dict(status=None), dict(out=None), dict(layout=5), dict(G=0),
               dict(N=0), dict(N=-2), dict(N=70000), dict(H=6), dict(W=-1), dict(H=1 << 20, W=1 << 20)):
        rc = ss(**kw)
        assert rc == L.RISP_E_INVALID, (kw, rc)
        assert b'risp_ssim_u8_store' in lib.risp_last_error(), kw
    assert ss(pos=odd) == L.RISP_E_ALIGN and ss(layout=0, y=ctypes.c_void_p((1 << 20) + 2)) == L.RISP_E_ALIGN
