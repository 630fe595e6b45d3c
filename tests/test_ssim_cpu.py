"""Per-image SSIM without a GPU: the numpy oracle (oracle/ssim_oracle.py) against an independent brute-force restatement of
its definition, its properties, skimage itself where it is installed, the host conversion `metrics.ssim_from_sums`, and
argument validation of the C entry point."""
import ctypes

import numpy as np
import pytest

from oracle import ssim_oracle as S

C1 = 49 ** 2 * (0.01 * 255) ** 2
C2 = 49 * 48 * (0.03 * 255) ** 2


def brute_ssim(img1, img2):
    """The definition term by term: explicit 7x7 integer sums per interior pixel, then the fp64 ratio of exact integers."""
    a, b = img1.astype(np.int64), img2.astype(np.int64)
    H, W, C = a.shape
    total = 0.0
    for c in range(C):
        x, y = a[..., c], b[..., c]
        vals = []
        for h in range(3, H - 3):
            for w in range(3, W - 3):
                wx, wy = x[h - 3:h + 4, w - 3:w + 4], y[h - 3:h + 4, w - 3:w + 4]
                sa, sb = int(wx.sum()), int(wy.sum())
                saa, sbb, sab = int((wx * wx).sum()), int((wy * wy).sum()), int((wx * wy).sum())
                p1, q1 = 2 * sa * sb, sa * sa + sb * sb
                p2, q2 = 2 * (49 * sab - sa * sb), (49 * saa - sa * sa) + (49 * sbb - sb * sb)
                vals.append((p1 + C1) * (p2 + C2) / ((q1 + C1) * (q2 + C2)))
        total += float(np.mean(vals))
    return total / C


def pairs():
    rng = np.random.default_rng(21)
    out = []
    for (H, W, C) in [(7, 7, 3), (9, 13, 3), (12, 8, 1), (10, 11, 4)]:
        a = rng.integers(0, 256, (H, W, C), dtype=np.uint8)
        b = rng.integers(0, 256, (H, W, C), dtype=np.uint8)
        out.append((a, b))
        near = np.clip(a.astype(int) + rng.integers(-3, 4, a.shape), 0, 255).astype(np.uint8)
        out.append((a, near))                                            # correlated pair
    flat = np.full((11, 14, 3), 200, np.uint8)
    out.append((flat, (flat.astype(int) + rng.integers(-1, 2, flat.shape)).astype(np.uint8)))
    return out


def test_oracle_equals_brute_force_definition():
    for a, b in pairs():
        assert abs(S.calculate_ssim(a, b) - brute_ssim(a, b)) <= 1e-12, a.shape


def test_oracle_properties():
    for a, b in pairs():
        assert S.calculate_ssim(a, a) == 1.0
        assert S.calculate_ssim(a, b) == S.calculate_ssim(b, a)
    for shape in [(6, 9, 3), (9, 6, 3), (6, 6, 1)]:
        z = np.zeros(shape, np.uint8)
        with pytest.raises(ValueError):
            S.calculate_ssim(z, z)
    # the (N,C,H,W) float form quantises like tensor2bgr: NaN -> 0, out-of-range values clip
    rng = np.random.default_rng(4)
    y = rng.random((2, 3, 9, 10)).astype(np.float32) * 1.4 - 0.2
    y[0, 0, 0, 0] = np.nan
    gt = rng.random((2, 3, 9, 10)).astype(np.float32)
    q = lambda v: np.transpose(np.clip(np.nan_to_num(v * np.float32(255), nan=0.0), 0, 255), (1, 2, 0)).astype(np.uint8)
    ref = [brute_ssim(q(y[n]), q(gt[n])) for n in range(2)]
    assert np.abs(S.ssim(y, gt) - ref).max() <= 1e-12


def test_oracle_equals_skimage():
    skm = pytest.importorskip('skimage.metrics', reason='skimage is not installed')
    for a, b in pairs():
        try:
            ref = skm.structural_similarity(a, b, channel_axis=-1, data_range=255)
        except TypeError:                                                 # skimage < 0.19
            ref = skm.structural_similarity(a, b, multichannel=True, data_range=255)
        assert abs(S.calculate_ssim(a, b) - ref) <= 1e-12, a.shape


def test_ssim_from_sums():
    import torch
    from reconfigisp_b200.metrics import ssim_from_sums
    C, H, W = 3, 3000, 4000
    one = C * (H - 6) * (W - 6) * 2 ** 32
    assert one < 2 ** 63
    got = ssim_from_sums([one, 0, -one // 2, one // 4], C, H, W)
    assert got.dtype == np.float64 and got.shape == (4,)
    assert got.tolist() == [1.0, 0.0, -0.5, 0.25]
    arr = np.array([one, 12345], dtype=np.int64)
    ref = ssim_from_sums(arr, C, H, W)
    assert np.array_equal(ssim_from_sums(torch.from_numpy(arr), C, H, W), ref)
    assert np.array_equal(ssim_from_sums(list(arr), C, H, W), ref)
    assert ref[1] == 12345 / one
    with pytest.raises(ValueError):
        ssim_from_sums([0], 3, 6, 10)


def test_ssim_entry_point_rejects_bad_arguments_without_a_gpu():
    """Validation happens before any CUDA call: null pointers, bad shapes and an unknown layout come back as RISP_E_INVALID
    naming the entry point, a misaligned fp32 operand or output as RISP_E_ALIGN."""
    from reconfigisp_b200 import _build, _lib as L
    lib = ctypes.CDLL(_build.LIB)
    lib.risp_last_error.restype = ctypes.c_char_p
    fn = lib.risp_ssim_u8
    fn.restype = ctypes.c_int
    fn.argtypes = [t for t, _ in L.PROTOS['risp_ssim_u8'][1]]
    assert [n for _, n in L.PROTOS['risp_ssim_u8'][1]] == ['y', 'y_layout', 'gt', 'ssim_sum_out', 'N', 'C', 'H', 'W',
                                                           'stream']
    assert L.ENUMS['RISP_IMG_F32_NCHW'] == 0 and L.ENUMS['RISP_IMG_U8_NHWC'] == 1
    fake = 1 << 20                       # 16-byte aligned, never dereferenced: validation fails first

    def call(y=fake, layout=0, gt=fake, out=fake, N=1, C=3, H=7, W=7):
        return fn(y, layout, gt, out, N, C, H, W, None)

    bad = [dict(y=None), dict(gt=None), dict(out=None), dict(N=0), dict(N=65536), dict(C=0), dict(C=-1), dict(H=6),
           dict(W=6), dict(H=-7), dict(layout=2), dict(layout=-1), dict(C=1 << 20, H=2054, W=1030)]
    for layout in (0, 1):
        for kw in bad:
            kw = dict(dict(layout=layout), **kw)
            rc = call(**kw)
            assert rc == L.RISP_E_INVALID, (kw, rc)
            assert b'risp_ssim_u8' in lib.risp_last_error(), kw
    assert (1 << 20) * 2048 * 1024 >= 2 ** 31
    for kw in (dict(gt=fake + 2), dict(out=fake + 4), dict(y=fake + 1, layout=0)):
        rc = call(**kw)
        assert rc == L.RISP_E_ALIGN, (kw, rc)
        assert b'risp_ssim_u8' in lib.risp_last_error(), kw
