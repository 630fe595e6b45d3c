"""The evaluation metric without a GPU: the host PSNR conversion against the numpy restatement of the reference's
tensor2bgr + calculate_psnr (oracle/metrics_oracle.py), and argument validation of the new C entry points."""
import ctypes

import numpy as np
import pytest

from oracle import metrics_oracle as M


def test_psnr_from_sse_is_the_reference_psnr_bit_for_bit():
    from reconfigisp_b200.metrics import psnr_from_sse
    rng = np.random.default_rng(3)
    N, C, H, W = 6, 3, 17, 23
    a = rng.integers(0, 256, (N, H, W, C), dtype=np.uint8)
    b = a.copy()
    b[1] = rng.integers(0, 256, (H, W, C), dtype=np.uint8)       # unrelated images
    b[2, 3, 4, 1] ^= 1                                           # one code off by one
    b[3] = 255 - a[3]                                            # large differences
    b[4] = 0
    b[4, ..., 0] = 255                                           # worst case on one channel
    # b[0], b[5]: identical -> inf
    sse = ((a.astype(np.int64) - b.astype(np.int64)) ** 2).reshape(N, -1).sum(1)
    ref = np.array([M.calculate_psnr(a[n], b[n]) for n in range(N)])
    got = psnr_from_sse(sse, C * H * W)
    assert got.dtype == np.float64 and got.shape == (N,)
    assert np.isinf(got[0]) and np.isinf(got[5]) and np.isfinite(got[1:5]).all()
    assert np.array_equal(got, ref)                              # bit for bit, inf included
    import torch
    assert np.array_equal(psnr_from_sse(torch.from_numpy(sse), C * H * W), ref)
    assert np.array_equal(psnr_from_sse(list(sse), C * H * W), ref)
    # 12 MP worst case: the sum does not fit 32 bits; int64 on the way in, exact
    big = 3 * 3000 * 4000 * 65025
    assert big > 2 ** 32 and psnr_from_sse([big], 3 * 3000 * 4000)[0] == 20 * np.log10(255.0 / 255.0)


def test_oracle_codes_are_tensor2bgr():
    """q(v) on the edge values: below 0, above 1, NaN, exact k/255 points (the code comes back) and their fp32 neighbours."""
    k = np.arange(256, dtype=np.float32)
    exact = k / np.float32(255)
    assert np.array_equal(M.tensor2bgr(exact.reshape(1, 1, -1))[0, :, 0], np.arange(256))
    below = np.nextafter(exact, np.float32(-1))
    codes = M.tensor2bgr(below.reshape(1, 1, -1))[0, :, 0].astype(int)
    assert ((codes == np.arange(256)) | (codes == np.arange(256) - 1)).all() and codes[0] == 0
    odd = np.array([-0.5, 1.5, np.nan, np.inf, -np.inf, 0.999], dtype=np.float32).reshape(1, 1, -1)
    assert M.tensor2bgr(odd)[0, :, 0].tolist() == [0, 255, 0, 255, 0, 254]
    y = np.zeros((1, 3, 2, 2), np.float32)
    gt = np.ones((1, 3, 2, 2), np.float32)
    assert M.sse_u8(y, gt).tolist() == [12 * 65025]


def _lib():
    from reconfigisp_b200 import _build, _lib as L
    lib = ctypes.CDLL(_build.LIB)
    lib.risp_last_error.restype = ctypes.c_char_p
    for name in ('risp_pipeline_eval', 'risp_sse_u8'):
        fn = getattr(lib, name)
        fn.restype = ctypes.c_int
        fn.argtypes = [t for t, _ in L.PROTOS[name][1]]
    lib.risp_pipeline_eval_workspace.restype = ctypes.c_size_t
    lib.risp_pipeline_eval_workspace.argtypes = [ctypes.c_int] * 3
    return lib, L


def test_eval_entry_points_reject_bad_arguments_without_a_gpu():
    """Validation happens before any CUDA call: null pointers, bad shapes and unknown demosaic kinds come back as
    RISP_E_INVALID with the entry point's name in the message."""
    lib, L = _lib()
    fake = ctypes.c_void_p(1 << 20)            # 16-byte aligned, never dereferenced: validation fails first
    ops_, off, iarg = L.iarr([L.ENUMS['RISP_OP_GAMMA']]), L.iarr([0]), L.iarr([0])
    ws = 1 << 20

    def ev(raw=fake, gt=fake, sse=fake, N=1, H=8, W=8, dm=1, params=fake, work=fake):
        return lib.risp_pipeline_eval(raw, gt, None, sse, N, H, W, dm, 1.0, ops_, off, iarg, 1, params, 0, work, ws, None)

    for kw in (dict(raw=None), dict(gt=None), dict(sse=None), dict(N=0), dict(H=2), dict(dm=7), dict(params=None),
               dict(work=None)):
        rc = ev(**kw)
        assert rc == L.RISP_E_INVALID, (kw, rc)
        assert b'risp_pipeline_eval' in lib.risp_last_error(), kw
    # geometry the fused kernels need (like risp_pipeline_fwd): odd H / W % 4 != 0 are alignment errors
    assert ev(H=7) == L.RISP_E_ALIGN and ev(W=6) == L.RISP_E_ALIGN
    assert lib.risp_pipeline_eval_workspace(0, 8, 8) == 0 and lib.risp_pipeline_eval_workspace(4, 3000, 4000) > 0

    def sse(y=fake, gt=fake, out=fake, N=1, C=3, H=5, W=7):
        return lib.risp_sse_u8(y, gt, out, N, C, H, W, None)

    for kw in (dict(y=None), dict(gt=None), dict(out=None), dict(N=0), dict(C=0), dict(H=-1), dict(W=0), dict(N=70000)):
        rc = sse(**kw)
        assert rc == L.RISP_E_INVALID, (kw, rc)
        assert b'risp_sse_u8' in lib.risp_last_error(), kw
