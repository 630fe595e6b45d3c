"""Evaluation metrics of the reference, per image of the 8-bit outputs: PSNR (test.py, test_split.py: `tensor2bgr` ->
`util.calculate_psnr`) and SSIM (utils/util_path_restore.py: `get_ssim`, skimage `compare_ssim(a, b, multichannel=True)`;
the definition is stated in oracle/metrics_oracle.py).

The squared code differences are summed on the device (`ops.sse_u8`, `ops.pipeline_eval`, `_Universal.evaluate`), exactly
and without a host sync; `psnr_from_sse` is the only step that reads them back.  A validation loop can keep the sums on the
device and convert once:

    sums = [net.evaluate(x, gt)[0] for x, gt in loader]
    values = psnr_from_sse(torch.cat(sums), 3 * H * W)

SSIM is summed on the device too, as exact int64 sums of rint(S * 2^32) per image (`ops.ssim_u8`,
`_Universal.evaluate(..., ssim=True)`), and `ssim_from_sums` is its only host sync:

    res = [net.evaluate(x, gt, ssim=True) for x, gt in loader]
    psnrs = psnr_from_sse(torch.cat([r[0] for r in res]), 3 * H * W)
    ssims = ssim_from_sums(torch.cat([r[2] for r in res]), 3, H, W)

For the tiled 12 MP path, `psnr(split_inference(..., clip01=True), gt)`: its clip to [0, 1] followed by truncation gives
the same codes as tensor2bgr.  SSIM takes the blend kernel's 8-bit image directly, which is the same image:
`ssim(split_inference(..., uint8=True), gt)`.
"""
import math

import numpy as np
import torch

from . import ops


def psnr_from_sse(sse, values_per_image):
    """PSNR_n = 20 log10(255 / sqrt(sse_n / values_per_image)) in float64, inf where sse_n == 0 (util.calculate_psnr on
    the two 8-bit images).  sse: int64 sums (a CUDA or CPU tensor, an array or a list) -> float64 numpy array."""
    if torch.is_tensor(sse):
        sse = sse.detach().cpu().numpy()
    s = np.asarray(sse, dtype=np.int64).reshape(-1)
    n = float(values_per_image)
    out = np.empty(s.shape, dtype=np.float64)
    for i, v in enumerate(s.tolist()):
        mse = float(v) / n
        out[i] = float('inf') if mse == 0 else 20 * math.log10(255.0 / math.sqrt(mse))
    return out


def psnr(y, gt):
    """Per-image PSNR of the 8-bit images of y and gt, fp32 (N,C,H,W) or (C,H,W) CUDA tensors -> float64 numpy (N,)."""
    sse = ops.sse_u8(y, gt)
    C, H, W = y.shape[-3:]
    return psnr_from_sse(sse, C * H * W)


def ssim_from_sums(sums, C, H, W):
    """SSIM_n = sums_n / (2^32 C (H-6)(W-6)) in float64, correctly rounded (the mean over channels and interior pixels of
    skimage's per-pixel S).  sums: int64 sums of `ops.ssim_u8` (a CUDA or CPU tensor, an array or a list) -> float64 numpy
    array.  Identical images give exactly 1.0."""
    if torch.is_tensor(sums):
        sums = sums.detach().cpu().numpy()
    s = np.asarray(sums, dtype=np.int64).reshape(-1)
    if H < 7 or W < 7:
        raise ValueError('ssim_from_sums: the 7x7 window needs H and W >= 7, got %d x %d' % (H, W))
    den = (int(C) * (int(H) - 6) * (int(W) - 6)) << 32
    return np.array([v / den for v in s.tolist()], dtype=np.float64)      # int / int: correctly rounded


def ssim(y, gt):
    """Per-image SSIM of the 8-bit images of y and gt -> float64 numpy (N,).  y: fp32 (N,C,H,W) / (C,H,W) or uint8
    (N,H,W,C) / (H,W,C) CUDA tensor (`split_inference(..., uint8=True)`, `pipeline_eval(..., u8=True)`); gt: fp32
    (N,C,H,W) / (C,H,W)."""
    sums = ops.ssim_u8(y, gt)
    C, H, W = gt.shape[-3:]
    return ssim_from_sums(sums, C, H, W)
