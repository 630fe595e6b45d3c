"""Evaluation metric of the reference: PSNR of the 8-bit images, per image (test.py, test_split.py: `tensor2bgr` ->
`util.calculate_psnr`).

The squared code differences are summed on the device (`ops.sse_u8`, `ops.pipeline_eval`, `_Universal.evaluate`), exactly
and without a host sync; `psnr_from_sse` is the only step that reads them back.  A validation loop can keep the sums on the
device and convert once:

    sums = [net.evaluate(x, gt)[0] for x, gt in loader]
    values = psnr_from_sse(torch.cat(sums), 3 * H * W)

For the tiled 12 MP path, `psnr(split_inference(..., clip01=True), gt)`: its clip to [0, 1] followed by truncation gives
the same codes as tensor2bgr.
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
