"""numpy restatement of the reference's evaluation metric: test.py / test_split.py turn every output and its GT into 8-bit
images with `util.tensor2bgr` and score them with `util.calculate_psnr` (utils/util.py:118, 141; the file is not in the
reference tree, SURVEY §3.3-§4 cites it).  Test infrastructure only.

For each image n of a batch (N,3,H,W):
  q(v)     = uint8(trunc(min(max(fl32(v*255), 0), 255)))    (NaN -> 0), applied to the output AND the GT
  SSE_n    = sum_{c,h,w} (q(y) - q(gt))^2                  exact integer (up to 3*255^2 per pixel: 64 bits)
  PSNR_n   = 20 log10(255 / sqrt(SSE_n / (3HW)))            float64, inf when SSE_n == 0
For GT decoded from 8-bit codes q gives the code back (trunc(fl32(fl32(c/255)*255)) == c for all 256 codes)."""
import math

import numpy as np


def tensor2bgr(x):
    """(C,H,W) float -> (H,W,C) uint8 = trunc(clip(fl32(x*255), 0, 255)); NaN -> 0."""
    v = np.asarray(x, dtype=np.float32) * np.float32(255.0)
    v = np.clip(np.nan_to_num(v, nan=0.0), 0, 255)
    return np.transpose(v, (1, 2, 0)).astype(np.uint8)


def calculate_psnr(img1, img2):
    """PSNR of two 8-bit images in float64: inf when they are equal."""
    img1, img2 = img1.astype(np.float64), img2.astype(np.float64)
    mse = np.mean((img1 - img2) ** 2)
    if mse == 0:
        return float('inf')
    return 20 * math.log10(255.0 / math.sqrt(mse))


def sse_u8(y, gt):
    """(N,C,H,W) float pair -> int64 (N,) sums of squared differences of the tensor2bgr codes."""
    y, gt = np.asarray(y), np.asarray(gt)
    return np.array([int(((tensor2bgr(a).astype(np.int64) - tensor2bgr(b).astype(np.int64)) ** 2).sum())
                     for a, b in zip(y, gt)], dtype=np.int64)


def psnr(y, gt):
    """(N,C,H,W) float pair -> float64 (N,) per-image PSNR of the 8-bit images."""
    return np.array([calculate_psnr(tensor2bgr(a), tensor2bgr(b)) for a, b in zip(np.asarray(y), np.asarray(gt))],
                    dtype=np.float64)
