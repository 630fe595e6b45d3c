"""numpy restatement of the reference's second evaluation metric, per-image SSIM of the 8-bit images.  Test infrastructure
only.

The reference's `get_ssim` (utils/util_path_restore.py:3 imports skimage.measure.compare_ssim for it) is not in the reference
tree, so this is the definition chosen and stated here: skimage 0.16 `compare_ssim(a, b, multichannel=True)` with its
defaults, applied to the tensor2bgr codes of metrics_oracle.py (the codes the PSNR uses), so data_range is 255.

For an image pair (C,H,W) with codes a = q(y), b = q(gt) (q(v) = trunc(clip(fl32(v*255), 0, 255)), NaN -> 0), for every
channel and every INTERIOR pixel h in [3, H-3), w in [3, W-3), take the integer sums over its 7x7 window Sa, Sb, Saa, Sbb,
Sab.  Then
  P1 = 2 Sa Sb                    Q1 = Sa^2 + Sb^2
  P2 = 2 (49 Sab - Sa Sb)         Q2 = (49 Saa - Sa^2) + (49 Sbb - Sb^2)
  S  = (P1 + c1)(P2 + c2) / ((Q1 + c1)(Q2 + c2))
  c1 = 49^2 (0.01*255)^2 = 15612.5025      c2 = 49*48 (0.03*255)^2 = 137644.92
  SSIM_n = mean over the C channels of the mean of S over the (H-6)(W-6) interior pixels
This is skimage's formula exactly (uniform 7x7 filter, sample covariance 49/48, K1 = 0.01, K2 = 0.03, the border of 3 pixels
cropped before the mean); the factors 2401 and 2352 cancel in the ratio.  H or W below 7 is a ValueError, as in skimage.

P1, Q1, P2, Q2 are integers below 3.2e8.  The device kernel (risp_ssim.cu) forms them exactly in int32 before any rounding:
in fp32 the moments 49 Saa - Sa^2 lose S to cancellation on flat regions.  After that fp32 suffices (about 5e-7 per pixel);
its division is correctly rounded, so identical images give exactly 1 and swapped operands the same bits, and S does not
depend on where a running window started.  The device returns rint(S * 2^32) summed per image in int64.
"""
import numpy as np
from scipy.ndimage import uniform_filter

from oracle.metrics_oracle import tensor2bgr

C1 = (0.01 * 255) ** 2
C2 = (0.03 * 255) ** 2


def calculate_ssim(img1, img2):
    """SSIM of two (H,W,C) (or (H,W)) 8-bit images in float64: skimage 0.16 compare_ssim(img1, img2, multichannel=True)
    restated with scipy.ndimage.uniform_filter."""
    a, b = np.asarray(img1), np.asarray(img2)
    if a.shape != b.shape:
        raise ValueError('calculate_ssim: shapes differ, %s and %s' % (a.shape, b.shape))
    if a.ndim == 2:
        a, b = a[..., None], b[..., None]
    H, W = a.shape[:2]
    if H < 7 or W < 7:
        raise ValueError('calculate_ssim: the 7x7 window needs H and W >= 7, got %d x %d' % (H, W))
    cov_norm = 49.0 / 48.0
    vals = []
    for ch in range(a.shape[2]):
        x, y = a[..., ch].astype(np.float64), b[..., ch].astype(np.float64)
        ux, uy = uniform_filter(x, size=7), uniform_filter(y, size=7)
        uxx, uyy, uxy = uniform_filter(x * x, size=7), uniform_filter(y * y, size=7), uniform_filter(x * y, size=7)
        vx, vy, vxy = cov_norm * (uxx - ux * ux), cov_norm * (uyy - uy * uy), cov_norm * (uxy - ux * uy)
        s = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux ** 2 + uy ** 2 + C1) * (vx + vy + C2))
        vals.append(s[3:-3, 3:-3].mean())
    return float(np.mean(vals))


def ssim(y, gt):
    """(N,C,H,W) float pair -> float64 (N,) per-image SSIM of the 8-bit images (tensor2bgr codes)."""
    return np.array([calculate_ssim(tensor2bgr(a), tensor2bgr(b)) for a, b in zip(np.asarray(y), np.asarray(gt))],
                    dtype=np.float64)
