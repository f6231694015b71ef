"""float64 CPU restatement of the validation metrics.  TEST INFRASTRUCTURE ONLY.

Restated from the published algorithms the reference calls (humanrf/trainer.py:373-419 and
actorshq/evaluation/evaluate.py:76-85):

  * ``bounding_rect``  -- cv2.boundingRect of a binary mask: the smallest upright box (x, y, w, h) holding every
    non-zero pixel, (0, 0, 0, 0) for an empty mask.
  * ``ssim``           -- skimage.metrics.structural_similarity(im1, im2, channel_axis=2, data_range=R) with its
    defaults: 7x7 uniform filter (scipy.ndimage, ``reflect`` boundaries), sample covariance (49/48), K1 = 0.01,
    K2 = 0.03, the map cropped by 3 pixels on every side, the mean of the channel means.
  * ``compute_psnr``   -- evaluate.py's compute_psnr on CHW images.
  * ``evaluate_one_image`` -- Trainer.evaluate_one_image without LPIPS.

Parity with skimage is pinned only where skimage is installed (tests/test_metrics_cpu.py).
"""
from __future__ import annotations

import numpy as np
from scipy.ndimage import uniform_filter

WIN = 7


def bounding_rect(mask):
    ys, xs = np.nonzero(np.asarray(mask).reshape(np.asarray(mask).shape[:2]) > 0)
    if xs.size == 0:
        return (0, 0, 0, 0)
    return (int(xs.min()), int(ys.min()), int(xs.max() - xs.min() + 1), int(ys.max() - ys.min() + 1))


def _ssim_channel(x, y, data_range):
    f = lambda z: uniform_filter(z, size=WIN, mode="reflect")  # noqa: E731
    ux, uy, uxx, uyy, uxy = f(x), f(y), f(x * x), f(y * y), f(x * y)
    cov_norm = WIN * WIN / (WIN * WIN - 1.0)
    vx, vy, vxy = cov_norm * (uxx - ux * ux), cov_norm * (uyy - uy * uy), cov_norm * (uxy - ux * uy)
    c1, c2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    s = (2 * ux * uy + c1) * (2 * vxy + c2) / ((ux * ux + uy * uy + c1) * (vx + vy + c2))
    p = (WIN - 1) // 2
    return s[p:-p, p:-p].mean(dtype=np.float64)


def ssim(im1, im2, data_range, roi=None):
    """Mean SSIM of two HWC images over roi = (x, y, w, h) (None: the whole image)."""
    a, b = np.asarray(im1, np.float64), np.asarray(im2, np.float64)
    if roi is not None:
        x, y, w, h = roi
        a, b = a[y:y + h, x:x + w], b[y:y + h, x:x + w]
    if a.shape != b.shape or a.ndim != 3:
        raise ValueError("images must be HWC of the same shape")
    if a.shape[0] < WIN or a.shape[1] < WIN:
        raise ValueError("win_size exceeds image extent")
    return float(np.mean([_ssim_channel(a[..., c], b[..., c], float(data_range)) for c in range(a.shape[2])]))


def compute_psnr(im1, im2, mask=None):
    """evaluate.py:compute_psnr on CHW images: the per-pixel channel mean of the squared error, averaged over the
    pixels with mask > 0."""
    mse = np.square(np.asarray(im1, np.float64) - np.asarray(im2, np.float64)).mean(0).reshape(-1)
    if mask is not None:
        mse = mse[np.asarray(mask).reshape(-1) > 0]
    with np.errstate(divide="ignore"):
        return float(-10 * np.log10(mse.mean()))


def evaluate_one_image(pred, gt_rgba, background=0.0, ray_mask=None):
    """pred [H,W,3], gt_rgba [H,W,4] in [0,1]; ray_mask [H,W] (None: every pixel).  Returns psnr, ssim and roi."""
    pred = np.asarray(pred, np.float64)
    gt_rgba = np.asarray(gt_rgba, np.float64)
    H, W = pred.shape[:2]
    rm = np.ones((H, W), bool) if ray_mask is None else np.asarray(ray_mask).reshape(H, W) > 0
    bg = np.broadcast_to(np.asarray(background, np.float64), (3,))
    a = gt_rgba[..., 3:4]
    gt = np.where(rm[..., None], gt_rgba[..., :3] * a + bg * (1 - a), bg)
    alpha = np.where(rm, gt_rgba[..., 3], 0.0)
    roi = bounding_rect(alpha > 0)
    psnr = compute_psnr(pred.transpose(2, 0, 1), gt.transpose(2, 0, 1), rm)
    x, y, w, h = roi
    s = ssim(pred, gt, 1.0, roi) if w >= WIN and h >= WIN else float("nan")
    return {"psnr": psnr, "ssim": s, "roi": roi}
