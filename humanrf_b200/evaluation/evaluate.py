"""Validation metrics on the device: the PSNR / SSIM half of actorshq/evaluation/evaluate.py and of
Trainer.evaluate_one_image (humanrf/trainer.py:373-419).  LPIPS (pretrained AlexNet weights) and VMAF (ffmpeg + vmaf)
are not provided.

``mask_bounding_rect``, ``ssim``, ``psnr`` and ``evaluate_image`` take CUDA tensors and return CUDA tensors without
synchronising, so a validation loop can queue them behind the render and read everything at the end.
``compute_psnr`` / ``compute_ssim`` mirror evaluate.py's functions and return Python floats (one read each).
"""
from __future__ import annotations

from typing import Optional, Sequence, Union

import torch

from .. import _lib as L

_WIN = 7
_SSIM, _PSNR = 1, 2


def _image(t: torch.Tensor, name: str) -> torch.Tensor:
    L.require_cuda(t, name)
    if t.dim() != 3 or t.shape[2] != 3:
        raise ValueError(f"{name} must be an HWC image with 3 channels, got shape {tuple(t.shape)}")
    if t.dtype not in (torch.float32, torch.uint8):
        raise RuntimeError(f"Tensor {name} has dtype {t.dtype}, expected torch.float32 or torch.uint8")
    return t


def _pair(im1: torch.Tensor, im2: torch.Tensor):
    _image(im1, "im1"), _image(im2, "im2")
    if im1.shape != im2.shape or im1.dtype != im2.dtype or im1.device != im2.device:
        raise ValueError("im1 and im2 must have the same shape, dtype and device")
    return im1.shape[0], im1.shape[1]


def _binary_mask(mask: torch.Tensor, height: int, width: int, name: str) -> torch.Tensor:
    """uint8 [H, W] view of mask > 0 (mask: bool, uint8 or float, H*W elements, e.g. [H, W] or [H, W, 1])."""
    if mask.device.type != "cuda":
        raise RuntimeError(f"Tensor is not on the expected device: {name}")
    if mask.numel() != height * width:
        raise ValueError(f"{name} has {mask.numel()} elements, expected {height} x {width}")
    m = mask if mask.dtype == torch.bool else mask > 0
    return m.contiguous().view(torch.uint8).view(height, width)


def _metrics(im1, im2, what, height, width, row_stride, roi=None, data_range=1.0, psnr_mask=None):
    """Launches hrf_image_metrics; returns its float64 [4] device result (SSIM, PSNR, squared error, pixel count)."""
    out = torch.empty(4, dtype=torch.float64, device=im1.device)
    ws = torch.empty(int(L.lib().hrf_image_metrics_workspace_bytes(height, width)), dtype=torch.uint8, device=im1.device)
    L.check(L.lib().hrf_image_metrics(im1.data_ptr(), im2.data_ptr(), int(im1.dtype == torch.uint8), height, width,
                                      row_stride, L.ptr(roi), float(data_range), L.ptr(psnr_mask), what, out.data_ptr(),
                                      ws.data_ptr(), L.stream()))
    return out


def mask_bounding_rect(mask: torch.Tensor) -> torch.Tensor:
    """cv2.boundingRect(mask > 0) on the device: int32 [4] (x, y, w, h); (0, 0, 0, 0) for an empty mask.
    mask: [H, W] or [H, W, 1], bool / uint8 / float."""
    if mask.dim() == 3 and mask.shape[2] == 1:
        mask = mask[..., 0]
    if mask.dim() != 2:
        raise ValueError(f"mask must be [H, W] or [H, W, 1], got shape {tuple(mask.shape)}")
    H, W = mask.shape
    m = _binary_mask(mask, H, W, "mask")
    box = torch.empty(4, dtype=torch.int32, device=m.device)
    L.check(L.lib().hrf_mask_bbox(m.data_ptr(), H, W, box.data_ptr(), L.stream()))
    return box


def ssim(im1: torch.Tensor, im2: torch.Tensor, data_range: Optional[float] = None,
         roi: Union[None, Sequence[int], torch.Tensor] = None) -> torch.Tensor:
    """Mean SSIM of two HWC images (skimage.metrics.structural_similarity(im1, im2, channel_axis=2) defaults) over roi:
    None (the whole image), a host (x, y, w, h), or a device int32 [4] such as mask_bounding_rect returns.
    data_range defaults to 255 for uint8 and must be given for float32.  Returns a 0-dim float64 device tensor; a device
    ROI narrower or shorter than 7 pixels gives NaN."""
    H, W = _pair(im1, im2)
    if data_range is None:
        if im1.dtype != torch.uint8:
            raise ValueError("data_range must be given for floating-point images")
        data_range = 255.0
    if H < _WIN or W < _WIN:
        raise ValueError("win_size exceeds image extent: both image dimensions must be at least 7")
    if isinstance(roi, torch.Tensor):
        L.require_cuda(roi, "roi", torch.int32)
        if roi.numel() != 4 or roi.device != im1.device:
            raise ValueError("roi must be an int32 [4] tensor (x, y, w, h) on the images' device")
        return _metrics(im1, im2, _SSIM, H, W, 3 * W, roi=roi, data_range=data_range)[0]
    if roi is None:
        return _metrics(im1, im2, _SSIM, H, W, 3 * W, data_range=data_range)[0]
    x, y, w, h = (int(v) for v in roi)
    if x < 0 or y < 0 or x + w > W or y + h > H:
        raise ValueError(f"roi {tuple(roi)} lies outside the {W} x {H} image")
    if w < _WIN or h < _WIN:
        raise ValueError("win_size exceeds image extent: both ROI dimensions must be at least 7")
    # a host ROI is a view: its first pixel and the image's row stride, no copy and no upload
    return _metrics(im1[y:, x:], im2[y:, x:], _SSIM, h, w, 3 * W, data_range=data_range)[0]


def psnr(im1: torch.Tensor, im2: torch.Tensor, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """PSNR of two HWC images: -10 log10 of the per-pixel channel mean of the squared error averaged over the pixels
    with mask > 0 (all pixels when mask is None).  uint8 images are read as value / 255.  Returns a 0-dim float64 device
    tensor; identical images give +inf."""
    H, W = _pair(im1, im2)
    m = None if mask is None else _binary_mask(mask, H, W, "mask")
    return _metrics(im1, im2, _PSNR, H, W, 3 * W, data_range=255.0 if im1.dtype == torch.uint8 else 1.0, psnr_mask=m)[1]


def evaluate_image(pred: torch.Tensor, gt_rgba: torch.Tensor, background: Union[float, torch.Tensor] = 0.0,
                   ray_mask: Optional[torch.Tensor] = None) -> dict:
    """Trainer.evaluate_one_image without LPIPS, on the device.  pred: float32 [H, W, 3] rendered image (the background
    outside the ray mask); gt_rgba: float32 [H, W, 4] in [0, 1]; ray_mask: [H, W] of the pixels that were rendered as
    rays (None: all).  The ground truth is rgb * a + background * (1 - a) on ray-masked pixels and the background
    elsewhere; PSNR is over the ray-masked pixels (trainer.py:218-222); SSIM (data_range 1) is over the bounding box of
    alpha > 0 on ray-masked pixels.  Returns {"psnr", "ssim": 0-dim float64, "roi": int32 [4]}, all device tensors."""
    _image(pred, "pred")
    H, W = pred.shape[0], pred.shape[1]
    if pred.dtype != torch.float32:
        raise RuntimeError(f"Tensor pred has dtype {pred.dtype}, expected torch.float32")
    L.require_cuda(gt_rgba, "gt_rgba", torch.float32)
    if tuple(gt_rgba.shape) != (H, W, 4):
        raise ValueError(f"gt_rgba must be [{H}, {W}, 4], got shape {tuple(gt_rgba.shape)}")
    if H < _WIN or W < _WIN:
        raise ValueError("win_size exceeds image extent: both image dimensions must be at least 7")
    bg = background.to(pred.device, torch.float32, non_blocking=True) if isinstance(background, torch.Tensor) \
        else float(background)
    a = gt_rgba[..., 3:4]
    gt = gt_rgba[..., :3] * a + bg * (1 - a)
    alpha = gt_rgba[..., 3]
    rm = None
    if ray_mask is not None:
        rm = _binary_mask(ray_mask, H, W, "ray_mask")
        on = rm.view(torch.bool)
        gt = torch.where(on.unsqueeze(-1), gt, bg)
        alpha = torch.where(on, alpha, 0.0)
    roi = mask_bounding_rect(alpha)
    out = _metrics(pred, gt.contiguous(), _SSIM | _PSNR, H, W, 3 * W, roi=roi, data_range=1.0, psnr_mask=rm)
    return {"psnr": out[1], "ssim": out[0], "roi": roi}


def compute_psnr(im1: torch.Tensor, im2: torch.Tensor, mask: Optional[torch.Tensor] = None) -> float:
    """evaluate.py:compute_psnr: CHW images in [0, 1], mask of H*W elements (e.g. [H, W, 1]) or None."""
    if im1.dim() != 3 or im1.shape[0] != 3 or im2.shape != im1.shape:
        raise ValueError("compute_psnr takes two CHW images with 3 channels of the same shape")
    return float(psnr(im1.permute(1, 2, 0).contiguous(), im2.permute(1, 2, 0).contiguous(), mask))


def compute_ssim(im1: torch.Tensor, im2: torch.Tensor) -> float:
    """evaluate.py:compute_ssim: HWC uint8 images, data_range 255."""
    if im1.dtype != torch.uint8 or im2.dtype != torch.uint8:
        raise ValueError("compute_ssim takes HWC uint8 images")
    return float(ssim(im1, im2))
