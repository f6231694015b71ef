#!/usr/bin/env python
"""Times validation metrics on the device against the CPU route the reference takes.

For images of 1028 x 752 (the bench's --mode image size) and 4112 x 3008 (full ActorsHQ resolution) with an elliptic
foreground covering 28 % of the pixels, it records:
  * evaluate_image (composite, bounding box, PSNR + SSIM) per call, CUDA events, L2 warm (back-to-back calls) and
    L2 flushed (a 256 MB write between calls, outside the timed window);
  * the two kernels alone: hrf_mask_bbox and hrf_image_metrics (SSIM over the box + masked PSNR);
  * the CPU route: copy pred and gt to the host, then skimage's structural_similarity if it is importable, otherwise
    the float64 oracle (oracle/metrics.py), on the same images; which one ran is in "cpu_route";
  * the algorithmic bytes of the metrics kernel (2 images x H x W x 3 x 4 B) over its time.
The card name and power limit are read in the same run.

    python scripts/metrics_times.py --out metrics_times_out
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from humanrf_b200 import _lib as L  # noqa: E402
from humanrf_b200.evaluation import evaluate as ev  # noqa: E402
from oracle import metrics as om  # noqa: E402


def images(H, W, dev, seed=0):
    """pred [H,W,3], gt_rgba [H,W,4]: a textured ellipse on a black background (28 % of the pixels), pred = gt + noise."""
    g = torch.Generator(device=dev).manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H, device=dev), torch.arange(W, device=dev), indexing="ij")
    k = (0.28 * 4 / np.pi) ** 0.5
    inside = ((xx - W / 2) / (0.5 * k * W)) ** 2 + ((yy - H / 2) / (0.5 * k * H)) ** 2 <= 1.0
    a = inside.float().unsqueeze(-1)
    rgb = torch.rand(H, W, 3, generator=g, device=dev) * a
    pred = (rgb + 0.03 * torch.randn(H, W, 3, generator=g, device=dev) * a).clamp(0, 1).contiguous()
    return pred, torch.cat([rgb, a], -1).contiguous(), float(inside.float().mean())


def event_time(fn, reps, flush=None):
    """Mean ms per call over reps calls; with flush, each call is timed alone after overwriting L2."""
    if flush is None:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            fn()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / reps
    total = 0.0
    for _ in range(reps):
        flush.fill_(1)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        total += s.elapsed_time(e)
    return total / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for metrics_times.json")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--cpu-reps", type=int, default=3)
    a = ap.parse_args()
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    try:
        from skimage.metrics import structural_similarity  # noqa: F401
        cpu_route = "skimage.metrics.structural_similarity + cv2.boundingRect (float32, as trainer.py:373-419)"
    except ImportError:
        structural_similarity = None
        cpu_route = "oracle/metrics.py (float64 numpy/scipy; skimage is not installed)"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    res = {"card": card, "cpu_route": cpu_route, "reps": a.reps, "sizes": []}
    for W, H in ((1028, 752), (4112, 3008)):
        pred, gt_rgba, frac = images(H, W, dev)
        gt = (gt_rgba[..., :3] * gt_rgba[..., 3:]).contiguous()
        alpha = gt_rgba[..., 3].contiguous()
        roi = ev.mask_bounding_rect(alpha)
        lib = L.lib()
        m8 = (alpha > 0).view(torch.uint8)
        box = torch.empty(4, dtype=torch.int32, device=dev)
        ws = torch.empty(int(lib.hrf_image_metrics_workspace_bytes(H, W)), dtype=torch.uint8, device=dev)
        res_out = torch.empty(4, dtype=torch.float64, device=dev)

        def full():
            ev.evaluate_image(pred, gt_rgba)

        def bbox_kernel():
            L.check(lib.hrf_mask_bbox(m8.data_ptr(), H, W, box.data_ptr(), L.stream()))

        def metrics_kernel():
            L.check(lib.hrf_image_metrics(pred.data_ptr(), gt.data_ptr(), 0, H, W, 3 * W, roi.data_ptr(), 1.0, None, 3,
                                          res_out.data_ptr(), ws.data_ptr(), L.stream()))

        for fn in (full, bbox_kernel, metrics_kernel):      # warm-up: module load, allocator
            for _ in range(20):
                fn()
        torch.cuda.synchronize()
        row = {"width": W, "height": H, "object_fraction": round(frac, 4), "roi": roi.tolist(),
               "roi_fraction": round(roi[2].item() * roi[3].item() / (H * W), 4)}
        for name, fn in (("evaluate_image", full), ("hrf_mask_bbox", bbox_kernel), ("hrf_image_metrics", metrics_kernel)):
            row[f"{name}_ms_l2_warm"] = round(event_time(fn, a.reps), 5)
            row[f"{name}_ms_l2_flushed"] = round(event_time(fn, max(a.reps // 4, 10), flush), 5)
        nbytes = 2 * H * W * 3 * 4
        row["metrics_kernel_bytes"] = nbytes
        row["metrics_kernel_GBps_l2_flushed"] = round(nbytes / (row["hrf_image_metrics_ms_l2_flushed"] * 1e-3) / 1e9, 1)
        r = ev.evaluate_image(pred, gt_rgba)
        row["device_psnr"], row["device_ssim"] = float(r["psnr"]), float(r["ssim"])

        # the CPU route: D2H, then composite + bounding box + crop + SSIM + PSNR on the host
        times, d2h = [], []
        for _ in range(a.cpu_reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            p_h, g_h = pred.cpu().numpy(), gt_rgba.cpu().numpy()
            t1 = time.perf_counter()
            if structural_similarity is not None:
                import cv2

                gth = g_h[..., :3] * g_h[..., 3:]
                x, y, w, h = cv2.boundingRect(((g_h[..., 3] > 0) * 255).astype(np.uint8))
                s = structural_similarity(p_h[y:y + h, x:x + w], gth[y:y + h, x:x + w], channel_axis=2, data_range=1.0)
                ps = om.compute_psnr(p_h.transpose(2, 0, 1), gth.transpose(2, 0, 1))
            else:
                o = om.evaluate_one_image(p_h, g_h)
                s, ps = o["ssim"], o["psnr"]
            t2 = time.perf_counter()
            d2h.append((t1 - t0) * 1e3)
            times.append((t2 - t0) * 1e3)
        row["cpu_route_ms"] = round(float(np.median(times)), 2)
        row["cpu_route_d2h_ms"] = round(float(np.median(d2h)), 2)
        row["cpu_ssim"], row["cpu_psnr"] = float(s), float(ps)
        res["sizes"].append(row)
        print(json.dumps(row), flush=True)
    (out / "metrics_times.json").write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({"card": card, "cpu_route": cpu_route}))


if __name__ == "__main__":
    main()
