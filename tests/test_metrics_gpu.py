"""Device PSNR / SSIM / mask bounding box (humanrf_b200.evaluation.evaluate) against the float64 oracle
(oracle/metrics.py)."""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from humanrf_b200.evaluation import evaluate as ev
from oracle import metrics as om

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent


def pair(shape, dtype, seed=0):
    """A textured image and a noisy copy of it, as numpy arrays."""
    rng = np.random.default_rng(seed)
    a = rng.random(shape + (3,))
    b = np.clip(a + 0.08 * rng.standard_normal(a.shape), 0, 1)
    if dtype == "uint8":
        return (a * 255).round().astype(np.uint8), (b * 255).round().astype(np.uint8)
    return a.astype(np.float32), b.astype(np.float32)


def flat_background_pair(seed=0):
    """1028 x 752, flat 0.3718 background with a textured object: the case fp32 moments without a shift get wrong."""
    rng = np.random.default_rng(seed)
    H, W, bg = 752, 1028, 0.3718
    gt = np.full((H, W, 3), bg)
    pr = np.full((H, W, 3), bg + 0.0123)
    gt[200:500, 300:700] = rng.random((300, 400, 3))
    pr[200:500, 300:700] = np.clip(gt[200:500, 300:700] + 0.05 * rng.standard_normal((300, 400, 3)), 0, 1)
    return gt.astype(np.float32), pr.astype(np.float32)


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


R = {"float32": 1.0, "uint8": 255.0}


@pytest.mark.parametrize("dtype", ["float32", "uint8"])
@pytest.mark.parametrize("shape", [(7, 7), (8, 13), (37, 45), (50, 97), (752, 1028), (3008, 4112)])
def test_ssim_matches_oracle(cuda, shape, dtype):
    a, b = pair(shape, dtype, seed=shape[0])
    got = ev.ssim(dev(a), dev(b), data_range=R[dtype])
    assert got.dtype == torch.float64 and got.dim() == 0
    assert abs(float(got) - om.ssim(a, b, R[dtype])) < 1e-5


@pytest.mark.parametrize("dtype", ["float32", "uint8"])
def test_ssim_rois_match_oracle(cuda, dtype):
    H, W = 61, 83
    a, b = pair((H, W), dtype, seed=11)
    rois = [(0, 0, W, H), (5, 7, 40, 30), (0, 10, 20, 20), (10, 0, 33, 17), (W - 20, 3, 20, 30), (4, H - 9, 50, 9),
            (0, 0, 7, 7), (12, 4, 7, 50), (30, 20, 45, 7), (W - 7, H - 7, 7, 7)]
    A, B = dev(a), dev(b)
    for roi in rois:
        want = om.ssim(a, b, R[dtype], roi)
        host = float(ev.ssim(A, B, data_range=R[dtype], roi=roi))
        device = float(ev.ssim(A, B, data_range=R[dtype], roi=torch.tensor(roi, dtype=torch.int32, device=cuda)))
        assert abs(host - want) < 1e-5, roi
        assert abs(device - want) < 1e-5, roi


def test_ssim_flat_background(cuda):
    gt, pr = flat_background_pair()
    for roi in (None, (250, 150, 500, 400)):
        want = om.ssim(pr, gt, 1.0, roi)
        assert abs(float(ev.ssim(dev(pr), dev(gt), data_range=1.0, roi=roi)) - want) < 1e-5


@pytest.mark.parametrize("dtype", ["float32", "uint8"])
def test_ssim_identical_images_is_one(cuda, dtype):
    a, _ = pair((101, 77), dtype, seed=3)
    A = dev(a)
    assert abs(float(ev.ssim(A, A.clone(), data_range=R[dtype])) - 1.0) < 1e-7


def test_ssim_small_or_empty_rois(cuda):
    a, b = pair((40, 40), "float32")
    A, B = dev(a), dev(b)
    for roi in [(0, 0, 0, 0), (3, 3, 6, 20), (3, 3, 20, 6), (38, 38, 10, 10)]:
        got = ev.ssim(A, B, data_range=1.0, roi=torch.tensor(roi, dtype=torch.int32, device=cuda))
        assert torch.isnan(got).item(), roi
    with pytest.raises(ValueError):
        ev.ssim(A, B, data_range=1.0, roi=(0, 0, 6, 20))
    with pytest.raises(ValueError):
        ev.ssim(A[:6], B[:6].contiguous(), data_range=1.0)
    with pytest.raises(ValueError):
        ev.ssim(A, B)                                     # float images need data_range
    with pytest.raises(RuntimeError):
        ev.ssim(A.double(), B.double(), data_range=1.0)
    with pytest.raises(RuntimeError):
        ev.ssim(A.transpose(0, 1), B.transpose(0, 1), data_range=1.0)


def test_ssim_uint8_default_range(cuda):
    a, b = pair((64, 48), "uint8", seed=8)
    assert float(ev.ssim(dev(a), dev(b))) == float(ev.ssim(dev(a), dev(b), data_range=255))


@pytest.mark.parametrize("mask_dtype", [None, "float", "uint8", "bool"])
@pytest.mark.parametrize("dtype", ["float32", "uint8"])
def test_psnr_matches_oracle(cuda, dtype, mask_dtype):
    a, b = pair((75, 131), dtype, seed=5)
    m = np.random.default_rng(6).random((75, 131)) > 0.4
    mask = None if mask_dtype is None else dev({"float": m.astype(np.float32), "uint8": m.astype(np.uint8) * 7,
                                                "bool": m}[mask_dtype])
    got = ev.psnr(dev(a), dev(b), mask)
    r = R[dtype]
    want = om.compute_psnr(a.transpose(2, 0, 1) / r, b.transpose(2, 0, 1) / r, None if mask is None else m)
    assert got.dtype == torch.float64 and got.dim() == 0
    assert abs(float(got) - want) < 1e-4
    assert float(ev.psnr(dev(a), dev(a), mask)) == np.inf


def bbox_masks():
    rng = np.random.default_rng(3)
    yield rng.random((75, 131)) > 0.7
    yield np.zeros((75, 131), bool)
    one = np.zeros((75, 131), bool)
    one[17, 23] = True
    yield one
    border = np.zeros((75, 131), bool)
    border[0, 5] = border[74, 130] = True
    yield border
    edge = np.zeros((752, 1028), bool)
    edge[100:752, 0:300] = True
    yield edge


@pytest.mark.parametrize("mask_dtype", ["float", "uint8", "bool"])
def test_mask_bounding_rect_equals_cv2(cuda, mask_dtype):
    cv2 = pytest.importorskip("cv2")
    for m in bbox_masks():
        t = dev({"float": m.astype(np.float32) * 0.5, "uint8": m.astype(np.uint8), "bool": m}[mask_dtype])
        got = tuple(ev.mask_bounding_rect(t).tolist())
        assert got == tuple(cv2.boundingRect(m.astype(np.uint8) * 255)) == om.bounding_rect(m)
        assert got == tuple(ev.mask_bounding_rect(t.unsqueeze(-1)).tolist())


@pytest.fixture(scope="module")
def rendered_pair(cuda):
    """A teacher radiance field rendered through TileShardedRenderer (the ground truth) and a perturbed student,
    set up as examples/train_synthetic.py does.  Returns (pred [H,W,3], gt_rgba [H,W,4]) on the device."""
    sys.path.insert(0, str(ROOT / "examples"))
    import train_synthetic as ts
    from humanrf_b200.dataset.data_loader import DataLoader
    from humanrf_b200.dataset.occupancy_grid_native import OccupanyGrid
    from humanrf_b200.parallel import TileShardedRenderer

    torch.manual_seed(0)
    frames = list(range(15, 21))
    teacher = ts.smooth_teacher(cuda, frames)
    ds = ts.TeacherDataset(teacher, cuda, num_cameras=6, frames=frames, width=96, height=72, G=64)
    ds._images = {(c, f): np.zeros((72, 96, 3), np.float32) for c in range(6) for f in frames}
    M = DataLoader.Mode
    boot = DataLoader(ds, "cuda", M.TEST, DataLoader.OutputMode.RAYS_AND_SAMPLES, DataLoader.SpacePruningMode.OCCUPANCY_GRID,
                      batch_size=8192, camera_numbers=tuple(range(6)), frame_numbers=tuple(frames), max_buffer_size=1,
                      render_sequence=[(0, frames[0])])
    og = OccupanyGrid(64, 2)
    cam = ts.camera_tables(boot, og, ds)(5, frames[0])
    n = cam["width"] * cam["height"]
    gt = TileShardedRenderer(teacher, og, rays_per_batch=8192).render_range(cam, 0, n).clamp(0, 1)
    student = ts.smooth_teacher(cuda, frames)
    g = torch.Generator(device=cuda).manual_seed(1)
    with torch.no_grad():
        for fg in student.feature_grids:
            for p in fg.grids():
                p.add_(0.3 * torch.randn(p.shape, generator=g, device=cuda))
    student._native = None
    pred = TileShardedRenderer(student, og, rays_per_batch=8192).render_range(cam, 0, n).clamp(0, 1)
    H, W = cam["height"], cam["width"]
    alpha = (gt.sum(-1, keepdim=True) > 1e-3).float()
    return pred.view(H, W, 3).contiguous(), torch.cat([gt, alpha], -1).view(H, W, 4).contiguous()


@pytest.mark.parametrize("with_ray_mask", [False, True])
def test_evaluate_image_matches_oracle(rendered_pair, with_ray_mask):
    pred, gt_rgba = rendered_pair
    H, W = pred.shape[:2]
    ray_mask = None
    if with_ray_mask:
        yy, xx = np.mgrid[:H, :W]
        ray_mask = dev((xx + yy) % 5 != 0)
    out = ev.evaluate_image(pred, gt_rgba, 0.0, ray_mask)
    want = om.evaluate_one_image(pred.cpu().numpy(), gt_rgba.cpu().numpy(), 0.0,
                                 None if ray_mask is None else ray_mask.cpu().numpy())
    x, y, w, h = want["roi"]
    assert w >= 7 and h >= 7
    assert tuple(out["roi"].tolist()) == want["roi"]
    assert abs(float(out["psnr"]) - want["psnr"]) < 1e-4
    assert abs(float(out["ssim"]) - want["ssim"]) < 1e-5
    assert 0.0 < want["ssim"] < 1.0 - 1e-6                 # the pair differs


def test_evaluate_image_background_and_mirrors(rendered_pair):
    pred, gt_rgba = rendered_pair
    bg = torch.tensor([0.2, 0.5, 0.9])
    pred_bg = pred + bg.to(pred.device) * (1 - gt_rgba[..., 3:4])
    out = ev.evaluate_image(pred_bg.contiguous(), gt_rgba, bg)
    want = om.evaluate_one_image(pred_bg.cpu().numpy(), gt_rgba.cpu().numpy(), bg.numpy())
    assert abs(float(out["psnr"]) - want["psnr"]) < 1e-4
    assert abs(float(out["ssim"]) - want["ssim"]) < 1e-5
    # evaluate.py's mirrors equal the device results on the same inputs
    gt = (gt_rgba[..., :3] * gt_rgba[..., 3:]).contiguous()
    m = gt_rgba[..., 3:].contiguous()
    assert ev.compute_psnr(pred.permute(2, 0, 1), gt.permute(2, 0, 1), m) == float(ev.psnr(pred, gt, m))
    p8, g8 = (pred * 255).round().to(torch.uint8), (gt * 255).round().to(torch.uint8)
    assert ev.compute_ssim(p8, g8) == float(ev.ssim(p8, g8, data_range=255))
    assert abs(ev.compute_ssim(p8, g8) - om.ssim(p8.cpu().numpy(), g8.cpu().numpy(), 255.0)) < 1e-5


def test_metrics_are_bitwise_reproducible(cuda):
    gt, pr = flat_background_pair(seed=2)
    P, G = dev(pr), dev(gt)
    rgba = torch.cat([G, (G[..., :1] != G[0, 0, 0]).float()], -1).contiguous()
    r1 = ev.evaluate_image(P, rgba)
    r2 = ev.evaluate_image(P, rgba)
    for k in ("psnr", "ssim", "roi"):
        assert torch.equal(r1[k], r2[k]), k
    assert torch.equal(ev.ssim(P, G, data_range=1.0), ev.ssim(P, G, data_range=1.0))


def test_evaluate_image_never_synchronises(rendered_pair):
    pred, gt_rgba = rendered_pair
    H, W = pred.shape[:2]
    ray_mask = torch.ones(H, W, dtype=torch.bool, device=pred.device)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = ev.evaluate_image(pred, gt_rgba, 0.0, ray_mask)
        out2 = ev.evaluate_image(pred, gt_rgba, 0.3)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert np.isfinite(float(out["psnr"])) and np.isfinite(float(out2["ssim"]))
