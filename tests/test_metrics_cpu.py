"""CPU checks of the float64 metrics oracle (oracle/metrics.py) that the device PSNR / SSIM are compared with."""
import numpy as np
import pytest

from oracle import metrics as om


def brute_ssim(im1, im2, data_range):
    """SSIM by definition: explicit symmetric padding (scipy's `reflect`) and one 7x7 window per pixel."""
    out = []
    c1, c2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    for c in range(im1.shape[2]):
        x = np.pad(np.asarray(im1[..., c], np.float64), 3, mode="symmetric")
        y = np.pad(np.asarray(im2[..., c], np.float64), 3, mode="symmetric")
        H, W = im1.shape[:2]
        vals = []
        for i in range(3, H - 3):
            for j in range(3, W - 3):
                wx, wy = x[i:i + 7, j:j + 7], y[i:i + 7, j:j + 7]
                ux, uy = wx.mean(), wy.mean()
                vx = ((wx - ux) ** 2).sum() / 48
                vy = ((wy - uy) ** 2).sum() / 48
                vxy = ((wx - ux) * (wy - uy)).sum() / 48
                vals.append((2 * ux * uy + c1) * (2 * vxy + c2) / ((ux * ux + uy * uy + c1) * (vx + vy + c2)))
        out.append(np.mean(vals))
    return float(np.mean(out))


@pytest.mark.parametrize("shape", [(7, 7), (8, 13), (13, 20)])
def test_oracle_ssim_equals_windowed_definition(shape):
    rng = np.random.default_rng(sum(shape))
    a = rng.random(shape + (3,))
    b = np.clip(a + 0.1 * rng.standard_normal(a.shape), 0, 1)
    assert abs(om.ssim(a, b, 1.0) - brute_ssim(a, b, 1.0)) < 1e-12
    u = rng.integers(0, 256, shape + (3,)).astype(np.uint8)
    v = rng.integers(0, 256, shape + (3,)).astype(np.uint8)
    assert abs(om.ssim(u, v, 255.0) - brute_ssim(u, v, 255.0)) < 1e-12


def test_oracle_ssim_constant_images_closed_form():
    a, b = 0.3718, 0.6
    c1 = 1e-4
    got = om.ssim(np.full((9, 11, 3), a), np.full((9, 11, 3), b), 1.0)
    assert abs(got - (2 * a * b + c1) / (a * a + b * b + c1)) < 1e-12


def test_oracle_ssim_identical_images_and_small_sizes():
    a = np.random.default_rng(0).random((10, 12, 3))
    assert abs(om.ssim(a, a, 1.0) - 1.0) < 1e-12
    assert abs(om.ssim(a, a, 1.0, roi=(2, 1, 7, 8)) - 1.0) < 1e-12
    with pytest.raises(ValueError):
        om.ssim(a[:6], a[:6], 1.0)
    with pytest.raises(ValueError):
        om.ssim(a, a, 1.0, roi=(0, 0, 6, 10))


def test_oracle_psnr():
    rng = np.random.default_rng(1)
    a, b = rng.random((3, 5, 4)), rng.random((3, 5, 4))
    mask = rng.random((5, 4, 1)) > 0.5
    mse = ((a - b) ** 2).mean(0)[mask[..., 0]].mean()
    assert om.compute_psnr(a, b, mask) == pytest.approx(-10 * np.log10(mse), abs=1e-12)
    assert om.compute_psnr(a, a) == np.inf


def _masks():
    rng = np.random.default_rng(3)
    yield rng.random((40, 57)) > 0.7
    yield np.zeros((40, 57), bool)
    one = np.zeros((40, 57), bool)
    one[17, 23] = True
    yield one
    border = np.zeros((40, 57), bool)
    border[0, 5] = border[39, 56] = True
    yield border
    blob = np.zeros((40, 57), bool)
    blob[10:30, 0:20] = True
    yield blob


def test_oracle_bounding_rect_equals_cv2():
    cv2 = pytest.importorskip("cv2")
    for m in _masks():
        assert om.bounding_rect(m) == tuple(cv2.boundingRect(m.astype(np.uint8) * 255))


def test_oracle_evaluate_one_image_pieces():
    rng = np.random.default_rng(4)
    H, W = 20, 30
    gt = np.zeros((H, W, 4))
    gt[5:15, 8:22, :3] = rng.random((10, 14, 3))
    gt[5:15, 8:22, 3] = 1.0
    pred = np.clip(gt[..., :3] + 0.05 * rng.standard_normal((H, W, 3)), 0, 1)
    r = om.evaluate_one_image(pred, gt, 0.0)
    assert r["roi"] == (8, 5, 14, 10)
    assert r["ssim"] == pytest.approx(om.ssim(pred, gt[..., :3], 1.0, (8, 5, 14, 10)), abs=1e-15)
    assert r["psnr"] == pytest.approx(om.compute_psnr(pred.transpose(2, 0, 1), gt[..., :3].transpose(2, 0, 1)), abs=1e-12)


def test_oracle_ssim_equals_skimage():
    skm = pytest.importorskip("skimage.metrics")
    rng = np.random.default_rng(5)
    a = rng.random((31, 40, 3)).astype(np.float32)
    b = np.clip(a + 0.05 * rng.standard_normal(a.shape), 0, 1).astype(np.float32)
    # skimage computes float32 inputs in float32
    assert abs(om.ssim(a, b, 1.0) - skm.structural_similarity(a, b, channel_axis=2, data_range=1.0)) < 1e-5
    u = (a * 255).astype(np.uint8)
    v = (b * 255).astype(np.uint8)
    assert abs(om.ssim(u, v, 255.0) - skm.structural_similarity(u, v, channel_axis=2)) < 1e-12
