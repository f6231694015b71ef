"""Differential tests against REAL builds of the reference's first-party CUDA (compiled from its unmodified sources by
oracle/build_ref.py; ray_sampler.cu through oracle/glm_shim).  What those builds returned for the inputs below is
stored in tests/golden/reference_cuda.npz (written by tests/golden/make_reference_cuda_golden.py on a B200), so the
comparison runs without them."""
import functools
from pathlib import Path

import numpy as np
import pytest
import torch

from scene import make_scene

pytestmark = pytest.mark.gpu
GOLDEN = Path(__file__).resolve().parent / "golden" / "reference_cuda.npz"
COMPOSE_STRIDE, VECTOR_GRAD_STRIDE = 57, 93      # stored: every 57th element of the feature outputs, every 93rd of the vector gradient


@functools.lru_cache(maxsize=None)
def reference_outputs():
    return dict(np.load(GOLDEN))


def compose_inputs(device):
    g = torch.Generator().manual_seed(0)
    n, F, VR = 5000, 32, 2048
    feats = [torch.randn(n, F, generator=g).half().to(device) for _ in range(4)]
    vec = (torch.randn(4, VR, F, generator=g) * 0.1).to(device)
    coords = torch.rand(n, 4, generator=g)
    coords[:50] = 0.0; coords[50:100] = 1.0                      # clamped taps at both ends
    coords[:, 3] = torch.randint(0, 6, (n,), generator=g).float() / 6   # few distinct time taps (atomic contention)
    coords = coords.to(device)
    dout = torch.randn(n, F, generator=g).half().to(device)
    return feats, vec, coords, dout


def strided(x, stride):
    return x.reshape(-1)[::stride].float().cpu()


def test_tensor_composition_matches_reference_extension(cuda):
    from humanrf_b200.scene_representation import tensor_composition_native as ours

    R = reference_outputs()
    feats, vec, coords, dout = compose_inputs(cuda)
    b = ours.compose_tensors_forward(*feats, vec, coords)
    rb = ours.compose_tensors_backward(*feats, vec, coords, dout)
    torch.cuda.synchronize()
    for name, x in zip(("fwd", "bwd0", "bwd1", "bwd2", "bwd3", "bwd4"), (b, *rb[:5])):
        assert list(x.shape) == R[f"compose_{name}_shape"].tolist() and str(x.dtype) == str(R[f"compose_{name}_dtype"]), name
    a = torch.from_numpy(R["compose_fwd"]).float()
    diff = (a - strided(b, COMPOSE_STRIDE)).abs()
    print("compose fwd max abs diff", diff.max().item())
    assert (diff <= 2e-3 * a.abs() + 1e-6).all()                 # <= 1-2 fp16 ulp (reference is built with --use_fast_math)
    for k in range(4):
        x = torch.from_numpy(R[f"compose_bwd{k}"]).float()
        d = (x - strided(rb[k], COMPOSE_STRIDE)).abs()
        assert (d <= 2e-3 * x.abs() + 1e-6).all()
    np.testing.assert_allclose(strided(rb[4], VECTOR_GRAD_STRIDE).numpy(), R["compose_bwd4"], rtol=2e-3,
                               atol=2e-3 * float(R["compose_bwd4_absmax"]))


def sampler_inputs(device):
    """Scene, occupancy grids on the device, and the arguments of get_samples_occupancy_minmax around the grid handles."""
    sc = make_scene(num_images=3, width=128, height=96, G=128)
    B = len(sc["grids"])
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)
    rng = np.random.default_rng(1)
    idx = torch.from_numpy(rng.integers(0, B * 128 * 96, 8192).astype(np.int64)).to(device)
    rgba, lm = torch.from_numpy(sc["rgba_big"]) if "rgba_big" in sc else torch.from_numpy(
        rng.integers(0, 256, (B * 128 * 96, 4)).astype(np.uint8)), torch.zeros(B * 128 * 96, dtype=torch.bool)
    head = (rgba, lm, t(sc["frame_numbers"]), t(sc["camera_numbers"]))
    tail = (t(sc["landscape"]), idx, t(sc["inverse_krs"]), t(sc["camera_origins"]), t(sc["aabb"]), sc["G"], 128, 96, 4e-4, False)
    return sc, [t(g) for g in sc["grids"]], head, tail


def test_sampler_against_reference_build(cuda):
    """Measured mismatch of the canonical-IEEE sampler vs the reference's --use_fast_math + hardware-texture build."""
    from humanrf_b200.dataset import ray_sampler_native as rs
    from humanrf_b200.dataset.occupancy_grid_native import OccupanyGrid

    R = reference_outputs()
    sc, grids_dev, head, tail = sampler_inputs(cuda)
    og = OccupanyGrid(sc["G"], len(grids_dev))
    oh = torch.tensor([og.add_grid(g) for g in grids_dev], dtype=torch.int64, device=cuda)
    b = rs.get_samples_occupancy_minmax(*head, oh, *tail)
    torch.cuda.synchronize()
    mb = b[6].cpu().numpy()
    ma = np.unpackbits(R["sampler_mask_bits"])[:mb.size].astype(bool)
    mask_mismatch = (ma != mb).mean()
    both = ma & mb
    # per-ray comparison on rays both keep
    ia, ib = np.cumsum(ma) - 1, np.cumsum(mb) - 1
    sel_a, sel_b = ia[both], ib[both]
    da, db = R["sampler_dirs"][sel_a], b[1].cpu().numpy()[sel_b]
    mma, mmb = R["sampler_minmax"][sel_a], b[5].cpu().numpy()[sel_b]
    ca = R["sampler_counts"][sel_a]
    cb = np.bincount(b[8].cpu().numpy(), minlength=mb.sum())[sel_b]
    n_ref = int(R["sampler_num_samples"])
    print(f"ray-mask mismatch rate {mask_mismatch:.2e}; dir max|d| {np.abs(da - db).max():.2e}; "
          f"tmin/tmax max|d| {np.abs(mma - mmb).max():.2e}; rays with different sample count {(ca != cb).mean():.2e}; "
          f"total samples ref {n_ref} ours {b[7].numel()}")
    rgba_a = torch.from_numpy(R["sampler_rgba_u8"]).float() / 255.0        # the reference's rgba[kept] / 255.0
    np.testing.assert_array_equal(rgba_a.numpy()[sel_a], b[2].cpu().numpy()[sel_b])   # rgba gather
    np.testing.assert_array_equal(R["sampler_frame_numbers"][sel_a], b[3].cpu().numpy()[sel_b])   # frame numbers
    assert [str(b[i].dtype) for i in (6, 7, 8)] == R["sampler_dtypes"].tolist()
    assert mask_mismatch < 5e-3
    assert np.abs(da - db).max() < 1e-5
    assert np.abs(mma - mmb).max() < 5e-3            # one coarse march step is 0.5/G = 3.9e-3
    assert (ca != cb).mean() < 0.05
    assert abs(n_ref - b[7].numel()) < 0.01 * n_ref
    del og
