"""SURVEY 8f-4 on the GPU: visual-hull carving bit-exact against the oracle and statistically against the reference's
own extension (its answer stored in tests/golden/reference_cuda.npz); adaptive temporal partitioning against the
reference's golden decisions."""
import numpy as np
import pytest
import torch

from oracle import occupancy_tools as O
from scene import carve_scene, occupancy_sequence
from test_occupancy_tools_cpu import golden_cases
from test_ref_parity_gpu import reference_outputs

pytestmark = pytest.mark.gpu


def _carve(sc, thr, G, cuda):
    from humanrf_b200.toolbox import occupancy_grid_generation_native as ours

    return ours.generate_from_masks(torch.from_numpy(sc["masks"]).to(cuda), torch.from_numpy(sc["projection_matrices"]).to(cuda),
                                    torch.from_numpy(sc["landscape"]).to(cuda), thr, G, sc["width"], sc["height"])


@pytest.mark.parametrize("thr,G", [(1, 40), (6, 64), (12, 33)])
def test_carve_bit_exact_vs_oracle(cuda, thr, G):
    sc = carve_scene(num_cameras=12, width=96, height=72, seed=thr)
    want = O.generate_from_masks(sc["masks"], sc["projection_matrices"], sc["landscape"], thr, G, 96, 72)
    got = _carve(sc, thr, G, cuda).cpu().numpy()
    assert got.shape == (G, G, G) and got.dtype == np.uint8
    assert (got == want).all(), f"{(got != want).sum()} voxels differ"
    assert 0 < (got == 255).sum() < G ** 3


def test_carve_rejects_wrong_mask_size(cuda):
    sc = carve_scene(num_cameras=4, width=32, height=24)
    with pytest.raises(RuntimeError, match="width\\*height"):
        _carve(dict(sc, width=31), 1, 8, cuda)


def reference_carve_args(device):
    """Full-size carve: G=256, 24 cameras of 512x384, threshold 20."""
    sc = carve_scene(num_cameras=24, width=512, height=384, seed=5)
    return (torch.from_numpy(sc["masks"]).to(device), torch.from_numpy(sc["projection_matrices"]).to(device),
            torch.from_numpy(sc["landscape"]).to(device), 20, 256, 512, 384)


def test_carve_vs_reference_extension(cuda):
    """Full-size carve (G=256, 24 cameras) against the reference's kernel built from its unmodified source (it returns
    0 or 255 per voxel; the occupied voxels are stored as a bit mask).  The reference is compiled with --use_fast_math
    (approximate divides), so a voxel whose projection lands within an ulp of a pixel boundary may sample a
    neighbouring mask pixel: a handful of voxels out of 16.7 M."""
    args = reference_carve_args(cuda)
    G = args[4]
    want = torch.from_numpy(np.unpackbits(reference_outputs()["carve_occupied_bits"])[:G ** 3].reshape(G, G, G) * 255).to(cuda)
    from humanrf_b200.toolbox import occupancy_grid_generation_native as ours

    got = ours.generate_from_masks(*args)
    torch.cuda.synchronize()
    assert got.shape == want.shape and got.dtype == want.dtype
    diff = int((want != got).sum())
    occ = int((want == 255).sum())
    def ms(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fn(); e0.record()
        for _ in range(5):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 5

    print(f"carve vs reference: {diff} of {G ** 3} voxels differ, {occ} occupied; ours {ms(lambda: ours.generate_from_masks(*args)):.3f} ms")
    assert 0 < occ < G ** 3 and diff <= 2e-5 * G ** 3


class _DS:
    def __init__(self, grids):
        self.grids = grids

    def get_occupancy_grid(self, frame_number):
        return self.grids[frame_number]


def test_partitioning_matches_reference_golden(cuda):
    from humanrf_b200.adaptive_temporal_partitioning import compute_adaptive_segment_sizes

    for name, n, speed, thr, seed, sizes in golden_cases():
        grids = occupancy_sequence(n, speed, G=48, seed=seed)
        assert compute_adaptive_segment_sizes(_DS(grids), list(range(n)), thr, device=cuda) == sizes, name


def test_union_count_odd_sizes(cuda):
    from humanrf_b200 import _lib as L

    rng = np.random.default_rng(0)
    for n in (1, 31, 33, 1000, 48 ** 3 + 7):
        a, b = [(rng.random(n) < 0.3).astype(np.uint8) * 255 for _ in range(2)]
        a[: n // 7] = 17                                              # values other than 255 are not occupied
        bits = torch.zeros((n + 31) // 32, dtype=torch.int32, device=cuda)
        cnt = torch.zeros(1, dtype=torch.int64, device=cuda)
        for g, want in ((a, (a == 255).sum()), (b, ((a == 255) | (b == 255)).sum())):
            t = torch.from_numpy(g).to(cuda)
            L.check(L.lib().hrf_occupancy_union_count(bits.data_ptr(), t.data_ptr(), n, cnt.data_ptr(), L.stream()))
            assert int(cnt.item()) == int(want)
