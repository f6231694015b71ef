"""CPU suite: host logic and oracle against the golden vectors generated from the reference
(tests/golden/make_golden.py), layout tables, and the C-ABI export list."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from humanrf_b200.dataset.cameras import inverse_kr, projection_matrix_world2pixel
from humanrf_b200.dataset.input_batch import InputBatch
from humanrf_b200.input import merge_input_batches
from humanrf_b200.scene_representation.grid_layout import GridLayout, mlp_blob_permutation, segment_log2_hashmap_size
from humanrf_b200.utils.activation import truncated_exp
from humanrf_b200.utils.loss import bce_loss
from oracle import field as ofield
from oracle import hashgrid, rendering

ROOT = Path(__file__).resolve().parent.parent
G = np.load(ROOT / "tests/golden/reference_host.npz")
FIELDS = ["ray_origins", "ray_directions", "minmaxes", "rgba", "ray_masks", "frame_numbers", "unique_frame_numbers",
          "camera_numbers", "sample_distances", "ray_indices"]


@pytest.mark.parametrize("case", ["a", "b", "c", "d"])
def test_merge_input_batches_matches_reference(case):
    nb = int(G[f"merge_{case}_nb"])
    budget = int(G[f"merge_{case}_budget"])
    batches = []
    for bi in range(nb):
        kw = {f: torch.from_numpy(G[f"merge_{case}_in{bi}_{f}"]) for f in FIELDS}
        batches.append(InputBatch(width=64, height=48, **kw))
    out = merge_input_batches(batches, None if budget < 0 else budget)
    for f in FIELDS:
        got = getattr(out, f)
        if f == "unique_frame_numbers":
            got = torch.sort(got.reshape(-1))[0]
        exp = G[f"merge_{case}_out_{f}"]
        assert got.dtype == torch.from_numpy(exp).dtype, f
        np.testing.assert_array_equal(got.numpy(), exp, err_msg=f)
    assert out.width == 64 and out.height == 48


def test_truncated_exp_matches_reference():
    for impl in (truncated_exp, ofield.truncated_exp):
        x = torch.from_numpy(G["texp_x"]).clone().requires_grad_(True)
        y = impl(x)
        y.backward(torch.from_numpy(G["texp_dy"]))
        np.testing.assert_array_equal(y.detach().numpy(), G["texp_y"])
        np.testing.assert_array_equal(x.grad.numpy(), G["texp_dx"])


def test_bce_loss_matches_reference():
    for impl in (bce_loss, rendering.bce_loss):
        out = impl(torch.from_numpy(G["bce_pred"]), torch.from_numpy(G["bce_target"]))
        np.testing.assert_array_equal(out.numpy(), G["bce_out"])


def test_inverse_kr_matches_reference_camera():
    for i, cp in enumerate(G["cam_params"]):
        w2p = projection_matrix_world2pixel(1028, 752, cp[:3], cp[3:], np.array([1.773863, 1.773863 * 1028 / 752]),
                                            np.array([0.5, 0.5]))
        np.testing.assert_allclose(np.linalg.inv(w2p), G["cam_world2pixel_inv_full"][i], rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(inverse_kr(w2p), G["cam_inverse_krs"][i], rtol=2e-6, atol=1e-7)


def test_grid_layout_matches_oracle_and_survey():
    # SURVEY 8: entries per grid for log2T = 19..15
    expected = {19: 6984576, 18: 3695768, 17: 1947288, 16: 1015808, 15: 524288}
    for l2, total in expected.items():
        lay = GridLayout(l2)
        sc, rs, of, sz, hs, tot = hashgrid.level_table(l2)
        assert lay.n_entries == tot == total
        np.testing.assert_array_equal(lay.scale, sc)
        np.testing.assert_array_equal(lay.res, rs)
        np.testing.assert_array_equal(lay.offset, of)
        np.testing.assert_array_equal(lay.size, sz)
        assert lay.hashed_mask == sum(1 << i for i, h in enumerate(hs) if h)
    lay = GridLayout(19)
    assert list(lay.res[:4]) == [32, 43, 56, 74] and lay.hashed_mask == 0xFFF0
    np.testing.assert_allclose(lay.scale[[5, 10, 15]], [127.000015, 511.00018, 2047.0015], rtol=1e-6)
    assert [segment_log2_hashmap_size(s, 19) for s in (6, 12, 25, 50, 100)] == [15, 16, 17, 18, 19]
    assert [ofield.segment_log2_hashmap_size(s) for s in (6, 12, 25, 50, 100)] == [15, 16, 17, 18, 19]


def test_mlp_blob_permutation():
    for emb, n in ((0, 10240), (2, 11264)):
        dst, src = mlp_blob_permutation(emb)
        assert sorted(src.tolist()) == list(range(n)) and len(set(dst.tolist())) == n and dst.max() < 22528 // 2
    dst, src = mlp_blob_permutation(0)
    # element (n=9, k=17) of the first layer [64,32]: core (kg=2, ng=1), row 1, col 1
    assert src[dst.tolist().index((2 * 8 + 1) * 64 + 1 * 8 + 1)] == 9 * 32 + 17
    # colour W2 follows colour W1 [64,K]: byte 6144 + 128*K
    dst48, src48 = mlp_blob_permutation(2)
    assert dst48[src48.tolist().index(3072 + 64 * 48)] == (6144 + 128 * 48) // 2
    assert dst[src.tolist().index(3072 + 64 * 32)] == (6144 + 128 * 32) // 2


def test_c_abi_exports_every_declared_symbol():
    from humanrf_b200 import _lib

    header = (ROOT / "include/humanrf_b200.h").read_text()
    declared = sorted(set(re.findall(r"\b(hrf_[a-z0-9_]+)\s*\(", header)))
    assert declared == _lib.exported_symbols()
    if not _lib.LIB_PATH.exists():
        pytest.skip("library not built yet (python -m humanrf_b200.build)")
    handle = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in declared:
        assert hasattr(handle, name), name
    assert _lib.lib().hrf_version() >= 1


def test_product_does_not_import_oracle():
    for p in (ROOT / "humanrf_b200").rglob("*.py"):
        src = p.read_text()
        assert "import oracle" not in src and "from oracle" not in src, p


def test_dropin_maps_reference_import_paths(tmp_path):
    """Every module the drop-in replaces exists in the reference (its module list is stored in
    tests/golden/reference_python.json), and the reference's import paths resolve to ours with its package tree (namespace
    packages, no __init__.py) on sys.path."""
    import json
    import sys

    import humanrf_b200.dropin as dropin

    modules = json.loads((ROOT / "tests/golden/reference_python.json").read_text())["modules"]
    assert set(dropin._MAP) <= set(modules)
    for name in modules:
        (tmp_path / Path(*name.split(".")[:-1])).mkdir(parents=True, exist_ok=True)
    ref = str(tmp_path)
    sys.path.insert(0, ref)
    try:
        dropin.install()
        from humanrf.scene_representation.humanrf import HumanRF as A
        from humanrf_b200.scene_representation.humanrf import HumanRF as B
        import humanrf.volume_rendering as vr
        import actorshq.dataset.ray_sampler_native as rs

        assert A is B and hasattr(vr, "prune_samples") and hasattr(rs, "get_samples_occupancy_minmax")
    finally:
        sys.path.remove(ref)
        for k in list(sys.modules):
            if k.startswith(("humanrf.", "actorshq.")) or k in ("humanrf", "actorshq"):
                del sys.modules[k]


def test_bench_reads_roofline_evidence_of_the_default_kernels():
    """bench.py fills roofline.traffic and the unit percentages from the newest committed `ncu --set full` export that holds the
    kernel it names: the default scatter generation for the train line, the fused forward for the render line."""
    import sys

    sys.path.insert(0, str(ROOT))
    import bench

    for kernel in ("grid_scatter_v3_kernel", "field_forward_kernel"):
        prof = bench.committed_ncu(kernel)
        assert prof is not None and kernel in prof["kernel_name"], kernel
        assert prof["source"].startswith("profiles/r2") and prof["source"].endswith("_raw.csv")
        assert prof["traffic"] > 1e6 and 0 < prof["issue_slots_pct"] <= 100 and 0 < prof["l2_pct"] <= 100
    assert bench.committed_ncu("no_such_kernel") is None


def test_reference_arm_line_follows_the_bench_contract(monkeypatch, capsys):
    """`bench.py --impl reference`: one JSON line with the b200 arm's metric / unit, impl, cpu_baseline (kind, cores, sample) and an
    e2e that repeats the value with zero copies.  (The CPU oracle run itself is replaced by a stub: it takes minutes.)"""
    import argparse
    import json
    import sys

    sys.path.insert(0, str(ROOT))
    import bench

    monkeypatch.setattr(bench, "cpu_oracle_rate", lambda mode, steps, warmup, budget_s: (
        123.0, 8, "stub sample", {"seconds_per_step": 2.0, "rays_per_step": 246}))
    monkeypatch.setattr(bench, "dist_info", lambda: (0, 1, 0))
    bench.run_reference(argparse.Namespace(mode="train", steps=3, warmup=1, gpus=1))
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == bench.METRIC["train"] and line["unit"] == "rays/s"
    assert line["value"] == 123.0 and line["higher_is_better"] is True and line["steps"] == 3 and line["warmup"] == 1
    assert line["cpu_baseline"] == {"value": 123.0, "unit": "rays/s", "cores": 8, "kind": "port", "sample": "stub sample"}
    assert line["e2e"] == {"value": 123.0, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # ranks other than 0 print nothing
    monkeypatch.setattr(bench, "dist_info", lambda: (1, 2, 1))
    bench.run_reference(argparse.Namespace(mode="train", steps=3, warmup=1, gpus=2))
    assert capsys.readouterr().out.strip() == ""


def test_cpu_oracle_bench_runs_a_tiny_train_step():
    """oracle/cpu_bench.py end to end at one ray per worker (two workers): prune pass, forward, loss, autograd backward, Adam."""
    import json
    import subprocess
    import sys

    out = subprocess.run([sys.executable, str(ROOT / "oracle" / "cpu_bench.py"), "--mode", "train", "--rays-per-worker", "1",
                          "--workers", "2", "--steps", "1", "--warmup", "1", "--samples-per-ray", "64"],
                         capture_output=True, text=True, check=True, timeout=600).stdout.strip().splitlines()[-1]
    r = json.loads(out)
    assert r["rays_per_step"] == 2 and r["cores"] == 2 and r["rays_per_s"] > 0 and "Adam" in r["sample"]
