"""Differential tests against the reference's first-party pure-Python pieces of the path, on randomized inputs.  The
reference's answers for exactly these inputs are stored in tests/golden/reference_python.json and .npz (written by
tests/golden/make_reference_python_golden.py from a reference checkout), so the comparisons run without one: the
inputs are rebuilt here from the same seeds and our side is run live."""
import dataclasses
import functools
import hashlib
import json
import types
from pathlib import Path

import numpy as np
import pytest
import torch

GOLDEN = Path(__file__).resolve().parent / "golden"


@functools.lru_cache(maxsize=None)
def _golden():
    return json.loads((GOLDEN / "reference_python.json").read_text()), dict(np.load(GOLDEN / "reference_python.npz"))


@pytest.fixture(scope="module")
def ref():
    """The reference's stored answers: (JSON document, arrays)."""
    return _golden()


def surface(cls):
    """Dataclass fields with their defaults, and public members (JSON-able: an absent default is "MISSING")."""
    fields = [[f.name, "MISSING" if f.default is dataclasses.MISSING else repr(f.default)] for f in dataclasses.fields(cls)]
    return fields, sorted(m for m in dir(cls) if not m.startswith("_"))


def test_dataclass_surfaces_match(ref):
    from humanrf_b200.dataset.input_batch import InputBatch
    from humanrf_b200.scene_representation.query_io import QueryInput, QueryOutput

    want = ref[0]["surfaces"]
    for cls in (InputBatch, QueryInput, QueryOutput):
        assert list(surface(cls)) == want[cls.__name__], cls.__name__


FIELDS = ["ray_origins", "ray_directions", "minmaxes", "rgba", "ray_masks", "frame_numbers", "unique_frame_numbers",
          "camera_numbers", "sample_distances", "ray_indices"]


def _batch(cls, rng, num_rays, masked):
    counts = rng.integers(0, 9, num_rays)
    ri = np.repeat(np.arange(num_rays), counts)
    mask = np.ones((num_rays + masked, 1), bool)
    mask[rng.permutation(num_rays + masked)[:masked]] = False
    fr = rng.integers(15, 40, (num_rays, 1)).astype(np.int32)
    t = torch.from_numpy
    return cls(ray_origins=t(rng.normal(size=(num_rays, 3)).astype(np.float32)),
               ray_directions=t(rng.normal(size=(num_rays, 3)).astype(np.float32)),
               minmaxes=t(rng.random((num_rays, 2)).astype(np.float32)), rgba=t(rng.random((num_rays, 4)).astype(np.float32)),
               ray_masks=t(mask), frame_numbers=t(fr), unique_frame_numbers=torch.unique(t(fr)).view(-1, 1),
               camera_numbers=t(rng.integers(0, 160, (num_rays, 1)).astype(np.int32)),
               sample_distances=t(rng.random((int(counts.sum()), 1)).astype(np.float32)), ray_indices=t(ri.astype(np.int64)),
               width=64, height=48)


def merge_cases(cls):
    """60 random configurations of merge_input_batches, batches built with `cls`: (case, batches, budget, total samples)."""
    rng = np.random.default_rng(7)
    for case in range(60):
        nb = int(rng.integers(1, 5))
        specs = [(int(rng.integers(1, 30)), int(rng.integers(0, 5))) for _ in range(nb)]
        r2 = np.random.default_rng(int(rng.integers(0, 2 ** 31)))
        batches = [_batch(cls, r2, *s) for s in specs]
        total = sum(b.sample_distances.shape[0] for b in batches)
        yield case, batches, [None, max(1, total // 2), max(1, total - 1), total, total + 5, 1][case % 6], total


def merged_fields(out):
    """Each field of a merged batch as "dtype shape digest", the digest a 96-bit prefix of the SHA-256 of its bytes
    (unique frame numbers sorted first)."""
    res = {}
    for f in FIELDS:
        x = getattr(out, f)
        if f == "unique_frame_numbers":
            x = torch.sort(x.reshape(-1))[0]
        digest = hashlib.sha256(np.ascontiguousarray(x.numpy()).tobytes()).hexdigest()[:24]
        res[f] = f"{str(x.dtype).replace('torch.', '')} {'x'.join(map(str, x.shape))} {digest}"
    return res


def test_merge_input_batches_randomized(ref):
    """input.py:10-55 incl. the sample-budget cut-off and its `cumsum < cutoff` behaviour, 60 random configurations."""
    from humanrf_b200.dataset.input_batch import InputBatch
    from humanrf_b200.input import merge_input_batches

    want = ref[0]["merge"]
    checked_cut = 0
    for case, batches, budget, total in merge_cases(InputBatch):
        if budget is not None and budget < total:
            checked_cut += 1
        out = merge_input_batches(batches, budget)
        got = merged_fields(out)
        for f in FIELDS:
            assert got[f] == want[case]["fields"][f], (case, f)
        assert [out.width, out.height] == want[case]["size"]
    assert len(want) == 60 and checked_cut >= 15


def truncated_exp_inputs():
    g = torch.Generator().manual_seed(3)
    for scale in (1.0, 9.0, 30.0):
        yield scale, torch.randn(513, generator=g) * scale, torch.randn(513, generator=g)
    pred = torch.rand(777, 1, generator=g) * 1.6 - 0.3
    yield "bce", pred, (torch.rand(777, 1, generator=g) > 0.4).float()


def test_truncated_exp_and_bce_randomized(ref):
    from humanrf_b200.utils.activation import truncated_exp
    from humanrf_b200.utils.loss import bce_loss

    arrays = ref[1]
    for scale, x, dy in truncated_exp_inputs():
        if scale == "bce":
            assert torch.equal(bce_loss(x, dy), torch.from_numpy(arrays["bce_out"]))
            continue
        xi = x.clone().requires_grad_(True)
        y = truncated_exp(xi)
        y.backward(dy)
        assert torch.equal(y.detach(), torch.from_numpy(arrays[f"texp_{scale:g}_y"]))
        assert torch.equal(xi.grad, torch.from_numpy(arrays[f"texp_{scale:g}_dx"]))


def partitioning_cases():
    """12 random occupancy sequences (occasional growth, jumps) and thresholds: (grids, threshold)."""
    rng = np.random.default_rng(11)
    for case in range(12):
        n = int(rng.integers(3, 140))
        base = rng.random((12, 12, 12)) < 0.2
        grids, cur = [], base.copy()
        for f in range(n):
            if rng.random() < [0.05, 0.3, 0.8][case % 3]:
                cur = cur | (rng.random(cur.shape) < 0.02)    # occasional growth of the occupied set
            if rng.random() < 0.03:
                cur = rng.random(cur.shape) < 0.2             # a jump
            grids.append((cur * 255).astype(np.uint8))
        yield grids, [1.05, 1.25, 2.0][case % 3]


def test_segment_size_rules_and_partitioning_randomized(ref):
    """adaptive_temporal_partitioning.py:28-107 against the oracle restatement (the GPU implementation is compared with
    the same reference decisions through tests/golden/partitioning.npz)."""
    from humanrf_b200 import adaptive_temporal_partitioning as ours
    from oracle import occupancy_tools as O

    want = ref[0]["partitioning"]
    assert list(ours.PREDEFINED_SEGMENT_SIZES) == want["predefined"] == list(O.PREDEFINED_SEGMENT_SIZES)
    for n in range(1, 260):
        assert ours.get_segment_size(n) == want["segment_size"][n - 1] == O.get_segment_size(n)
        assert ours.get_final_segment_size(n) == want["final_segment_size"][n - 1] == O.get_final_segment_size(n)
    cases = list(partitioning_cases())
    assert len(cases) == len(want["sizes"])
    for case, (grids, thr) in enumerate(cases):
        assert O.compute_adaptive_segment_sizes(grids, thr) == want["sizes"][case], case


MODEL_CASES = [((50,), 15, 50, 0), ((25, 12, 100, 6), 0, 140, 2), ((6, 6), 3, 9, 0)]


def model_case_key(segment_sizes, first, count, cam_emb):
    return f"{'-'.join(map(str, segment_sizes))}_{first}_{count}_{cam_emb}"


def model_kwargs(cam_emb):
    from humanrf_b200.synthetic import MODEL_KW

    return {**MODEL_KW, "camera_embedding_dim": cam_emb, "temporal_partitioning": "adaptive", "fixed_segment_size": 6}


@pytest.mark.parametrize("segment_sizes,first,count,cam_emb", MODEL_CASES)
def test_model_constructor_against_the_reference(ref, segment_sizes, first, count, cam_emb):
    """humanrf.py:68-156 + decomposition4d.py:73-122 as the reference ran them (only tcnn was a recording stub): frame LUTs,
    per-segment hash-map sizes, encoding / network configs, state-dict key names and the shapes of the first-party
    tensors."""
    from humanrf_b200.scene_representation.grid_layout import GridLayout
    from humanrf_b200.scene_representation.humanrf import HumanRF

    key = model_case_key(segment_sizes, first, count, cam_emb)
    theirs, arrays = ref[0]["model"][key], ref[1]
    ours = HumanRF(sorted_frame_numbers=tuple(range(first, first + count)), segment_sizes=segment_sizes, **model_kwargs(cam_emb))
    # frame -> segment / local-time look-up tables
    for name in ("frame_numbers_to_segment_numbers", "frame_numbers_to_normalized_local_frame_numbers"):
        assert torch.equal(getattr(ours, name), torch.from_numpy(arrays[f"model_{key}_{name}"])), name
    assert [ours.num_frames, ours.num_segments, ours.total_feature_dim, ours.density_scale] == theirs["scalars"]
    # what the reference asks tcnn for, segment by segment
    calls = theirs["calls"]
    enc = [c for c in calls if c[0] == "Encoding"]
    assert len(enc) == 4 * len(segment_sizes)
    for s, fg in enumerate(ours.feature_grids):
        for c in enc[4 * s:4 * s + 4]:
            cfg = c[2]
            assert c[1] == 3 and cfg["otype"] == "HashGrid" and cfg["n_levels"] == 16 and cfg["n_features_per_level"] == 2
            assert cfg["log2_hashmap_size"] == fg.layout.log2_hashmap_size
            assert cfg["base_resolution"] == 32 and np.float32(cfg["per_level_scale"]) == np.float32(np.exp(np.log(2048 / 32) / 15))
            assert GridLayout(cfg["log2_hashmap_size"]).n_params == fg.layout.n_params
    net = [c for c in calls if c[0] == "Network"][0]
    assert net[1:3] == [32, 16] and net[3] == {"otype": "FullyFusedMLP", "activation": "ReLU", "output_activation": "None",
                                              "n_neurons": 64, "n_hidden_layers": 1}
    col = [c for c in calls if c[0] == "NetworkWithInputEncoding"][0]
    assert col[1:3] == [18 + cam_emb, 3] and col[4]["output_activation"] == "Sigmoid" and col[4]["n_hidden_layers"] == 2
    assert col[3]["nested"][0] == {"n_dims_to_encode": 3, "otype": "SphericalHarmonics", "degree": 4}
    # state dict: same keys in the same order, same shapes (first-party tensors: vectors, LUT buffers, embeddings)
    assert [[k, list(v.shape), str(v.dtype)] for k, v in ours.state_dict().items()] == theirs["state_dict"]
    # optimiser parameter groups (humanrf.py:210-220)
    assert [[len(list(g["params"])), g["lr"]] for g in ours.get_params(1e-2)] == theirs["param_groups"]


def closed_form_scene(QueryOutput):
    """The stand-in for the scene representation both sides render: a Gaussian blob whose density depends on the frame."""

    class Scene:
        def density(self, q):
            r2 = (q.positions ** 2).sum(1)
            return QueryOutput(density=2500.0 * torch.exp(-60.0 * r2) * (1.0 + 0.25 * (q.frame_numbers.reshape(-1) % 3).float()))

        def __call__(self, q):
            return QueryOutput(density=self.density(q).density, radiance=torch.sigmoid(3.0 * q.positions + q.directions))

    return Scene()


def prune_render_rays():
    from helpers import synthetic_rays

    return synthetic_rays(64, 40, tuple(range(15, 27)), ragged=True, seed=8)


def prune_render_background():
    return torch.rand(64, 3, generator=torch.Generator().manual_seed(1))


def merge_render_parts():
    g = torch.Generator().manual_seed(9)
    return [(torch.rand(n, 3, generator=g), torch.rand(n, 1, generator=g)) for n in (3, 0, 5)]


def test_prune_and_render_glue_against_the_reference(ref):
    """The reference's own prune_samples / render / merge_render_outputs (volume_rendering.py:26-150), run on the CPU with
    `nerfacc` replaced by the oracle's restatement of its three functions and a closed-form stand-in for the scene
    representation, against the oracle: pins everything the oracle restates AROUND nerfacc (positions, jitter, alpha,
    t_ends = t + step, mask application, background blend, output shapes).  nerfacc's own arithmetic stays unpinned."""
    from humanrf_b200.scene_representation.query_io import QueryOutput
    from humanrf_b200.volume_rendering import RenderOutput as OurRenderOutput
    from oracle import rendering as R

    doc, arrays = ref
    b = prune_render_rays()
    o, d, fr, ri = b["o"], b["d"], b["frames"].view(-1, 1), b["ri"]
    scene = closed_form_scene(QueryOutput)
    bg = prune_render_background()
    for is_training in (False, True):
        tag = "train" if is_training else "eval"
        want = {k: torch.from_numpy(arrays[f"render_{tag}_{k}"]) for k in ("t", "ri", "color", "wsum", "color_nobg")}
        torch.manual_seed(5)
        t = b["t"].view(-1, 1) + (torch.rand_like(b["t"].view(-1, 1)) * R.STEP if is_training else 0)
        pos = o[ri] + t * d[ri]
        sigma = scene.density(types.SimpleNamespace(positions=pos, frame_numbers=fr[ri])).density
        keep = R.prune_mask(sigma, ri)
        assert 0 < int(keep.sum()) < keep.numel()
        assert torch.equal(want["t"], t[keep]) and torch.equal(want["ri"], ri[keep])
        assert want["t"].shape == (int(keep.sum()), 1)
        # render the survivors
        tk, rk = t[keep], ri[keep]
        pk = o[rk] + tk * d[rk]
        q = types.SimpleNamespace(positions=pk, directions=d[rk], frame_numbers=fr[rk])
        col, ws = R.render(tk, scene.density(q).density, scene(q).radiance, rk, 64, bg)
        assert torch.equal(want["color"], col) and torch.equal(want["wsum"], ws)
        assert want["color"].shape == (64, 3) and want["wsum"].shape == (64, 1)
        assert torch.equal(want["color_nobg"], R.render(tk, scene.density(q).density, scene(q).radiance, rk, 64, None)[0])
    # merge_render_outputs: same concatenation, same error for a field that is not a tensor
    c = OurRenderOutput.merge_render_outputs([OurRenderOutput(color=a, weights_sum=w) for a, w in merge_render_parts()])
    assert torch.equal(c.color, torch.from_numpy(arrays["merge_color"]))
    assert torch.equal(c.weights_sum, torch.from_numpy(arrays["merge_wsum"]))
    with pytest.raises(RuntimeError) as err:
        OurRenderOutput.merge_render_outputs([OurRenderOutput(color=torch.rand(2, 3))])
    assert str(err.value) == doc["merge_render_outputs_error"]


SCENE_SIZES, SCENE_EMB = (6, 12, 6), 2
SCENE_ROWS = 256            # samples whose reference outputs are stored (a fixed subset of the batch)


def scene_glue_inputs():
    """Oracle model and ray batch of the scene-representation glue comparison: (model, positions, directions, frames,
    cameras, ray batch)."""
    from helpers import positions_of, synthetic_rays
    from oracle import field as OF

    frames = tuple(range(15, 15 + sum(SCENE_SIZES)))
    om = OF.make_model(SCENE_SIZES, frames, seed=5, table_init="trained", bf16=False, table_std=0.5, camera_embedding_dim=SCENE_EMB)
    b = synthetic_rays(96, 24, frames, ragged=True, seed=12, n_distinct_frames=len(frames))
    ri = b["ri"]
    return om, positions_of(b), b["d"][ri], b["frames"][ri].view(-1, 1), b["cams"][ri].view(-1, 1), b


def test_scene_representation_glue_against_the_reference(ref):
    """The reference's HumanRF.density / forward and Decomposition4D.forward (humanrf.py:158-208, decomposition4d.py:124-135)
    as run with every tcnn module and the composition extension answering through the ORACLE's restatement of that one
    module, against the oracle.  What is compared is therefore the glue the oracle restates around them: frame -> segment
    routing, the +0.5 shift, local time, grid axis selection (xyz, xyt, yzt, xzt), composition call,
    truncated_exp * density_scale, geometry-feature slicing, (d+1)/2, camera embeddings while training / zeros
    otherwise.  The reference stores the composed features in fp16, hence the tolerances."""
    arrays = ref[1]
    om, pos, dirs, fr, cams, b = scene_glue_inputs()
    touched = set(om.f2s[b["frames"].numpy()].tolist())
    assert len(touched) == 3                                                 # all three segments are exercised
    rows = torch.from_numpy(arrays["scene_rows"])
    assert rows.numel() == SCENE_ROWS
    radiance = {}
    for is_training in (True, False):
        tag = "train" if is_training else "eval"
        with torch.no_grad():
            sigma, geo, rgb = om.forward(pos, dirs, fr.view(-1), cams.view(-1) if is_training else None)
        assert ref[0]["scene_shapes"][tag] == [list(sigma.shape), [pos.shape[0], 15], list(rgb.shape)]
        density, geometry, radiance[tag] = (torch.from_numpy(arrays[f"scene_{tag}_{k}"]) for k in ("density", "geometry", "radiance"))
        rel = ((density - sigma[rows]).abs() / sigma[rows].abs().clamp_min(1e-3)).max().item()
        dg = (geometry.float() - geo[rows]).abs().max().item()
        dc = (radiance[tag] - rgb[rows]).abs().max().item()
        print(f"is_training={is_training}: density rel {rel:.2e}, geometry abs {dg:.2e}, radiance abs {dc:.2e}")
        assert rel < 2e-3 and dg < 2e-3 and dc < 1e-3       # measured 5e-5 / 5e-5 / 5e-6 (the fp16 feature buffer)
    # the embedding really is dropped at evaluation: the two passes differ in radiance only
    assert (radiance["eval"] - radiance["train"]).abs().max() > 1e-3
