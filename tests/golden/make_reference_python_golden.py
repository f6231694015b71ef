"""Writes tests/golden/reference_python.json and reference_python.npz: the reference's answers for the inputs of
tests/test_reference_live_cpu.py (and the module list test_host_cpu.py checks the drop-in against), computed by
IMPORTING a reference checkout read-only and running its first-party Python on the CPU.

    HUMANRF_REFERENCE=/path/to/humanrf python tests/golden/make_reference_python_golden.py

tinycudann and nerfacc are not needed: tcnn is replaced by a stub that records the configs it is built with, nerfacc
and the tcnn modules' forward passes by the oracle's restatement (as described in each test)."""
import contextlib
import io
import json
import os
import re
import sys
import types
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
REF = Path(os.environ["HUMANRF_REFERENCE"]).resolve()
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]

import test_reference_live_cpu as T  # noqa: E402  (the tests' input builders)
from humanrf_b200.scene_representation.grid_layout import GridLayout, MLP_SIGMA_PARAMS, mlp_color_params  # noqa: E402
from humanrf_b200.synthetic import MODEL_KW  # noqa: E402
from oracle import field as OF  # noqa: E402
from oracle import hashgrid  # noqa: E402
from oracle import rendering as R  # noqa: E402

sys.path.insert(0, str(REF))
# adaptive_temporal_partitioning imports VolumetricDataset only for an annotation (needs cv2 etc.): stub it
_vd = types.ModuleType("actorshq.dataset.volumetric_dataset")
_vd.VolumetricDataset = object
sys.modules["actorshq.dataset.volumetric_dataset"] = _vd
import actorshq.dataset.input_batch as ref_ib  # noqa: E402
import humanrf.adaptive_temporal_partitioning as ref_atp  # noqa: E402
import humanrf.input as ref_input  # noqa: E402
import humanrf.scene_representation.query_io as ref_qio  # noqa: E402
import humanrf.utils.activation as ref_act  # noqa: E402
import humanrf.utils.loss as ref_loss  # noqa: E402

doc, arrays = {}, {}

# ---- module paths (what the drop-in maps must exist in the reference)
mods = {".".join(p.relative_to(REF).with_suffix("").parts) for pkg in ("humanrf", "actorshq") for p in (REF / pkg).rglob("*.py")
        if "third_party" not in p.parts and p.name != "setup.py"}
for setup in (REF / "humanrf" / "setup.py", REF / "actorshq" / "setup.py"):
    mods |= set(re.findall(r'CUDAExtension\(\s*name="([\w.]+)"', setup.read_text()))
doc["modules"] = sorted(mods)

# ---- dataclass surfaces
doc["surfaces"] = {c.__name__: list(T.surface(c)) for c in (ref_ib.InputBatch, ref_qio.QueryInput, ref_qio.QueryOutput)}

# ---- merge_input_batches
doc["merge"] = []
for case, batches, budget, _ in T.merge_cases(ref_ib.InputBatch):
    out = ref_input.merge_input_batches(batches, budget)
    doc["merge"].append({"fields": T.merged_fields(out), "size": [out.width, out.height]})

# ---- truncated_exp / bce_loss
for scale, x, dy in T.truncated_exp_inputs():
    if scale == "bce":
        arrays["bce_out"] = ref_loss.bce_loss(x, dy).numpy()
        continue
    xi = x.clone().requires_grad_(True)
    y = ref_act.truncated_exp(xi)
    y.backward(dy)
    arrays[f"texp_{scale:g}_y"], arrays[f"texp_{scale:g}_dx"] = y.detach().numpy(), xi.grad.numpy()


# ---- adaptive temporal partitioning
class _DS:
    def __init__(self, grids):
        self.grids = grids

    def get_occupancy_grid(self, frame_number):
        return self.grids[frame_number].copy()       # the reference ORs into the first grid of a cluster in place


sizes = []
for grids, thr in T.partitioning_cases():
    with contextlib.redirect_stderr(io.StringIO()):      # tqdm bar
        sizes.append([int(s) for s in ref_atp.compute_adaptive_segment_sizes(_DS(grids), list(range(len(grids))), thr)])
doc["partitioning"] = {"predefined": list(ref_atp.PREDEFINED_SEGMENT_SIZES),
                       "segment_size": [ref_atp.get_segment_size(n) for n in range(1, 260)],
                       "final_segment_size": [ref_atp.get_final_segment_size(n) for n in range(1, 260)], "sizes": sizes}

# ---- the reference's HumanRF with tinycudann replaced by a recording stub (parameter sizes follow our layout rule, so
#      the sizes of tcnn tensors are not evidence; the configs, names and first-party tensors are)
calls = []


class _Flat(torch.nn.Module):
    def __init__(self, n):
        super().__init__()
        self.params = torch.nn.Parameter(torch.zeros(n))


class Encoding(_Flat):
    def __init__(self, n_input_dims, encoding_config, **kw):
        calls.append(["Encoding", n_input_dims, dict(encoding_config)])
        c = encoding_config
        fin = c["base_resolution"] * c["per_level_scale"] ** (c["n_levels"] - 1)
        super().__init__(GridLayout(c["log2_hashmap_size"], c["n_levels"], c["base_resolution"], int(round(fin))).n_params)


class Network(_Flat):
    def __init__(self, n_input_dims, n_output_dims, network_config, **kw):
        calls.append(["Network", n_input_dims, n_output_dims, dict(network_config)])
        super().__init__(MLP_SIGMA_PARAMS)


class NetworkWithInputEncoding(_Flat):
    def __init__(self, n_input_dims, n_output_dims, encoding_config, network_config, **kw):
        calls.append(["NetworkWithInputEncoding", n_input_dims, n_output_dims, dict(encoding_config), dict(network_config)])
        super().__init__(mlp_color_params(n_input_dims - 18))


tcnn = types.ModuleType("tinycudann")
tcnn.Encoding, tcnn.Network, tcnn.NetworkWithInputEncoding = Encoding, Network, NetworkWithInputEncoding
sys.modules["tinycudann"] = tcnn
sys.modules["humanrf.scene_representation.tensor_composition_native"] = types.ModuleType("tensor_composition_native")
nerfacc = types.ModuleType("nerfacc")
nerfacc.render_visibility = lambda alphas, ray_indices, early_stop_eps, alpha_thre, n_rays: \
    R.render_visibility(alphas, ray_indices, early_stop_eps, alpha_thre)


def render_weight_from_density(t_starts, t_ends, sigmas, ray_indices, n_rays):
    sdt = sigmas.reshape(-1) * (t_ends - t_starts).reshape(-1)
    return (torch.exp(-R._exclusive_by_ray(sdt, ray_indices, "sum")) * (1.0 - torch.exp(-sdt))).unsqueeze(-1)


nerfacc.render_weight_from_density = render_weight_from_density
nerfacc.accumulate_along_rays = lambda weights, ray_indices, values=None, n_rays=None: R.accumulate(weights, ray_indices, values, n_rays)
sys.modules["nerfacc"] = nerfacc
import humanrf.scene_representation.decomposition4d as d4  # noqa: E402
import humanrf.scene_representation.humanrf as ref_model  # noqa: E402
import humanrf.volume_rendering as vr  # noqa: E402

doc["model"] = {}
for segment_sizes, first, count, cam_emb in T.MODEL_CASES:
    calls.clear()
    key = T.model_case_key(segment_sizes, first, count, cam_emb)
    m = ref_model.HumanRF(sorted_frame_numbers=tuple(range(first, first + count)), segment_sizes=segment_sizes,
                          **T.model_kwargs(cam_emb))
    for name in ("frame_numbers_to_segment_numbers", "frame_numbers_to_normalized_local_frame_numbers"):
        arrays[f"model_{key}_{name}"] = getattr(m, name).numpy()
    doc["model"][key] = {"scalars": [m.num_frames, m.num_segments, m.total_feature_dim, m.density_scale],
                         "calls": json.loads(json.dumps(calls)),
                         "state_dict": [[k, list(v.shape), str(v.dtype)] for k, v in m.state_dict().items()],
                         "param_groups": [[len(list(g["params"])), g["lr"]] for g in m.get_params(1e-2)]}

# ---- prune_samples / render / merge_render_outputs with nerfacc answered by the oracle
b = T.prune_render_rays()
o, d, fr, ri = b["o"], b["d"], b["frames"].view(-1, 1), b["ri"]
scene = T.closed_form_scene(ref_qio.QueryOutput)
bg = T.prune_render_background()
for is_training in (False, True):
    tag = "train" if is_training else "eval"
    ib = ref_ib.InputBatch(ray_origins=o, ray_directions=d, frame_numbers=fr, unique_frame_numbers=torch.unique(fr).view(-1, 1),
                           camera_numbers=torch.zeros_like(fr), sample_distances=b["t"].clone().view(-1, 1), ray_indices=ri.clone(),
                           rgba=b["rgba"], width=8, height=8)
    torch.manual_seed(5)
    vr.prune_samples(ib, scene, is_training=is_training)
    out = vr.render(ib, scene, bg, is_training=is_training)
    nobg = vr.render(ib, scene, None, is_training=is_training)
    arrays.update({f"render_{tag}_t": ib.sample_distances.numpy(), f"render_{tag}_ri": ib.ray_indices.numpy(),
                   f"render_{tag}_color": out.color.numpy(), f"render_{tag}_wsum": out.weights_sum.numpy(),
                   f"render_{tag}_color_nobg": nobg.color.numpy()})
merged = vr.RenderOutput.merge_render_outputs([vr.RenderOutput(color=a, weights_sum=w) for a, w in T.merge_render_parts()])
arrays["merge_color"], arrays["merge_wsum"] = merged.color.numpy(), merged.weights_sum.numpy()
try:
    vr.RenderOutput.merge_render_outputs([vr.RenderOutput(color=torch.rand(2, 3))])
    raise SystemExit("the reference's merge_render_outputs accepted a field that is not a tensor")
except RuntimeError as e:
    doc["merge_render_outputs_error"] = str(e)

# ---- HumanRF.density / forward with the tcnn modules and the composition extension answered by the oracle
om, pos, dirs, fr, cams, b = T.scene_glue_inputs()
frames = tuple(range(15, 15 + sum(T.SCENE_SIZES)))
calls.clear()
theirs = ref_model.HumanRF(sorted_frame_numbers=frames, segment_sizes=T.SCENE_SIZES, **{**MODEL_KW, "camera_embedding_dim": T.SCENE_EMB})
d4.Decomposition4D.to = lambda self, *a, **k: self                       # the reference parks idle segments on the CPU
d4.tensor_composition_native.compose_tensors_forward = \
    lambda xyz, xyt, yzt, xzt, vectors, coords: OF.compose(xyz.float(), xyt.float(), yzt.float(), xzt.float(), vectors, coords).half()
for s, fg in enumerate(theirs.feature_grids):
    with torch.no_grad():
        fg.vectors.copy_(om.segments[s].vectors)
    for k, name in enumerate(("xyz_encoding", "xyt_encoding", "yzt_encoding", "xzt_encoding")):
        getattr(fg, name).forward = (lambda x, s=s, k=k: hashgrid.encode(om.segments[s].grids[k], x.float(), om.segments[s].log2T).half())
theirs.sigma_net.forward = lambda f: torch.relu(f.float() @ om.w_sigma[0].t()) @ om.w_sigma[1].t()


def color_net(x):                                                        # [ (d+1)/2 | geo 15 | embedding E ] -> rgb
    dd, rest = x[:, :3].float() * 2 - 1, x[:, 3:].float()
    inp = torch.cat((OF.sh4(dd), rest, torch.ones((x.shape[0], 48 - 16 - rest.shape[1]))), dim=1)
    w1, w2, w3 = om.w_color
    h = torch.relu(torch.relu(inp @ w1.t()) @ w2.t())
    return torch.sigmoid((h @ w3.t())[:, :3])


theirs.color_net.forward = color_net
with torch.no_grad():
    theirs.camera_embeddings.weight.copy_(om.camera_embeddings)
rows = np.sort(np.random.default_rng(0).choice(pos.shape[0], T.SCENE_ROWS, replace=False))
arrays["scene_rows"] = rows.astype(np.int64)
doc["scene_shapes"] = {}
for is_training in (True, False):
    tag = "train" if is_training else "eval"
    q = ref_qio.QueryInput(is_training=is_training, positions=pos, directions=dirs, frame_numbers=fr,
                           unique_frame_numbers=torch.unique(b["frames"]).view(-1, 1), camera_numbers=cams)
    with torch.no_grad():
        out, dens = theirs(q), theirs.density(q)
    assert torch.equal(out.density, dens.density)
    doc["scene_shapes"][tag] = [list(out.density.shape), list(out.geometry_features.shape), list(out.radiance.shape)]
    arrays[f"scene_{tag}_density"] = out.density[rows].numpy()
    arrays[f"scene_{tag}_geometry"] = out.geometry_features[rows].numpy()
    arrays[f"scene_{tag}_radiance"] = out.radiance[rows].numpy()



def dumps(doc):
    """JSON with one line per entry of each top-level list or object (readable diffs, no line per number)."""
    def body(v):
        if isinstance(v, dict) and v:
            return "{\n" + ",\n".join(f"  {json.dumps(k)}: {json.dumps(x)}" for k, x in v.items()) + "\n }"
        if isinstance(v, list) and v and all(isinstance(x, (dict, list)) for x in v):
            return "[\n" + ",\n".join(f"  {json.dumps(x)}" for x in v) + "\n ]"
        return json.dumps(v)
    return "{\n" + ",\n".join(f" {json.dumps(k)}: {body(v)}" for k, v in doc.items()) + "\n}\n"


(HERE / "reference_python.json").write_text(dumps(doc))
np.savez_compressed(HERE / "reference_python.npz", **arrays)
print("wrote", HERE / "reference_python.json", HERE / "reference_python.npz", len(arrays), "arrays")
