"""Writes tests/golden/reference_cuda.npz: what the reference's own CUDA extensions return for the inputs of the GPU
tests that compare with them (test_ref_parity_gpu.py, test_occupancy_tools_gpu.py::test_carve_vs_reference_extension).
The extensions are the builds of the reference's unmodified sources that oracle/build_ref.py leaves in oracle/_ref/.
Needs a CUDA device:

    HUMANRF_REFERENCE=/path/to/humanrf python oracle/build_ref.py        # once, where the reference checkout is
    python tests/golden/make_reference_cuda_golden.py [OUT.npz]           # on the GPU machine

Outputs too large to store whole are sampled at the strides the tests read them with."""
import importlib
import sys
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests"), str(ROOT / "oracle" / "_ref")]

import test_occupancy_tools_gpu as TO  # noqa: E402
import test_ref_parity_gpu as TP  # noqa: E402

dev = torch.device("cuda:0")
out = {}

# ---- visual-hull carving: 0 / 255 per voxel, stored as a bit mask of the occupied voxels
carve = importlib.import_module("occupancy_grid_generation_native")
args = TO.reference_carve_args(dev)
G = args[4]
grid = carve.generate_from_masks(*args).cpu().numpy()
assert grid.shape == (G, G, G) and grid.dtype == np.uint8 and set(np.unique(grid).tolist()) <= {0, 255}
out["carve_occupied_bits"] = np.packbits(grid.reshape(-1) == 255)

# ---- tensor composition, forward and backward
compose = importlib.import_module("tensor_composition_native")
feats, vec, coords, dout = TP.compose_inputs(dev)
res = [compose.compose_tensors_forward(*feats, vec, coords), *compose.compose_tensors_backward(*feats, vec, coords, dout)[:5]]
for name, x in zip(("fwd", "bwd0", "bwd1", "bwd2", "bwd3", "bwd4"), res):
    out[f"compose_{name}_shape"] = np.asarray(x.shape, np.int64)
    out[f"compose_{name}_dtype"] = np.asarray(str(x.dtype))
    stride = TP.VECTOR_GRAD_STRIDE if name == "bwd4" else TP.COMPOSE_STRIDE
    out[f"compose_{name}"] = x.reshape(-1)[::stride].cpu().numpy()
out["compose_bwd4_absmax"] = np.asarray(res[5].abs().max().item(), np.float32)

# ---- ray sampler over the reference's texture-backed occupancy grid
sampler, occ = importlib.import_module("ray_sampler_native"), importlib.import_module("occupancy_grid_native")
sc, grids_dev, head, tail = TP.sampler_inputs(dev)
rog = occ.OccupanyGrid(sc["G"], len(grids_dev))
rh = torch.tensor([rog.add_grid(g) for g in grids_dev], dtype=torch.int64, device=dev)
a = [x.cpu() for x in sampler.get_samples_occupancy_minmax(*head, rh, *tail)]
kept = int(a[6].sum())
rgba_u8 = torch.round(a[2] * 255.0).to(torch.uint8)
assert torch.equal(rgba_u8.float() / 255.0, a[2])                      # rgba[kept] / 255.0 is recovered exactly
out.update(sampler_mask_bits=np.packbits(a[6].numpy()), sampler_dirs=a[1].numpy(), sampler_minmax=a[5].numpy(),
           sampler_rgba_u8=rgba_u8.numpy(), sampler_frame_numbers=a[3].numpy(),
           sampler_counts=np.bincount(a[8].numpy(), minlength=kept).astype(np.int32),
           sampler_num_samples=np.asarray(a[7].numel(), np.int64),
           sampler_dtypes=np.asarray([str(a[i].dtype) for i in (6, 7, 8)]))
del rog

dst = Path(sys.argv[1]) if len(sys.argv) > 1 else HERE / "reference_cuda.npz"
dst.parent.mkdir(parents=True, exist_ok=True)
np.savez_compressed(dst, **out)
print("wrote", dst, {k: v.shape for k, v in out.items()})
