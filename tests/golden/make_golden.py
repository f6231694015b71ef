"""Generates tests/golden/reference_host.npz by IMPORTING the reference (the checkout HUMANRF_REFERENCE
names, read-only) and running its pure-torch first-party functions on seeded inputs:

  humanrf/input.py:10-55                 merge_input_batches (incl. the sample-budget cut-off)
  humanrf/utils/activation.py:6-39       truncated_exp forward / backward
  humanrf/utils/loss.py:4-10             bce_loss
  actorshq/dataset/camera_data.py:93-102 projection_matrix_world2pixel -> inverse_krs (data_loader.py:194-207)

Run:  HUMANRF_REFERENCE=/path/to/humanrf python tests/golden/make_golden.py
"""
import os
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, os.environ["HUMANRF_REFERENCE"])
from actorshq.dataset.camera_data import CameraData  # noqa: E402
from actorshq.dataset.input_batch import InputBatch  # noqa: E402
from humanrf.input import merge_input_batches  # noqa: E402
from humanrf.utils.activation import truncated_exp  # noqa: E402
from humanrf.utils.loss import bce_loss  # noqa: E402

OUT = Path(__file__).resolve().parent / "reference_host.npz"
g = torch.Generator().manual_seed(123)
data = {}


def make_batch(num_rays, masked, seed):
    gg = torch.Generator().manual_seed(seed)
    counts = torch.randint(0, 7, (num_rays,), generator=gg)
    ri = torch.repeat_interleave(torch.arange(num_rays), counts)
    n = int(counts.sum())
    mask = torch.ones(num_rays + masked, 1, dtype=torch.bool)
    mask[torch.randperm(num_rays + masked, generator=gg)[:masked]] = False
    fr = torch.randint(15, 23, (num_rays, 1), generator=gg, dtype=torch.int32)
    return InputBatch(
        ray_origins=torch.randn(num_rays, 3, generator=gg), ray_directions=torch.randn(num_rays, 3, generator=gg),
        minmaxes=torch.rand(num_rays, 2, generator=gg), rgba=torch.rand(num_rays, 4, generator=gg), ray_masks=mask,
        frame_numbers=fr, unique_frame_numbers=torch.unique(fr).view(-1, 1),
        camera_numbers=torch.randint(0, 160, (num_rays, 1), generator=gg, dtype=torch.int32),
        sample_distances=torch.rand(n, 1, generator=gg), ray_indices=ri.long(), width=64, height=48)


FIELDS = ["ray_origins", "ray_directions", "minmaxes", "rgba", "ray_masks", "frame_numbers", "unique_frame_numbers",
          "camera_numbers", "sample_distances", "ray_indices"]
cases = {"a": ([(11, 3, 1), (7, 2, 2), (13, 0, 3)], None), "b": ([(11, 3, 1), (7, 2, 2), (13, 0, 3)], 40),
         "c": ([(5, 0, 9)], 3), "d": ([(9, 4, 4), (9, 1, 5)], 10 ** 6)}
for name, (specs, budget) in cases.items():
    batches = [make_batch(*s) for s in specs]
    for bi, b in enumerate(batches):
        for f in FIELDS:
            data[f"merge_{name}_in{bi}_{f}"] = getattr(b, f).numpy()
    data[f"merge_{name}_nb"] = np.array(len(batches))
    data[f"merge_{name}_budget"] = np.array(-1 if budget is None else budget)
    out = merge_input_batches(batches, budget)
    for f in FIELDS:
        v = getattr(out, f)
        data[f"merge_{name}_out_{f}"] = (torch.sort(v.reshape(-1))[0] if f == "unique_frame_numbers" else v).numpy()

x = (torch.randn(257, generator=g) * 9).requires_grad_(True)
y = truncated_exp(x)
dy = torch.randn(257, generator=g)
y.backward(dy)
data["texp_x"], data["texp_y"], data["texp_dy"], data["texp_dx"] = x.detach().numpy(), y.detach().numpy(), dy.numpy(), x.grad.numpy()

pred = torch.rand(301, 1, generator=g) * 1.4 - 0.2
target = (torch.rand(301, 1, generator=g) > 0.5).float()
data["bce_pred"], data["bce_target"], data["bce_out"] = pred.numpy(), target.numpy(), bce_loss(pred, target).numpy()

rot = torch.randn(6, 3, generator=g).numpy()
cams, invs = [], []
for i in range(6):
    cam = CameraData(name=f"c{i}", width=1028, height=752, rotation_axisangle=rot[i] * 0.7,
                     translation=np.array([2.0 * np.cos(i), 0.3 * i - 0.5, 2.0 * np.sin(i)]),
                     focal_length=np.array([1.773863, 1.773863 * 1028 / 752]), principal_point=np.array([0.5, 0.5]))
    cams.append(np.concatenate([cam.rotation_axisangle, cam.translation]))
    invs.append(np.linalg.inv(cam.projection_matrix_world2pixel()))
data["cam_params"] = np.stack(cams)
# data_loader.py:194-207 : inv(world2pixel)[:3,:3] transposed, float32
data["cam_inverse_krs"] = np.stack(invs)[..., :3, :3].transpose(0, 2, 1).astype(np.float32)
data["cam_world2pixel_inv_full"] = np.stack(invs)

np.savez_compressed(OUT, **data)
print("wrote", OUT, len(data), "arrays")
