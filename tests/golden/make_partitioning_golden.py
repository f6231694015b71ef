"""Generates tests/golden/partitioning.npz by running the REFERENCE's compute_adaptive_segment_sizes
(humanrf/adaptive_temporal_partitioning.py of the reference checkout HUMANRF_REFERENCE names) on synthetic occupancy
sequences.  Run:  HUMANRF_REFERENCE=/path/to/humanrf python tests/golden/make_partitioning_golden.py"""
import os
import sys
import types
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, os.environ["HUMANRF_REFERENCE"])
sys.path.insert(0, str(HERE.parent.parent))
# the reference module imports VolumetricDataset only for a type annotation; avoid its heavy imports
stub = types.ModuleType("actorshq.dataset.volumetric_dataset")
stub.VolumetricDataset = object
for name in ("actorshq", "actorshq.dataset"):
    sys.modules.setdefault(name, types.ModuleType(name))
sys.modules["actorshq.dataset.volumetric_dataset"] = stub
from humanrf.adaptive_temporal_partitioning import compute_adaptive_segment_sizes  # noqa: E402

sys.path.insert(0, str(HERE.parent))
from scene import occupancy_sequence  # noqa: E402


class _DS:
    def __init__(self, grids):
        self.grids = grids

    def get_occupancy_grid(self, frame_number):
        return self.grids[frame_number].copy()      # the reference mutates the first grid of a cluster in place


out = {}
cases = [("slow", 130, 0.002, 1.25), ("fast", 90, 0.02, 1.25), ("burst", 160, None, 1.25), ("tight", 70, 0.006, 1.05),
         ("short", 5, 0.01, 1.25), ("exact", 100, 0.0, 1.25)]
for name, n, speed, thr in cases:
    grids = occupancy_sequence(n, speed, G=48, seed=len(name) * 7 + n)
    sizes = compute_adaptive_segment_sizes(_DS(grids), list(range(n)), thr)
    out[name + "_sizes"] = np.asarray(sizes, np.int32)
    out[name + "_args"] = np.asarray([n, -1.0 if speed is None else speed, thr, len(name) * 7 + n], np.float64)
    print(name, sizes)
np.savez_compressed(HERE / "partitioning.npz", **out)
