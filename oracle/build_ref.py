"""TEST INFRASTRUCTURE ONLY.  Compiles the reference's own first-party CUDA extensions from the
sources where they lie in the reference checkout named by HUMANRF_REFERENCE (nothing is copied) into
oracle/_ref/, so that tests/golden/make_reference_cuda_golden.py can record what the real thing computes:

  tensor_composition_native  <- humanrf/scene_representation/native/tensor_composition.cu
  occupancy_grid_native      <- actorshq/dataset/native/occupancy_grid.cu
  ray_sampler_native         <- actorshq/dataset/native/ray_sampler.cu   (+ oracle/glm_shim: GLM is absent here)
  occupancy_grid_generation_native <- actorshq/toolbox/native/occupancy_grid_generation.cu   (+ oracle/glm_shim)

Flags follow humanrf/setup.py:17 and actorshq/setup.py:17-29 (--use_fast_math) with the arch
pinned to sm_100.  tinycudann / nerfacc are not part of the reference checkout and cannot be built.
Run:  HUMANRF_REFERENCE=/path/to/humanrf python oracle/build_ref.py   (a few minutes per extension; skipped when up to date)
"""
from __future__ import annotations

import os
import shutil
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
OUT = HERE / "_ref"

EXTS = {
    "tensor_composition_native": ("humanrf/scene_representation/native/tensor_composition.cu", []),
    "occupancy_grid_native": ("actorshq/dataset/native/occupancy_grid.cu", []),
    "ray_sampler_native": ("actorshq/dataset/native/ray_sampler.cu", [HERE / "glm_shim"]),
    "occupancy_grid_generation_native": ("actorshq/toolbox/native/occupancy_grid_generation.cu", [HERE / "glm_shim"]),
}


def build(names=None, verbose=False):
    ref = os.environ.get("HUMANRF_REFERENCE")
    if not ref or not Path(ref).is_dir():
        print("HUMANRF_REFERENCE does not name a reference checkout; skipping oracle/_ref build")
        return {}
    ref = Path(ref)
    os.environ["TORCH_CUDA_ARCH_LIST"] = "10.0"
    from torch.utils.cpp_extension import load  # noqa: WPS433

    OUT.mkdir(exist_ok=True)
    built = {}
    for name, (rel, extra_inc) in EXTS.items():
        if names and name not in names:
            continue
        src = ref / rel
        final = OUT / f"{name}.so"
        if final.exists() and final.stat().st_mtime >= src.stat().st_mtime:
            built[name] = final
            continue
        bdir = OUT / f"_build_{name}"
        bdir.mkdir(exist_ok=True)
        try:
            load(name=name, sources=[str(src)], build_directory=str(bdir),
                 extra_include_paths=[str(ref / "actorshq/toolbox/native")] + [str(p) for p in extra_inc],
                 extra_cuda_cflags=["--use_fast_math"], is_python_module=False, verbose=verbose)
            shutil.copy(bdir / f"{name}.so", final)
            built[name] = final
            print("built", final)
        except Exception as e:  # noqa: BLE001
            print(f"could not build {name}: {e}", file=sys.stderr)
        shutil.rmtree(bdir, ignore_errors=True)
    return built


if __name__ == "__main__":
    build(sys.argv[1:] or None, verbose=True)
