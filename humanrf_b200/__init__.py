"""humanrf_b200 -- B200-native (sm_100a) implementation of HumanRF's per-ray hot path.

Host-side mirror of the reference's interfaces for that path (same names, argument meaning and
error behaviour) on top of the C ABI in include/humanrf_b200.h:

  reference module                                        here
  humanrf/scene_representation/{humanrf,query_io}.py   -> humanrf_b200.scene_representation
  humanrf/volume_rendering.py                          -> humanrf_b200.volume_rendering
  humanrf/input.py, actorshq/dataset/input_batch.py    -> humanrf_b200.input, humanrf_b200.dataset.input_batch
  actorshq/dataset/native/ray_sampler.cu  (pybind)     -> humanrf_b200.dataset.ray_sampler_native
  actorshq/dataset/native/occupancy_grid.cu (pybind)   -> humanrf_b200.dataset.occupancy_grid_native
  humanrf/scene_representation/native/tensor_composition.cu -> humanrf_b200.scene_representation.tensor_composition_native
  humanrf/utils/{activation,loss}.py                   -> humanrf_b200.utils
  actorshq/evaluation/evaluate.py (PSNR, SSIM)         -> humanrf_b200.evaluation.evaluate
"""
__version__ = "0.1.0"
