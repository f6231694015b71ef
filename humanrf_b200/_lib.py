"""ctypes binding of libhumanrf_b200.so (the C ABI declared in include/humanrf_b200.h).

The product path has NO fallback: if the shared library is missing or fails to load, every
entry point raises (``lib()`` raises ``RuntimeError``).  PyTorch is used only for device
memory and streams; tensors cross the boundary as raw device pointers.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libhumanrf_b200.so"
N_LEVELS = 16
MLP_BLOB_BYTES = 22528

vp, i64, i32, u32, u64, f32 = C.c_void_p, C.c_int64, C.c_int32, C.c_uint32, C.c_uint64, C.c_float


class SamplerParams(C.Structure):
    _fields_ = [("frame_numbers", vp), ("camera_numbers", vp), ("grid_handles", vp), ("landscape_modes", vp),
                ("inverse_krs", vp), ("camera_origins", vp), ("aabb", vp), ("rgba_pool", vp), ("light_mask", vp), ("light_mask_rays", vp),
                ("grid_resolution", i32), ("image_width", i32), ("image_height", i32), ("step", f32),
                ("occupancy", i32), ("filter_light_bloom", i32), ("want_samples", i32)]


class Segment(C.Structure):
    _fields_ = [("grid", vp * 4), ("vectors", vp), ("level_offset", u32 * N_LEVELS), ("level_size", u32 * N_LEVELS),
                ("hashed_mask", u32), ("n_entries", u32), ("vectors_t", vp)]


class Field(C.Structure):
    _fields_ = [("segments", vp), ("frame_to_segment", vp), ("frame_to_tlocal", vp), ("mlp_blob", vp),
                ("level_scale", f32 * N_LEVELS), ("level_res", u32 * N_LEVELS), ("num_segments", i32),
                ("lut_size", i32), ("vec_res", i32), ("density_scale", f32), ("camera_embeddings", vp),
                ("camera_embedding_dim", i32), ("num_cameras", i32), ("color_in_width", i32)]


class Samples(C.Structure):
    _fields_ = [("positions", vp), ("directions", vp), ("frame_numbers", vp), ("ray_origins", vp),
                ("ray_directions", vp), ("ray_frame_numbers", vp), ("sample_distances", vp), ("ray_indices", vp),
                ("num_samples", i64), ("camera_numbers", vp), ("ray_camera_numbers", vp), ("use_camera_embeddings", i32),
                ("num_samples_dev", vp)]


class SegmentGrads(C.Structure):
    _fields_ = [("grid", vp * 4), ("vectors", vp)]


class AdamTensor(C.Structure):
    _fields_ = [("param", vp), ("exp_avg", vp), ("exp_avg_sq", vp), ("grad", vp), ("shadow_bf16", vp), ("blob_perm", vp),
                ("active", vp), ("step", vp), ("n", i64), ("first_block", i64), ("vectors_t", vp), ("vec_res", i32)]


ADAM_BLOCK_ELEMS = 4096
DP_MAX_WORLD = 8


class DpPeers(C.Structure):
    _fields_ = [("grad", vp * DP_MAX_WORLD), ("shadow", vp * DP_MAX_WORLD), ("world", i32), ("rank", i32)]


class DpTensor(C.Structure):
    _fields_ = [("param", vp), ("exp_avg", vp), ("exp_avg_sq", vp), ("grad_offset", i64), ("shadow_offset", i64),
                ("local_shadow_bf16", vp), ("blob_perm", vp), ("active", vp), ("step", vp), ("n", i64),
                ("shard_begin", i64), ("shard_end", i64), ("first_block", i64), ("sharded", i32), ("vec_res", i32),
                ("vectors_t", vp)]


_SIGNATURES = {
    "hrf_last_error": (C.c_char_p, []),
    "hrf_version": (C.c_int, []),
    "hrf_device_info": (C.c_int, [C.POINTER(C.c_int)]),
    "hrf_occgrid_create": (C.c_int, [u64, C.c_int, C.POINTER(vp)]),
    "hrf_occgrid_destroy": (C.c_int, [vp]),
    "hrf_occgrid_add": (C.c_int, [vp, vp, u64, u64, u64, vp, C.POINTER(i64)]),
    "hrf_occgrid_lookup": (C.c_int, [i64, C.c_int, vp, i64, vp, vp]),
    "hrf_sampler_rays": (C.c_int, [C.POINTER(SamplerParams), vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp]),
    "hrf_sampler_workspace_bytes": (i64, [i64]),
    "hrf_sampler_samples": (C.c_int, [C.POINTER(SamplerParams), i64, vp, vp, vp, vp, vp, vp, vp, vp]),
    "hrf_field_forward": (C.c_int, [C.POINTER(Field), C.POINTER(Samples), C.c_int, C.c_int, vp, vp, vp, vp, vp, vp]),
    "hrf_field_forward_from_features": (C.c_int, [C.POINTER(Field), C.POINTER(Samples), vp, vp, vp, vp, vp]),
    "hrf_render_fused_workspace_bytes": (i64, [i64]),
    "hrf_render_fused": (C.c_int, [C.POINTER(Field), C.POINTER(Samples), vp, i64, f32, vp, vp, vp, vp, vp, vp, vp]),
    "hrf_density_early_stop_workspace_bytes": (i64, [i64]),
    "hrf_field_density_early_stop": (C.c_int, [C.POINTER(Field), C.POINTER(Samples), vp, i64, f32, f32, vp, vp, vp, vp, vp]),
    "hrf_ray_offsets": (C.c_int, [vp, i64, i64, vp, vp]),
    "hrf_prune": (C.c_int, [vp, vp, vp, vp, i64, f32, f32, f32, vp, vp, vp, vp, vp, vp, vp]),
    "hrf_composite_forward": (C.c_int, [vp, vp, vp, vp, i64, f32, vp, vp, vp, vp, vp]),
    "hrf_composite_backward": (C.c_int, [vp, vp, vp, vp, i64, f32, vp, vp, vp, vp, vp, vp]),
    "hrf_field_backward": (C.c_int, [C.POINTER(Field), C.POINTER(Samples), vp, vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp]),
    "hrf_field_backward_mlp": (C.c_int, [C.POINTER(Field), C.POINTER(Samples), vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "hrf_field_backward_tables": (C.c_int, [C.POINTER(Field), C.POINTER(Samples), vp, vp, vp, i64, vp, C.c_int, C.c_int, vp]),
    "hrf_train_loss": (C.c_int, [vp, vp, vp, vp, i64, f32, f32, vp, vp, vp, vp, vp]),
    "hrf_adam_multi": (C.c_int, [vp, C.c_int, i64, f32, f32, f32, f32, f32, C.c_int, vp]),
    "hrf_peer_alloc": (C.c_int, [i64, C.POINTER(vp)]),
    "hrf_peer_free": (C.c_int, [vp]),
    "hrf_peer_export": (C.c_int, [vp, vp]),
    "hrf_peer_open": (C.c_int, [vp, C.POINTER(vp)]),
    "hrf_peer_close": (C.c_int, [vp]),
    "hrf_dp_reduce_adam": (C.c_int, [C.POINTER(DpPeers), vp, C.c_int, i64, i64, C.c_int, f32, f32, f32, f32, f32, vp]),
    "hrf_compose_tensors_forward": (C.c_int, [vp, vp, vp, vp, vp, vp, i64, C.c_int, C.c_int, vp, vp]),
    "hrf_compose_tensors_backward": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, i64, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp]),
    "hrf_adam_step": (C.c_int, [vp, vp, vp, vp, vp, i64, f32, f32, f32, f32, C.c_int, f32, vp]),
    "hrf_cast_bf16": (C.c_int, [vp, vp, i64, vp]),
    "hrf_transpose_vectors": (C.c_int, [vp, vp, C.c_int, vp]),
    "hrf_occupancy_from_masks": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]),
    "hrf_occupancy_union_count": (C.c_int, [vp, vp, i64, vp, vp]),
    "hrf_mask_bbox": (C.c_int, [vp, C.c_int, C.c_int, vp, vp]),
    "hrf_image_metrics_workspace_bytes": (i64, [C.c_int, C.c_int]),
    "hrf_image_metrics": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, i64, vp, f32, vp, C.c_int, vp, vp, vp]),
    "hrf_selftest_umma": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, u32, u32, u32, u32, u32, u32, u32, u32,
                                    C.c_int, vp]),
}

_lib = None


def exported_symbols():
    """Names every C-ABI entry point include/humanrf_b200.h declares (used by the CPU test)."""
    return sorted(_SIGNATURES)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m humanrf_b200.build` "
                "(there is no CPU or PyTorch fallback for the hot path)")
        handle = C.CDLL(str(LIB_PATH), mode=os.RTLD_LOCAL if hasattr(os, "RTLD_LOCAL") else 0)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int) -> None:
    """Mirror of the reference's std::runtime_error -> Python RuntimeError convention."""
    if rc != 0:
        msg = lib().hrf_last_error()
        raise RuntimeError(f"humanrf_b200: {msg.decode() if msg else 'error'} (code {rc})")


def ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def require_cuda(t: torch.Tensor, name: str, dtype=None) -> torch.Tensor:
    """CHECK_CONTIGUITY_AND_DEVICE (actorshq/toolbox/native/utils.cuh:5-19)."""
    if not t.is_contiguous():
        raise RuntimeError(f"Tensor not contiguous: {name}")
    if t.device.type != "cuda":
        raise RuntimeError(f"Tensor is not on the expected device: {name}")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"Tensor {name} has dtype {t.dtype}, expected {dtype}")
    return t
