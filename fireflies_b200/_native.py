"""ctypes binding of ``libffb200.so`` (see ``include/ffb200.h``).

There is NO CPU fallback: every function here raises if the shared library is missing or a tensor is
not a contiguous CUDA tensor of the expected dtype.  PyTorch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FFB_LIB") or os.path.join(_HERE, "_lib", "libffb200.so")   # FFB_LIB: kernel A/B builds (scripts/ab_build.py)

FFB_MAX_MESHES = 32
MODE_TRAIN, MODE_EVAL, MODE_INJECTED = 0, 1, 2
SAMPLER_UNIFORM, SAMPLER_SCALAR_TO_VEC3, SAMPLER_GAUSSIAN = 0, 1, 2
ENTITY_PLAIN, ENTITY_MESH = 0, 1


class SplatDesc(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("ts0", C.c_int32), ("ts1", C.c_int32),
                ("sigma", C.c_float), ("num_std_sum", C.c_int32), ("num_std_softor", C.c_int32),
                ("pts_batch_stride", C.c_int64)]


class Sampler(C.Structure):
    _fields_ = [("kind", C.c_int32), ("dim", C.c_int32), ("aliased", C.c_int32), ("step", C.c_float),
                ("vmin", C.c_float * 3), ("vmax", C.c_float * 3), ("cur", C.c_float * 3),
                ("mean", C.c_float * 3), ("std", C.c_float * 3)]


class Entity(C.Structure):
    _fields_ = [("kind", C.c_int32), ("parent", C.c_int32), ("randomizable", C.c_int32),
                ("s_translation", C.c_int32), ("s_rotation", C.c_int32), ("s_scale", C.c_int32),
                ("centroid", C.c_float * 3), ("_pad", C.c_float), ("world", C.c_float * 16)]


class MeshTable(C.Structure):
    _fields_ = [("M", C.c_int32), ("voff", C.c_int32 * (FFB_MAX_MESHES + 1)), ("entity", C.c_int32 * FFB_MAX_MESHES),
                ("nframes", C.c_int32 * FFB_MAX_MESHES), ("frames", C.c_void_p * FFB_MAX_MESHES)]


class PostDesc(C.Structure):
    _fields_ = [("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("blur_ky", C.c_int32), ("blur_kx", C.c_int32),
                ("blur_sy", C.c_float), ("blur_sx", C.c_float), ("noise", C.c_int32), ("noise_mean", C.c_float),
                ("noise_std", C.c_float), ("seed", C.c_uint64), ("frame0", C.c_uint64)]


class PerlinParams(C.Structure):
    _fields_ = [("res0", C.c_int32), ("res1", C.c_int32), ("octaves", C.c_int32), ("_pad", C.c_int32),
                ("persistence", C.c_double), ("angle_offset", C.c_int64)]


# symbol -> (restype, argtypes); the complete export list of include/ffb200.h
_P = C.c_void_p
SIGNATURES = {
    "ffb_version": (C.c_int, []),
    "ffb_last_error_string": (C.c_char_p, []),
    "ffb_splat_workspace_bytes": (C.c_size_t, [C.POINTER(SplatDesc)]),
    "ffb_splat_prepare": (C.c_int, [C.POINTER(SplatDesc), _P, _P, C.c_size_t, _P, _P]),
    "ffb_splat_fwd": (C.c_int, [C.POINTER(SplatDesc), _P, _P, _P, C.c_int, _P, _P]),
    "ffb_splat_bwd": (C.c_int, [C.POINTER(SplatDesc), _P, _P, _P, C.c_int, _P, _P, _P, _P]),
    "ffb_splat_bwd_l1": (C.c_int, [C.POINTER(SplatDesc), _P, _P, _P, C.c_int, _P, _P, _P, _P]),
    "ffb_fold_allreduce": (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P, C.c_int32, C.c_int32, C.c_uint32, _P, _P, _P]),
    "ffb_reduce_sample_groups": (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P]),
    "ffb_reduce_over_samples": (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P]),
    "ffb_splat_dense_fwd": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P]),
    "ffb_splat_dense_bwd": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P, _P]),
    "ffb_splat_dense_px_fwd": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P]),
    "ffb_splat_dense_px_bwd": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P, _P]),
    "ffb_lines_dense_fwd": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P]),
    "ffb_lines_dense_bwd": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P, _P]),
    "ffb_lines_reduce_fwd": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P, _P]),
    "ffb_lines_reduce_bwd": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P, _P, _P]),
    "ffb_depth_dense_fwd": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P]),
    "ffb_depth_dense_bwd": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P, _P, _P, _P]),
    "ffb_depth_softor_fwd": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P]),
    "ffb_l1_loss_fwd_bwd": (C.c_int, [_P, _P, C.c_int, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "ffb_sample": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_uint64, C.c_uint64, _P, _P, _P]),
    "ffb_uniform_between": (C.c_int, [_P, _P, _P, C.c_int64, _P, _P]),
    "ffb_sample_anim_index": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_uint64, C.c_uint64, _P, _P]),
    "ffb_compose_world": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.c_int32, _P, _P]),
    "ffb_transform_vertices": (C.c_int, [C.POINTER(MeshTable), _P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "ffb_transform_points": (C.c_int, [_P, C.c_int64, _P, C.c_int, _P, _P]),
    "ffb_transform_points_bwd": (C.c_int, [_P, C.c_int64, _P, C.c_int, _P, _P, _P]),
    "ffb_rays_to_ndc": (C.c_int, [_P, C.c_int32, _P, _P, _P]),
    "ffb_clamp_to_fov": (C.c_int, [_P, C.c_int32, _P, _P, C.c_float, C.c_float, _P, _P]),
    "ffb_silhouette": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P]),
    "ffb_perlin_texture": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, _P, _P, _P, _P, _P, _P]),
    "ffb_perlin_texture_batch": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_uint64, C.c_uint64, C.c_int32, _P, _P, C.c_int64,
                                           _P, _P, _P, _P, _P, _P, _P]),
    "ffb_respawn_rays": (C.c_int, [_P, C.c_int32, _P, _P, C.c_float, C.c_float, _P, C.c_uint64, C.c_uint64, _P, _P, _P]),
    "ffb_postprocess": (C.c_int, [C.POINTER(PostDesc), _P, _P, _P, _P, _P]),
    "ffb_blur_bwd": (C.c_int, [C.POINTER(PostDesc), _P, _P, _P]),
    "ffb_nurbs_curve_eval": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, C.c_int32, _P, _P]),
    "ffb_curve_pose": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, C.c_int32, C.c_double, _P, _P, _P, _P, _P]),
    "ffb_ray_plane": (C.c_int, [_P, _P, _P, _P, C.c_int32, _P, _P]),
    "ffb_sphere_sphere": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P]),
}

_lib: Optional[C.CDLL] = None
launch_count = 0      # kernels launched through this binding (bench.py reports it as gpu_launches)


def lib() -> C.CDLL:
    """Load libffb200.so (once).  Raises RuntimeError when it has not been built -- no fallback."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m fireflies_b200._build` "
                "(or __graft_entry__.build()).  fireflies_b200 has no CPU/PyTorch fallback.")
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)          # AttributeError if the export is missing
            fn.restype, fn.argtypes = res, args
        _lib = h
    return _lib


E_UNSUPPORTED = -4     # FFB_E_UNSUPPORTED: a fused path does not cover this case; the caller uses the unfused calls


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().ffb_last_error_string().decode(errors="replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")


def require_cuda(t: torch.Tensor, dtype: torch.dtype, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{name}: fireflies_b200 kernels need a CUDA tensor (got {getattr(t, 'device', type(t))}); "
                           "there is no CPU path")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: tensor must be contiguous")
    return t


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def count(n: int = 1) -> None:
    global launch_count
    launch_count += n
