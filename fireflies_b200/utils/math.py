"""Math primitives -- drop-in for ``fireflies/utils/math.py``.

Matrix *builders* run on the host exactly like the reference (python ``math.cos`` on the angle, i.e. fp64
trig rounded to fp32 -- utils/math.py:24-60); the per-vertex work (``transform_points`` /
``transform_directions``) runs in ``libffb200.so``.  The batched path never calls the builders: the compose
kernel evaluates the same fp64-trig-then-round arithmetic on the device.
"""
from __future__ import annotations

import math
import random

import torch
import torch.nn.functional as F

from .. import _native as nat


def uniformBetweenValues(a: float, b: float) -> float:
    return random.uniform(a, b)


def getYawTransform(alpha: float, _device) -> torch.Tensor:        # utils/math.py:24-34 (about Z)
    c, s = math.cos(alpha), math.sin(alpha)
    return torch.tensor([[c, -s, 0], [s, c, 0], [0, 0, 1]], device=_device)


def getPitchTransform(alpha: float, _device) -> torch.Tensor:      # utils/math.py:37-47 (about Y)
    c, s = math.cos(alpha), math.sin(alpha)
    return torch.tensor([[c, 0, s], [0, 1, 0], [-s, 0, c]], device=_device)


def getRollTransform(alpha: float, _device) -> torch.Tensor:       # utils/math.py:50-60 (about X)
    c, s = math.cos(alpha), math.sin(alpha)
    return torch.tensor([[1, 0, 0], [0, c, -s], [0, s, c]], device=_device)


def getZTransform(alpha: float, _device) -> torch.Tensor:          # utils/math.py:12-21
    return getYawTransform(alpha, _device)


def getYTransform(alpha: float, _device) -> torch.Tensor:
    return getPitchTransform(alpha, _device)


def getXTransform(alpha: float, _device) -> torch.Tensor:
    return getRollTransform(alpha, _device)


def vector_dot(A: torch.Tensor, B: torch.Tensor) -> torch.Tensor:
    return torch.sum(A * B, dim=-1)


def rotation_matrix_from_vectors(v1, v2):
    """utils/math.py:67-105 (Rodrigues)."""
    v1 = F.normalize(v1, dim=0)
    v2 = F.normalize(v2, dim=0)
    cross = torch.linalg.cross(v1, v2)
    dot = torch.dot(v1, v2)
    skew = torch.zeros(3, 3, dtype=torch.float32, device=v1.device)
    skew[0, 1], skew[0, 2] = -cross[2], cross[1]
    skew[1, 0], skew[1, 2] = cross[2], -cross[0]
    skew[2, 0], skew[2, 1] = -cross[1], cross[0]
    return torch.eye(3, device=v1.device) + skew + torch.mm(skew, skew) * (1 - dot) / torch.norm(cross) ** 2


def rotation_matrix_from_vectors_with_fixed_up(v1, v2, up_vector=torch.tensor([0.0, 0.0, 1.0])):
    """utils/math.py:108-159.  The reference computes the Rodrigues matrix, uses it only to measure the angle between the
    rotated and the original up vector, and returns ``eye + normalize(skew, dim=0) * angle`` -- reproduced as written."""
    up_vector = F.normalize(up_vector.to(v1.device), dim=0)
    rotation_matrix = rotation_matrix_from_vectors(v1, v2)
    cross = torch.linalg.cross(F.normalize(v1, dim=0), F.normalize(v2, dim=0))
    skew = torch.zeros(3, 3, dtype=torch.float32, device=v1.device)
    skew[0, 1], skew[0, 2] = -cross[2], cross[1]
    skew[1, 0], skew[1, 2] = cross[2], -cross[0]
    skew[2, 0], skew[2, 1] = -cross[1], cross[0]
    correction_angle = torch.acos(torch.dot(torch.mv(rotation_matrix, up_vector), up_vector))
    return torch.eye(3, device=v1.device) + F.normalize(skew, dim=0) * correction_angle


def singleRandomBetweenTensors(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    assert a.size() == b.size()
    assert a.device == b.device
    rands = random.uniform(0, 1)
    return rands * (b - a) + b          # sic: the reference adds b (utils/math.py:162-167)


def randomBetweenTensors(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """utils/math.py:170-175: ``torch.rand(a.shape)*(b-a)+a`` -- same global torch generator stream as the
    reference; the affine map runs in the sampling kernel (injected-variate mode)."""
    assert a.size() == b.size()
    assert a.device == b.device
    from ..sampling.base import _lerp_native
    return _lerp_native(a, b, torch.rand(a.shape, device=a.device))


def normalize(tensor: torch.Tensor) -> torch.Tensor:
    tensor = tensor - tensor.amin()
    return tensor / tensor.amax()


def normalize_channelwise(tensor: torch.Tensor, dim: int = -1, device=torch.device("cuda")) -> torch.Tensor:
    indices = [i for i in range(tensor.dim()) if i != (dim % tensor.dim())]
    tensor = tensor - tensor.amin(indices)
    return tensor / tensor.amax(indices)


def convert_points_to_homogeneous(points: torch.Tensor) -> torch.Tensor:
    return F.pad(points, pad=(0, 1), mode="constant", value=1.0)


def toMat4x4(mat: torch.Tensor, addOne: bool = True) -> torch.Tensor:
    mat4x4 = F.pad(mat, pad=(0, 1, 0, 1), mode="constant", value=0.0)
    if addOne:
        mat4x4[3, 3] = 1.0
    return mat4x4


def convert_points_from_homogeneous(points: torch.Tensor) -> torch.Tensor:
    return points[..., :-1] / points[..., -1:]


def convert_points_to_nonhomogeneous(points: torch.Tensor) -> torch.Tensor:
    return F.pad(points, pad=(0, 1), mode="constant", value=0.0)


class _TransformFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points, transform, as_directions):
        pts = nat.require_cuda(points.detach().float().contiguous(), torch.float32, "points")
        T = nat.require_cuda(transform.detach().float().contiguous(), torch.float32, "transform")
        if pts.dim() != 2 or pts.shape[1] != 3 or T.shape != (4, 4):
            raise ValueError("transform_points expects points [V,3] and a [4,4] transform")
        out = torch.empty_like(pts)
        nat.check(nat.lib().ffb_transform_points(pts.data_ptr(), pts.shape[0], T.data_ptr(), int(as_directions),
                                                 out.data_ptr(), nat.stream()), "ffb_transform_points")
        nat.count()
        ctx.save_for_backward(pts, T)
        ctx.dirs = as_directions
        ctx.t_dtype = transform.dtype
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        pts, T = ctx.saved_tensors
        g = g.contiguous().float()
        L = nat.lib()
        if not ctx.needs_input_grad[1]:
            d = torch.empty_like(pts)
            nat.check(L.ffb_transform_points_bwd(pts.data_ptr(), pts.shape[0], T.data_ptr(), int(ctx.dirs),
                                                 g.data_ptr(), d.data_ptr(), nat.stream()), "ffb_transform_points_bwd")
            nat.count()
            return d, None, None
        d = torch.empty_like(pts) if ctx.needs_input_grad[0] else None
        d_T = torch.empty(16, dtype=torch.float32, device=pts.device)
        ws = torch.empty(L.ffb_transform_bwd_workspace_bytes(pts.shape[0]), dtype=torch.uint8, device=pts.device)
        nat.check(L.ffb_transform_points_bwd_full(pts.data_ptr(), pts.shape[0], T.data_ptr(), int(ctx.dirs), g.data_ptr(),
                                                  nat.ptr(d), d_T.data_ptr(), ws.data_ptr() if ws.numel() else None, ws.numel(),
                                                  nat.stream()), "ffb_transform_points_bwd_full")
        nat.count(2 if ws.numel() else 1)
        return d, d_T.view(4, 4).to(ctx.t_dtype), None


def transform_points(points: torch.Tensor, transform: torch.Tensor) -> torch.Tensor:
    """utils/math.py:220-228: ``(T @ [x,y,z,1])[:3] / w``.  Differentiable w.r.t. ``points`` and ``transform`` (the
    transform's gradient has its shape and dtype).  CUDA tensors only.  First derivatives only: differentiating the
    gradient again (``create_graph=True``) raises."""
    return _TransformFn.apply(points, transform, False)


def transform_directions(points: torch.Tensor, transform: torch.Tensor) -> torch.Tensor:
    """utils/math.py:231-235: ``(T @ [x,y,z,0])[:3]``.  Differentiable w.r.t. ``points`` and ``transform`` (row 3 and
    column 3 of its gradient are zero).  CUDA tensors only; first derivatives only, as :func:`transform_points`."""
    return _TransformFn.apply(points, transform, True)
