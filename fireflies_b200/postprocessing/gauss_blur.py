"""``fireflies/postprocessing/gauss_blur.py`` -- kornia ``gaussian_blur2d`` semantics (reflect border, separable)
evaluated by the TMA-staged blur kernel; :func:`gaussian_blur2d` is the differentiable form of the same blur."""
import ctypes as C
import numbers

import numpy as np
import torch

from . import base
from .. import _native as nat


class GaussianBlur(base.BasePostProcessingFunction):
    def __init__(self, kernel_size, sigma, probability: float):
        super().__init__(probability)
        self._kernel_size = kernel_size
        self._sigma = sigma

    def spec(self):
        return (tuple(int(k) for k in self._kernel_size), tuple(float(s) for s in self._sigma))

    def post_process(self, image: np.ndarray) -> np.ndarray:
        x = self._to_device(image)
        return base.run_postprocess(x, blur=self.spec())[0].cpu().numpy()


def _pair(v, conv, name):
    if torch.is_tensor(v) or (isinstance(v, (tuple, list)) and any(torch.is_tensor(e) for e in v)):
        raise NotImplementedError(f"gaussian_blur2d: tensor-valued {name} (per-batch or differentiable) is not supported; "
                                  "pass python numbers")
    if isinstance(v, numbers.Number):
        return conv(v), conv(v)
    v = tuple(v)
    if len(v) != 2:
        raise ValueError(f"gaussian_blur2d: {name} must be a number or a (y, x) pair")
    return conv(v[0]), conv(v[1])


def blur_spec(kernel_size, sigma):
    """``((ky, kx), (sy, sx))`` from kornia-style arguments (a number stands for both axes)."""
    return _pair(kernel_size, int, "kernel_size"), _pair(sigma, float, "sigma")


def gaussian_blur2d_backward(grad: torch.Tensor, kernel_size, sigma, out: torch.Tensor = None) -> torch.Tensor:
    """Adjoint of the blur (``ffb_blur_bwd``): the gradient w.r.t. the input of ``gaussian_blur2d`` given ``grad``, the
    gradient w.r.t. its output.  ``grad`` f32 CUDA ``[..., H, W]``; ``out``: optional tensor of the same shape to write into."""
    (ky, kx), (sy, sx) = blur_spec(kernel_size, sigma)
    g = nat.require_cuda(grad.contiguous(), torch.float32, "grad")
    H, W = g.shape[-2:]
    B = g.numel() // max(H * W, 1)
    res = torch.empty_like(g) if out is None else nat.require_cuda(out, torch.float32, "out")
    if res.shape != g.shape:
        raise ValueError("gaussian_blur2d_backward: `out` must have the shape of `grad`")
    d = nat.PostDesc(B, H, W, ky, kx, sy, sx, 0, 0.0, 0.0, 0, 0)
    nat.check(nat.lib().ffb_blur_bwd(C.byref(d), g.data_ptr(), res.data_ptr(), nat.stream()), "ffb_blur_bwd")
    nat.count()
    return res


class _GaussianBlur2dFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, spec):
        H, W = x.shape[-2:]
        frames = x.detach().reshape(-1, H, W)
        ctx.spec = spec
        return base.run_postprocess(frames, blur=spec).view(x.shape)

    @staticmethod
    def backward(ctx, g):
        return gaussian_blur2d_backward(g, *ctx.spec), None


def gaussian_blur2d(input: torch.Tensor, kernel_size, sigma, border_type: str = "reflect", separable: bool = True) -> torch.Tensor:
    """``kornia.filters.gaussian_blur2d`` (0.7.1 signature) on the device, differentiable w.r.t. ``input``.

    ``input`` f32 CUDA ``[B, C, H, W]``, blurred as ``B*C`` frames by the kernel behind :class:`GaussianBlur` (bit-identical
    to ``run_postprocess(..., blur=...)``); the backward is the blur's adjoint kernel.  ``kernel_size`` / ``sigma``: ``(y, x)``
    pairs or one number for both axes; odd sizes up to 15 with ``kernel_size // 2`` below the image side.  Only kornia's
    default ``border_type="reflect"`` exists; the blur is always evaluated separably (``separable=False`` changes only
    rounding in kornia).  No gradient w.r.t. ``sigma``."""
    if border_type != "reflect":
        raise ValueError(f"gaussian_blur2d: border_type={border_type!r} is not implemented (only 'reflect')")
    spec = blur_spec(kernel_size, sigma)
    x = nat.require_cuda(input.contiguous(), torch.float32, "input")
    if x.dim() != 4:
        raise ValueError(f"gaussian_blur2d: input must be [B, C, H, W], got {tuple(x.shape)}")
    return _GaussianBlur2dFn.apply(x, spec)
