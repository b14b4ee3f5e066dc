"""Laser splat -- drop-in for ``fireflies/graphics/rasterization.py`` backed by ``libffb200.so``.

Same function names, argument order, defaults and return orientation as the reference (cited per
function); the work is done by the fused sm_100a splat-reduce kernels (``csrc/ffb_splat.cu``).
There is no CPU path: CPU tensors / ``device="cpu"`` raise.

Additions (not in the reference): :func:`splat_reduce` -- the fused, batched entry point the
pattern-optimisation path uses (both reductions in one pass, ``B`` scene samples per launch).
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Sequence, Tuple, Union

import torch

from .. import _native as nat

__all__ = [
    "rasterize_points", "softor", "sum", "baked_sum", "baked_sum_2", "baked_softor", "baked_softor_2",
    "rasterize_points_baked_sum", "rasterize_points_baked_softor", "splat_reduce", "splat_windows", "l1_loss",
]

_builtin_sum = sum


def _ts(texture_size) -> Tuple[int, int]:
    v = texture_size.tolist() if torch.is_tensor(texture_size) else list(texture_size)
    if len(v) != 2:
        raise ValueError("texture_size must have two entries")
    return int(v[0]), int(v[1])


def _sigma(sigma) -> float:
    if torch.is_tensor(sigma):
        return float(sigma.detach().reshape(-1)[0].item())
    return float(sigma)


def _device_ok(device) -> None:
    if device is not None and torch.device(device).type != "cuda":
        raise RuntimeError(f"fireflies_b200 has no CPU path (device={device!r}); the splat runs on sm_100a only")


def _points(points: torch.Tensor) -> torch.Tensor:
    if not points.is_cuda:
        raise RuntimeError("fireflies_b200: `points` must be a CUDA tensor; there is no CPU path")
    if points.dtype != torch.float32:
        points = points.float()
    return points.contiguous()


class _SplatPlan:
    """Descriptor + binning workspace of one fused splat call (kept alive for the backward)."""

    def __init__(self, points: torch.Tensor, B: int, sigma: float, ts0: int, ts1: int, num_std_sum: int, num_std_softor: int,
                 windows: bool = False):
        shared = points.dim() == 2
        N = points.shape[-2]
        if not shared and points.shape[0] != B:
            raise ValueError("points batch dimension does not match B")
        self.desc = nat.SplatDesc(B, N, ts0, ts1, sigma, num_std_sum, num_std_softor, 0 if shared else N * 2)
        self.B, self.N, self.ts0, self.ts1, self.shared = B, N, ts0, ts1, shared
        L = nat.lib()
        nbytes = L.ffb_splat_workspace_bytes(C.byref(self.desc))
        if nbytes == 0:
            nat.check(-1, "ffb_splat_workspace_bytes")
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=points.device)
        self.windows = None
        if windows:
            self.windows = torch.empty((1 if shared else B, N, 2, 2, 3), dtype=torch.int32, device=points.device)
        nat.check(L.ffb_splat_prepare(C.byref(self.desc), points.data_ptr(), self.ws.data_ptr(), nbytes,
                                      nat.ptr(self.windows), nat.stream()), "ffb_splat_prepare")
        nat.count()

    def forward(self, points, want_sum: bool, want_softor: bool, sum_transposed: bool, out=None):
        """``out``: optional ``(sum, softor)`` tensors to write into (contiguous, e.g. slices of a larger batch along dim 0)."""
        dev = points.device
        out_s = out_o = None
        if want_sum:
            shape = (self.B, self.ts0, self.ts1) if sum_transposed else (self.B, self.ts1, self.ts0)
            out_s = out[0] if out is not None else torch.empty(shape, dtype=torch.float32, device=dev)
            assert tuple(out_s.shape) == shape and out_s.is_contiguous()
        if want_softor:
            out_o = out[1] if out is not None else torch.empty((self.B, self.ts1, self.ts0), dtype=torch.float32, device=dev)
            assert tuple(out_o.shape) == (self.B, self.ts1, self.ts0) and out_o.is_contiguous()
        nat.check(nat.lib().ffb_splat_fwd(C.byref(self.desc), points.data_ptr(), self.ws.data_ptr(), nat.ptr(out_s),
                                          int(sum_transposed), nat.ptr(out_o), nat.stream()), "ffb_splat_fwd")
        nat.count()
        return out_s, out_o

    def backward(self, points, g_sum, g_softor, sum_transposed: bool, saved_softor=None, out=None) -> torch.Tensor:
        """``saved_softor``: the forward's soft-OR output (what autograd saves for ``prod``'s backward); the production kernel
        rebuilds the per-texel product instead (8 instead of 12 B/texel) and reads it only for soft-OR windows tighter than
        their no-op radius and for textures the TMA unit cannot describe.  ``out``: optional
        ``[B,N,2]`` tensor to write into."""
        d_pts = out if out is not None else torch.empty((self.B, self.N, 2), dtype=torch.float32, device=points.device)
        nat.check(nat.lib().ffb_splat_bwd(C.byref(self.desc), points.data_ptr(), self.ws.data_ptr(), nat.ptr(g_sum),
                                          int(sum_transposed), nat.ptr(g_softor), nat.ptr(saved_softor), d_pts.data_ptr(),
                                          nat.stream()), "ffb_splat_bwd")
        nat.count(2)      # memset + kernel
        return d_pts


    def backward_l1(self, points, out_sum, out_softor, sum_transposed: bool, out=None):
        """Fused ``L1Loss(softor, sum).backward()`` (rasterization.py:589-599): returns ``(loss [B], d_pts [B,N,2])`` or
        ``None`` when the fused kernel does not cover the case (the caller then runs the loss and the backward
        separately).  ``out``: optional ``(loss, d_pts)`` tensors to write into."""
        if sum_transposed and self.ts0 != self.ts1:
            return None
        d_pts = out[1] if out is not None else torch.empty((self.B, self.N, 2), dtype=torch.float32, device=points.device)
        loss = out[0] if out is not None else torch.empty(self.B, dtype=torch.float32, device=points.device)
        rc = nat.lib().ffb_splat_bwd_l1(C.byref(self.desc), points.data_ptr(), self.ws.data_ptr(), out_sum.data_ptr(),
                                        int(sum_transposed), out_softor.data_ptr(), loss.data_ptr(), d_pts.data_ptr(), nat.stream())
        if rc == nat.E_UNSUPPORTED:
            return None
        nat.check(rc, "ffb_splat_bwd_l1")
        nat.count(3)      # two memsets + kernel
        return loss, d_pts


def reduce_over_samples(x: torch.Tensor) -> torch.Tensor:
    """``x.sum(0)`` in a fixed order (deterministic): folds per-sample pattern gradients."""
    x = nat.require_cuda(x, torch.float32, "x")
    row = x[0].numel()
    # texture-sized rows: fold 8 samples per level at streaming bandwidth (a CTA that walks all B planes loses to TLB reach)
    while x.shape[0] > 8 and row >= 1 << 16 and row % 4 == 0 and x.data_ptr() % 16 == 0:
        G = (x.shape[0] + 7) // 8
        part = torch.empty((G,) + tuple(x.shape[1:]), dtype=torch.float32, device=x.device)
        nat.check(nat.lib().ffb_reduce_sample_groups(x.data_ptr(), x.shape[0], row, part.data_ptr(), nat.stream()),
                  "ffb_reduce_sample_groups")
        nat.count()
        x = part
    out = torch.empty(x.shape[1:], dtype=torch.float32, device=x.device)
    nat.check(nat.lib().ffb_reduce_over_samples(x.data_ptr(), x.shape[0], row, out.data_ptr(), nat.stream()),
              "ffb_reduce_over_samples")
    nat.count()
    return out


class _SplatReduceFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points, B, sigma, ts0, ts1, num_std_sum, num_std_softor, want_sum, want_softor, sum_transposed):
        pts = _points(points.detach())
        plan = _SplatPlan(pts, B, sigma, ts0, ts1, num_std_sum, num_std_softor)
        out_s, out_o = plan.forward(pts, want_sum, want_softor, sum_transposed)
        ctx.plan, ctx.pts, ctx.flags = plan, pts, (want_sum, want_softor, sum_transposed)
        empty = pts.new_empty(0)
        outs = (out_s if want_sum else empty, out_o if want_softor else empty)
        ctx.mark_non_differentiable(*[o for o, w in zip(outs, (want_sum, want_softor)) if not w])
        if want_softor:
            ctx.save_for_backward(outs[1])      # like torch.prod's backward, keep the output (version-checked)
        return outs

    @staticmethod
    def backward(ctx, g_sum, g_softor):
        want_sum, want_softor, sum_t = ctx.flags
        gs = g_sum.contiguous().float() if (want_sum and g_sum is not None) else None
        go = g_softor.contiguous().float() if (want_softor and g_softor is not None) else None
        if gs is None and go is None:
            return (None,) * 10
        plan = ctx.plan
        d = plan.backward(ctx.pts, gs, go, sum_t, ctx.saved_tensors[0] if go is not None else None)
        if plan.shared:
            d = d[0] if plan.B == 1 else reduce_over_samples(d)
        return (d,) + (None,) * 9


def splat_reduce(points: torch.Tensor, sigma, texture_size, num_std_sum: Optional[int] = 4,
                 num_std_softor: Optional[int] = 5, reduce: Sequence[str] = ("sum", "softor"),
                 sum_transposed: bool = False, batch: Optional[int] = None):
    """Fused splat + reduction for ``B`` scene samples in one launch.

    ``points``: ``[N,2]`` (one pattern, optionally replicated over ``batch`` samples) or ``[B,N,2]``.
    ``num_std_*``: footprint multiplier of the reference's ``baked_*`` functions, ``None``/0 = dense
    semantics (``rasterize_points`` + ``sum``/``softor``).  Returns ``(sum, softor)`` with ``None`` for a
    reduction that was not requested; each is ``[B, ts1, ts0]`` (``sum``: ``[B, ts0, ts1]`` if
    ``sum_transposed``, baked_sum_2's orientation), or without the leading axis when ``points`` is
    ``[N,2]`` and ``batch`` is None.  Differentiable w.r.t. ``points``.
    """
    ts0, ts1 = _ts(texture_size)
    want_sum, want_softor = "sum" in reduce, "softor" in reduce
    if not (want_sum or want_softor):
        raise ValueError("reduce must name 'sum' and/or 'softor'")
    squeeze = points.dim() == 2 and batch is None
    B = points.shape[0] if points.dim() == 3 else (1 if batch is None else int(batch))
    out_s, out_o = _SplatReduceFn.apply(points, B, _sigma(sigma), ts0, ts1, int(num_std_sum or 0), int(num_std_softor or 0),
                                        want_sum, want_softor, bool(sum_transposed))
    out_s = (out_s[0] if squeeze else out_s) if want_sum else None
    out_o = (out_o[0] if squeeze else out_o) if want_softor else None
    return out_s, out_o


def splat_windows(points: torch.Tensor, sigma, texture_size, num_std_sum: int = 4, num_std_softor: int = 5) -> torch.Tensor:
    """int32 ``[N,2,2,3]`` (``[B,N,2,2,3]`` for batched points): per point, per reduction (sum, softor), per
    axis, the ``(wo, rs, re)`` slice triple the reference clips its footprint with
    (fireflies/graphics/rasterization.py:199-230).  The splat path's integer outputs."""
    ts0, ts1 = _ts(texture_size)
    pts = _points(points.detach())
    B = pts.shape[0] if pts.dim() == 3 else 1
    plan = _SplatPlan(pts, B, _sigma(sigma), ts0, ts1, num_std_sum, num_std_softor, windows=True)
    return plan.windows[0] if pts.dim() == 2 else plan.windows


class _DenseFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points, sigma, ts0, ts1, in_pixels=False):
        pts = _points(points.detach())
        N = pts.shape[0]
        out = torch.empty((N, ts1, ts0), dtype=torch.float32, device=pts.device)
        fn = nat.lib().ffb_splat_dense_px_fwd if in_pixels else nat.lib().ffb_splat_dense_fwd
        nat.check(fn(pts.data_ptr(), N, ts0, ts1, sigma, out.data_ptr(), nat.stream()), "ffb_splat_dense_fwd")
        nat.count()
        ctx.pts, ctx.args = pts, (sigma, ts0, ts1, in_pixels)
        return out

    @staticmethod
    def backward(ctx, g):
        sigma, ts0, ts1, in_pixels = ctx.args
        g = g.contiguous().float()
        d = torch.empty_like(ctx.pts)
        fn = nat.lib().ffb_splat_dense_px_bwd if in_pixels else nat.lib().ffb_splat_dense_bwd
        nat.check(fn(ctx.pts.data_ptr(), ctx.pts.shape[0], ts0, ts1, sigma, g.data_ptr(), d.data_ptr(), nat.stream()), "ffb_splat_dense_bwd")
        nat.count(2)
        return d, None, None, None, None


# --------------------------------------------------------------------------------------------------
# reference-compatible surface
# --------------------------------------------------------------------------------------------------
def rasterize_points(points: torch.Tensor, sigma: float, texture_size: torch.Tensor,
                     device: torch.device = torch.device("cuda")) -> torch.Tensor:
    """fireflies/graphics/rasterization.py:7-37 -- dense ``[N, ts[1], ts[0]]`` tensor
    ``exp(-(((c - p0*ts0)^2 + (r - p1*ts1)^2)/sigma)^2)``.  Kept for API compatibility (N*H*W floats);
    the optimisation path uses the fused reductions instead."""
    _device_ok(device)
    ts0, ts1 = _ts(texture_size)
    return _DenseFn.apply(points, _sigma(sigma), ts0, ts1)


def rasterize_points_in_non_ndc(points: torch.Tensor, sigma: float, texture_size: torch.Tensor,
                                device: torch.device = torch.device("cuda")) -> torch.Tensor:
    """fireflies/graphics/rasterization.py:38-63 -- ``rasterize_points`` for points already in texel units (no scaling by
    ``texture_size``): ``points[:,0]`` pairs with the column index, ``points[:,1]`` with the row index."""
    _device_ok(device)
    ts0, ts1 = _ts(texture_size)
    return _DenseFn.apply(points, _sigma(sigma), ts0, ts1, True)


def softor(texture: torch.Tensor, dim=0, keepdim: bool = False) -> torch.Tensor:
    """fireflies/graphics/rasterization.py:156-157."""
    return 1 - torch.prod(1 - texture, dim=dim, keepdim=keepdim)


def sum(texture: torch.Tensor, dim=0, keepdim: bool = False) -> torch.Tensor:  # noqa: A001 (reference name)
    """fireflies/graphics/rasterization.py:160-161."""
    return torch.sum(texture, dim=dim, keepdim=keepdim)


def baked_sum(points, sigma, texture_size, num_std: int = 4, device: torch.device = torch.device("cuda")) -> torch.Tensor:
    """fireflies/graphics/rasterization.py:164-237 -> ``[ts[1], ts[0]]``."""
    _device_ok(device)
    return splat_reduce(points, sigma, texture_size, num_std_sum=num_std, reduce=("sum",))[0]


def baked_sum_2(points, sigma, texture_size, num_std: int = 4, device: torch.device = torch.device("cuda")) -> torch.Tensor:
    """fireflies/graphics/rasterization.py:240-318 -> ``[ts[0], ts[1]]`` (the reference returns the
    un-transposed accumulator here, SURVEY.md A-3)."""
    _device_ok(device)
    return splat_reduce(points, sigma, texture_size, num_std_sum=num_std, reduce=("sum",), sum_transposed=True)[0]


def baked_softor(points, sigma, texture_size, num_std: int = 5, device: torch.device = torch.device("cuda")) -> torch.Tensor:
    """fireflies/graphics/rasterization.py:321-392 -> ``[ts[1], ts[0]]``."""
    _device_ok(device)
    return splat_reduce(points, sigma, texture_size, num_std_softor=num_std, reduce=("softor",))[1]


def baked_softor_2(points, sigma, texture_size, num_std: int = 5, device: torch.device = torch.device("cuda")) -> torch.Tensor:
    """fireflies/graphics/rasterization.py:395-472 -> ``[ts[1], ts[0]]``."""
    _device_ok(device)
    return splat_reduce(points, sigma, texture_size, num_std_softor=num_std, reduce=("softor",))[1]


def rasterize_points_baked_softor(points, sigma, texture_size, device: torch.device = torch.device("cuda")) -> torch.Tensor:
    """fireflies/graphics/rasterization.py:475-503 (full-frame soft-OR, no footprint)."""
    _device_ok(device)
    return splat_reduce(points, sigma, texture_size, num_std_softor=None, reduce=("softor",))[1]


def rasterize_points_baked_sum(points, sigma, texture_size, device: torch.device = torch.device("cuda")) -> torch.Tensor:
    """fireflies/graphics/rasterization.py:507-535 (full-frame sum, no footprint)."""
    _device_ok(device)
    return splat_reduce(points, sigma, texture_size, num_std_sum=None, reduce=("sum",))[0]


class _L1Fn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b, b_transposed):
        a_ = nat.require_cuda(a.detach().contiguous(), torch.float32, "a")
        b_ = nat.require_cuda(b.detach().contiguous(), torch.float32, "b")
        ctx.single = a_.dim() == 2                          # one texture pair ([ts1, ts0]): scalar loss, like torch.nn.L1Loss
        if ctx.single:
            a_, b_ = a_.unsqueeze(0), b_.unsqueeze(0)
        B, ts1, ts0 = a_.shape
        loss = torch.empty(B, dtype=torch.float32, device=a_.device)
        ga, gb = torch.empty_like(a_), torch.empty_like(b_)
        nat.check(nat.lib().ffb_l1_loss_fwd_bwd(a_.data_ptr(), b_.data_ptr(), int(b_transposed), B, ts0, ts1,
                                                loss.data_ptr(), ga.data_ptr(), gb.data_ptr(), nat.stream()), "ffb_l1_loss_fwd_bwd")
        nat.count(2)
        ctx.save_for_backward(ga, gb)
        return loss[0] if ctx.single else loss

    @staticmethod
    def backward(ctx, g):
        ga, gb = ctx.saved_tensors
        g = g.reshape(-1, 1, 1)
        da, db = ga * g, gb * g
        return (da[0], db[0], None) if ctx.single else (da, db, None)


def l1_loss(a: torch.Tensor, b: torch.Tensor, b_transposed: bool = False) -> torch.Tensor:
    """Per-sample ``torch.nn.L1Loss()(a, b)`` (mean |a-b|) for ``a`` ``[B,ts1,ts0]`` and ``b`` in the same or the
    transposed (``baked_sum_2``) layout -- the loss of the in-tree pattern optimisation
    (fireflies/graphics/rasterization.py:589-599).  Returns ``[B]`` (a scalar for one ``[ts1,ts0]`` pair)."""
    return _L1Fn.apply(a, b, b_transposed)


# --------------------------------------------------------------------------------------------------
# line and depth rasterisers (SURVEY.md 8(f) row 2)
# --------------------------------------------------------------------------------------------------
def _lines(lines: torch.Tensor) -> torch.Tensor:
    lines = nat.require_cuda(lines.float().contiguous(), torch.float32, "lines")
    if lines.dim() != 3 or lines.shape[1:] != (2, 2):
        raise ValueError("lines must be [L, 2, 2] (start / end x X / Y)")
    if lines.data_ptr() % 16 != 0:
        lines = lines.clone()           # the kernels read each line as one float4; a fresh allocation is 16-byte aligned
    return lines


class _LinesDenseFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lines, sigma, ts0, ts1):
        ln = _lines(lines.detach())
        L = ln.shape[0]
        out = torch.empty((L, ts1, ts0), dtype=torch.float32, device=ln.device)
        nat.check(nat.lib().ffb_lines_dense_fwd(ln.data_ptr(), L, ts0, ts1, sigma, out.data_ptr(), nat.stream()), "ffb_lines_dense_fwd")
        nat.count()
        ctx.ln, ctx.args = ln, (sigma, ts0, ts1)
        return out

    @staticmethod
    def backward(ctx, g):
        sigma, ts0, ts1 = ctx.args
        g = g.contiguous().float()
        d = torch.empty_like(ctx.ln)
        nat.check(nat.lib().ffb_lines_dense_bwd(ctx.ln.data_ptr(), ctx.ln.shape[0], ts0, ts1, sigma, g.data_ptr(), d.data_ptr(),
                                                nat.stream()), "ffb_lines_dense_bwd")
        nat.count(2)
        return d, None, None, None


class _LinesReduceFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lines, sigma, ts0, ts1, want_sum, want_softor):
        ln = _lines(lines.detach())
        L = ln.shape[0]
        out_s = torch.empty((ts1, ts0), dtype=torch.float32, device=ln.device) if want_sum else None
        out_o = torch.empty((ts1, ts0), dtype=torch.float32, device=ln.device) if want_softor else None
        nat.check(nat.lib().ffb_lines_reduce_fwd(ln.data_ptr(), L, ts0, ts1, sigma, nat.ptr(out_s), nat.ptr(out_o), nat.stream()),
                  "ffb_lines_reduce_fwd")
        nat.count()
        ctx.ln, ctx.args = ln, (sigma, ts0, ts1, want_sum, want_softor)
        empty = ln.new_empty(0)
        outs = (out_s if want_sum else empty, out_o if want_softor else empty)
        ctx.mark_non_differentiable(*[o for o, w in zip(outs, (want_sum, want_softor)) if not w])
        return outs

    @staticmethod
    def backward(ctx, g_sum, g_softor):
        sigma, ts0, ts1, want_sum, want_softor = ctx.args
        gs = g_sum.contiguous().float() if (want_sum and g_sum is not None) else None
        go = g_softor.contiguous().float() if (want_softor and g_softor is not None) else None
        d = torch.zeros_like(ctx.ln)
        if gs is not None or go is not None:
            nat.check(nat.lib().ffb_lines_reduce_bwd(ctx.ln.data_ptr(), ctx.ln.shape[0], ts0, ts1, sigma, nat.ptr(gs), nat.ptr(go),
                                                     d.data_ptr(), nat.stream()), "ffb_lines_reduce_bwd")
            nat.count(2)
        return d, None, None, None, None, None


def rasterize_lines(lines: torch.Tensor, sigma: float, texture_size: torch.Tensor,
                    device: torch.device = torch.device("cuda")) -> torch.Tensor:
    """fireflies/graphics/rasterization.py:107-153 -- dense ``[L, ts[1], ts[0]]`` squared-distance transform of the
    segments ``lines[L,2,2]``, ``exp(-(d2*d2)/(sigma*sigma))``.  Deviation: the reference scales the caller's ``lines``
    by ``texture_size`` IN PLACE (:122-123); here ``lines`` is left untouched."""
    _device_ok(device)
    ts0, ts1 = _ts(texture_size)
    return _LinesDenseFn.apply(lines, _sigma(sigma), ts0, ts1)


def lines_reduce(lines: torch.Tensor, sigma, texture_size, reduce: Tuple[str, ...] = ("sum", "softor")):
    """``(rasterize_lines(...).sum(0), softor(rasterize_lines(...)))`` without the ``[L,H,W]`` tensor (what
    test_line_reg, rasterization.py:684-697, and the epipolar regulariser compute).  Entries not named in ``reduce``
    come back as ``None``."""
    ts0, ts1 = _ts(texture_size)
    s, o = _LinesReduceFn.apply(lines, _sigma(sigma), ts0, ts1, "sum" in reduce, "softor" in reduce)
    return (s if "sum" in reduce else None), (o if "softor" in reduce else None)


class _DepthFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points, depth_vals, sigma, ts0, ts1):
        pts = _points(points.detach())
        dv = nat.require_cuda(depth_vals.detach().float().reshape(-1).contiguous(), torch.float32, "depth_vals")
        N = pts.shape[0]
        if dv.numel() != N:
            raise ValueError("depth_vals must hold one value per point")
        out = torch.empty((N, ts1, ts0), dtype=torch.float32, device=pts.device)
        nat.check(nat.lib().ffb_depth_dense_fwd(pts.data_ptr(), dv.data_ptr(), N, ts0, ts1, sigma, out.data_ptr(), nat.stream()),
                  "ffb_depth_dense_fwd")
        nat.count()
        ctx.pts, ctx.dv, ctx.args, ctx.dshape = pts, dv, (sigma, ts0, ts1), depth_vals.shape
        return out

    @staticmethod
    def backward(ctx, g):
        sigma, ts0, ts1 = ctx.args
        g = g.contiguous().float()
        N = ctx.pts.shape[0]
        d_pts, d_dv = torch.empty_like(ctx.pts), torch.empty_like(ctx.dv)
        scratch = torch.empty((N, 3), dtype=torch.float32, device=g.device)
        nat.check(nat.lib().ffb_depth_dense_bwd(ctx.pts.data_ptr(), ctx.dv.data_ptr(), N, ts0, ts1, sigma, g.data_ptr(),
                                                scratch.data_ptr(), d_pts.data_ptr(), d_dv.data_ptr(), nat.stream()), "ffb_depth_dense_bwd")
        nat.count(3)
        return d_pts, d_dv.reshape(ctx.dshape), None, None, None


def rasterize_depth(points: torch.Tensor, depth_vals: torch.Tensor, sigma: float, texture_size: torch.Tensor,
                    device: torch.device = torch.device("cuda")) -> torch.Tensor:
    """fireflies/graphics/rasterization.py:66-104 -- ``rasterize_points`` normalised by its per-point maximum over the
    frame and scaled by ``depth_vals [N,1]`` -> ``[N, ts[1], ts[0]]``."""
    _device_ok(device)
    ts0, ts1 = _ts(texture_size)
    return _DepthFn.apply(points, depth_vals, _sigma(sigma), ts0, ts1)


def subsampled_point_raster(ndc_points: torch.Tensor, num_subsamples: int, sigma, sensor_size):
    """fireflies/graphics/rasterization.py:538-549 -- per pyramid level ``i`` the soft-OR (keepdim) over the points of
    ``rasterize_depth`` at ``sensor_size // 2**i``; one fused launch per level, no ``[N,H,W]`` tensor.  Forward only
    (the reference uses it for the depth regulariser's target)."""
    pts = _points(ndc_points[:, 0:2].detach())
    dv = nat.require_cuda(ndc_points[:, 2].detach().float().contiguous(), torch.float32, "depth")
    ss = torch.as_tensor(sensor_size).cpu()
    out = []
    for i in range(num_subsamples):
        ts0, ts1 = _ts(ss // 2 ** i)
        o = torch.empty((1, ts1, ts0), dtype=torch.float32, device=pts.device)
        nat.check(nat.lib().ffb_depth_softor_fwd(pts.data_ptr(), dv.data_ptr(), pts.shape[0], ts0, ts1, _sigma(sigma), o.data_ptr(),
                                                 nat.stream()), "ffb_depth_softor_fwd")
        nat.count()
        out.append(o)
    return out
