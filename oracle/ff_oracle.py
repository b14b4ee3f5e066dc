"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the Fireflies hot path.

This module is the *oracle*: an independent CPU (torch fp32 / numpy) restatement
of the reference algorithms on the north-star path, written from the formulas in
SURVEY.md section 8(a).  It is NOT part of the product: ``fireflies_b200`` never
imports it; only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs do, as the checker or as the timed
CPU baseline.

Parity status: the reference ships no tests, golden vectors or fixtures
(SURVEY.md section 4), so parity is *unpinned by the reference itself*.  We pin
the oracle against the reference's own code: ``oracle/make_golden.py`` imports a
checkout of the original Fireflies project named by ``FIREFLIES_REF``
(``oracle/ref_loader.py``) and writes ``tests/golden/*.npz``;
``tests/test_oracle_golden.py`` checks every function here against those fixtures
(and against the live reference when ``FIREFLIES_REF`` is set).  Third-party
arithmetic that is absent from the reference and not installed (kornia 0.7.1
``gaussian_blur2d``, geomdl 5.3.1 ``NURBS.Curve``) is restated from its published
algorithm and pinned against independent implementations that ARE installed
(OpenCV, scipy): see ``gaussian_blur2d``, ``silhouette`` and the NURBS section
below.  ``cv2.circle`` is the real OpenCV in the fixtures.

All citations are ``path:line`` relative to the root of the original Fireflies project.
"""
from __future__ import annotations

import math
import random as _pyrandom
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

F32 = torch.float32


# ----------------------------------------------------------------------------
# a1/a2: dense splat and its reductions  (fireflies/graphics/rasterization.py:7-37,156-161)
# ----------------------------------------------------------------------------
def _as_ts(texture_size) -> Tuple[int, int]:
    ts = [int(v) for v in (texture_size.tolist() if torch.is_tensor(texture_size) else texture_size)]
    return ts[0], ts[1]


def _sigma_f32(sigma) -> torch.Tensor:
    if torch.is_tensor(sigma):
        return sigma.detach().to(F32).reshape(-1)[0]
    return torch.tensor(float(sigma), dtype=F32)


def splat_dense(points: torch.Tensor, sigma, texture_size) -> torch.Tensor:
    """``out[n,r,c] = exp(-(((c - p[n,0]*ts0)^2 + (r - p[n,1]*ts1)^2)/sigma)^2)``, shape ``[N, ts1, ts0]``.

    Follows rasterize_points (graphics/rasterization.py:18-35): pixel centres are the
    integer indices, ``points[:,0]`` pairs with the last (column) axis.
    """
    ts0, ts1 = _as_ts(texture_size)
    scale = torch.tensor([ts0, ts1], dtype=F32)
    P = points.to(F32) * scale                                     # :18
    cols = torch.arange(ts0, dtype=F32).view(1, 1, ts0)            # :21-25 (second meshgrid output)
    rows = torch.arange(ts1, dtype=F32).view(1, ts1, 1)
    dc = cols - P[:, 0].view(-1, 1, 1)                              # :29
    dr = rows - P[:, 1].view(-1, 1, 1)                              # :30
    d2 = dc * dc + dr * dr                                          # :32-34
    u = d2 / _sigma_f32(sigma)
    return torch.exp(-(u * u))                                      # :35


def softor(tex: torch.Tensor, dim: int = 0) -> torch.Tensor:
    """``1 - prod(1 - g)``  (graphics/rasterization.py:156-157)."""
    return 1 - torch.prod(1 - tex, dim=dim)


def reduce_sum(tex: torch.Tensor, dim: int = 0) -> torch.Tensor:
    """``sum(g)``  (graphics/rasterization.py:160-161)."""
    return torch.sum(tex, dim=dim)


# ----------------------------------------------------------------------------
# f2: line and depth rasterisers (SURVEY 8(f) row 2)
# (fireflies/graphics/rasterization.py:38-104, 107-153, 538-549)
# ----------------------------------------------------------------------------
def rasterize_lines(lines: torch.Tensor, sigma, texture_size) -> torch.Tensor:
    """Squared point-to-segment distance transform, ``exp(-(d2*d2)/(sigma*sigma))``, shape ``[L, ts1, ts0]``.

    Follows rasterize_lines (graphics/rasterization.py:107-153) without its in-place scaling of the caller's
    tensor (:122-123): ``lines[L,2,2]`` = (start, end) x (x, y), scaled by ``texture_size``; ``t0`` with the
    ``finfo.eps`` guard (:142), the three boolean-masked branches (:145-149).
    """
    ts0, ts1 = _as_ts(texture_size)
    scale = torch.tensor([ts0, ts1], dtype=F32)
    a = (lines[:, 0, :].to(F32) * scale).permute(1, 0).unsqueeze(-1).unsqueeze(-1)      # [2,L,1,1]  :122,125
    b = (lines[:, 1, :].to(F32) * scale).permute(1, 0).unsqueeze(-1).unsqueeze(-1)
    L = lines.shape[0]
    y, x = torch.meshgrid(torch.arange(0, ts1), torch.arange(0, ts0), indexing="ij")    # :128-132
    xy = torch.stack([x.unsqueeze(0).repeat(L, 1, 1), y.unsqueeze(0).repeat(L, 1, 1)])  # integer grid, promoted below
    pa = xy - a                                                                          # :140
    pb = xy - b
    m = b - a
    t0 = (pa * m).sum(dim=0) / ((m * m).sum(dim=0) + torch.finfo().eps)                  # :142
    patm = xy - (a + t0.unsqueeze(0) * m)
    d = (t0 <= 0) * (pa * pa).sum(dim=0) + (t0 > 0) * (t0 < 1) * (patm * patm).sum(dim=0) + (t0 >= 1) * (pb * pb).sum(dim=0)
    s = _sigma_f32(sigma)
    return torch.exp(-(d * d) / (s * s))                                                 # :153


def splat_dense_px(points_px: torch.Tensor, sigma, texture_size) -> torch.Tensor:
    """rasterize_points_in_non_ndc (graphics/rasterization.py:38-63): the dense splat for points in texel units."""
    ts0, ts1 = _as_ts(texture_size)
    cols = torch.arange(ts0, dtype=F32).view(1, 1, ts0)
    rows = torch.arange(ts1, dtype=F32).view(1, ts1, 1)
    dc = cols - points_px[:, 0].to(F32).view(-1, 1, 1)             # :52  (y grid = column index) - points[:, 0]
    dr = rows - points_px[:, 1].to(F32).view(-1, 1, 1)             # :53
    d2 = dc * dc + dr * dr
    return torch.exp(-torch.pow(d2 / _sigma_f32(sigma), 2))         # :58


def rasterize_depth(points: torch.Tensor, depth_vals: torch.Tensor, sigma, texture_size) -> torch.Tensor:
    """rasterize_depth (graphics/rasterization.py:66-104): the dense point splat, normalised by its per-point maximum
    over the frame (:96-99), scaled by the point's depth (:104).  ``depth_vals`` is ``[N,1]``."""
    g = splat_dense(points, sigma, texture_size)
    g = g / g.max(dim=2, keepdim=True)[0].max(dim=1, keepdim=True)[0]
    return g * depth_vals.to(F32).unsqueeze(-1)


def subsampled_point_raster(ndc_points: torch.Tensor, num_subsamples: int, sigma, sensor_size) -> List[torch.Tensor]:
    """subsampled_point_raster (graphics/rasterization.py:538-549): soft-OR (keepdim) of rasterize_depth at
    ``sensor_size // 2**i``."""
    out = []
    ss = torch.as_tensor(sensor_size)
    for i in range(num_subsamples):
        d = rasterize_depth(ndc_points[:, 0:2], ndc_points[:, 2:3], sigma, ss // 2 ** i)
        out.append((1 - torch.prod(1 - d, dim=0, keepdim=True)))
    return out


# ----------------------------------------------------------------------------
# a3-a5: footprint-limited ("baked") splat-reduce
# (fireflies/graphics/rasterization.py:164-237, 240-318, 321-392, 395-472)
# ----------------------------------------------------------------------------
def footprint_size(sigma, num_std: int) -> Tuple[int, int]:
    """(footprint, half) -- graphics/rasterization.py:180-182 (odd(floor(sqrt(sigma))*num_std))."""
    root = float(torch.sqrt(_sigma_f32(sigma)).item())
    fp = math.floor(root) * int(num_std)
    if fp % 2 == 0:
        fp += 1
    return fp, int((fp - 1) / 2)


def baked_windows(points: torch.Tensor, sigma, texture_size, num_std: int) -> torch.Tensor:
    """Integer clip rectangles of every point's footprint: int32 ``[N, 2, 3]`` = per axis
    ``(wo, rs, re)`` -- the texture origin, footprint start and footprint end that the
    reference slices with (graphics/rasterization.py:199-230 / 275-304).  Axis 0 pairs with
    ``points[:,0]`` / ``texture_size[0]``.  These are the "index outputs" of the splat path
    and are compared bit-exactly.
    """
    ts0, ts1 = _as_ts(texture_size)
    fp, half = footprint_size(sigma, num_std)
    P = points.detach().to(F32) * torch.tensor([ts0, ts1], dtype=F32)
    fo = torch.floor(P - half)                                      # :186 / :258
    out = torch.zeros(P.shape[0], 2, 3, dtype=torch.int32)
    for ax, ts in ((0, ts0), (1, ts1)):
        wo = fo[:, ax].to(torch.int32)
        rs = torch.where(wo < 0, wo.abs(), torch.zeros_like(wo))    # :214-220
        wo = torch.clamp(wo, min=0)
        re = torch.where(wo + fp >= ts, ts - wo, torch.full_like(wo, fp))  # :222-226
        out[:, ax, 0], out[:, ax, 1], out[:, ax, 2] = wo, rs, re
    return out


def _footprint_values(points: torch.Tensor, sigma, texture_size, num_std: int):
    """Per-point footprint values ``[N, fp, fp]`` (axis 1 <-> points[:,0]) and the
    texture index of every footprint cell plus a validity mask reproducing the
    reference's slice clipping."""
    ts0, ts1 = _as_ts(texture_size)
    fp, half = footprint_size(sigma, num_std)
    P = points.to(F32) * torch.tensor([ts0, ts1], dtype=F32)       # :174
    mid = P - torch.floor(P) + half                                 # :184 / :256
    k = torch.arange(fp, dtype=F32)
    d0 = k.view(1, fp, 1) - mid[:, 0].view(-1, 1, 1)                # :194 / :269
    d1 = k.view(1, 1, fp) - mid[:, 1].view(-1, 1, 1)                # :195 / :270
    d2 = d0 * d0 + d1 * d1
    u = d2 / _sigma_f32(sigma)
    vals = torch.exp(-(u * u))                                      # :197 / :273
    win = baked_windows(points, sigma, texture_size, num_std).to(torch.int64)
    ki = torch.arange(fp, dtype=torch.int64)
    idx, ok = [], []
    for ax in (0, 1):
        wo, rs, re = win[:, ax, 0:1], win[:, ax, 1:2], win[:, ax, 2:3]
        n = torch.clamp(re - rs, min=0)                             # slice length (empty if re<rs)
        inside = (ki.view(1, -1) >= rs) & (ki.view(1, -1) < rs + n)
        idx.append(wo + (ki.view(1, -1) - rs))
        ok.append(inside)
    tex_idx = idx[0].unsqueeze(2) * ts1 + idx[1].unsqueeze(1)       # tex is [ts0, ts1]
    mask = ok[0].unsqueeze(2) & ok[1].unsqueeze(1)
    mask = mask & (idx[0].unsqueeze(2) < ts0) & (idx[1].unsqueeze(1) < ts1)
    return vals, tex_idx, mask, (ts0, ts1)


def baked_sum(points, sigma, texture_size, num_std: int = 4, transposed: bool = False) -> torch.Tensor:
    """Footprint-limited ``sum``.  ``transposed=False`` gives baked_sum's orientation
    ``[ts1, ts0]`` (= ``splat_dense(...).sum(0)``, graphics/rasterization.py:237);
    ``transposed=True`` gives baked_sum_2's ``[ts0, ts1]`` (:318)."""
    vals, tex_idx, mask, (ts0, ts1) = _footprint_values(points, sigma, texture_size, num_std)
    tex = torch.zeros(ts0 * ts1, dtype=F32)
    tex = tex.index_put((tex_idx[mask],), vals[mask], accumulate=True)
    tex = tex.view(ts0, ts1)
    return tex if transposed else tex.T


def baked_softor(points, sigma, texture_size, num_std: int = 5) -> torch.Tensor:
    """Footprint-limited soft-OR, orientation ``[ts1, ts0]`` for both reference variants
    (graphics/rasterization.py:392, 472)."""
    vals, tex_idx, mask, (ts0, ts1) = _footprint_values(points, sigma, texture_size, num_std)
    tex = torch.ones(ts0 * ts1, dtype=F32)
    tex = tex.scatter_reduce(0, tex_idx[mask], 1 - vals[mask], reduce="prod", include_self=True)
    return (1 - tex.view(ts0, ts1)).T


def baked_sum_sequential(points, sigma, texture_size, num_std: int = 4) -> torch.Tensor:
    """Point-by-point variant (accumulation in index order like the reference's loop,
    graphics/rasterization.py:176-235); used on small cases to validate the scatter form."""
    vals, tex_idx, mask, (ts0, ts1) = _footprint_values(points, sigma, texture_size, num_std)
    tex = torch.zeros(ts0 * ts1, dtype=F32)
    for i in range(vals.shape[0]):
        tex = tex.index_put((tex_idx[i][mask[i]],), vals[i][mask[i]], accumulate=True)
    return tex.view(ts0, ts1).T


def baked_softor_sequential(points, sigma, texture_size, num_std: int = 5) -> torch.Tensor:
    vals, tex_idx, mask, (ts0, ts1) = _footprint_values(points, sigma, texture_size, num_std)
    tex = torch.ones(ts0 * ts1, dtype=F32)
    for i in range(vals.shape[0]):
        upd = torch.ones_like(tex).index_put((tex_idx[i][mask[i]],), 1 - vals[i][mask[i]])
        tex = tex * upd
    return (1 - tex.view(ts0, ts1)).T


def l1_loss(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """``torch.nn.L1Loss()(a, b)`` as used by test_point_reg (graphics/rasterization.py:591-599)."""
    return (a - b).abs().mean()


def splat_grad_analytic(points, sigma, texture_size, g_sum, g_softor,
                        num_std_sum: Optional[int] = None, num_std_softor: Optional[int] = None):
    """Closed-form ``d/d points`` of ``<g_sum, S> + <g_softor, O>`` in float64 (SURVEY 8(a) a7):
    ``dg/dp0 = 4 g u (c-P0) ts0 / sigma`` and ``dO/dg_n = prod_{m!=n}(1-g_m)``.
    Independent of torch autograd; windows ``None`` = dense.  ``g_sum``/``g_softor`` are in the
    dense ``[ts1, ts0]`` orientation."""
    ts0, ts1 = _as_ts(texture_size)
    sig = float(_sigma_f32(sigma))
    P = (points.detach().to(F32) * torch.tensor([ts0, ts1], dtype=F32)).double()
    c = torch.arange(ts0, dtype=torch.float64).view(1, 1, ts0)
    r = torch.arange(ts1, dtype=torch.float64).view(1, ts1, 1)
    dc = c - P[:, 0].view(-1, 1, 1)
    dr = r - P[:, 1].view(-1, 1, 1)
    u = (dc * dc + dr * dr) / sig
    g = torch.exp(-u * u)

    def window_mask(num_std):
        if num_std is None:
            return torch.ones_like(g, dtype=torch.bool)
        win = baked_windows(points, sigma, texture_size, num_std).to(torch.int64)
        ci = torch.arange(ts0).view(1, 1, ts0)
        ri = torch.arange(ts1).view(1, ts1, 1)
        lo0, n0 = win[:, 0, 0].view(-1, 1, 1), torch.clamp(win[:, 0, 2] - win[:, 0, 1], min=0).view(-1, 1, 1)
        lo1, n1 = win[:, 1, 0].view(-1, 1, 1), torch.clamp(win[:, 1, 2] - win[:, 1, 1], min=0).view(-1, 1, 1)
        return (ci >= lo0) & (ci < lo0 + n0) & (ri >= lo1) & (ri < lo1 + n1)

    ms, mo = window_mask(num_std_sum), window_mask(num_std_softor)
    om = torch.where(mo, 1 - g, torch.ones_like(g))
    excl = torch.empty_like(g)
    for n in range(g.shape[0]):
        others = torch.cat([om[:n], om[n + 1:]], dim=0)
        excl[n] = others.prod(dim=0) if others.shape[0] else torch.ones_like(g[0])
    coef = torch.zeros_like(g)
    if g_sum is not None:
        coef = coef + ms * g_sum.double().unsqueeze(0)
    if g_softor is not None:
        coef = coef + mo * g_softor.double().unsqueeze(0) * excl
    q = coef * 4.0 * g * u / sig
    d0 = (q * dc).sum(dim=(1, 2)) * ts0
    d1 = (q * dr).sum(dim=(1, 2)) * ts1
    return torch.stack([d0, d1], dim=1)


# ----------------------------------------------------------------------------
# a14-a17: math primitives, compose, vertex transform
# (fireflies/utils/math.py:24-60,170-175,199-235; entity/base.py:194-244; entity/mesh.py:131-165)
# ----------------------------------------------------------------------------
def _trig32(alpha) -> Tuple[float, float]:
    # utils/math.py:24-60: python math.cos/sin on the fp32 angle (fp64 trig), rounded to fp32
    a = float(alpha)
    return math.cos(a), math.sin(a)


def yaw(alpha) -> torch.Tensor:      # utils/math.py:24-34  (rotation about Z)
    c, s = _trig32(alpha)
    return torch.tensor([[c, -s, 0], [s, c, 0], [0, 0, 1]], dtype=F32)


def pitch(alpha) -> torch.Tensor:    # utils/math.py:37-47  (rotation about Y)
    c, s = _trig32(alpha)
    return torch.tensor([[c, 0, s], [0, 1, 0], [-s, 0, c]], dtype=F32)


def roll(alpha) -> torch.Tensor:     # utils/math.py:50-60  (rotation about X)
    c, s = _trig32(alpha)
    return torch.tensor([[1, 0, 0], [0, c, -s], [0, s, c]], dtype=F32)


def to_mat4(m3: torch.Tensor) -> torch.Tensor:     # utils/math.py:203-209
    out = torch.zeros(4, 4, dtype=F32)
    out[:3, :3] = m3
    out[3, 3] = 1.0
    return out


def rotation_from_sample(r: Sequence[float]) -> torch.Tensor:
    """entity/base.py:194-207: ``Pitch(r[2]) @ Yaw(r[1]) @ Roll(r[0])`` (so ``rotate_z`` spins about Y)."""
    return to_mat4(pitch(r[2]) @ yaw(r[1]) @ roll(r[0]))


def translation_from_sample(t: Sequence[float]) -> torch.Tensor:   # entity/base.py:209-218
    m = torch.eye(4, dtype=F32)
    m[0, 3], m[1, 3], m[2, 3] = float(t[0]), float(t[1]), float(t[2])
    return m


def scale_from_sample(s: Sequence[float]) -> torch.Tensor:         # entity/mesh.py:131-139
    m = torch.eye(4, dtype=F32)
    m[0, 0], m[1, 1], m[2, 2] = float(s[0]), float(s[1]), float(s[2])
    return m


def centroid_mat(c: Sequence[float]) -> torch.Tensor:              # entity/base.py:43,51-54
    m = torch.zeros(4, 4, dtype=F32)
    m[0, 3], m[1, 3], m[2, 3] = float(c[0]), float(c[1]), float(c[2])
    return m


def compose_world(t, r, s, centroid, world, has_scale: bool) -> torch.Tensor:
    """``(T + C) @ R [@ S] @ W``  (entity/mesh.py:145-150 with scale, entity/base.py:224-228 without)."""
    m = (translation_from_sample(t) + centroid_mat(centroid)) @ rotation_from_sample(r)
    if has_scale:
        m = m @ scale_from_sample(s)
    return m @ world.to(F32)


def chain_world(locals_: List[torch.Tensor], parent: Sequence[int]) -> List[torch.Tensor]:
    """``world = parent.world() @ local`` recursively (entity/base.py:239-244); parent[i] = -1 for roots."""
    out: List[Optional[torch.Tensor]] = [None] * len(locals_)

    def rec(i):
        if out[i] is None:
            out[i] = locals_[i].clone() if parent[i] < 0 else rec(parent[i]) @ locals_[i]
        return out[i]

    return [rec(i) for i in range(len(locals_))]


def transform_points(points: torch.Tensor, T: torch.Tensor) -> torch.Tensor:
    """utils/math.py:220-228: homogeneous ``T @ [x,y,z,1]`` then divide by w."""
    ph = torch.cat([points.to(F32), torch.ones(points.shape[0], 1, dtype=F32)], dim=1)
    q = torch.matmul(T.to(F32).unsqueeze(0), ph.unsqueeze(-1)).squeeze(-1)
    return q[:, :3] / q[:, 3:4]


def transform_directions(dirs: torch.Tensor, T: torch.Tensor) -> torch.Tensor:
    """utils/math.py:231-235: ``T @ [x,y,z,0]``, no divide."""
    dh = torch.cat([dirs.to(F32), torch.zeros(dirs.shape[0], 1, dtype=F32)], dim=1)
    q = torch.matmul(T.to(F32).unsqueeze(0), dh.unsqueeze(-1)).squeeze(-1)
    return q[:, :3]


def uniform_between(a: torch.Tensor, b: torch.Tensor, u: torch.Tensor) -> torch.Tensor:
    """utils/math.py:170-175 with the ``torch.rand`` variates ``u`` injected: ``u*(b-a)+a``."""
    assert a.shape == b.shape
    return u.to(F32) * (b.to(F32) - a.to(F32)) + a.to(F32)


# ----------------------------------------------------------------------------
# a11-a13: sampler state machines, reproducing the aliasing quirks
# (fireflies/sampling/base.py:54-74, uniform_scalar_to_vec3.py:18-38, animation.py:27-45)
# ----------------------------------------------------------------------------
class EvalStepper:
    """Bit-reproduction of ``Sampler.sample_eval`` (sampling/base.py:64-74) *including* its
    aliasing: the returned value is the post-increment ``_current_step``; on wrap
    ``_current_step`` aliases ``_min_range`` so later increments drift the range itself and
    wrapping is decided against the (un-drifted) ``_max_range``.  ``start`` is the value
    ``_current_step`` was cloned from at construction (sampling/base.py:26-30)."""

    def __init__(self, min_range, max_range, start, step: float = 0.01):
        self.min = torch.as_tensor(min_range, dtype=F32).clone().reshape(-1)
        self.max = torch.as_tensor(max_range, dtype=F32).clone().reshape(-1)
        self.cur = torch.as_tensor(start, dtype=F32).clone().reshape(-1)
        self.step = step
        self.aliased = False

    def sample(self) -> torch.Tensor:
        if bool((self.min == self.max).all()):                      # :65-66
            return self.min.clone()
        self.cur += self.step                                       # :68-69 (alias -> post-increment)
        if self.aliased:
            self.min = self.cur                                     # same storage in the reference
        ret = self.cur
        if bool((self.cur > self.max).any()):                       # :71-72
            self.cur = self.min
            self.aliased = True
            # reference returns the tensor object that held the overflowing value
        return ret.clone()


class AnimationStepper:
    """sampling/animation.py:27-37: eval walks ``min..max`` inclusive; train = ``random.randint``."""

    def __init__(self, min_train, max_train, min_eval, max_eval, step: int = 1):
        self.min_train, self.max_train = int(min_train), int(max_train)
        self.min_eval, self.max_eval = int(min_eval), int(max_eval)
        self.step = int(step)
        self.cur = int(min_eval)

    def sample_eval(self) -> int:
        s = self.cur
        self.cur += self.step
        if self.cur > self.max_eval:
            self.cur = self.min_eval
        return s

    def sample_train(self, rng: _pyrandom.Random = _pyrandom) -> int:
        return rng.randint(self.min_train, self.max_train - 1)


# ----------------------------------------------------------------------------
# a8/a9: laser <-> NDC glue  (fireflies/projection/laser.py:19-37,199-206,262-296; utils/io.py:14-68)
# ----------------------------------------------------------------------------
def build_projection_matrix(fov_deg: float, near: float, far: float) -> torch.Tensor:
    """utils/io.py:14-68 (pytorch3d-style K mapping to NDC [-1,1]); Mitsuba-free stand-in."""
    K = torch.zeros(4, 4, dtype=F32)
    t = torch.tan(torch.tensor((math.pi / 180) * fov_deg) / 2.0)
    max_y = t * near
    min_y = -max_y
    max_x = max_y * 1.0
    min_x = -max_x
    K[0, 0] = 2.0 * near / (max_x - min_x)
    K[1, 1] = 2.0 * near / (max_y - min_y)
    K[0, 2] = (max_x + min_x) / (max_x - min_x)
    K[1, 2] = (max_y + min_y) / (max_y - min_y)
    K[3, 2] = -1.0
    K[2, 2] = -1.0 * far / (far - near)
    K[2, 3] = -(far * near) / (far - near)
    return K


def uniform_rays(angle: float, nx: int, ny: int) -> torch.Tensor:
    """projection/laser.py:19-37 -- row index is ``x*nx + y`` (only a bijection for nx == ny)."""
    rays = torch.zeros(nx * ny, 3, dtype=F32)
    for x in range(nx):
        for y in range(ny):
            rays[x * nx + y] = torch.tensor(
                [math.tan((x - (nx - 1) / 2) * angle), math.tan((y - (ny - 1) / 2) * angle), -1.0])
    return rays / torch.linalg.norm(rays, dim=-1, keepdim=True)


_FLIP_Y = torch.diag(torch.tensor([1.0, -1.0, 1.0, 1.0]))


def rays_to_ndc(rays: torch.Tensor, K: torch.Tensor) -> torch.Tensor:
    """projection/laser.py:262-275."""
    return transform_points(rays, K.to(F32) @ _FLIP_Y)


def ndc_to_world(points: torch.Tensor, K: torch.Tensor) -> torch.Tensor:
    """projection/laser.py:277-290."""
    return transform_points(points, (K.to(F32) @ _FLIP_Y).inverse())


def clamp_to_fov(rays: torch.Tensor, K: torch.Tensor, clamp_val: float = 0.95) -> torch.Tensor:
    """projection/laser.py:199-206 (returns the new, renormalised rays)."""
    ndc = rays_to_ndc(rays, K)
    ndc[:, 0:2] = torch.clamp(ndc[:, 0:2], 1 - clamp_val, clamp_val)
    w = ndc_to_world(ndc, K)
    return w / torch.linalg.norm(w, dim=-1, keepdim=True)


# ----------------------------------------------------------------------------
# a19-a21: post-processing  (fireflies/postprocessing/*.py; kornia 0.7.1 restated)
# ----------------------------------------------------------------------------
def gaussian_kernel1d(ksize: int, sigma: float) -> torch.Tensor:
    """kornia 0.7.1 ``get_gaussian_kernel1d``: ``x = i - k//2`` (+0.5 for even k),
    ``exp(-x^2 / (2 sigma^2))`` normalised to sum 1.  kornia itself is not installed; the taps are pinned against
    ``cv2.getGaussianKernel`` (tests/test_oracle_golden.py::test_blur_restatement_against_opencv_and_scipy)."""
    x = torch.arange(ksize, dtype=F32) - ksize // 2
    if ksize % 2 == 0:
        x = x + 0.5
    g = torch.exp(-x.pow(2.0) / (2 * float(sigma) ** 2))
    return g / g.sum()


def gaussian_blur2d(img: torch.Tensor, kernel_size: Tuple[int, int], sigma: Tuple[float, float]) -> torch.Tensor:
    """kornia 0.7.1 ``filters.gaussian_blur2d(x, (ky,kx), (sy,sx))`` with its defaults
    ``border_type='reflect'``, ``separable=True`` -- restated as reflect padding followed by a
    horizontal then a vertical 1-D correlation (postprocessing/gauss_blur.py:18-28 call site).
    ``img`` is ``[..., H, W]``.  Pinned against two independent implementations that are in the image:
    ``cv2.GaussianBlur(BORDER_REFLECT_101)`` and ``scipy.ndimage.correlate1d(mode="mirror")``; the residual caveat is
    only that kornia 0.7.1's defaults are as recalled (reflect border, separable)."""
    ky, kx = int(kernel_size[0]), int(kernel_size[1])
    sy, sx = float(sigma[0]), float(sigma[1])
    lead = img.shape[:-2]
    x = img.to(F32).reshape(-1, 1, img.shape[-2], img.shape[-1])
    wx = gaussian_kernel1d(kx, sx).view(1, 1, 1, kx)
    wy = gaussian_kernel1d(ky, sy).view(1, 1, ky, 1)
    x = torch.nn.functional.pad(x, (kx // 2, (kx - 1) // 2, 0, 0), mode="reflect")
    x = torch.nn.functional.conv2d(x, wx)
    x = torch.nn.functional.pad(x, (0, 0, ky // 2, (ky - 1) // 2), mode="reflect")
    x = torch.nn.functional.conv2d(x, wy)
    return x.reshape(*lead, x.shape[-2], x.shape[-1])


def white_noise(img: np.ndarray, noise: np.ndarray) -> np.ndarray:
    """postprocessing/white_noise.py:16-20 with the normal variates injected (already scaled
    by ``mean``/``std``): fp64 draw added into the fp32 image, then clip to [0,1]."""
    out = img.astype(np.float32, copy=True)
    out += noise
    return np.clip(out, 0, 1)


def post_process(img: np.ndarray, blur: Optional[dict], noise: Optional[dict], gates: Sequence[bool],
                 noise_values: Optional[np.ndarray] = None) -> np.ndarray:
    """PostProcessor.post_process (postprocessing/postprocessor.py:14-19) for the chain
    ``[GaussianBlur, WhiteNoise]`` with the Bernoulli gates (postprocessing/base.py:10-14) injected."""
    out = img.copy()
    gi = 0
    if blur is not None:
        if gates[gi]:
            out = gaussian_blur2d(torch.tensor(out), blur["kernel_size"], blur["sigma"]).numpy()
        gi += 1
    if noise is not None:
        if gates[gi]:
            out = white_noise(out, noise_values)
        gi += 1
    return out


def bernoulli_gates(probabilities: Sequence[float], rng: _pyrandom.Random) -> List[bool]:
    """postprocessing/base.py:10-11: one ``random.uniform(0,1) < p`` per function, in chain order."""
    return [rng.uniform(0, 1) < p for p in probabilities]


# ----------------------------------------------------------------------------
# f4: Perlin material textures (SURVEY 8(f) row 4)
# (fireflies/sampling/noise_texture_lerp.py:8-98)
# ----------------------------------------------------------------------------
def perlin_2d(shape, res, angles01: torch.Tensor) -> torch.Tensor:
    """rand_perlin_2d (noise_texture_lerp.py:8-50) with its ``torch.rand(res[0]+1, res[1]+1)`` draw passed in."""
    import math
    fade = lambda t: 6 * t ** 5 - 15 * t ** 4 + 10 * t ** 3  # noqa: E731  (:8)
    delta = (res[0] / shape[0], res[1] / shape[1])
    d = (shape[0] // res[0], shape[1] // res[1])
    grid = torch.stack(torch.meshgrid(torch.arange(0, res[0], delta[0]), torch.arange(0, res[1], delta[1]), indexing="ij"), dim=-1) % 1
    angles = 2 * math.pi * angles01
    gradients = torch.stack((torch.cos(angles), torch.sin(angles)), dim=-1)

    def tile_grads(s1, s2):
        return gradients[s1[0]:s1[1], s2[0]:s2[1]].repeat_interleave(d[0], 0).repeat_interleave(d[1], 1)

    def dot(grad, shift):
        return (torch.stack((grid[:shape[0], :shape[1], 0] + shift[0], grid[:shape[0], :shape[1], 1] + shift[1]), dim=-1)
                * grad[:shape[0], :shape[1]]).sum(dim=-1)

    n00 = dot(tile_grads([0, -1], [0, -1]), [0, 0])
    n10 = dot(tile_grads([1, None], [0, -1]), [-1, 0])
    n01 = dot(tile_grads([0, -1], [1, None]), [0, -1])
    n11 = dot(tile_grads([1, None], [1, None]), [-1, -1])
    t = fade(grid[:shape[0], :shape[1]])
    return math.sqrt(2) * torch.lerp(torch.lerp(n00, n10, t[..., 0]), torch.lerp(n01, n11, t[..., 0]), t[..., 1])


def perlin_octaves(shape, res, octaves: int, persistence: float, angles: List[torch.Tensor]) -> torch.Tensor:
    """rand_perlin_2d_octaves (noise_texture_lerp.py:53-62)."""
    noise = torch.zeros(shape)
    frequency, amplitude = 1, 1
    for o in range(octaves):
        noise += amplitude * perlin_2d(shape, (frequency * res[0], frequency * res[1]), angles[o])
        frequency *= 2
        amplitude *= persistence
    return noise


def noise_texture_lerp(noise: torch.Tensor, color_a: torch.Tensor, color_b: torch.Tensor) -> torch.Tensor:
    """NoiseTextureLerpSampler.sample_train after the noise (noise_texture_lerp.py:86-98)."""
    tex = (noise - noise.min()) / (noise.max() - noise.min())
    col_a = torch.ones_like(tex).unsqueeze(0).repeat(3, 1, 1) * color_a.unsqueeze(-1).unsqueeze(-1)
    col_b = torch.ones_like(tex).unsqueeze(0).repeat(3, 1, 1) * color_b.unsqueeze(-1).unsqueeze(-1)
    return torch.lerp(col_a, col_b, tex.unsqueeze(0).repeat(3, 1, 1))


def silhouette(image: torch.Tensor, cx: int, cy: int, r: int) -> torch.Tensor:
    """ApplySilhouette.post_process (postprocessing/apply_silhouette.py:17-40) with the disc drawn analytically
    (``(x-cx)^2 + (y-cy)^2 <= r^2``, which is exactly what the filled ``cv2.circle`` rasterises -- pinned against the reference
    run with the real OpenCV, tests/golden/postprocess.npz::silhouette_*), blurred with the restated kornia
    gaussian_blur2d (11,11)/(5,5) and multiplied into the image."""
    H, W = image.shape
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    mask = (((xx - cx) ** 2 + (yy - cy) ** 2) <= r * r).to(F32)
    return image * gaussian_blur2d(mask, (11, 11), (5.0, 5.0))


# ----------------------------------------------------------------------------
# NURBS-curve camera path  (fireflies/entity/curve.py:48-96, utils/io.py:77-108)
# ----------------------------------------------------------------------------
# The curve arithmetic lives in geomdl==5.3.1 (requirements.txt:16), which is NOT under /root/reference and is not
# installed.  The evaluator is pinned against an independent implementation that is in the image (scipy.interpolate.BSpline on
# homogeneous control points, tests/test_oracle_golden.py::test_nurbs_evaluator_against_scipy_bspline); what stays unpinned is
# only geomdl's conventions around it, as recalled.  It is restated from the published algorithms geomdl implements
# (Piegl & Tiller, "The NURBS Book": knot span search, A2.2 BasisFuns, A4.1 CurvePoint) with geomdl's conventions as
# recalled from its 5.3.1 sources: knot vectors are normalised to [0, 1] on assignment, the span is found by a linear
# walk, evaluation is Python floats (fp64), control points without weights get weight 1.  Anchors: Bernstein closed
# form, the rational quadratic arc, partition of unity (tests/test_oracle_golden.py) and the reference's own Curve
# methods run on top of this evaluator (oracle/make_golden.py::curve_cases).
def nurbs_normalize_knots(knots: Sequence[float]) -> List[float]:
    k0, k1 = float(knots[0]), float(knots[-1])
    return [float("{:.18f}".format((float(k) - k0) / (k1 - k0))) for k in knots]


def nurbs_find_span(degree: int, knots: Sequence[float], n_ctrl: int, t: float) -> int:
    span = degree + 1
    while span < n_ctrl and knots[span] <= t:
        span += 1
    return span - 1


def nurbs_basis(degree: int, knots: Sequence[float], span: int, t: float) -> List[float]:
    """The degree+1 non-vanishing B-spline basis functions at t (NURBS Book A2.2)."""
    left, right, N = [0.0] * (degree + 1), [0.0] * (degree + 1), [1.0] * (degree + 1)
    for j in range(1, degree + 1):
        left[j] = t - knots[span + 1 - j]
        right[j] = knots[span + j] - t
        saved = 0.0
        for r in range(j):
            temp = N[r] / (right[r + 1] + left[j - r])
            N[r] = saved + right[r + 1] * temp
            saved = left[j - r] * temp
        N[j] = saved
    return N


def nurbs_curve_point(ctrlpts: Sequence[Sequence[float]], knots: Sequence[float], degree: int, t: float,
                      weights: Optional[Sequence[float]] = None) -> List[float]:
    """Rational curve point in fp64 (NURBS Book A4.1): ``knots`` already normalised, ``t`` in [0, 1]."""
    n = len(ctrlpts)
    w = [1.0] * n if weights is None else [float(x) for x in weights]
    span = nurbs_find_span(degree, knots, n, t)
    N = nurbs_basis(degree, knots, span, t)
    acc = [0.0, 0.0, 0.0, 0.0]
    for i in range(degree + 1):
        c = span - degree + i
        pw = [float(ctrlpts[c][0]) * w[c], float(ctrlpts[c][1]) * w[c], float(ctrlpts[c][2]) * w[c], w[c]]
        for d in range(4):
            acc[d] = acc[d] + N[i] * pw[d]
    return [acc[0] / acc[3], acc[1] / acc[3], acc[2] / acc[3]]


def rotation_matrix_from_vectors(v1: torch.Tensor, v2: torch.Tensor) -> torch.Tensor:
    """utils/math.py:67-105 (Rodrigues), fp32."""
    v1 = torch.nn.functional.normalize(v1, dim=0)
    v2 = torch.nn.functional.normalize(v2, dim=0)
    c = torch.linalg.cross(v1, v2)
    d = torch.dot(v1, v2)
    K = torch.tensor([[0, -c[2], c[1]], [c[2], 0, -c[0]], [-c[1], c[0], 0]], dtype=F32)
    return torch.eye(3) + K + torch.mm(K, K) * (1 - d) / torch.norm(c) ** 2


def rotation_matrix_from_vectors_with_fixed_up(v1, v2, up=None) -> torch.Tensor:
    """utils/math.py:108-159: the Rodrigues matrix is computed and then DISCARDED -- the function returns
    ``eye + normalize(K, dim=0) * acos(dot(R @ up, up))`` (column-normalised skew matrix times the correction angle)."""
    up = torch.tensor([0.0, 0.0, 1.0]) if up is None else up
    v1n = torch.nn.functional.normalize(v1, dim=0)
    v2n = torch.nn.functional.normalize(v2, dim=0)
    up = torch.nn.functional.normalize(up, dim=0)
    c = torch.linalg.cross(v1n, v2n)
    K = torch.tensor([[0, -c[2], c[1]], [c[2], 0, -c[0]], [-c[1], c[0], 0]], dtype=F32)
    R = rotation_matrix_from_vectors(v1, v2)
    angle = torch.acos(torch.dot(torch.mv(R, up), up))
    return torch.eye(3) + torch.nn.functional.normalize(K, dim=0) * angle


def curve_pose(ctrlpts, knots, degree: int, t: float, world: torch.Tensor, weights=None, dt: float = 0.001) -> torch.Tensor:
    """Curve.randomize's matrix (entity/curve.py:48-96): ``T(C(t)) @ toMat4x4(R([0,1,0] -> d)) @ W`` with
    ``d = C(t + dt) - C(t)`` (fp32 difference of the fp64 points rounded to fp32), x and z negated."""
    p1 = torch.tensor(nurbs_curve_point(ctrlpts, knots, degree, t + dt, weights), dtype=F32)
    p0 = torch.tensor(nurbs_curve_point(ctrlpts, knots, degree, t, weights), dtype=F32)
    d = p1 - p0
    d[0] *= -1.0
    d[2] *= -1.0
    R = to_mat4(rotation_matrix_from_vectors(torch.tensor([0.0, 1.0, 0.0]), d))
    T = torch.eye(4)
    T[0:3, 3] = p0
    return T @ R @ world


# ----------------------------------------------------------------------------
# Poisson-disk initialisation  (fireflies/sampling/poisson.py:16-116, projection/laser.py:94-145)
# ----------------------------------------------------------------------------
def bridson(radius: np.ndarray, k: int = 30, rng=np.random):
    """Bridson's Poisson-disk sampling with a per-cell radius map, consuming the numpy stream draw for draw like the
    reference: 2 draws for the seed point, then per round one ``randint`` (which active point) and per attempt one draw
    for the distance in [r, 2r) and one for the angle; a round does not stop at its first accepted point; an active point
    is retired only when all k attempts failed.  Occupancy test: any occupied cell in the square window of half-width
    ``ceil(r)`` around the candidate's cell (poisson.py:82-98)."""
    H, W = radius.shape
    occ = np.zeros((H, W), dtype=bool)
    first = (rng.random() * H, rng.random() * W)
    occ[int(np.floor(first[0])), int(np.floor(first[1]))] = True
    active, pts = [first], [first]
    while active:
        a = rng.randint(len(active))
        ay, ax = active[a]
        cy, cx = int(np.floor(ay)), int(np.floor(ax))
        found = False
        for _ in range(k):
            dist = radius[cy, cx] * (rng.random() + 1)
            ang = 2 * np.pi * rng.random()
            ny, nx = ay + dist * np.sin(ang), ax + dist * np.cos(ang)
            if not (0 <= nx <= W and 0 <= ny <= H):
                continue
            gy, gx = int(np.floor(ny)), int(np.floor(nx))
            rr = int(np.ceil(radius[gy, gx]))     # IndexError at ny == H / nx == W exactly, like the reference
            if occ[max(gy - rr, 0):min(gy + rr + 1, H), max(gx - rr, 0):min(gx + rr + 1, W)].any():
                continue
            active.append((ny, nx)); pts.append((ny, nx))
            occ[gy, gx] = True
            found = True
        if not found:
            del active[a]
    return len(pts), np.array(pts)


def blue_noise_rays(samples: np.ndarray, image_size_x: int, image_size_y: int, K: torch.Tensor) -> torch.Tensor:
    """Laser.generate_blue_noise_rays after the sampler (laser.py:115-145): samples / size -> (x, y, -1) -> K^-1 ->
    normalise -> flip z.  ``torch.tensor(fp64 samples)`` stays fp64 until it is copied into the fp32 ray tensor."""
    ps = torch.tensor(samples) / torch.tensor([image_size_x, image_size_y])
    temp = torch.ones([ps.shape[0], 3]) * -1.0
    temp[:, 0:2] = ps
    rays = transform_points(temp, K.inverse())
    rays = rays / torch.linalg.norm(rays, dim=-1, keepdims=True)
    rays[:, 2] *= -1.0
    return rays


def poisson_radius(image_size_x: int, image_size_y: int, num_beams: int) -> float:
    r = math.sqrt((image_size_x * image_size_y) / (math.pi * num_beams))    # laser.py:109-112
    return r + r / 4.0


# ----------------------------------------------------------------------------
# Batched intersections  (fireflies/utils/intersections.py:5-33)
# ----------------------------------------------------------------------------
def ray_plane(origin, direction, plane_origin, plane_normal) -> torch.Tensor:
    denom = torch.sum(plane_normal * direction, dim=1)
    denom = torch.where(torch.abs(denom) < 0.000001, denom / denom, denom)     # 0/0 -> NaN for exactly parallel rays
    return (torch.sum((plane_origin - origin) * plane_normal, dim=1) / denom)[:, None]


def sphere_sphere(a, ra, b, rb) -> torch.Tensor:
    return (a - b).pow(2).sum(dim=1, keepdim=True) <= (ra + rb).pow(2)
