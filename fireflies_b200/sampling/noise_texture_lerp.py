"""``fireflies/sampling/noise_texture_lerp.py`` -- Perlin-noise material textures, same interface.

The octave sum, the min/max normalisation and the colour lerp run in libffb200 (``ffb_perlin_texture``).  The random
draws are made exactly where the reference makes them -- ``random.randint`` / ``random.uniform`` for the lattice
resolution, octave count and persistence, ``torch.rand`` on the CPU generator for the lattice angles
(noise_texture_lerp.py:21,77-79) -- so a seeded run consumes both streams identically.

:func:`perlin_texture_batch` makes B textures in one call (``ffb_perlin_texture_batch``), with the parameters and
lattice angles either given or drawn on the device from Philox; ``SceneBatch`` uses it for texture samplers.
"""
from __future__ import annotations

import ctypes as C
import random
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import torch

from .. import _native as nat
from . import base


def perlin_angles(res, octaves: int) -> List[torch.Tensor]:
    """The ``torch.rand(res[0]+1, res[1]+1)`` draws of rand_perlin_2d_octaves, octave by octave (:21, :57-61)."""
    out, f = [], 1
    for _ in range(octaves):
        out.append(torch.rand(f * res[0] + 1, f * res[1] + 1))
        f *= 2
    return out


def perlin_texture(shape, res, octaves: int, persistence: float, angles: List[torch.Tensor], color_a=None, color_b=None,
                   device=torch.device("cuda")):
    """``rand_perlin_2d_octaves(shape, res, octaves, persistence)`` from given lattice draws -> ``(noise [H,W], texture
    [3,H,W] or None)``; the texture is ``lerp(color_a, color_b, (noise - min) / (max - min))`` (:80-98)."""
    H, W = int(shape[0]), int(shape[1])
    ang = torch.cat([a.reshape(-1).float() for a in angles]).to(device)
    noise = torch.empty((H, W), dtype=torch.float32, device=device)
    mm = torch.empty(2, dtype=torch.int32, device=device)
    out = ca = cb = None
    if color_a is not None:
        ca = nat.require_cuda(color_a.detach().float().reshape(3).contiguous().to(device), torch.float32, "color_a")
        cb = nat.require_cuda(color_b.detach().float().reshape(3).contiguous().to(device), torch.float32, "color_b")
        out = torch.empty((3, H, W), dtype=torch.float32, device=device)
    nat.check(nat.lib().ffb_perlin_texture(ang.data_ptr(), H, W, int(res[0]), int(res[1]), int(octaves), float(persistence),
                                           nat.ptr(ca), nat.ptr(cb), noise.data_ptr(), mm.data_ptr(), nat.ptr(out), nat.stream()),
              "ffb_perlin_texture")
    nat.count(3 if out is not None else 2)
    return noise, out


PERLIN_TILE = 512      # FFB_PERLIN_TILE: drawn textures need H and W multiples of this (64 * 2^3, the largest res * 2^(octaves-1))


@dataclass
class PerlinDraws:
    """The parameters and device buffers of B textures made by :func:`perlin_texture_batch`."""
    noise: torch.Tensor      # [B,H,W] octave sums
    minmax: torch.Tensor     # [B,2] int32, ordered-int extrema of each sample's noise
    raw: torch.Tensor        # [B,8] int32: ffb_perlin_params per sample

    @property
    def res(self) -> torch.Tensor:
        """[B,2] int32 lattice resolution (drawn: ``2^k`` twice)."""
        return self.raw[:, 0:2]

    @property
    def octaves(self) -> torch.Tensor:
        return self.raw[:, 2]

    @property
    def persistence(self) -> torch.Tensor:
        return self.raw.view(torch.float64)[:, 2]

    @property
    def angle_offset(self) -> torch.Tensor:
        return self.raw.view(torch.int64)[:, 3]


def _colour(c, device) -> torch.Tensor:
    return torch.as_tensor(c).detach().to(device=device, dtype=torch.float32).reshape(3).contiguous()


def perlin_texture_batch(shape, B: int, color_a, color_b, *, seed: int, sample0: int, row: int = 0,
                         params: Optional[Sequence[Tuple]] = None, angles: Optional[Sequence[List[torch.Tensor]]] = None,
                         out: Optional[Tuple[torch.Tensor, PerlinDraws]] = None, device=torch.device("cuda")):
    """B textures ``lerp(color_a, color_b, (noise - min) / (max - min))`` -> ``(textures [B,3,H,W], draws)``.

    Drawn (``params=None``): sample ``b`` is keyed by ``(seed, sample0 + b, row)`` (include/ffb200.h gives the Philox
    keying), so the result does not depend on how samples are split over calls; ``H`` and ``W`` must be multiples of
    512.  Injected: ``params[b] = (res, octaves, persistence)`` (``res`` an int or a pair) and ``angles[b]`` the list
    :func:`perlin_angles` returns; each sample then equals :func:`perlin_texture` of the same draws bit for bit.
    ``out``: the return value of an earlier call with the same ``B`` and shape, overwritten in place."""
    H, W, B = int(shape[0]), int(shape[1]), int(B)
    dev = torch.device(device)
    if out is None:
        tex = torch.empty((B, 3, H, W), dtype=torch.float32, device=dev)
        draws = PerlinDraws(torch.empty((B, H, W), dtype=torch.float32, device=dev),
                            torch.empty((B, 2), dtype=torch.int32, device=dev),
                            torch.zeros((B, 8), dtype=torch.int32, device=dev))
    else:
        tex, draws = out
        if tuple(tex.shape) != (B, 3, H, W) or tuple(draws.noise.shape) != (B, H, W):
            raise ValueError(f"perlin_texture_batch: `out` holds {tuple(tex.shape)} textures, not {(B, 3, H, W)}")
    ca, cb = _colour(color_a, dev), _colour(color_b, dev)
    host, ang = None, None
    if params is not None:
        if angles is None or len(params) != B or len(angles) != B:
            raise ValueError("perlin_texture_batch: injected mode needs B parameter tuples and B angle lists")
        host, flat, off = (nat.PerlinParams * B)(), [], 0
        for b, ((res, octaves, persistence), a) in enumerate(zip(params, angles)):
            r0, r1 = (res, res) if isinstance(res, int) else res
            host[b] = nat.PerlinParams(int(r0), int(r1), int(octaves), 0, float(persistence), off)
            flat.append(torch.cat([x.reshape(-1).float() for x in a]))
            off += flat[-1].numel()
        ang = torch.cat(flat).to(dev)
    elif angles is not None:
        raise ValueError("perlin_texture_batch: angles are drawn on the device unless params are given")
    nat.check(nat.lib().ffb_perlin_texture_batch(B, H, W, int(seed), int(sample0), int(row),
                                                 None if host is None else C.cast(host, C.c_void_p), nat.ptr(ang),
                                                 0 if ang is None else ang.numel(), draws.raw.data_ptr(), ca.data_ptr(),
                                                 cb.data_ptr(), draws.noise.data_ptr(), draws.minmax.data_ptr(), tex.data_ptr(),
                                                 nat.stream()), "ffb_perlin_texture_batch")
    nat.count(3)
    return tex, draws


def rand_perlin_2d(shape, res, fade=None, device=torch.device("cuda")) -> torch.Tensor:
    """noise_texture_lerp.py:8-50: one octave; draws ``torch.rand(res[0]+1, res[1]+1)`` like the reference.  Only the
    reference's default quintic fade is compiled into the kernel."""
    if fade is not None:
        raise NotImplementedError("rand_perlin_2d: only the default fade 6t^5 - 15t^4 + 10t^3 is supported")
    return perlin_texture(shape, res, 1, 1.0, perlin_angles(res, 1), device=device)[0]


def rand_perlin_2d_octaves(shape, res, octaves=1, persistence=0.5, device=torch.device("cuda")) -> torch.Tensor:
    """noise_texture_lerp.py:53-62."""
    return perlin_texture(shape, res, octaves, persistence, perlin_angles(res, octaves), device=device)[0]


class NoiseTextureLerpSampler(base.Sampler):
    _KIND = None          # no sampler-table record: its samples are textures; SceneBatch draws them with perlin_texture_batch
    def __init__(self, color_a: torch.Tensor, color_b: torch.Tensor, texture_shape: List[int], eval_step_size: float = 0.01,
                 device: torch.device = torch.device("cuda")) -> None:
        super().__init__(torch.tensor([0.0], device=device), torch.tensor([1.0], device=device), eval_step_size, device)
        self._color_a = color_a
        self._color_b = color_b
        self._texture_shape = texture_shape

    def sample_train(self) -> torch.Tensor:
        i = 2 ** random.randint(1, 6)
        octaves = random.randint(1, 4)
        persistence = random.uniform(0.1, 2.0)
        angles = perlin_angles((i, i), octaves)
        return perlin_texture(self._texture_shape, (i, i), octaves, persistence, angles, self._color_a, self._color_b, self._device)[1]

    # the reference's eval mode is its train mode (:100-102)
    def sample_eval(self) -> torch.Tensor:
        return self.sample_train()
