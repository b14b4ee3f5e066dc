"""B200-native batched path: randomise B scene samples and run the pattern-optimisation step in a handful
of launches.  This is what the reference's per-sample loop (``scene.randomize()`` -> render -> ``backward``,
SURVEY.md section 3 (C)-(E)) becomes when B samples are processed at once.

* :class:`SceneBatch`  -- ``Scene.randomize()`` for B samples: sampling (Philox / eval stepping), 4x4 compose
  with parent chains, vertex transform with animation gather, Perlin material textures.  3-4 launches (plus 3 per
  texture attribute), no host sync.
* :class:`PatternStep` -- splat fwd (sum + soft-OR) -> loss -> splat bwd -> fold over samples -> allreduce.
* :class:`TextureStep` -- the blurred projector texture from the laser rays, and its backward for B rendered samples.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from . import _native as nat
from .entity import Mesh, Transformable
from .entity.base import _ENT_INTS, _ENT_WORDS
from .graphics import rasterization as R
from .sampling import AnimationSampler, NoiseTextureLerpSampler, Sampler
from .sampling.base import _WORDS as _SMP_WORDS
from .sampling.base import rehome
from .sampling.noise_texture_lerp import PERLIN_TILE, perlin_texture_batch


@dataclass
class BatchResult:
    """B randomised scene samples on the device (see :class:`SceneBatch`)."""
    world: torch.Tensor                 # [B,E,4,4]
    sampled: torch.Tensor               # [B,S,3]
    vertices: Optional[torch.Tensor]    # [B,Vtot,3] (padded slots) or None
    batch: "SceneBatch"
    textures: Dict[Tuple[str, str], tuple] = field(default_factory=dict)   # (entity, key) -> ([B,3,H,W], PerlinDraws)

    def mesh_vertices(self, name: str) -> torch.Tensor:
        off, n = self.batch._mesh_slices[name]
        return self.vertices[:, off:off + n]

    def entity_world(self, name: str) -> torch.Tensor:
        return self.world[:, self.batch._entity_index[name]]

    def attribute(self, entity_name: str, key: str) -> torch.Tensor:
        """``[B,dim]`` sampled values, or ``[B,3,H,W]`` for a texture attribute."""
        if (entity_name, key) in self.textures:
            return self.textures[(entity_name, key)][0]
        row, dim = self.batch._attr_rows[(entity_name, key)]
        return self.sampled[:, row, :dim]

    # ---- hand-off to Mitsuba (SURVEY.md 8(f) row 1; reference: Scene.update_*, scene.py:243-342) ----------------------
    def to_host(self):
        """ONE device->host copy (pinned, asynchronous + one event wait) of every 4x4 matrix and sampled attribute of all B
        samples.  The reference pays a `.tolist()` / `.item()` sync per entity and attribute (scene.py:257-342).  Textures
        stay on the device."""
        if getattr(self, "_host", None) is None:
            B = self.world.shape[0]
            nw, ns = self.world[0].numel(), self.sampled[0].numel()
            stage = torch.empty((B, nw + ns), dtype=torch.float32, device=self.world.device)
            stage[:, :nw] = self.world.reshape(B, nw)
            stage[:, nw:] = self.sampled.reshape(B, ns)
            host = torch.empty((B, nw + ns), dtype=torch.float32, pin_memory=True)
            host.copy_(stage, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            self._host = (host[:, :nw].reshape(self.world.shape).numpy(), host[:, nw:].reshape(self.sampled.shape).numpy())
        return self._host

    def write_sample(self, b: int, update: bool = True) -> None:
        """Write scene sample ``b`` into the Mitsuba parameter map, like ``Scene.randomize()``'s update_* tail
        (scene.py:243-342, 371-384), from the host copy made by :meth:`to_host` -- no further device syncs.  Mesh vertices
        and textures are handed over as slices of the device buffers (``Float32`` / ``TensorXf`` take them through
        DLPack / ``__cuda_array_interface__`` without a copy)."""
        sb, sc = self.batch, self.batch.scene
        params, T = sc._mitsuba_params, sc._types
        world, sampled = self.to_host()
        for m in sb.meshes:
            off, n = sb._mesh_slices[m.name()]
            params[m.name() + ".vertex_positions"] = T.Float32(self.vertices[b, off:off + n].reshape(-1))
        for e in sb.entities:
            if isinstance(e, Mesh) or not e.randomizable():
                continue
            name = e.name()
            if name + ".to_world" in params.keys():
                params[name + ".to_world"] = T.Transform4f(world[b, sb._entity_index[name]].tolist())
        for (name, key), (row, dim) in sb._attr_rows.items():
            joined = name + "." + key
            tp = type(params[joined])
            params[joined] = tp(float(sampled[b, row, 0])) if dim == 1 else tp(sampled[b, row, :dim].tolist())
        for (name, key), (tex, _) in self.textures.items():
            joined = name + "." + key
            params[joined] = type(params[joined])(tex[b])
        if update:
            params.update()


class SceneBatch:
    def __init__(self, scene, seed: int = 0):
        self.scene = scene
        self.seed = int(seed)
        self.device = torch.device(scene.device())
        self._next_sample = 0
        # ---- entities, parents before children ----
        # The compose kernel walks the table once, so every parent row must precede its children -- whichever list the parent
        # lives in (a light parented to the camera, two children of one parent, ...): depth-first over the parent() links.
        pool: List[Transformable] = list(scene._meshes) + list(scene._lights)
        for e in (scene._camera, scene._projector):
            if e is not None:
                pool.append(e)
        ents: List[Transformable] = []

        def place(e, chain=()):
            if any(e is x for x in ents):
                return
            if any(e is x for x in chain):
                raise ValueError(f"SceneBatch: parent cycle through entity {e.name()!r}")
            par = e.parent()
            if par is not None:
                if not any(par is x for x in pool):
                    raise ValueError(f"SceneBatch: parent {par.name()!r} of {e.name()!r} is not an entity of this scene")
                place(par, chain + (e,))
            ents.append(e)

        for e in pool:
            place(e)
        self.entities = ents
        self._entity_index = {e.name(): i for i, e in enumerate(ents)}
        # ---- sampler table ----
        samplers: List[Sampler] = []
        self._attr_rows: Dict[Tuple[str, str], Tuple[int, int]] = {}
        # texture samplers get rows of their own, numbered in attribute order: (entity, key) -> (row, [H, W], color_a, color_b)
        self._textures: Dict[Tuple[str, str], tuple] = {}
        trs_rows = []
        for e in ents:
            rows = []
            for s in (e._translation_sampler, e._rotation_sampler, getattr(e, "_scale_sampler", None)):
                if s is None:
                    rows.append(-1)
                else:
                    rows.append(len(samplers))
                    samplers.append(s)
            trs_rows.append(rows)
        for e in ents + list(scene._materials):
            if isinstance(e, Mesh) or not e.randomizable():
                continue
            for key, s in list(e._float_attributes.items()) + list(e._vec3_attributes.items()):
                if isinstance(s, NoiseTextureLerpSampler):
                    self._add_texture(e.name(), key, s)
                    continue
                self._attr_rows[(e.name(), key)] = (len(samplers), 3 if getattr(s, "_KIND", None) == nat.SAMPLER_SCALAR_TO_VEC3 else s._dim)
                samplers.append(s)
        for s in samplers:
            if not isinstance(s, Sampler):
                raise TypeError("SceneBatch needs fireflies_b200.sampling.Sampler instances")
            if getattr(s, "_KIND", None) is None:
                raise NotImplementedError(f"SceneBatch: {type(s).__name__} has no device record (its samples are not 1-3 scalars); "
                                          "sample it per scene through its own sample() instead")
        self.samplers = samplers
        self.S = len(samplers)
        self.sampler_table = torch.zeros((max(self.S, 1), _SMP_WORDS), dtype=torch.int32, device=self.device)
        for i, s in enumerate(samplers):
            rehome(s, self.sampler_table[i])
        # ---- entity table ----
        self.E = len(ents)
        self._trs_rows = trs_rows
        self.entity_table = torch.zeros((max(self.E, 1), _ENT_WORDS), dtype=torch.int32, device=self.device)
        self.refresh()
        # ---- meshes ----
        self._mesh_slices: Dict[str, Tuple[int, int]] = {}
        self.meshes = [m for m in scene._meshes if m.randomizable()]
        self.mesh_tables: List[nat.MeshTable] = []
        self._frames_keepalive = []
        if self.meshes:
            self._build_meshes()

    def _add_texture(self, name: str, key: str, s: NoiseTextureLerpSampler) -> None:
        H, W = (int(x) for x in s._texture_shape)
        if H % PERLIN_TILE or W % PERLIN_TILE:
            raise ValueError(f"SceneBatch: the texture of {name}.{key} is {H}x{W}; batched Perlin textures need both sides to be "
                             f"multiples of {PERLIN_TILE} (the largest lattice resolution x 2^(octaves-1) the sampler draws)")
        colours = [torch.as_tensor(c).detach().to(self.device, torch.float32).reshape(3).contiguous() for c in (s._color_a, s._color_b)]
        self._textures[(name, key)] = (len(self._textures), (H, W), *colours)

    def refresh(self) -> None:
        """Re-read world matrices, centroids, flags and parent links from the python objects."""
        ints = np.full((max(self.E, 1), _ENT_INTS), -1, dtype=np.int32)
        cents, worlds = [], []
        for i, e in enumerate(self.entities):
            parent = -1
            if e.parent() is not None:
                parent = self._entity_index.get(e.parent().name(), -2)
                if not 0 <= parent < i:         # re-parented after construction: the row order no longer fits
                    raise ValueError(f"SceneBatch.refresh: parent {e.parent().name()!r} of {e.name()!r} does not precede it in the "
                                     "entity table; build a new SceneBatch after changing parent links")
            ints[i] = (e._KIND, parent, int(e.randomizable()), *self._trs_rows[i])
            cents.append(e._centroid_mat[0:3, 3].to(self.device).float())
            worlds.append(e._world.to(self.device).float().reshape(16))
        self.entity_table[:, :_ENT_INTS] = torch.from_numpy(ints).to(self.device)
        if self.E:
            fv = self.entity_table.view(torch.float32)
            fv[:, 6:9] = torch.stack(cents)
            fv[:, 10:26] = torch.stack(worlds)

    def _build_meshes(self) -> None:
        voff, chunks, anim = [0], [], []
        for m in self.meshes:
            if m._animated and m._animation_func is not None:
                raise NotImplementedError("python animation callbacks cannot be batched; use frame data")
            V = m._vertices.shape[0]
            slot = (V + 3) // 4 * 4                              # 16-byte aligned slots
            v = torch.zeros((slot, 3), dtype=torch.float32, device=self.device)
            v[:V] = m._vertices.float()
            chunks.append(v)
            self._mesh_slices[m.name()] = (voff[-1], V)
            voff.append(voff[-1] + slot)
            anim.append(m if (m._animated and m._anim_data_train is not None and m._anim_data_eval is not None) else None)
        self.verts = torch.cat(chunks)
        self.Vtot = voff[-1]
        self._anim_meshes = anim
        M = len(self.meshes)
        if M > nat.FFB_MAX_MESHES:
            raise NotImplementedError(f"more than {nat.FFB_MAX_MESHES} randomizable meshes per launch")
        self._voff = voff
        if any(a is not None for a in anim):
            self._anim_cur = torch.tensor([(a._animation_sampler._current_step if a is not None else 0) for a in anim],
                                          dtype=torch.int32, device=self.device)

    def _mesh_table(self, train: bool) -> nat.MeshTable:
        # the table only changes when a mesh's animation frames do: cache it per mode (keyed by the frame tensors' addresses)
        key = (train, tuple((id(a._anim_data_train), id(a._anim_data_eval)) if a is not None else None for a in self._anim_meshes))
        cached = getattr(self, "_mt_cache", {}).get(train)
        if cached is not None and cached[0] == key:
            return cached[1]
        mt = self._build_mesh_table(train)
        if not hasattr(self, "_mt_cache"):
            self._mt_cache, self._mt_keep = {}, {}
        self._mt_cache[train] = (key, mt)
        self._mt_keep[train] = list(self._frames_keepalive)
        return mt

    def _build_mesh_table(self, train: bool) -> nat.MeshTable:
        mt = nat.MeshTable()
        mt.M = len(self.meshes)
        self._frames_keepalive = []
        for i, m in enumerate(self.meshes):
            mt.voff[i] = self._voff[i]
            mt.entity[i] = self._entity_index[m.name()]
            a = self._anim_meshes[i]
            if a is not None:
                frames = a._anim_data_train if train else a._anim_data_eval
                V = m._vertices.shape[0]
                slot = self._voff[i + 1] - self._voff[i]
                if frames.shape[1] != slot:                      # pad frames to the slot size once
                    key = "_ffb_frames_train" if train else "_ffb_frames_eval"
                    if getattr(a, key, None) is None:
                        p = torch.zeros((frames.shape[0], slot, 3), dtype=torch.float32, device=self.device)
                        p[:, :V] = frames
                        setattr(a, key, p)
                    frames = getattr(a, key)
                self._frames_keepalive.append(frames)
                mt.nframes[i] = frames.shape[0]
                mt.frames[i] = frames.data_ptr()
            else:
                mt.nframes[i] = 0
                mt.frames[i] = None
        mt.voff[mt.M] = self._voff[mt.M]
        return mt

    def randomize(self, B: int, sample0: Optional[int] = None, variates: Optional[torch.Tensor] = None,
                  out: Optional[BatchResult] = None) -> BatchResult:
        """B scene samples.  Train mode: sample ``sample0 + b`` depends only on (seed, sample0 + b, sampler row)
        -- identical for any batch split or rank layout.  Eval mode: B successive ``sample_eval`` steps per
        sampler.  ``variates`` ([B,S,3]) switches the scalar samplers to injected mode (parity tests).  Texture
        samplers draw from Philox in every mode (the reference's eval mode is its train mode), keyed by
        (seed, sample0 + b, texture row).  ``out``: a ``BatchResult`` of an earlier
        call with the same ``B`` whose tensors are overwritten and returned (no allocation: a loop that runs ahead of the
        device otherwise makes the caching allocator grow by one vertex buffer per step in flight, and a ``cudaMalloc`` of
        B x V x 12 bytes blocks the host for 10-90 ms -- ``scripts/stall_probe2.py``)."""
        L = nat.lib()
        if out is not None and (out.sampled.shape[0] != B or out.batch is not self):
            raise ValueError("SceneBatch.randomize: `out` must be a BatchResult of this SceneBatch with the same B")
        train = bool(self.scene._train)
        mode = nat.MODE_INJECTED if variates is not None else (nat.MODE_TRAIN if train else nat.MODE_EVAL)
        if sample0 is None:
            sample0 = self._next_sample
            self._next_sample += B
        S, E = self.S, self.E
        sampled = out.sampled if out is not None else torch.empty((B, max(S, 1), 3), dtype=torch.float32, device=self.device)
        if S:
            v = None if variates is None else nat.require_cuda(variates.contiguous(), torch.float32, "variates")
            nat.check(L.ffb_sample(self.sampler_table.data_ptr(), S, B, mode, self.seed, int(sample0), nat.ptr(v),
                                   sampled.data_ptr(), nat.stream()), "ffb_sample")
            nat.count()
        world = out.world if out is not None else torch.empty((B, max(E, 1), 4, 4), dtype=torch.float32, device=self.device)
        if E:
            nat.check(L.ffb_compose_world(self.entity_table.data_ptr(), E, B, sampled.data_ptr(), S, world.data_ptr(),
                                          nat.stream()), "ffb_compose_world")
            nat.count()
        verts = None
        idx = None
        if self.meshes:
            mt = self._mesh_table(train)
            if any(a is not None for a in self._anim_meshes):
                M = len(self.meshes)
                lo = [(a._animation_sampler._min_integer_train if train else a._animation_sampler._min_integer_eval) if a else 0
                      for a in self._anim_meshes]
                hi = [(a._animation_sampler._max_integer_train if train else a._animation_sampler._max_integer_eval) if a else 0
                      for a in self._anim_meshes]
                key = (train, tuple(lo), tuple(hi))
                if getattr(self, "_anim_range_key", None) != key:      # two tiny H2D copies only when the ranges change
                    self._anim_range = (torch.tensor(lo, dtype=torch.int32, device=self.device),
                                        torch.tensor(hi, dtype=torch.int32, device=self.device))
                    self._anim_range_key = key
                amin, amax = self._anim_range
                idx = getattr(out, "_anim_idx", None) if out is not None else None
                if idx is None or tuple(idx.shape) != (B, M):
                    idx = torch.empty((B, M), dtype=torch.int32, device=self.device)
                nat.check(L.ffb_sample_anim_index(amin.data_ptr(), amax.data_ptr(), self._anim_cur.data_ptr(), M, B,
                                                  nat.MODE_TRAIN if train else nat.MODE_EVAL, self.seed, int(sample0),
                                                  idx.data_ptr(), nat.stream()), "ffb_sample_anim_index")
                nat.count()
            verts = out.vertices if out is not None and out.vertices is not None else torch.empty((B, self.Vtot, 3), dtype=torch.float32, device=self.device)
            nat.check(L.ffb_transform_vertices(C.byref(mt), self.verts.data_ptr(), E, B, nat.ptr(idx), world.data_ptr(),
                                               verts.data_ptr(), nat.stream()), "ffb_transform_vertices")
            nat.count()
        textures = {k: perlin_texture_batch(shape, B, ca, cb, seed=self.seed, sample0=int(sample0), row=row,
                                            out=out.textures[k] if out is not None else None, device=self.device)
                     for k, (row, shape, ca, cb) in self._textures.items()}
        if out is not None:
            out.textures = textures
            out._host = None                                # the cached host copy belongs to the overwritten samples
            out._anim_idx = idx
            return out
        res = BatchResult(world, sampled, verts, self, textures)
        res._anim_idx = idx                                 # kept for reuse through `out=`
        return res


class PatternStep:
    """One pattern-optimisation step over B scene samples on this rank.

    Mirrors the only in-tree optimisation loop of the reference (``test_point_reg``,
    fireflies/graphics/rasterization.py:586-607): ``summed = baked_sum_2``, ``softored = baked_softor_2``,
    ``loss = L1(softored, summed)``, backward to ``points`` -- for B samples at once, preceded by the batched scene
    randomisation.  With ``upstream`` the loss stage is skipped and the given texture gradients (e.g. from the
    renderer's backward pass) are consumed instead.  The only collective is the allreduce of ``d loss/d points``.
    The ``BatchResult`` a step returns stays valid through the next step and is reused by the one after
    (``rotate_results=False``: a fresh one per step).
    """

    def __init__(self, n_points: int, texture_size, sigma: float, batch: int, scene_batch: Optional[SceneBatch] = None,
                 num_std_sum: int = 4, num_std_softor: int = 5, sum_transposed: bool = True, per_sample_points: bool = True,
                 device="cuda", process_group=None, fuse_loss: bool = True, rotate_results: bool = True):
        self.N, self.B = int(n_points), int(batch)
        self.ts0, self.ts1 = R._ts(texture_size)
        self.sigma = float(sigma)
        self.ns, self.no, self.sum_t = int(num_std_sum), int(num_std_softor), bool(sum_transposed)
        self.scene_batch = scene_batch
        self.per_sample = per_sample_points
        self.device = torch.device(device)
        self.pg = process_group
        self.fuse_loss = bool(fuse_loss)      # False: loss and texture gradients through ffb_l1_loss_fwd_bwd, then the plain backward
        self.pts_dev = torch.empty((self.B if per_sample_points else 1, self.N, 2), dtype=torch.float32, device=self.device)
        # per_sample_points=False: one pattern for all scenes of the step -> see _shared_pattern
        self._pat_dev = torch.empty((self.N, 2), dtype=torch.float32, device=self.device)
        self.last = None
        self._side: Optional[torch.cuda.Stream] = None
        # rotate_results: the randomised samples are written into two alternating BatchResults (the one returned by step i is
        # overwritten by step i + 2); False: fresh tensors every step, like SceneBatch.randomize
        self._res_ring = [None, None] if rotate_results else None
        self._res_turn = 0

    def _allreduce(self, t: torch.Tensor) -> None:
        from .parallel import allreduce_sum_
        allreduce_sum_(t, self.pg)

    def forward_backward(self, points: torch.Tensor, upstream: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
                         sample0: Optional[int] = None, marks: Optional[dict] = None, randomize: bool = True):
        """points: ``[N,2]`` or ``[B,N,2]`` (device, or pinned host -> copied inside).  Returns
        ``(loss [B] or None, dpoints [N,2] summed over the B samples and all ranks, BatchResult or None)``.
        ``marks``: a dict that receives one CUDA event per phase boundary (``start, prepare, fwd, bwd, end`` on the calling stream,
        ``randomize0 / randomize1`` on the side stream) -- how ``bench.py`` times the kernels of the step it measures.
        Phases are wrapped in NVTX ranges (``ffb.randomize / prepare / fwd / bwd / fold``)."""
        nvtx = torch.cuda.nvtx

        def mark(name, stream=None):
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(stream) if stream is not None else ev.record()
                marks[name] = ev
        # the scene randomisation (HBM-bound vertex transform) does not depend on the pattern: it runs on a side stream
        # next to the latency-bound binning kernel and joins before the fold
        res = None
        mark("start")
        if self.scene_batch is not None and randomize:
            cur = torch.cuda.current_stream()
            if self._side is None:
                self._side = torch.cuda.Stream(device=self.device)
            self._side.wait_stream(cur)
            with torch.cuda.stream(self._side):
                nvtx.range_push("ffb.randomize")
                mark("randomize0", self._side)
                # two rotating result buffers: the samples of step i stay valid through step i + 1 (`self.last`), nothing is
                # allocated per step.  Safe without further events: this stream has just waited for everything the calling
                # stream has enqueued, which includes every consumer of the buffer written two steps ago.
                ring = self._res_ring
                slot = self._res_turn = (self._res_turn + 1) % len(ring) if ring is not None else 0
                res = self.scene_batch.randomize(self.B, sample0=sample0, out=ring[slot] if ring is not None else None)
                if ring is not None:
                    ring[slot] = res
                mark("randomize1", self._side)
                nvtx.range_pop()
        if not self.per_sample:
            self.pts_dev.copy_(points.unsqueeze(0) if points.dim() == 2 else points, non_blocking=True)
            loss, dp, s, o = self._shared_pattern(self.pts_dev[0], upstream)
            return self._finish(loss, dp, s, o, res)
        if points.dim() == 2:
            # one pattern for every sample: binned once (a [N,2] plan), while the B textures and the per-sample gradients against
            # the per-sample upstream gradients stay as they are
            self._pat_dev.copy_(points, non_blocking=True)
            pts = self._pat_dev
        else:
            self.pts_dev.copy_(points, non_blocking=True)
            pts = self.pts_dev
        nvtx.range_push("ffb.prepare")
        plan = R._SplatPlan(pts, self.B, self.sigma, self.ts0, self.ts1, self.ns, self.no)
        nvtx.range_pop()
        mark("prepare")
        nvtx.range_push("ffb.fwd")
        s, o = plan.forward(pts, True, True, self.sum_t)
        nvtx.range_pop()
        mark("fwd")
        loss = None
        d = None
        nvtx.range_push("ffb.bwd")
        if upstream is None:
            # rasterization.py:589-599: L1(softored, summed) -- the reference compares against the transposed sum as-is
            fused = plan.backward_l1(pts, s, o, self.sum_t) if self.fuse_loss else None
            if fused is not None:
                loss, d = fused
            else:
                loss = torch.empty(self.B, dtype=torch.float32, device=self.device)
                gs, go = torch.empty_like(s), torch.empty_like(o)
                nat.check(nat.lib().ffb_l1_loss_fwd_bwd(o.data_ptr(), s.data_ptr(), 0, self.B, self.ts0, self.ts1, loss.data_ptr(),
                                                        go.data_ptr(), gs.data_ptr(), nat.stream()), "ffb_l1_loss_fwd_bwd")
                nat.count(2)
        else:
            gs, go = upstream
        if d is None:
            d = plan.backward(pts, gs, go, self.sum_t, o)
        nvtx.range_pop()
        mark("bwd")
        nvtx.range_push("ffb.fold")
        out = self._finish(loss, None, s, o, res, per_sample=d)
        nvtx.range_pop()
        mark("end")
        return out

    def capture(self, points: torch.Tensor, upstream: Optional[Tuple[torch.Tensor, torch.Tensor]] = None):
        """CUDA-graph form of the step for small, launch-bound problems (the reference's own loop, rasterization.py:583-607, runs
        100 points into 512^2 for one sample: ten kernels of a few microseconds each).  Captures bin + splat forward + loss +
        backward + fold once and returns ``replay(points) -> (loss, dpoints)``; the tensors are overwritten by every replay.
        The scene randomisation is not captured (its sample index is a host-side kernel argument): call
        ``scene_batch.randomize`` next to the replay.  One rank only (the exchange agrees on its path with a host read)."""
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.pg) > 1:
            raise NotImplementedError("PatternStep.capture: single rank only")
        static_pts = torch.empty_like(points, device=self.device)
        static_pts.copy_(points)
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):                              # warm-up: one-time attribute / occupancy queries happen outside the capture
                self.forward_backward(static_pts, upstream=upstream, randomize=False)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loss, dp, _ = self.forward_backward(static_pts, upstream=upstream, randomize=False)

        def replay(new_points: Optional[torch.Tensor] = None):
            if new_points is not None:
                static_pts.copy_(new_points, non_blocking=True)
            graph.replay()
            return loss, dp
        replay.graph = graph
        return replay

    def _finish(self, loss, dp, s, o, res, per_sample=None):
        if res is not None:
            cur = torch.cuda.current_stream()
            cur.wait_stream(self._side)
            for t in (res.world, res.sampled, res.vertices):      # produced on the side stream, consumed by the caller on this one
                if t is not None:
                    t.record_stream(cur)
            for tex, _ in res.textures.values():
                tex.record_stream(cur)
        if per_sample is not None:
            from .parallel import fold_allreduce
            dp = fold_allreduce(per_sample, self.pg)        # fold over the samples + the step's only exchange, one kernel on NVLink
        else:
            self._allreduce(dp)
        self.last = (s, o, res)
        return loss, dp, res

    def _shared_pattern(self, pts: torch.Tensor, upstream):
        """One pattern for all B scenes of the step (``per_sample_points=False``: what data-parallel pattern optimisation
        does -- the scenes differ, the projector texture does not).  The B textures are one texture, and the backward is
        linear in the upstream texture gradients, so they are folded over the samples first (a streaming read of
        2 x B textures) and ONE splat backward runs on the folded gradients: the per-sample splat work disappears, the
        step is bounded by reading the upstream gradients once."""
        plan = R._SplatPlan(pts, 1, self.sigma, self.ts0, self.ts1, self.ns, self.no)
        s, o = plan.forward(pts, True, True, self.sum_t)                    # [1, ...]: the texture every scene is rendered with
        if upstream is None:
            fused = plan.backward_l1(pts, s, o, self.sum_t) if self.fuse_loss else None
            if fused is not None:
                loss1, d = fused
            else:
                loss1 = torch.empty(1, dtype=torch.float32, device=self.device)
                gs, go = torch.empty_like(s), torch.empty_like(o)
                nat.check(nat.lib().ffb_l1_loss_fwd_bwd(o.data_ptr(), s.data_ptr(), 0, 1, self.ts0, self.ts1, loss1.data_ptr(),
                                                        go.data_ptr(), gs.data_ptr(), nat.stream()), "ffb_l1_loss_fwd_bwd")
                nat.count(2)
                d = plan.backward(pts, gs, go, self.sum_t, o)
            return loss1.expand(self.B), d[0] * float(self.B), s.expand(self.B, -1, -1), o.expand(self.B, -1, -1)
        gs, go = upstream
        gs1 = R.reduce_over_samples(gs).unsqueeze(0) if gs.shape[0] > 1 else gs
        go1 = R.reduce_over_samples(go).unsqueeze(0) if go.shape[0] > 1 else go
        d = plan.backward(pts, gs1, go1, self.sum_t, o)
        return None, d[0], s.expand(self.B, -1, -1), o.expand(self.B, -1, -1)

    def step_host(self, points_host: torch.Tensor, out_host: torch.Tensor, loss_host: torch.Tensor, sample0: Optional[int] = None):
        """End-to-end step with HOST buffers: pinned ``points_host`` [N,2] in, ``out_host`` [N,2] (gradient) and
        ``loss_host`` [B] out; returns after the device->host copies have completed."""
        loss, dp, _ = self.forward_backward(points_host, sample0=sample0)
        out_host.copy_(dp, non_blocking=True)
        loss_host.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return loss_host, out_host


class TextureStep:
    """The projector-texture optimisation step for B rendered scene samples per rank, with one exchange per step.

    ``texture()`` builds the texture the renderer reads (:meth:`Laser.projector_texture`: the dense splat sum of the rays'
    NDC xy, Gaussian-blurred, in channel 1 of ``[ts1, ts0, 3]``) from ``laser._rays`` and keeps what the backward needs.
    ``backward(g_tex)`` takes the renderer's gradients w.r.t. that texture for this rank's samples (``[B, ts1, ts0, 3]`` or
    ``[ts1, ts0, 3]``) and returns ``d loss / d rays`` ``[N, 3]`` summed over the samples and all ranks of
    ``process_group``, also accumulated into ``laser._rays.grad`` the way autograd would (so ``torch.optim.Adam([laser._rays])``
    works unchanged).  When ``laser._perspective`` requires grad, the same pass of the ray projection's backward also gives
    ``d loss / d _perspective`` [4, 4], which travels in the same exchange and is accumulated into ``laser._perspective.grad``
    in its dtype.  Every scene of the step sees the same texture and every backward stage is linear in the upstream
    gradient, so the B gradients are folded first and the blur adjoint, the splat backward and the ray projection's backward
    run once per step.  No autograd graph is built; the step's buffers are allocated by the first call and reused (the
    returned tensor is overwritten by the next ``backward``)."""

    def __init__(self, laser, sigma: float, texture_size, blur=((5, 5), (3.0, 3.0)), process_group=None):
        from .postprocessing.gauss_blur import blur_spec
        self.laser = laser
        self.sigma = R._sigma(sigma)
        self.ts0, self.ts1 = R._ts(texture_size)
        self.blur = None if blur is None else blur_spec(blur[0], blur[1])
        self.pg = process_group
        self._saved = None                  # (rays, M, pts, plan) of the last texture()
        self._bufs = None

    def texture(self) -> torch.Tensor:
        from .postprocessing.base import run_postprocess
        L = nat.lib()
        rays = nat.require_cuda(self.laser._rays.detach().float().contiguous(), torch.float32, "laser._rays")
        M = self.laser._M().detach()
        N = rays.shape[0]
        ndc = torch.empty_like(rays)
        nat.check(L.ffb_transform_points(rays.data_ptr(), N, M.data_ptr(), 0, ndc.data_ptr(), nat.stream()), "ffb_transform_points")
        nat.count()
        pts = ndc[:, 0:2].contiguous()
        plan = R._SplatPlan(pts, 1, self.sigma, self.ts0, self.ts1, 0, 0)
        s, _ = plan.forward(pts, True, False, False)                        # [1, ts1, ts0]
        if self.blur is not None:
            s = run_postprocess(s, blur=self.blur)
        tex = torch.zeros((self.ts1, self.ts0, 3), dtype=torch.float32, device=rays.device)
        tex[..., 1] = s[0]
        self._saved = (rays, M, pts, plan)
        return tex

    def _buffers(self, N: int, dev) -> dict:
        b = self._bufs
        if b is None or b["d_rays"].shape[0] != N or b["d_rays"].device != dev:
            d_ndc = torch.zeros((N, 3), dtype=torch.float32, device=dev)        # column 2 stays 0: d ndc = (dx, dy, 0)
            packed = torch.empty(3 * N + 16, dtype=torch.float32, device=dev)   # [d_rays, d_perspective]: one exchange
            b = self._bufs = {"g1": torch.empty((1, self.ts1, self.ts0), dtype=torch.float32, device=dev),
                              "g_in": torch.empty((1, self.ts1, self.ts0), dtype=torch.float32, device=dev),
                              "d_pts": torch.empty((1, N, 2), dtype=torch.float32, device=dev),
                              "d_ndc": d_ndc, "packed": packed, "d_rays": packed[:3 * N].view(N, 3),
                              "d_K": packed[3 * N:].view(4, 4),
                              "ws": torch.empty(nat.lib().ffb_transform_bwd_workspace_bytes(N), dtype=torch.uint8, device=dev)}
        return b

    def backward(self, g_tex: torch.Tensor) -> torch.Tensor:
        from .parallel import allreduce_sum_
        from .postprocessing.gauss_blur import gaussian_blur2d_backward
        if self._saved is None:
            raise RuntimeError("TextureStep.backward: call texture() first")
        rays, M, pts, plan = self._saved
        g = nat.require_cuda(g_tex.contiguous(), torch.float32, "g_tex")
        if g.dim() == 3:
            g = g.unsqueeze(0)
        if g.dim() != 4 or tuple(g.shape[1:]) != (self.ts1, self.ts0, 3):
            raise ValueError(f"TextureStep.backward: g_tex must be [B, {self.ts1}, {self.ts0}, 3] or [{self.ts1}, {self.ts0}, 3]")
        N = rays.shape[0]
        b = self._buffers(N, rays.device)
        folded = R.reduce_over_samples(g) if g.shape[0] > 1 else g[0]       # [ts1, ts0, 3]; channels 0 and 2 multiply constants
        b["g1"][0].copy_(folded[..., 1])
        g_sum = b["g1"]
        if self.blur is not None:
            g_sum = gaussian_blur2d_backward(b["g1"], *self.blur, out=b["g_in"])
        d_pts = plan.backward(pts, g_sum, None, False, out=b["d_pts"])
        b["d_ndc"][:, 0:2].copy_(d_pts[0])
        K = self.laser._perspective
        if not K.requires_grad:
            nat.check(nat.lib().ffb_transform_points_bwd(rays.data_ptr(), N, M.data_ptr(), 0, b["d_ndc"].data_ptr(), b["d_rays"].data_ptr(),
                                                         nat.stream()), "ffb_transform_points_bwd")
            nat.count()
            d_rays = allreduce_sum_(b["d_rays"], self.pg)
        else:
            ws = b["ws"]
            nat.check(nat.lib().ffb_transform_points_bwd_full(rays.data_ptr(), N, M.data_ptr(), 0, b["d_ndc"].data_ptr(),
                                                              b["d_rays"].data_ptr(), b["d_K"].data_ptr(),
                                                              ws.data_ptr() if ws.numel() else None, ws.numel(), nat.stream()),
                      "ffb_transform_points_bwd_full")
            nat.count(2 if ws.numel() else 1)
            b["d_K"][:, 1].neg_()                       # d_M -> d_perspective: M = K @ FLIP_Y, d_K = d_M @ FLIP_Y^T
            allreduce_sum_(b["packed"], self.pg)
            d_rays = b["d_rays"]
            _accumulate_grad(K, b["d_K"])
        _accumulate_grad(self.laser._rays, d_rays)
        return d_rays


def _accumulate_grad(target: torch.Tensor, d: torch.Tensor) -> None:
    """``target.grad += d`` in the target's dtype, creating the gradient on first use, the way autograd accumulates a leaf."""
    if target.grad is None:
        target.grad = d.to(target.dtype, copy=True)
    else:
        target.grad.add_(d.to(target.dtype))
