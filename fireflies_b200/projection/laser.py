"""``fireflies/projection/laser.py`` -- Laser, same interface.

Ray <-> NDC projection, the field-of-view clamp and the texture splat run in libffb200 on the device.
Deviations from the reference, all documented in DESIGN.md: ``generateTexture`` keeps the result on the
GPU (the reference forces the splat onto the CPU, laser.py:292-296); ``fireflies.utils.transforms.*`` (an empty
module in the reference) is read as ``fireflies.utils.math.*``; ``rays/origin/originPerRay`` use
``self._transformable.world()`` instead of the garbled attribute at laser.py:163-177.
"""
from __future__ import annotations

import math
from typing import List

import numpy as np
import torch

from .. import _native as nat
from ..graphics import rasterization
from ..postprocessing.gauss_blur import gaussian_blur2d
from ..sampling import poisson
from ..utils import math as ffmath
from .camera import Camera

_FLIP_Y = [[1.0, 0.0, 0.0, 0.0], [0.0, -1.0, 0.0, 0.0], [0.0, 0.0, 1.0, 0.0], [0.0, 0.0, 0.0, 1.0]]


class Laser(Camera):
    @staticmethod
    def generate_uniform_rays(intra_ray_angle: float, num_beams_x: int, num_beams_y: int,
                              device: torch.device = torch.device("cuda")) -> torch.Tensor:
        """laser.py:19-37 (row index ``x*num_beams_x + y`` as in the reference); set-up only, host math."""
        rays = torch.zeros((num_beams_y * num_beams_x, 3))
        for x in range(num_beams_x):
            for y in range(num_beams_y):
                rays[x * num_beams_x + y, :] = torch.tensor([
                    math.tan((x - (num_beams_x - 1) / 2) * intra_ray_angle),
                    math.tan((y - (num_beams_y - 1) / 2) * intra_ray_angle), -1.0])
        rays = rays / torch.linalg.norm(rays, dim=-1, keepdims=True)
        return rays.to(device)

    @staticmethod
    def generate_uniform_rays_by_count(num_beams_x: int, num_beams_y: int, intrinsic_matrix: torch.Tensor,
                                       device: torch.device = torch.device("cuda")) -> torch.Tensor:
        """laser.py:40-66."""
        laserRays = torch.zeros((num_beams_y * num_beams_x, 3), device=device)
        x_steps = torch.arange((1 / num_beams_x) / 2, 1, 1 / num_beams_x)
        y_steps = torch.arange((1 / num_beams_y) / 2, 1, 1 / num_beams_y)
        xy = torch.stack(torch.meshgrid(x_steps, y_steps, indexing="ij")).movedim(0, -1).reshape(-1, 2)
        laserRays[:, 0:2] = xy.to(device)
        laserRays[:, 2] = -1.0
        rays = ffmath.transform_points(laserRays, intrinsic_matrix.inverse())
        rays = rays / torch.linalg.norm(rays, dim=-1, keepdims=True)
        rays[:, 2] *= -1.0
        return rays

    @staticmethod
    def generate_random_rays(num_beams: int, intrinsic_matrix: torch.Tensor,
                             device: torch.device = torch.device("cuda")) -> torch.Tensor:
        """laser.py:69-92."""
        spawned = torch.ones([num_beams, 3], device=device) * 0.5 + (torch.rand([num_beams, 3], device=device) - 0.5) / 10.0
        spawned[:, 2] = -1.0
        rays = ffmath.transform_points(spawned, intrinsic_matrix.inverse())
        rays = rays / torch.linalg.norm(rays, dim=-1, keepdims=True)
        rays[:, 2] *= -1.0
        return rays

    @staticmethod
    def generate_blue_noise_rays(image_size_x: int, image_size_y: int, num_beams: int, intrinsic_matrix: torch.Tensor,
                                 device: torch.device = torch.device("cuda")) -> torch.Tensor:
        """laser.py:94-145: Poisson-disk samples (radius chosen for roughly ``num_beams`` points) in the image box,
        scaled to [0,1]^2, un-projected through the intrinsics, normalised, z flipped.  The sample count is whatever
        the dart throwing yields, as in the reference."""
        poisson_radius = math.sqrt((image_size_x * image_size_y) / (math.pi * num_beams))
        poisson_radius += poisson_radius / 4.0
        im = np.ones([image_size_x, image_size_y]) * poisson_radius
        _, poisson_samples = poisson.bridson(im)
        poisson_samples = torch.tensor(poisson_samples) / torch.tensor([image_size_x, image_size_y])     # fp64, like the reference
        temp = torch.ones([poisson_samples.shape[0], 3]) * -1.0
        temp[:, 0:2] = poisson_samples
        rays = ffmath.transform_points(temp.to(device), intrinsic_matrix.inverse())
        rays = rays / torch.linalg.norm(rays, dim=-1, keepdims=True)
        rays[:, 2] *= -1.0
        return rays

    def __init__(self, transformable, ray_directions, perspective: torch.Tensor, max_fov: float, near_clip: float = 0.01,
                 far_clip: float = 1000.0, device: torch.device = torch.device("cuda")):
        super().__init__(transformable, perspective, max_fov, near_clip, far_clip, device)
        self._rays = ray_directions.to(self.device)
        self.device = device

    def rays(self) -> torch.Tensor:
        return ffmath.transform_directions(self._rays, self._transformable.world())

    def origin(self) -> torch.Tensor:
        return self._transformable.world()

    def originPerRay(self) -> torch.Tensor:
        return self._transformable.world()[0:3, 3].unsqueeze(0).repeat(self._rays.shape[0], 1)

    def _M(self) -> torch.Tensor:
        flip = torch.tensor(_FLIP_Y, device=self._perspective.device)
        return (self._perspective.float() @ flip).contiguous()

    def initRandomRays(self):
        spawned = torch.rand(self._rays.shape, device=self.device) * 2.0 - 1.0
        spawned[:, 2] = 1.0
        self._rays = self.normalize(self.projectNDCPointsToWorld(spawned))

    def initPoissonDiskSamples(self, width, height, radius):
        return None                                   # a stub in the reference as well (laser.py:196-197)

    def clamp_to_fov(self, clamp_val: float = 0.95, epsilon: float = 0.0001) -> None:
        """laser.py:199-206, one fused launch (project, clamp, un-project, renormalise)."""
        M = self._M()
        Minv = M.inverse().contiguous()
        rays = nat.require_cuda(self._rays.detach().float().contiguous(), torch.float32, "rays")
        out = torch.empty_like(rays)
        nat.check(nat.lib().ffb_clamp_to_fov(rays.data_ptr(), rays.shape[0], M.data_ptr(), Minv.data_ptr(),
                                             float(1 - clamp_val), float(clamp_val), out.data_ptr(), nat.stream()),
                  "ffb_clamp_to_fov")
        nat.count()
        with torch.no_grad():
            self._rays[:] = out

    def _respawn(self, M, ndc, lo: float, hi: float, variates) -> None:
        """One launch, no host sync (``ffb_respawn_rays``).  New positions come from the device Philox stream keyed by
        (torch's seed, ray index, call counter) unless ``variates`` ([K,3], the reference's ``torch.rand(K, 3)`` rows in ray
        order) is given.  ``self.last_respawned`` (device int32) holds the number of respawned rays."""
        rays = nat.require_cuda(self._rays.detach(), torch.float32, "rays")
        Minv = self._M().inverse().contiguous()
        v = None
        if variates is not None:
            v = nat.require_cuda(variates.float().contiguous(), torch.float32, "variates")
            if v.dim() != 2 or v.shape[1] != 3:
                raise ValueError("variates must be [K, 3]")
            if v.shape[0] < rays.shape[0]:          # the kernel consumes one row per out-of-bounds ray, at most N: never read past the end
                v = torch.cat([v, v.new_zeros((rays.shape[0] - v.shape[0], 3))])
        self.last_respawned = torch.zeros(1, dtype=torch.int32, device=rays.device)
        self._respawn_calls = getattr(self, "_respawn_calls", 0) + 1
        nat.check(nat.lib().ffb_respawn_rays(rays.data_ptr(), rays.shape[0], nat.ptr(M), nat.ptr(ndc), float(lo), float(hi),
                                             Minv.data_ptr(), int(torch.initial_seed()) & (2 ** 64 - 1), self._respawn_calls,
                                             nat.ptr(v), self.last_respawned.data_ptr(), nat.stream()), "ffb_respawn_rays")
        nat.count()

    def randomize_laser_out_of_bounds(self, variates: torch.Tensor = None) -> None:
        """laser.py:208-231: rays whose projection through ``_perspective`` leaves (0, 1)^2 are respawned uniformly in NDC
        and all rays renormalised.  (The reference returns 0 when nothing was out of bounds, None otherwise; no caller
        uses the value and reading it would cost a host sync: this returns None, see ``last_respawned``.)"""
        self._respawn(self._perspective.float().contiguous(), None, 0.0, 1.0, variates)

    def randomize_camera_out_of_bounds(self, ndc_coords, variates: torch.Tensor = None) -> None:
        """laser.py:233-249: as above for camera-space coordinates supplied by the caller, bounds (-1, 1)."""
        ndc = nat.require_cuda(ndc_coords.detach().float().contiguous(), torch.float32, "ndc_coords")
        if ndc.shape != (self._rays.shape[0], 3):
            raise ValueError("ndc_coords must be [N, 3]")
        self._respawn(None, ndc, -1.0, 1.0, variates)

    def normalize(self, tensor: torch.Tensor) -> torch.Tensor:
        return tensor / torch.linalg.norm(tensor, dim=-1, keepdims=True)

    def normalize_rays(self) -> None:
        with torch.no_grad():
            self._rays[:] = self.normalize(self._rays)

    def setToWorld(self, to_world: torch.Tensor) -> None:
        self._transformable.set_world(to_world)

    def projectRaysToNDC(self) -> torch.Tensor:
        """laser.py:262-275: ``transform_points(rays, K @ FLIP_Y)`` (differentiable w.r.t. ``_rays`` and ``_perspective``)."""
        return ffmath.transform_points(self._rays, self._M())

    def projectNDCPointsToWorld(self, points: torch.Tensor) -> torch.Tensor:
        """laser.py:277-290 (differentiable w.r.t. ``points`` and ``_perspective``)."""
        return ffmath.transform_points(points, self._M().inverse())

    def generateTexture(self, sigma: float, texture_size: List[int]) -> torch.Tensor:
        """laser.py:292-296: dense ``[N, ts[1], ts[0]]`` splat of the rays' NDC xy (stays on the GPU)."""
        points = self.projectRaysToNDC()[:, 0:2]
        return rasterization.rasterize_points(points, sigma, texture_size)

    def generateTextureReduced(self, sigma: float, texture_size, reduce: str = "sum") -> torch.Tensor:
        """Fused replacement for ``generateTexture(...).sum(0)`` / ``softor(generateTexture(...))`` (what every
        caller of the reference does next, main.py:64-67): never materialises the ``[N,H,W]`` tensor."""
        points = self.projectRaysToNDC()[:, 0:2]
        s, o = rasterization.splat_reduce(points, sigma, texture_size, num_std_sum=None, num_std_softor=None, reduce=(reduce,))
        return s if reduce == "sum" else o

    def projector_texture(self, sigma: float, texture_size, blur=((5, 5), (3.0, 3.0))) -> torch.Tensor:
        """The projector texture the renderer reads (main.py:64-77): ``[ts[1], ts[0], 3]``, zeros in channels 0 and 2 and
        the Gaussian-blurred dense splat sum of the rays' NDC xy in channel 1.  ``blur`` = ``(kernel_size, sigma)`` as in
        ``kornia.filters.gaussian_blur2d``, None = no blur.  Differentiable w.r.t. ``_rays`` and ``_perspective``.  For B rendered
        samples per step see :class:`fireflies_b200.TextureStep`."""
        points = self.projectRaysToNDC()[:, 0:2]
        tex = rasterization.splat_reduce(points, sigma, texture_size, num_std_sum=None, num_std_softor=None, reduce=("sum",))[0]
        if blur is not None:
            tex = gaussian_blur2d(tex[None, None], blur[0], blur[1])[0, 0]
        zero = torch.zeros_like(tex)
        return torch.stack([zero, tex, zero]).movedim(0, -1)

    def render_epipolar_lines(self, sigma: float, texture_size: torch.Tensor, camera_to_world: torch.Tensor = None) -> torch.Tensor:
        """laser.py:298-325: the segments origin + [near_clip, far_clip] * ray, seen through ``camera_to_world`` (identity when
        omitted) and ``_perspective``, rasterised with ``rasterize_lines``.  The reference reads the camera pose through an
        attribute that does not exist (``self._fireflies.entity.Transformable.world()``, :304); the evident intent is the
        viewing camera's world matrix, which the caller passes here.  Differentiable w.r.t. ``_rays``, ``_perspective`` and
        ``camera_to_world``."""
        lo = self.originPerRay() + self._near_clip * self.rays()
        hi = self.originPerRay() + self._far_clip * self.rays()
        if camera_to_world is None:
            camera_to_world = torch.eye(4, device=self.device)
        w2c = camera_to_world.float().inverse()
        hi = ffmath.transform_points(ffmath.transform_points(hi, w2c), self._perspective)[:, 0:2]
        lo = ffmath.transform_points(ffmath.transform_points(lo, w2c), self._perspective)[:, 0:2]
        return rasterization.rasterize_lines(torch.stack([lo, hi], dim=1), sigma, texture_size)

    def save(self, filepath: str):
        import yaml
        save_dict = {"rays": self._rays.detach().cpu().numpy().tolist(), "fov": self._fov,
                     "near_clip": self._near_clip, "far_clip": self._far_clip}
        with open(filepath, "w") as file:
            yaml.dump(save_dict, file)
