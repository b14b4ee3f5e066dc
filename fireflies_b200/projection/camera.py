"""``fireflies/projection/camera.py``."""
import torch

from ..utils import math as ffmath


class Camera:
    id = 0
    MITSUBA_KEYS = {"fov": "x_fov", "f": "x_fov", "to_world": "to_world", "world": "to_world"}

    def __init__(self, transform, perspective: torch.Tensor, fov: float, near_clip: float = 0.01, far_clip: float = 1000.0,
                 device: torch.device = torch.device("cuda")):
        self.device = device
        self._transformable = transform
        self._perspective = perspective
        self._near_clip = near_clip
        self._far_clip = far_clip
        self._fov = fov
        self._key = self.generate_mitsuba_key()
        Camera.id += 1

    def full_key(self, key: str):
        return self._key + "." + Camera.MITSUBA_KEYS[key]

    def key(self) -> str:
        return self._key

    def near_clip(self) -> float:
        return self._near_clip

    def generate_mitsuba_key(self) -> str:
        if Camera.id == 0:
            return "PerspectiveCamera"
        return "PerspectiveCamera_{0}".format(Camera.id)    # the reference formats the builtin `id` (camera.py:50)

    def far_clip(self) -> float:
        return self._far_clip

    def fov(self):
        return self._fov

    def origin(self) -> torch.Tensor:
        return self._transformable.world()               # the reference calls a non-existent .origin() (camera.py:58-59)

    def world(self) -> torch.Tensor:
        return self._transformable.world()

    def randomize(self) -> None:
        self._transformable.randomize()

    def pointsToNDC(self, points) -> torch.Tensor:
        """camera.py:67-74: points through ``world().inverse()`` and ``_perspective``; differentiable w.r.t. ``points``, the pose
        and ``_perspective``."""
        view_space_points = ffmath.transform_points(points, self.world().inverse())
        return ffmath.transform_points(view_space_points, self._perspective)
