"""fireflies_b200 -- B200 (sm_100a) implementation of the Fireflies hot path.

Drop-in for the part of Henningson/Fireflies the project owns: ``import fireflies_b200 as fireflies``
(``fireflies.Scene(mi_params)``, ``train()/eval()/randomize()``, ``fireflies.entity``, ``fireflies.projection.Laser``,
``fireflies.sampling``, ``fireflies.postprocessing``, ``fireflies.graphics.rasterization``).  All compute runs in
``libffb200.so`` (hand-written CUDA, C ABI in ``include/ffb200.h``); there is no CPU fallback -- importing works
anywhere, calling a kernel without the library or a GPU raises.
"""
from . import _native  # noqa: F401
from . import utils  # noqa: F401
from . import sampling  # noqa: F401
from . import entity  # noqa: F401
from . import emitter  # noqa: F401
from . import material  # noqa: F401
from . import graphics  # noqa: F401
from . import projection  # noqa: F401
from . import postprocessing  # noqa: F401
from .scene import Scene
from .batch import SceneBatch, PatternStep, TextureStep  # noqa: F401

scene = Scene          # the README of the reference spells it ``ff.scene(mi_params)``

__version__ = "0.1.0"
