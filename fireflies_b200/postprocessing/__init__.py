from .base import BasePostProcessingFunction
from .white_noise import WhiteNoise
from .postprocessor import PostProcessor
from .gauss_blur import GaussianBlur, gaussian_blur2d
from .apply_silhouette import ApplySilhouette
