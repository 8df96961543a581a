"""B200-native differentiable Gaussian rasterizer: drop-in for the ``gsplat.rendering.rasterization``
call of li199603/easy_gaussian_splatting (/root/reference/model/gaussian.py:353-367)."""
from .rendering import rasterization, rasterization_camera_model, rasterization_from_parameters  # noqa: F401

__version__ = "0.1.0"
