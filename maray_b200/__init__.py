"""maray_b200 -- B200 (sm_100a) render path for Maray scenes.

The product is the C-ABI shared library `libmaray_cuda.so` (include/maray_cuda.h); this package is
its host-side mirror of the reference's render API (`render.py`) plus scene-authoring helpers
(`expr.py`, `scenes.py`).  There is no CPU or PyTorch fallback: render calls need the CUDA library
and a GPU.
"""
from . import expr  # noqa: F401
from .render import (CudaFunctions, CudaRenderer, MarayCudaError, RenderMethod, Report, Runtime, Textures, gen,  # noqa: F401
                     gen_to_image)
