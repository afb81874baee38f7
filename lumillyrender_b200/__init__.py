"""lumillyrender_b200 — B200-native (sm_100a) implementation of LumillyRender's per-pixel Monte Carlo
path-tracing loop behind the reference's scene-file surface.

The product is the C-ABI shared library (include/lumilly.h, built from csrc/ by build.py); this package is
the thin host-side mirror used by the tests, bench.py and the CLI wrapper.  No CPU fallback exists.
"""
from .capi import LumillyError, library_path, load_library  # noqa: F401
from .renderer import (Description, Film, MultiFilm, MultiScene, Scene, device_info, init, load_hdr, measure_hbm_read_gbs,  # noqa: F401
                       measure_l2_read_gbs, save_hdr, save_png)
from .assets import ensure_assets  # noqa: F401

REPO_ROOT = __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__)))
SCENES_DIR = __import__("os").path.join(REPO_ROOT, "scenes")
