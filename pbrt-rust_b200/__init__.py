"""B200-native wavefront path tracer behind pbrt-rust's PathIntegrator interface.

The package directory name contains a hyphen (it mirrors the reference's name); import it
with `importlib.import_module("pbrt-rust_b200")` or through `__graft_entry__.package()`.
"""
from . import api, host, paramset, plymesh, pbrtparser, scenes, spectrum  # noqa: F401
from .api import API, RenderJob  # noqa: F401
from .pbrtparser import pbrt_parse, pbrt_parse_string  # noqa: F401
from .host import (B200Error, BDPTIntegrator, DirectLightingIntegrator, WhittedIntegrator, VolPathIntegrator, Film, FlatScene, PathIntegrator, PerspectiveCamera, Sampler, Scene, SceneBuilder, Transform, bvh_build,  # noqa: F401
                   load_library, make_rays)
