"""TEST INFRASTRUCTURE -- ctypes binding of the BDPT oracle (oracle/oracle_bdpt.hpp, oracle/capi_bdpt.cpp -> liboracle_bdpt.so).

BDPTIntegrator on surfaces, with pbrt-v3's per-strategy films (visualizestrategies / visualizeweights).  It is a library of its own,
beside oracle.py's liboracle.so, built with the same compiler flags (oracle/Makefile).  Only tests/ import it."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

from . import oracle as O

HERE = Path(__file__).resolve().parent
LIB = HERE / "liboracle_bdpt.so"
CXXFLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fexcess-precision=standard", "-Wall", "-Wno-unused-function", "-pthread"]
_lib = None


def build(force=False):
    srcs = list(HERE.glob("*.hpp")) + [HERE / "capi_bdpt.cpp", HERE.parent / "include" / "pbrt_b200.h"]
    if force or not LIB.exists() or LIB.stat().st_mtime < max(s.stat().st_mtime for s in srcs):
        tmp = LIB.with_suffix(f".{os.getpid()}.tmp")
        r = subprocess.run([os.environ.get("CXX", "g++"), *CXXFLAGS, "-shared", "-o", str(tmp), str(HERE / "capi_bdpt.cpp")], cwd=HERE,
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"building {LIB.name} failed:\n{r.stderr}")
        tmp.replace(LIB)
    return LIB


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(str(LIB))
        L.orc_bdpt_render.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        _lib = L
    return _lib


def n_strategies(max_depth):
    return (max_depth + 1) * (max_depth + 6) // 2


def strategy_index(s, t):
    d = s + t - 2
    return s + d * (5 + d) // 2


def render(flat, integrator, nthreads=0, tile_range=None, sample_range=None, rgbw=None, splat=None, tile_interleave=None, tile_order=0,
           strategies=None, weighted=False):
    """BDPTIntegrator::render on the CPU -> ({r,g,b,w} sums [npix,4], splat RGB sums [npix,3], stats dict).  `strategies`: an array
    [n_strategies(max_depth), npix, 3] that receives the per-(s, t) films (unweighted, or MIS-weighted with weighted=True)."""
    film = integrator.film
    npix = film.height * film.width
    if rgbw is None:
        rgbw = np.zeros((npix, 4), np.float32)
    if splat is None:
        splat = np.zeros((npix, 3), np.float32)
    sd = flat.desc()
    rd = integrator.desc(tile_range, sample_range, tile_interleave=tile_interleave, tile_order=tile_order)
    stats = np.zeros(12, np.uint64)
    rc = lib().orc_bdpt_render(C.addressof(sd), C.addressof(rd), O.ptr(rgbw), O.ptr(splat), int(nthreads), O.ptr(stats), O.ptr(strategies),
                               int(bool(weighted)))
    if rc != 0:
        raise ValueError("the BDPT oracle renders the bdpt integrator (maxdepth >= 0) with the sobol or halton sampler only")
    return rgbw, splat, dict(zip(O.STAT_NAMES, (int(v) for v in stats)))


def resolve(rgbw, splat, spp, scale=1.0):
    """Film::write_image(1 / spp): weighted RGB plus the splat film over spp (both through RGB -> XYZ -> RGB), times scale."""
    img = O.film_resolve(rgbw, 1.0)
    sp = _xyz_round_trip(np.asarray(splat, np.float32).reshape(-1, 3))
    return ((img + sp / np.float32(spp)) * np.float32(scale)).astype(np.float32)


def _xyz_round_trip(rgb):
    to_xyz = np.array([[0.412453, 0.357580, 0.180423], [0.212671, 0.715160, 0.072169], [0.019334, 0.119193, 0.950227]], np.float32)
    to_rgb = np.array([[3.240479, -1.537150, -0.498535], [-0.969256, 1.875991, 0.041556], [0.055648, -0.204043, 1.057311]], np.float32)
    return (rgb @ to_xyz.T) @ to_rgb.T


def render_image(flat, integrator, **kw):
    rgbw, splat, stats = render(flat, integrator, **kw)
    film = integrator.film
    spp = integrator.sampler.spp if hasattr(integrator.sampler, "spp") else integrator.spp
    return resolve(rgbw, splat, spp, film.scale).reshape(film.height, film.width, 3), stats
