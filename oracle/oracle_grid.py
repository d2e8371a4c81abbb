"""TEST INFRASTRUCTURE -- ctypes binding of the grid-media oracle (oracle/oracle_grid.hpp, oracle/capi_grid.cpp -> liboracle_grid.so).

VolPathIntegrator for scenes whose media use density grids (GridDensityMedium).  It is a library of its own, beside oracle.py's
liboracle.so, built with the same compiler flags (oracle/Makefile).  Only tests/ import it."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

from . import oracle as O

HERE = Path(__file__).resolve().parent
LIB = HERE / "liboracle_grid.so"
CXXFLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fexcess-precision=standard", "-Wall", "-Wno-unused-function", "-pthread"]
_lib = None


def build(force=False):
    srcs = list(HERE.glob("*.hpp")) + [HERE / "capi_grid.cpp", HERE.parent / "include" / "pbrt_b200.h"]
    if force or not LIB.exists() or LIB.stat().st_mtime < max(s.stat().st_mtime for s in srcs):
        tmp = LIB.with_suffix(f".{os.getpid()}.tmp")
        subprocess.run([os.environ.get("CXX", "g++"), *CXXFLAGS, "-shared", "-o", str(tmp), str(HERE / "capi_grid.cpp")], check=True, cwd=HERE,
                       capture_output=True)
        tmp.replace(LIB)
    return LIB


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(str(LIB))
        L.orc_grid_render.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_uint64]
        L.orc_grid_density.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
        _lib = L
    return _lib


def render(flat, integrator, nthreads=0, tile_range=None, sample_range=None, rgbw=None, tile_interleave=None, tile_order=0):
    """oracle.render for a volpath scene with grid media (FlatScene.grids) -> ({r,g,b,w} sums [npix,4], stats dict)."""
    film = integrator.film
    if rgbw is None:
        rgbw = np.zeros((film.height * film.width, 4), np.float32)
    sd = flat.desc()
    rd = integrator.desc(tile_range, sample_range, tile_interleave=tile_interleave, tile_order=tile_order)
    stats = np.zeros(12, np.uint64)
    grids = flat.grid_table()
    rc = lib().orc_grid_render(C.addressof(sd), C.addressof(rd), O.ptr(rgbw), int(nthreads), O.ptr(stats), O.ptr(grids), len(grids))
    if rc != 0:
        raise ValueError("the grid-media oracle renders the volpath integrator only")
    return rgbw, dict(zip(O.STAT_NAMES, (int(v) for v in stats)))


def render_image(flat, integrator, **kw):
    rgbw, stats = render(flat, integrator, **kw)
    film = integrator.film
    return O.film_resolve(rgbw, film.scale).reshape(film.height, film.width, 3), stats


def grid_density(grid_row, points):
    """GridDensityMedium::density of one DENSITY_GRID_DTYPE row (FlatScene.grid_table()) at medium-space points [n, 3]."""
    pts = np.ascontiguousarray(points, np.float32).reshape(-1, 3)
    out = np.zeros(len(pts), np.float32)
    row = np.ascontiguousarray(np.asarray(grid_row).reshape(1))
    lib().orc_grid_density(O.ptr(row), O.ptr(pts), len(pts), O.ptr(out))
    return out
