"""Host side of the B200 path tracer: ctypes binding of include/pbrt_b200.h plus a
Python mirror of the pbrt-rust scene API for the PathIntegrator hot path.

The reference's host is Rust (`API::shape`, `API::world_end`, `make_scene`,
`RenderOptions::make_integrator`: src/core/api.rs:244-300,1493-1771); no Rust
toolchain exists in this image, so this module plays that role: it keeps graphics
state (CTM, current material, area light), flattens shapes into the SoA tables of
`pbrt_b200_scene_desc`, asks the library's host-side `pbrt_b200_bvh_build`
(mirror of BVHAccel::new) for the node array and hands everything to CUDA through
the C ABI.  Nothing here computes a hit or a pixel: without the CUDA library and a
GPU every compute call raises.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import warnings
from pathlib import Path

import numpy as np

from . import textures as T

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libpbrt_b200.so"
TABLES_PATH = _HERE / "tables" / "sobol_tables.npz"

f32 = np.float32
NO_HIT = 0xFFFFFFFF

# ---------------------------------------------------------------------------
# ctypes mirrors of include/pbrt_b200.h
# ---------------------------------------------------------------------------


class BvhNode(C.Structure):
    _fields_ = [("bounds", C.c_float * 6), ("offset", C.c_uint32), ("n_prims", C.c_uint16), ("axis", C.c_uint8), ("pad", C.c_uint8)]


NODE_DTYPE = np.dtype([("bounds", "<f4", 6), ("offset", "<u4"), ("n_prims", "<u2"), ("axis", "u1"), ("pad", "u1")])
PRIM_DTYPE = np.dtype([("shape_kind", "<u4"), ("shape_index", "<u4"), ("material", "<i4"), ("area_light", "<i4"), ("flags", "<u4"), ("creation_index", "<u4")])
SPHERE_DTYPE = np.dtype([("object_to_world", "<f4", 16), ("world_to_object", "<f4", 16), ("radius", "<f4"), ("flags", "<u4"), ("pad", "<f4", 2)])
MATERIAL_DTYPE = np.dtype([("type", "<u4"), ("remap_roughness", "<u4"), ("a", "<f4", 3), ("b", "<f4", 3), ("f0", "<f4"), ("f1", "<f4"), ("f2", "<f4"), ("textured", "<u4")])
LIGHT_DTYPE = np.dtype([("type", "<u4"), ("two_sided", "<u4"), ("L", "<f4", 3), ("pos", "<f4", 3), ("dir", "<f4", 3), ("shape_kind", "<u4"),
                        ("shape_index", "<u4"), ("shape_flags", "<u4"), ("area", "<f4"), ("cos_total_width", "<f4"), ("cos_falloff_start", "<f4"),
                        ("world_to_light", "<f4", 16), ("n_samples", "<u4")])
RAY_DTYPE = np.dtype([("o", "<f4", 3), ("t_max", "<f4"), ("d", "<f4", 3), ("time", "<f4")])
HIT_DTYPE = np.dtype([("prim", "<u4"), ("t", "<f4"), ("b0", "<f4"), ("b1", "<f4")])
assert NODE_DTYPE.itemsize == 32 and PRIM_DTYPE.itemsize == 24 and SPHERE_DTYPE.itemsize == 144
assert MATERIAL_DTYPE.itemsize == 48 and LIGHT_DTYPE.itemsize == 136 and RAY_DTYPE.itemsize == 32 and HIT_DTYPE.itemsize == 16

SHAPE_TRIANGLE, SHAPE_SPHERE, SHAPE_INSTANCE = 0, 1, 2
MEDIUM_DTYPE = np.dtype([("sigma_a", "<f4", 3), ("sigma_s", "<f4", 3), ("g", "<f4"), ("grid", "<u4")])                     # pbrt_b200_medium
DENSITY_GRID_DTYPE = np.dtype([("medium_to_world", "<f4", 16), ("world_to_medium", "<f4", 16), ("nx", "<u4"), ("ny", "<u4"), ("nz", "<u4"),
                               ("pad", "<u4"), ("density", "<u8")])                                                              # pbrt_b200_density_grid
assert DENSITY_GRID_DTYPE.itemsize == 152
MEDIUM_INTERFACE_DTYPE = np.dtype([("inside", "<i4"), ("outside", "<i4")])                                                   # pbrt_b200_medium_interface
OBJECT_DTYPE = np.dtype([("node_offset", "<u8"), ("n_nodes", "<u8"), ("prim_offset", "<u8"), ("n_prims", "<u8")])
INSTANCE_DTYPE = np.dtype([("prim_to_world", "<f4", 16), ("world_to_prim", "<f4", 16), ("object", "<u4"), ("pad", "<u4", 3)])
assert OBJECT_DTYPE.itemsize == 32 and INSTANCE_DTYPE.itemsize == 144
PRIM_REVERSE_ORIENTATION, PRIM_SWAPS_HANDEDNESS, PRIM_HAS_N, PRIM_HAS_S, PRIM_HAS_UV = 1, 2, 4, 8, 16
MAT_MATTE, MAT_PLASTIC, MAT_MIRROR, MAT_GLASS, MAT_METAL, MAT_UBER, MAT_SUBSTRATE = range(7)
LIGHT_POINT, LIGHT_DISTANT, LIGHT_SPOT, LIGHT_DIFFUSE, LIGHT_INFINITE = range(5)
SAMPLER_SOBOL, SAMPLER_HALTON, SAMPLER_ZEROTWO = range(3)
LIGHTS_UNIFORM, LIGHTS_POWER, LIGHTS_SPATIAL = range(3)
INTEGRATOR_PATH, INTEGRATOR_DIRECT_ONE, INTEGRATOR_DIRECT_ALL, INTEGRATOR_WHITTED, INTEGRATOR_VOLPATH, INTEGRATOR_BDPT = range(6)
BDPT_MAX_DEPTH = 64  # PBRT_B200_BDPT_MAX_DEPTH: the bdpt integrator keeps every subpath vertex of a sample in device memory
SPLIT = {"sah": 0, "middle": 2, "equal": 3}


class SceneDesc(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("pad", C.c_uint32),
                ("nodes", C.c_void_p), ("n_nodes", C.c_uint64),
                ("prims", C.c_void_p), ("n_prims", C.c_uint64),
                ("vertex_p", C.c_void_p), ("vertex_n", C.c_void_p), ("vertex_s", C.c_void_p), ("vertex_uv", C.c_void_p), ("n_vertices", C.c_uint64),
                ("tri_indices", C.c_void_p), ("n_triangles", C.c_uint64),
                ("spheres", C.c_void_p), ("n_spheres", C.c_uint64),
                ("materials", C.c_void_p), ("n_materials", C.c_uint64),
                ("lights", C.c_void_p), ("n_lights", C.c_uint64),
                ("objects", C.c_void_p), ("n_objects", C.c_uint64),
                ("instances", C.c_void_p), ("n_instances", C.c_uint64),
                ("n_top_nodes", C.c_uint64), ("n_top_prims", C.c_uint64),
                ("media", C.c_void_p), ("n_media", C.c_uint64), ("prim_media", C.c_void_p),
                ("textures", C.c_void_p), ("n_textures", C.c_uint64), ("mipmaps", C.c_void_p), ("n_mipmaps", C.c_uint64), ("material_ext", C.c_void_p)]


class CameraDesc(C.Structure):
    _fields_ = [("raster_to_camera", C.c_float * 16), ("camera_to_world", C.c_float * 16), ("lens_radius", C.c_float), ("focal_distance", C.c_float),
                ("shutter_open", C.c_float), ("shutter_close", C.c_float)]


class FilmDesc(C.Structure):
    _fields_ = [("full_resolution", C.c_int32 * 2), ("cropped_pixel_bounds", C.c_int32 * 4), ("filter_radius", C.c_float * 2),
                ("filter_table", C.c_float * 256), ("scale", C.c_float), ("max_sample_luminance", C.c_float)]


class SamplerDesc(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("samples_per_pixel", C.c_uint32), ("sample_bounds", C.c_int32 * 4), ("n_sampled_dimensions", C.c_uint32),
                ("pad", C.c_uint32), ("sobol_matrices32", C.c_void_p), ("vdc_matrices", C.c_void_p), ("vdc_matrices_inv", C.c_void_p)]


class IntegratorDesc(C.Structure):
    _fields_ = [("max_depth", C.c_int32), ("rr_threshold", C.c_float), ("pixel_bounds", C.c_int32 * 4), ("light_sample_strategy", C.c_uint32),
                ("kind", C.c_uint32), ("camera_medium", C.c_int32), ("reserved", C.c_uint32)]


class RenderDesc(C.Structure):
    _fields_ = [("camera", CameraDesc), ("film", FilmDesc), ("sampler", SamplerDesc), ("integrator", IntegratorDesc),
                ("tile_begin", C.c_uint32), ("tile_end", C.c_uint32), ("sample_begin", C.c_uint32), ("sample_end", C.c_uint32),
                ("paths_in_flight", C.c_uint32), ("flags", C.c_uint32),
                ("tile_group", C.c_uint32), ("tile_mod", C.c_uint32), ("tile_rem", C.c_uint32), ("tile_order", C.c_uint32)]


class RenderStats(C.Structure):
    _fields_ = [("camera_rays", C.c_uint64), ("intersection_tests", C.c_uint64), ("shadow_tests", C.c_uint64), ("zero_radiance_paths", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("device_ms", C.c_double), ("trace_closest_ms", C.c_double), ("trace_any_ms", C.c_double),
                ("shade_ms", C.c_double), ("finish_ms", C.c_double), ("iterations", C.c_uint64)]


RENDER_KEEP_ON_DEVICE = 1
RENDER_LAZY_SPATIAL = 2
RENDER_OVERWRITE = 4

EXPORTS = ["pbrt_b200_last_error", "pbrt_b200_abi_version", "pbrt_b200_device_count", "pbrt_b200_bvh_build", "pbrt_b200_scene_create", "pbrt_b200_scene_create_with_grids",
           "pbrt_b200_scene_destroy", "pbrt_b200_scene_world_bound", "pbrt_b200_intersect", "pbrt_b200_intersect_p", "pbrt_b200_intersect_dev",
           "pbrt_b200_intersect_p_dev", "pbrt_b200_render", "pbrt_b200_film_resolve", "pbrt_b200_light_distribution_lookup", "pbrt_b200_release_cached_memory", "pbrt_b200_tile_positions",
           "pbrt_b200_work_counter_open", "pbrt_b200_work_counter_fetch_add", "pbrt_b200_work_counter_fetch_max", "pbrt_b200_work_counter_load", "pbrt_b200_work_counter_store",
           "pbrt_b200_work_counter_close", "pbrt_b200_render_splat", "pbrt_b200_film_resolve_splat"]


class B200Error(RuntimeError):
    pass


_lib = None


def load_library():
    """dlopen the in-tree CUDA library.  There is no fallback: a missing library is an error."""
    global _lib
    if _lib is not None:
        return _lib
    import os
    path = Path(os.environ.get("PBRT_B200_LIB", LIB_PATH))  # a second build for before/after comparisons (csrc/Makefile NAME=...); still a CUDA library, never a fallback
    if not path.exists():
        raise B200Error(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (no CPU fallback exists)")
    lib = C.CDLL(str(path))
    lib.pbrt_b200_last_error.restype = C.c_char_p
    lib.pbrt_b200_bvh_build.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]
    lib.pbrt_b200_scene_create.argtypes = [C.POINTER(SceneDesc), C.c_int, C.POINTER(C.c_void_p)]
    lib.pbrt_b200_scene_create_with_grids.argtypes = [C.POINTER(SceneDesc), C.c_void_p, C.c_uint64, C.c_int, C.POINTER(C.c_void_p)]
    lib.pbrt_b200_scene_destroy.argtypes = [C.c_void_p]
    lib.pbrt_b200_scene_destroy.restype = None
    lib.pbrt_b200_scene_world_bound.argtypes = [C.c_void_p, C.c_void_p]
    lib.pbrt_b200_intersect.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
    lib.pbrt_b200_intersect_p.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
    lib.pbrt_b200_intersect_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    lib.pbrt_b200_intersect_p_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    lib.pbrt_b200_render.argtypes = [C.c_void_p, C.POINTER(RenderDesc), C.c_void_p, C.POINTER(RenderStats)]
    lib.pbrt_b200_film_resolve.argtypes = [C.c_void_p, C.c_uint64, C.c_float, C.c_void_p]
    lib.pbrt_b200_render_splat.argtypes = [C.c_void_p, C.POINTER(RenderDesc), C.c_void_p, C.c_void_p, C.POINTER(RenderStats)]
    lib.pbrt_b200_film_resolve_splat.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_float, C.c_float, C.c_void_p]
    lib.pbrt_b200_release_cached_memory.restype = None
    lib.pbrt_b200_light_distribution_lookup.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    lib.pbrt_b200_tile_positions.argtypes = [C.c_int, C.c_int, C.c_uint32]
    lib.pbrt_b200_tile_positions.restype = C.c_uint32
    lib.pbrt_b200_work_counter_open.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]
    lib.pbrt_b200_work_counter_fetch_add.argtypes = [C.c_void_p, C.c_uint64]
    lib.pbrt_b200_work_counter_fetch_add.restype = C.c_uint64
    lib.pbrt_b200_work_counter_fetch_max.argtypes = [C.c_void_p, C.c_uint64]
    lib.pbrt_b200_work_counter_fetch_max.restype = C.c_uint64
    lib.pbrt_b200_work_counter_load.argtypes = [C.c_void_p]
    lib.pbrt_b200_work_counter_load.restype = C.c_uint64
    lib.pbrt_b200_work_counter_store.argtypes = [C.c_void_p, C.c_uint64]
    lib.pbrt_b200_work_counter_store.restype = None
    lib.pbrt_b200_work_counter_close.argtypes = [C.c_void_p, C.c_int]
    lib.pbrt_b200_work_counter_close.restype = None
    _lib = lib
    return lib


def _check(rc, what):
    if rc != 0:
        msg = load_library().pbrt_b200_last_error().decode("utf-8", "replace")
        raise B200Error(f"{what} failed (code {rc}): {msg}")


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


_tables = None


def sampler_tables():
    """The reference crate's Sobol tables (src/core/sobolmatrices.rs), see tools/convert_tables.py."""
    global _tables
    if _tables is None:
        t = np.load(TABLES_PATH)
        _tables = {k: np.ascontiguousarray(t[k]) for k in ("sobol32", "vdc", "vdc_inv")}
    return _tables


# ---------------------------------------------------------------------------
# Transform (src/core/transform.rs), f32 arithmetic via numpy scalars
# ---------------------------------------------------------------------------


def _m4_inverse(m):
    """Matrix4x4::inverse, transform.rs:78-145 (Gauss-Jordan, full pivoting, f32)."""
    minv = np.array(m, dtype=f32).copy()
    indxc, indxr, ipiv = [0] * 4, [0] * 4, [0] * 4
    for i in range(4):
        irow = icol = 0
        big = f32(0)
        for j in range(4):
            if ipiv[j] != 1:
                for k in range(4):
                    if ipiv[k] == 0:
                        a = abs(minv[j, k])
                        if a >= big:
                            big, irow, icol = a, j, k
        ipiv[icol] += 1
        if irow != icol:
            minv[[irow, icol]] = minv[[icol, irow]]
        indxr[i], indxc[i] = irow, icol
        pivinv = f32(1) / minv[icol, icol]
        minv[icol, icol] = f32(1)
        minv[icol, :] = minv[icol, :] * pivinv
        for j in range(4):
            if j != icol:
                save = minv[j, icol]
                minv[j, icol] = f32(0)
                minv[j, :] = minv[j, :] - minv[icol, :] * save
    for i in range(4):
        j = 3 - i
        if indxr[j] != indxc[j]:
            minv[:, [indxr[j], indxc[j]]] = minv[:, [indxc[j], indxr[j]]]
    return minv


def _m4_mul(a, b):
    r = np.zeros((4, 4), dtype=f32)
    for i in range(4):
        for j in range(4):
            r[i, j] = a[i, 0] * b[0, j] + a[i, 1] * b[1, j] + a[i, 2] * b[2, j] + a[i, 3] * b[3, j]
    return r


class Transform:
    def __init__(self, m=None, m_inv=None):
        self.m = np.eye(4, dtype=f32) if m is None else np.array(m, dtype=f32)
        self.m_inv = _m4_inverse(self.m) if m_inv is None else np.array(m_inv, dtype=f32)

    def __mul__(self, o):  # transform.rs:647-656
        return Transform(_m4_mul(self.m, o.m), _m4_mul(o.m_inv, self.m_inv))

    def inverse(self):
        r = Transform(self.m_inv, self.m)
        r.inverse_of = self  # provenance only (scenefile.py writes `LookAt` for a camera built from look_at().inverse())
        return r

    @staticmethod
    def translate(d):  # transform.rs:255-271
        m, mi = np.eye(4, dtype=f32), np.eye(4, dtype=f32)
        m[:3, 3] = np.asarray(d, dtype=f32)
        mi[:3, 3] = -np.asarray(d, dtype=f32)
        return Transform(m, mi)

    @staticmethod
    def scale(x, y, z):  # transform.rs:273-289
        m = np.diag(np.array([x, y, z, 1], dtype=f32))
        mi = np.diag(np.array([f32(1) / f32(x), f32(1) / f32(y), f32(1) / f32(z), 1], dtype=f32))
        return Transform(m, mi)

    @staticmethod
    def rotate(theta_deg, axis):  # transform.rs:333-355
        a = np.asarray(axis, dtype=f32)
        a = a / f32(np.sqrt(f32(a[0] * a[0] + a[1] * a[1] + a[2] * a[2])))
        th = f32(math.pi / 180.0) * f32(theta_deg)
        s, c = f32(np.sin(th)), f32(np.cos(th))
        m = np.eye(4, dtype=f32)
        m[0, 0] = a[0] * a[0] + (1 - a[0] * a[0]) * c
        m[0, 1] = a[0] * a[1] * (1 - c) - a[2] * s
        m[0, 2] = a[0] * a[2] * (1 - c) + a[1] * s
        m[1, 0] = a[0] * a[1] * (1 - c) + a[2] * s
        m[1, 1] = a[1] * a[1] + (1 - a[1] * a[1]) * c
        m[1, 2] = a[1] * a[2] * (1 - c) - a[0] * s
        m[2, 0] = a[0] * a[2] * (1 - c) - a[1] * s
        m[2, 1] = a[1] * a[2] * (1 - c) + a[0] * s
        m[2, 2] = a[2] * a[2] + (1 - a[2] * a[2]) * c
        return Transform(m, m.T.copy())

    @staticmethod
    def look_at(pos, look, up):  # transform.rs:357-393 (returns world->camera; m_inv = camera->world)
        pos, look, up = (np.asarray(v, dtype=f32) for v in (pos, look, up))

        def nrm(v):
            return v * (f32(1) / f32(np.sqrt(f32(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]))))

        def cross(a, b):
            return np.cross(a.astype(np.float64), b.astype(np.float64)).astype(f32)

        d = nrm(look - pos)
        right = nrm(cross(nrm(up), d))
        new_up = cross(d, right)
        c2w = np.eye(4, dtype=f32)
        c2w[:3, 0], c2w[:3, 1], c2w[:3, 2], c2w[:3, 3] = right, new_up, d, pos
        r = Transform(_m4_inverse(c2w), c2w)
        r.lookat_args = (pos, look, up)
        return r

    @staticmethod
    def perspective(fov, n, f):  # transform.rs:399-411
        n, f = f32(n), f32(f)
        persp = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, f / (f - n), -f * n / (f - n)], [0, 0, 1, 0]], dtype=f32)
        inv_tan = f32(1) / f32(np.tan(f32(f32(math.pi / 180.0) * f32(fov)) / f32(2)))
        return Transform.scale(inv_tan, inv_tan, 1) * Transform(persp)

    def points(self, p):  # transform_point, transform.rs:413-431 (vectorised, f32, same op order)
        p = np.asarray(p, dtype=f32).reshape(-1, 3)
        m = self.m
        x, y, z = p[:, 0], p[:, 1], p[:, 2]
        xp = x * m[0, 0] + y * m[0, 1] + z * m[0, 2] + m[0, 3]
        yp = x * m[1, 0] + y * m[1, 1] + z * m[1, 2] + m[1, 3]
        zp = x * m[2, 0] + y * m[2, 1] + z * m[2, 2] + m[2, 3]
        wp = x * m[3, 0] + y * m[3, 1] + z * m[3, 2] + m[3, 3]
        out = np.stack([xp, yp, zp], axis=1).astype(f32)
        div = wp != f32(1)
        if div.any():
            out[div] = out[div] * (f32(1) / wp[div])[:, None]
        return out

    def vectors(self, v):  # transform.rs:496-508
        v = np.asarray(v, dtype=f32).reshape(-1, 3)
        m = self.m
        x, y, z = v[:, 0], v[:, 1], v[:, 2]
        return np.stack([x * m[0, 0] + y * m[0, 1] + z * m[0, 2], x * m[1, 0] + y * m[1, 1] + z * m[1, 2],
                         x * m[2, 0] + y * m[2, 1] + z * m[2, 2]], axis=1).astype(f32)

    def normals(self, n):  # transform.rs:529-541
        n = np.asarray(n, dtype=f32).reshape(-1, 3)
        mi = self.m_inv
        x, y, z = n[:, 0], n[:, 1], n[:, 2]
        return np.stack([x * mi[0, 0] + y * mi[1, 0] + z * mi[2, 0], x * mi[0, 1] + y * mi[1, 1] + z * mi[2, 1],
                         x * mi[0, 2] + y * mi[1, 2] + z * mi[2, 2]], axis=1).astype(f32)

    def bounds(self, b):  # transform_bounds, transform.rs:593-605: union of the 8 transformed corners
        b = np.asarray(b, f32)
        corners = np.array([[b[0 if i & 1 == 0 else 3], b[1 if i & 2 == 0 else 4], b[2 if i & 4 == 0 else 5]] for i in range(8)], f32)
        w = self.points(corners)
        return np.concatenate([w.min(0), w.max(0)]).astype(f32)

    def is_identity(self):  # transform.rs:229-238
        return bool(np.array_equal(self.m, np.eye(4, dtype=f32)))

    def swaps_handedness(self):  # transform.rs:638-644
        m = self.m
        det = (m[0, 0] * (m[1, 1] * m[2, 2] - m[1, 2] * m[2, 1]) - m[0, 1] * (m[1, 0] * m[2, 2] - m[1, 2] * m[2, 0]) +
               m[0, 2] * (m[1, 0] * m[2, 1] - m[1, 1] * m[2, 0]))
        return bool(det < 0)


class WorkCounter:
    """pbrt_b200_work_counter: a 64-bit counter in POSIX shared memory that the processes driving the GPUs of one box claim tile
    ranges from (the reference's shared tile queue, integrator.rs:291-296).  Host-only: works without a GPU."""

    def __init__(self, name, create):
        self.lib, self.name, self.owner = load_library(), name, bool(create)
        h = C.c_void_p()
        _check(self.lib.pbrt_b200_work_counter_open(name.encode(), 1 if create else 0, C.byref(h)), "pbrt_b200_work_counter_open")
        self.handle = h

    def fetch_add(self, n):
        return int(self.lib.pbrt_b200_work_counter_fetch_add(self.handle, C.c_uint64(int(n))))

    def fetch_max(self, v):
        return int(self.lib.pbrt_b200_work_counter_fetch_max(self.handle, C.c_uint64(int(v))))

    def load(self):
        return int(self.lib.pbrt_b200_work_counter_load(self.handle))

    def store(self, v):
        self.lib.pbrt_b200_work_counter_store(self.handle, C.c_uint64(int(v)))

    def close(self):
        if self.handle:
            self.lib.pbrt_b200_work_counter_close(self.handle, 1 if self.owner else 0)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---------------------------------------------------------------------------
# BVHAccel (host build through the library) and the flattened scene
# ---------------------------------------------------------------------------


# world_end() builds accelerators with this callable when no `builder` is passed; None = pbrt_b200_bvh_build.  bench.py's
# `--impl reference` arm points it at the oracle's builder so that the CPU arm never loads the product library (the two
# builders are byte-identical: tests/test_host_bvh.py).
DEFAULT_BVH_BUILDER = None


def bvh_build(prim_bounds, max_prims=4, split_method="sah"):
    """BVHAccel::new (bvh.rs:145-198) via pbrt_b200_bvh_build -> (nodes, ordered)."""
    lib = load_library()
    pb = np.ascontiguousarray(prim_bounds, dtype=f32).reshape(-1, 6)
    n = pb.shape[0]
    nodes = np.zeros(max(2 * n - 1, 1), dtype=NODE_DTYPE)
    ordered = np.zeros(max(n, 1), dtype=np.uint32)
    nn = C.c_uint64(0)
    _check(lib.pbrt_b200_bvh_build(_ptr(pb), n, int(max_prims), SPLIT[split_method], _ptr(nodes), _ptr(ordered), C.byref(nn)), "pbrt_b200_bvh_build")
    return nodes[: nn.value].copy(), ordered[:n].copy()


class DensityGrid:
    """The density field of a GridDensityMedium (grid.rs): density[(z * ny + y) * nx + x] over the unit box that medium_to_world
    (4x4, row-major) maps into the world; world_to_medium is its inverse as the Transform carries it."""

    def __init__(self, density, nx, ny, nz, medium_to_world, world_to_medium):
        self.density = np.ascontiguousarray(density, f32).reshape(-1)
        self.nx, self.ny, self.nz = int(nx), int(ny), int(nz)
        self.medium_to_world = np.ascontiguousarray(medium_to_world, f32).reshape(4, 4)
        self.world_to_medium = np.ascontiguousarray(world_to_medium, f32).reshape(4, 4)


class FlatScene:
    """The arrays behind `pbrt_b200_scene_desc` (owned here; the library copies them)."""

    def __init__(self):
        self.nodes = np.zeros(0, NODE_DTYPE)
        self.prims = np.zeros(0, PRIM_DTYPE)
        self.vertex_p = np.zeros((0, 3), f32)
        self.vertex_n = None
        self.vertex_s = None
        self.vertex_uv = None
        self.tri_indices = np.zeros((0, 3), np.uint32)
        self.spheres = np.zeros(0, SPHERE_DTYPE)
        self.materials = np.zeros(0, MATERIAL_DTYPE)
        self.lights = np.zeros(0, LIGHT_DTYPE)
        self.objects = np.zeros(0, OBJECT_DTYPE)
        self.instances = np.zeros(0, INSTANCE_DTYPE)
        self.n_top_nodes = self.n_top_prims = 0  # 0 = all of nodes / prims (no object instancing)
        self.media = np.zeros(0, MEDIUM_DTYPE)       # HomogeneousMedium / GridDensityMedium rows (volpath)
        self.grids = []                              # DensityGrid of each media row with grid = k > 0 (grids[k - 1])
        self.prim_media = None                       # MediumInterface per `prims` row, or None
        self.textures = np.zeros(0, T.TEXNODE_DTYPE)  # postfix texture programs (ABI v5)
        self.mipmaps = np.zeros(0, T.MIPMAP_DTYPE)    # rows point into the MipMap objects kept in mipmap_objects
        self.mipmap_objects = []
        self.material_ext = None                      # one MATERIAL_EXT row per material row when any is textured

    def desc(self):
        d = SceneDesc()
        d.abi_version = 5
        if len(self.textures):
            d.textures, d.n_textures = _ptr(self.textures), len(self.textures)
        if len(self.mipmaps):
            d.mipmaps, d.n_mipmaps = _ptr(self.mipmaps), len(self.mipmaps)
        if self.material_ext is not None:
            if len(self.material_ext) != len(self.materials):
                raise B200Error("FlatScene.material_ext must have one row per material row")
            d.material_ext = _ptr(self.material_ext)
        d.nodes, d.n_nodes = _ptr(self.nodes), len(self.nodes)
        d.prims, d.n_prims = _ptr(self.prims), len(self.prims)
        d.vertex_p, d.n_vertices = _ptr(self.vertex_p), len(self.vertex_p)
        d.vertex_n, d.vertex_s, d.vertex_uv = _ptr(self.vertex_n), _ptr(self.vertex_s), _ptr(self.vertex_uv)
        d.tri_indices, d.n_triangles = _ptr(self.tri_indices), len(self.tri_indices)
        d.spheres, d.n_spheres = _ptr(self.spheres), len(self.spheres)
        d.materials, d.n_materials = _ptr(self.materials), len(self.materials)
        d.lights, d.n_lights = _ptr(self.lights), len(self.lights)
        d.objects, d.n_objects = _ptr(self.objects), len(self.objects)
        d.instances, d.n_instances = _ptr(self.instances), len(self.instances)
        d.n_top_nodes, d.n_top_prims = self.n_top_nodes, self.n_top_prims
        if len(self.media):
            d.media, d.n_media = _ptr(self.media), len(self.media)
        if self.prim_media is not None and len(self.prim_media):
            if len(self.prim_media) != len(self.prims):
                raise B200Error("FlatScene.prim_media must have one row per primitive row")
            d.prim_media = _ptr(self.prim_media)
        return d

    def grid_table(self):
        """pbrt_b200_density_grid rows of `grids`; their density pointers stay valid while this FlatScene lives."""
        t = np.zeros(len(self.grids), DENSITY_GRID_DTYPE)
        for k, g in enumerate(self.grids):
            t[k]["medium_to_world"], t[k]["world_to_medium"] = g.medium_to_world.reshape(-1), g.world_to_medium.reshape(-1)
            t[k]["nx"], t[k]["ny"], t[k]["nz"], t[k]["density"] = g.nx, g.ny, g.nz, g.density.ctypes.data
        return t

    @property
    def world_bound(self):
        return self.nodes[0]["bounds"].copy() if len(self.nodes) else np.array([np.inf] * 3 + [-np.inf] * 3, f32)


def _tri_area(p0, p1, p2):
    """Triangle::area, triangle.rs:550-554: 0.5 * |(p1-p0) x (p2-p0)| with the f64 cross."""
    c = np.cross((p1 - p0).astype(np.float64), (p2 - p0).astype(np.float64)).astype(f32)
    return f32(0.5) * np.sqrt(c[..., 0] * c[..., 0] + c[..., 1] * c[..., 1] + c[..., 2] * c[..., 2]).astype(f32)


# copper eta/k as RGB: Spectrum::from_sampled of metal.rs:13-53 evaluated by
# tools/copper_rgb.py against the reference's CIE tables (src/core/cie.rs)
COPPER_N = (0.19999069, 0.92208463, 1.09987593)
COPPER_K = (3.90463543, 2.44763327, 2.13765264)


TEX_STACK_LIMIT = 8  # PB_TEX_STACK in csrc/texture.cuh


class TexturedMaterial:
    """A material row whose parameters come from pbrt_b200_material_ext: texture trees, a bump map, or uber / substrate."""

    def __init__(self, name, row, spectra, floats, bump):
        self.name, self.row, self.spectra, self.floats, self.bump = name, row, spectra, floats, bump

    def key(self):
        def k(x):
            return x.key() if T.is_texture(x) else np.asarray(x, f32).tobytes()

        return (self.row.tobytes(), tuple(k(x) for x in self.spectra), tuple(k(x) for x in self.floats), self.bump.key() if self.bump is not None else None)


class SceneBuilder:
    """Graphics state + shape/light factories of pbrt-rust's API (api.rs:552-806,1493-1546)."""

    def __init__(self):
        self.ctm = Transform()
        self._stack = []
        self.reverse_orientation = False
        self._material = self._mat_row("matte")  # api.rs default material: matte
        self._materials = []
        self._mat_index = {}
        self._area_light = None
        self._P, self._N, self._S, self._UV = [], [], [], []
        self._nverts = 0
        self._tris = []     # (indices[k,3] + base)
        self._prims = []    # rows of PRIM_DTYPE before ordering
        self._bounds = []
        self._spheres = []
        self._lights = []
        self.any_n = self.any_s = self.any_uv = False
        self._objects, self._instances, self._cur_object = {}, [], None
        # participating media (api.rs:1211-1258): named media are global (RenderOptions), the current interface is graphics state
        self._media, self._media_index = [], {}
        self._grids = []                # DensityGrid of each heterogeneous medium, in creation order
        self._medium_names = ("", "")   # (inside, outside) of GraphicsState
        self._pmedia = []               # one [n,2] int32 block per entry of self._prims: MediumInterface of each primitive row
        self.log = []  # every directive in call order (scenefile.py turns it back into a .pbrt file)

    # --- object instancing (api.rs:1593-1713) ---------------------------------
    def object_begin(self, name):
        self.log.append(("ObjectBegin", name))
        self._push()
        if self._cur_object is not None:
            raise B200Error("ObjectBegin called inside of instance definition")
        self._objects[name] = {"prims": [], "bounds": [], "pmedia": []}
        self._cur_object = name
        self._top = (self._prims, self._bounds, self._pmedia)
        self._prims, self._bounds, self._pmedia = self._objects[name]["prims"], self._objects[name]["bounds"], self._objects[name]["pmedia"]

    def object_end(self):
        if self._cur_object is None:
            raise B200Error("ObjectEnd called outside of instance definition")
        self._prims, self._bounds, self._pmedia = self._top
        self._cur_object = None
        self._pop()
        self.log.append(("ObjectEnd",))

    def object_instance(self, name):
        if self._cur_object is not None:
            raise B200Error("ObjectInstance can't be called inside instance definition")
        if name not in self._objects:
            raise B200Error(f'Unable to find instance named "{name}"')
        self.log.append(("ObjectInstance", name))
        if not self._objects[name]["prims"]:
            return  # api.rs:1684-1686: empty instance
        row = np.zeros(1, PRIM_DTYPE)
        row["shape_kind"], row["shape_index"], row["material"], row["area_light"] = SHAPE_INSTANCE, len(self._instances), -1, -1
        self._instances.append((name, self.ctm))
        self._prims.append(row)
        self._pmedia.append(np.full((1, 2), -1, np.int32))  # a TransformedPrimitive carries no interface; its GeometricPrimitives do
        self._bounds.append(None)  # TransformedPrimitive::world_bound needs the object's BVH: filled in by world_end

    # --- graphics state ---------------------------------------------------
    def _push(self):
        self._stack.append((self.ctm, self._material, self._area_light, self.reverse_orientation, self._medium_names))

    def _pop(self):
        self.ctm, self._material, self._area_light, self.reverse_orientation, self._medium_names = self._stack.pop()

    # --- participating media (api.rs:706-760,1211-1258) -----------------------
    def make_named_medium(self, name, type="homogeneous", sigma_a=(0.0011, 0.0024, 0.014), sigma_s=(2.55, 3.21, 3.77), g=0.0, scale=1.0, preset="",
                          density=None, nx=1, ny=1, nz=1, p0=(0.0, 0.0, 0.0), p1=(1.0, 1.0, 1.0)):
        """MakeNamedMedium (api.rs:1211-1241 -> make_medium :706-760): defaults as there; sigma_a / sigma_s are multiplied by `scale`.

        type="heterogeneous" is a GridDensityMedium (grid.rs): `density` holds nx * ny * nz values, x fastest, over the box p0..p1
        of the current transformation.  Its sigma_t is (sigma_a + sigma_s)[0], the first channel only, as the reference's
        constructor takes it; a sigma_t that is not the same in every channel draws a warning.  Where the reference logs an error and
        creates no medium -- `density` missing, or not nx * ny * nz values -- this raises B200Error, so that a smoke scene whose data
        failed to load is refused instead of rendered as vacuum."""
        kw = {"type": type, "sigma_a": tuple(np.asarray(sigma_a, f32).reshape(-1).tolist()) if not np.isscalar(sigma_a) else sigma_a,
              "sigma_s": tuple(np.asarray(sigma_s, f32).reshape(-1).tolist()) if not np.isscalar(sigma_s) else sigma_s, "g": g, "scale": scale}
        if type == "heterogeneous":
            kw.update({"nx": int(nx), "ny": int(ny), "nz": int(nz), "p0": tuple(np.asarray(p0, f32).tolist()), "p1": tuple(np.asarray(p1, f32).tolist()),
                       "density": None if density is None else np.asarray(density, f32).reshape(-1)})
        self.log.append(("MakeNamedMedium", name, kw))
        if type not in ("homogeneous", "heterogeneous"):
            raise B200Error(f'Medium "{type}" is outside the hot path (homogeneous, heterogeneous)')
        if preset:
            raise B200Error("named medium presets (get_medium_scattering_properties) are outside the hot path: give sigma_a / sigma_s")
        r = np.zeros(1, MEDIUM_DTYPE)[0]
        sa = np.full(3, sigma_a, f32) if np.isscalar(sigma_a) else np.asarray(sigma_a, f32)
        ss = np.full(3, sigma_s, f32) if np.isscalar(sigma_s) else np.asarray(sigma_s, f32)
        r["sigma_a"], r["sigma_s"], r["g"] = sa * f32(scale), ss * f32(scale), g
        if type == "heterogeneous":
            if density is None:
                raise B200Error(f'No "density" values provided for heterogeneous medium "{name}"')
            dens = np.asarray(density, f32).reshape(-1)
            if len(dens) != int(nx) * int(ny) * int(nz):
                raise B200Error(f'GridDensityMedium "{name}" has {len(dens)} density values; expected nx*ny*nz = {int(nx) * int(ny) * int(nz)}')
            st = r["sigma_a"] + r["sigma_s"]
            if not (st[0] == st[1] == st[2]):
                warnings.warn(f'GridDensityMedium "{name}" requires a spectrally uniform sigma_t; using the first channel, {float(st[0])}')
            pa, pb = np.asarray(p0, f32), np.asarray(p1, f32)
            m2w = self.ctm * Transform.translate(pa) * Transform.scale(*(pb - pa))
            self._grids.append(DensityGrid(dens, nx, ny, nz, m2w.m, m2w.m_inv))
            r["grid"] = len(self._grids)
        self._media_index[name] = len(self._media)  # HashMap::insert replaces the entry; primitives created earlier keep the old Arc
        self._media.append(r)

    def medium_interface(self, inside, outside=""):
        """MediumInterface (api.rs:1243-1258): names of the media inside / outside the shapes that follow ("" = none)."""
        self.log.append(("MediumInterface", inside, outside))
        self._medium_names = (inside, outside)

    def medium_index(self, name):
        """Row of `name` in FlatScene.media, -1 for "" (create_medium_interface, api.rs:382-403: an undefined name is an error there and None)."""
        if not name:
            return -1
        if name not in self._media_index:
            raise B200Error(f'Named medium "{name}" undefined')
        return self._media_index[name]

    def camera_medium(self):
        """Camera.medium: the OUTSIDE medium current at the Camera directive (api.rs:256,302-320 pass create_medium_interface().outside)."""
        return self.medium_index(self._medium_names[1])

    def _cur_pmedia(self, n):
        return np.tile(np.array([[self.medium_index(self._medium_names[0]), self.medium_index(self._medium_names[1])]], np.int32), (n, 1))

    def attribute_begin(self):
        self.log.append(("AttributeBegin",))
        self._push()

    def attribute_end(self):
        self._pop()
        self.log.append(("AttributeEnd",))

    def identity(self):
        self.log.append(("Identity",))
        self.ctm = Transform()

    def translate(self, x, y, z):
        self.log.append(("Translate", x, y, z))
        self.ctm = self.ctm * Transform.translate((x, y, z))

    def scale(self, x, y, z):
        self.log.append(("Scale", x, y, z))
        self.ctm = self.ctm * Transform.scale(x, y, z)

    def rotate(self, deg, x, y, z):
        self.log.append(("Rotate", deg, x, y, z))
        self.ctm = self.ctm * Transform.rotate(deg, (x, y, z))

    def transform(self, t):
        self.log.append(("ConcatTransform", t))
        self.ctm = self.ctm * t

    # --- materials (src/materials/*.rs create_* defaults) -------------------
    # parameter slots of pbrt_b200_material_ext, per material: (spectrum slots, float slots)
    MATERIAL_SLOTS = {"matte": (("Kd",), ("sigma",)), "plastic": (("Kd", "Ks"), ("roughness",)), "mirror": (("Kr",), ()),
                      "glass": (("Kr", "Kt"), ("uroughness", "vroughness", "eta")), "metal": (("eta", "k"), ("uroughness", "vroughness")),
                      "uber": (("Kd", "Ks", "Kr", "Kt", "opacity"), ("uroughness", "vroughness", "eta")),
                      "substrate": (("Kd", "Ks"), ("uroughness", "vroughness"))}
    MATERIAL_TYPES = {"matte": MAT_MATTE, "plastic": MAT_PLASTIC, "mirror": MAT_MIRROR, "glass": MAT_GLASS, "metal": MAT_METAL, "uber": MAT_UBER,
                      "substrate": MAT_SUBSTRATE}

    @staticmethod
    def _mat_row(name, **kw):
        """-> MATERIAL_DTYPE row (every parameter constant, one of the five hot materials) | TexturedMaterial | None.
        Parameter values are constants (scalar / RGB) or textures.Tex trees; "bumpmap" is a float texture."""
        if name in ("none", ""):
            return None
        if name not in SceneBuilder.MATERIAL_SLOTS:
            raise B200Error(f'Material "{name}" is outside the device path (matte, plastic, mirror, glass, metal, uber, substrate)')
        # create_* defaults (matte.rs:55-61, plastic.rs:72-80, mirror.rs:44-49, glass.rs:95-108, metal.rs:115-125, uber.rs:114-128,
        # substrate.rs:64-71); metal / uber fall back from u/vroughness to `roughness` (metal.rs:88-97, uber.rs:78-87)
        v = dict(kw)
        if name == "matte":
            v.setdefault("Kd", 0.5); v.setdefault("sigma", 0.0)
        elif name == "plastic":
            v.setdefault("Kd", 0.25); v.setdefault("Ks", 0.25); v.setdefault("roughness", 0.1)
        elif name == "mirror":
            v.setdefault("Kr", 0.9)
        elif name == "glass":
            v.setdefault("Kr", 1.0); v.setdefault("Kt", 1.0); v.setdefault("uroughness", 0.0); v.setdefault("vroughness", 0.0)
            v.setdefault("eta", v.get("index", 1.5))
        elif name == "metal":
            v.setdefault("eta", COPPER_N); v.setdefault("k", COPPER_K)
            rough = v.get("roughness", 0.01)
            v.setdefault("uroughness", rough); v.setdefault("vroughness", rough)
        elif name == "uber":
            v.setdefault("Kd", 0.25); v.setdefault("Ks", 0.25); v.setdefault("Kr", 0.0); v.setdefault("Kt", 0.0); v.setdefault("opacity", 1.0)
            rough = v.get("roughness", 0.1)
            v.setdefault("uroughness", rough); v.setdefault("vroughness", rough)
            v.setdefault("eta", v.get("index", 1.5))
        elif name == "substrate":
            v.setdefault("Kd", 0.5); v.setdefault("Ks", 0.5); v.setdefault("uroughness", 0.1); v.setdefault("vroughness", 0.1)
        sslots, fslots = SceneBuilder.MATERIAL_SLOTS[name]
        bump = v.get("bumpmap")
        if bump is not None and not T.is_texture(bump):
            bump = T.Tex.constant(bump)
        r = np.zeros(1, MATERIAL_DTYPE)[0]
        r["type"] = SceneBuilder.MATERIAL_TYPES[name]
        r["remap_roughness"] = 1 if v.get("remaproughness", True) else 0
        textured = bump is not None or name in ("uber", "substrate") or any(T.is_texture(v[k]) for k in sslots + fslots)

        def rgb(x):
            return np.zeros(3, f32) if T.is_texture(x) else (np.full(3, x, f32) if np.isscalar(x) or np.ndim(x) == 0 else np.asarray(x, f32))

        def flt(x):
            return f32(0.0) if T.is_texture(x) else f32(x)

        if name not in ("uber", "substrate"):
            for field, key in zip(("a", "b"), sslots):
                r[field] = rgb(v[key])
            for field, key in zip(("f0", "f1", "f2"), fslots):
                r[field] = flt(v[key])
        if not textured:
            return r
        r["textured"] = 1
        return TexturedMaterial(name, r, [v[k] for k in sslots], [v[k] for k in fslots], bump)

    def material(self, name, **kw):
        self.log.append(("Material", name, kw))
        self._material = self._mat_row(name, **kw)

    def _material_id(self):
        if self._material is None:
            return -1
        key = self._material.key() if isinstance(self._material, TexturedMaterial) else self._material.tobytes()
        if key not in self._mat_index:
            self._mat_index[key] = len(self._materials)
            self._materials.append(self._material if isinstance(self._material, TexturedMaterial) else self._material.copy())
        return self._mat_index[key]

    def _material_tables(self, fs):
        """materials[] (+ material_ext[], textures[], mipmaps[] when a row is textured) of the flat scene."""
        if not self._materials:
            return
        fs.materials = np.array([m.row if isinstance(m, TexturedMaterial) else m for m in self._materials], MATERIAL_DTYPE)
        if not any(isinstance(m, TexturedMaterial) for m in self._materials):
            return
        tabs = T.TextureTables()
        ext = np.zeros(len(self._materials), T.MATERIAL_EXT_DTYPE)
        for i, m in enumerate(self._materials):
            if not isinstance(m, TexturedMaterial):
                continue
            for k, val in enumerate(m.spectra):
                if T.is_texture(val):
                    ext[i]["s_tex"][k] = tabs.program(val)
                else:
                    ext[i]["s_const"][k] = np.full(3, val, f32) if np.isscalar(val) or np.ndim(val) == 0 else np.asarray(val, f32)
            for k, val in enumerate(m.floats):
                if T.is_texture(val):
                    ext[i]["f_tex"][k] = tabs.program(val)
                else:
                    ext[i]["f_const"][k] = f32(val)
            if m.bump is not None:
                ext[i]["bump"] = tabs.program(m.bump)
        fs.material_ext = ext
        fs.textures = tabs.node_array()
        fs.mipmap_objects = list(tabs.mipmaps)
        fs.mipmaps = tabs.mipmap_array()
        if tabs.max_depth > TEX_STACK_LIMIT:
            raise B200Error(f"texture expressions nest deeper than the device's value stack ({TEX_STACK_LIMIT} operands)")

    # --- lights ------------------------------------------------------------
    def area_light_source(self, name="diffuse", L=(1, 1, 1), scale=1.0, twosided=False, samples=1):  # diffuse.rs:178-195
        if name not in ("diffuse", "area"):
            raise B200Error(f'AreaLightSource "{name}" unknown')
        self.log.append(("AreaLightSource", name, {"L": L, "scale": scale, "twosided": twosided, **({"samples": int(samples)} if samples != 1 else {})}))
        self._area_light = (np.asarray(L, f32) * f32(scale) if not np.isscalar(L) else np.full(3, L * scale, f32), bool(twosided), max(int(samples), 1))

    def light_source(self, name, **kw):
        self.log.append(("LightSource", name, kw))
        r = np.zeros(1, LIGHT_DTYPE)[0]
        r["n_samples"] = 1

        def rgb(key, default):
            v = kw.get(key, default)
            return np.full(3, v, f32) if np.isscalar(v) else np.asarray(v, f32)

        sc = rgb("scale", 1.0)
        if name == "point":  # point.rs:99-106 (note the reference's translate(P.x, P.y, P.x) quirk)
            P = np.asarray(kw.get("from", (0, 0, 0)), f32)
            l2w = Transform.translate((P[0], P[1], P[0])) * self.ctm
            r["type"], r["L"], r["pos"] = LIGHT_POINT, rgb("I", 1.0) * sc, l2w.points([[0, 0, 0]])[0]
        elif name == "distant":  # distant.rs:124-132
            frm, to = np.asarray(kw.get("from", (0, 0, 0)), f32), np.asarray(kw.get("to", (0, 0, 1)), f32)
            w = self.ctm.vectors([frm - to])[0]
            w = w * (f32(1) / np.sqrt(f32(w[0] * w[0] + w[1] * w[1] + w[2] * w[2])))
            r["type"], r["L"], r["dir"] = LIGHT_DISTANT, rgb("L", 1.0) * sc, w
        elif name == "spot":  # spot.rs:119-146 (+ SpotLight::new :31-45)
            frm, to = np.asarray(kw.get("from", (0, 0, 0)), f32), np.asarray(kw.get("to", (0, 0, 1)), f32)
            d = to - frm
            d = d * (f32(1) / np.sqrt(f32(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])))
            if abs(d[0]) > abs(d[1]):  # vec3_coordinate_system, vector.rs:551-560 (division = multiply by the reciprocal)
                du = np.array([-d[2], 0, d[0]], f32) * (f32(1) / np.sqrt(f32(d[0] * d[0] + d[2] * d[2])))
            else:
                du = np.array([0, d[2], -d[1]], f32) * (f32(1) / np.sqrt(f32(d[1] * d[1] + d[2] * d[2])))
            d64, u64 = d.astype(np.float64), du.astype(np.float64)  # Vector3::cross is evaluated in f64 (vector.rs:339-353)
            dv = np.array([d64[1] * u64[2] - d64[2] * u64[1], d64[2] * u64[0] - d64[0] * u64[2], d64[0] * u64[1] - d64[1] * u64[0]]).astype(f32)
            m = np.array([[du[0], du[1], du[2], 0], [dv[0], dv[1], dv[2], 0], [d[0], d[1], d[2], 0], [0, 0, 0, 1]], f32)
            dirtoz = Transform(m)
            l2w = self.ctm * Transform.translate((frm[0], frm[1], frm[2])) * dirtoz.inverse()
            cone, delta = f32(kw.get("coneangle", 30.0)), f32(kw.get("conedeltaangle", 5.0))
            rad = lambda deg: f32(f32(np.pi) / f32(180.0)) * f32(deg)  # pbrt.rs:167-169
            r["type"], r["L"], r["pos"] = LIGHT_SPOT, rgb("I", 1.0) * sc, l2w.points([[0, 0, 0]])[0]
            r["cos_total_width"], r["cos_falloff_start"] = np.cos(rad(cone)), np.cos(rad(f32(cone - delta)))
            r["world_to_light"] = l2w.m_inv.reshape(-1)
        elif name == "infinite":  # infinite.rs, constant map only
            if kw.get("mapname"):
                raise B200Error("image-mapped infinite lights are outside the hot path")
            r["type"], r["L"], r["n_samples"] = LIGHT_INFINITE, rgb("L", 1.0) * sc, max(int(kw.get("samples", 1)), 1)
            # infinite.rs:128-156 takes sampled directions through light_to_world / world_to_light.  With the constant map of the hot path
            # the radiance does not depend on the direction, so the estimator stays unbiased under any CTM, but the 2x2 sin(theta)
            # importance map is not rotation invariant: under a non-identity CTM the reference draws a different sample set than
            # the identity-frame sampling done here (per-sample parity is lost, the expectation is not).  Say so instead of staying silent.
            if not np.allclose(self.ctm.m, np.eye(4, dtype=f32), atol=1e-6):
                import warnings
                warnings.warn('LightSource "infinite" under a non-identity CTM: directions are sampled in the world frame (the reference samples in the '
                              "light's frame, infinite.rs:128-156); the image is unbiased but not sample-for-sample identical to the reference's")
        else:
            raise B200Error(f'LightSource "{name}" is outside the hot path (point, spot, distant, infinite, diffuse area)')
        self._lights.append(r)

    # --- shapes --------------------------------------------------------------
    def shape(self, name, **kw):
        self.log.append(("Shape", name, kw))
        if name == "trianglemesh":
            return self._trianglemesh(**kw)
        if name == "sphere":
            return self._sphere(**kw)
        raise B200Error(f'Shape "{name}" is outside the hot path (trianglemesh, sphere)')

    def _trianglemesh(self, P, indices, N=None, S=None, uv=None):  # triangle.rs:33-73,657-760
        P = self.ctm.points(P)
        idx = np.asarray(indices, np.uint32).reshape(-1, 3)
        nv, nt = len(P), len(idx)
        base = self._nverts
        flags = (PRIM_REVERSE_ORIENTATION if self.reverse_orientation else 0) | (PRIM_SWAPS_HANDEDNESS if self.ctm.swaps_handedness() else 0)
        self._P.append(P)
        if N is not None:
            flags |= PRIM_HAS_N
            self.any_n = True
        if S is not None:
            flags |= PRIM_HAS_S
            self.any_s = True
        if uv is not None:
            flags |= PRIM_HAS_UV
            self.any_uv = True
        self._N.append(self.ctm.normals(N) if N is not None else np.zeros((nv, 3), f32))
        self._S.append(self.ctm.vectors(S) if S is not None else np.zeros((nv, 3), f32))
        self._UV.append(np.asarray(uv, f32).reshape(-1, 2) if uv is not None else np.zeros((nv, 2), f32))
        self._nverts += nv
        tri_base = sum(len(t) for t in self._tris)
        self._tris.append(idx + np.uint32(base))
        p0, p1, p2 = P[idx[:, 0]], P[idx[:, 1]], P[idx[:, 2]]
        lo = np.minimum(np.minimum(p0, p1), p2)
        hi = np.maximum(np.maximum(p0, p1), p2)
        self._bounds.append(np.concatenate([lo, hi], axis=1))
        rows = np.zeros(nt, PRIM_DTYPE)
        rows["shape_kind"] = SHAPE_TRIANGLE
        rows["shape_index"] = np.arange(tri_base, tri_base + nt, dtype=np.uint32)
        rows["material"] = self._material_id()
        rows["area_light"] = -1
        rows["flags"] = flags
        if self._area_light is not None and self._cur_object is not None:
            raise B200Error("Area lights not supported with object instancing (api.rs:1573-1575)")
        if self._area_light is not None:  # api.rs:1531-1546: one DiffuseAreaLight per shape
            L, two, nsamp = self._area_light
            lights = np.zeros(nt, LIGHT_DTYPE)
            lights["type"], lights["two_sided"], lights["L"] = LIGHT_DIFFUSE, int(two), L
            lights["shape_kind"], lights["shape_index"], lights["shape_flags"] = SHAPE_TRIANGLE, rows["shape_index"], flags
            lights["area"] = _tri_area(p0, p1, p2)
            lights["n_samples"] = nsamp
            first = len(self._lights)
            self._lights.extend(list(lights))
            rows["area_light"] = np.arange(first, first + nt, dtype=np.int32)
        self._prims.append(rows)
        self._pmedia.append(self._cur_pmedia(nt))

    def _sphere(self, radius=1.0):  # sphere.rs:397-432 (full sphere)
        o2w = self.ctm
        r = np.zeros(1, SPHERE_DTYPE)[0]
        r["object_to_world"], r["world_to_object"], r["radius"] = o2w.m.reshape(-1), o2w.m_inv.reshape(-1), radius
        flags = (PRIM_REVERSE_ORIENTATION if self.reverse_orientation else 0) | (PRIM_SWAPS_HANDEDNESS if o2w.swaps_handedness() else 0)
        r["flags"] = flags
        if self._area_light is not None and self._cur_object is not None:
            raise B200Error("Area lights not supported with object instancing (api.rs:1573-1575)")
        # Transform::transform_bounds of the object bound (transform.rs:593-605)
        rr = f32(radius)
        corners = np.array([[x, y, z] for x in (-rr, rr) for y in (-rr, rr) for z in (-rr, rr)], f32)
        wc = o2w.points(corners)
        self._bounds.append(np.concatenate([wc.min(0), wc.max(0)])[None, :])
        row = np.zeros(1, PRIM_DTYPE)
        row["shape_kind"], row["shape_index"], row["material"], row["area_light"], row["flags"] = SHAPE_SPHERE, len(self._spheres), self._material_id(), -1, flags
        if self._area_light is not None:  # api.rs:1531-1546 + DiffuseAreaLight::new (diffuse.rs:33-66): area = Sphere::area (sphere.rs:291-293)
            L, two, nsamp = self._area_light
            light = np.zeros(1, LIGHT_DTYPE)[0]
            light["type"], light["two_sided"], light["L"] = LIGHT_DIFFUSE, int(two), L
            light["shape_kind"], light["shape_index"], light["shape_flags"] = SHAPE_SPHERE, len(self._spheres), flags
            phi_max = f32(f32(np.pi) / f32(180.0)) * f32(360.0)  # radians(clamp(phimax, 0, 360)), sphere.rs:36
            light["area"] = phi_max * rr * (rr - (-rr))
            light["n_samples"] = nsamp
            row["area_light"] = len(self._lights)
            self._lights.append(light)
        self._spheres.append(r)
        self._prims.append(row)
        self._pmedia.append(self._cur_pmedia(1))

    # --- WorldEnd: make_scene (api.rs:244-251) -------------------------------
    def world_end(self, max_prims=4, split_method="sah", builder=None):
        fs = FlatScene()
        fs.source_log, fs.accelerator = self.log, (split_method, max_prims)
        nprim = sum(len(p) for p in self._prims)
        if self._P:
            fs.vertex_p = np.ascontiguousarray(np.concatenate(self._P), f32)
            fs.tri_indices = np.ascontiguousarray(np.concatenate(self._tris), np.uint32)
            if self.any_n:
                fs.vertex_n = np.ascontiguousarray(np.concatenate(self._N), f32)
            if self.any_s:
                fs.vertex_s = np.ascontiguousarray(np.concatenate(self._S), f32)
            if self.any_uv:
                fs.vertex_uv = np.ascontiguousarray(np.concatenate(self._UV), f32)
        if self._spheres:
            fs.spheres = np.array(self._spheres, SPHERE_DTYPE)
        self._material_tables(fs)
        if self._lights:
            fs.lights = np.array(self._lights, LIGHT_DTYPE)
        if self._cur_object is not None:
            raise B200Error("WorldEnd inside an object definition")
        build = builder or DEFAULT_BVH_BUILDER or bvh_build
        # ObjectInstance (api.rs:1663-1713): an object with more than one primitive gets its own accelerator, built with the
        # scene's accelerator parameters; TransformedPrimitive::world_bound = prim_to_world.motion_bounds(object bound)
        used, obj_tables, next_ci = {}, [], nprim
        for name, _ in self._instances:
            if name in used:
                continue
            o = self._objects[name]
            oprims = np.concatenate(o["prims"])
            opm = np.concatenate(o["pmedia"])
            obounds = np.ascontiguousarray(np.concatenate(o["bounds"]), f32)
            oprims["creation_index"] = np.arange(next_ci, next_ci + len(oprims), dtype=np.uint32)
            next_ci += len(oprims)
            if len(oprims) > 1:
                onodes, oorder = build(obounds, max_prims, split_method)
                oprims = oprims[oorder]
                opm = opm[oorder]
                wb = onodes[0]["bounds"].copy()
            else:
                onodes, wb = np.zeros(0, NODE_DTYPE), obounds[0].copy()
            used[name] = len(obj_tables)
            obj_tables.append((onodes, np.ascontiguousarray(oprims), wb, opm))
        if nprim:
            for k, bnd in enumerate(self._bounds):
                if bnd is None:
                    inst = int(self._prims[k]["shape_index"][0])
                    name, ctm = self._instances[inst]
                    self._bounds[k] = ctm.bounds(obj_tables[used[name]][2])[None, :]
            prims = np.concatenate(self._prims)
            prims["creation_index"] = np.arange(nprim, dtype=np.uint32)
            bounds = np.ascontiguousarray(np.concatenate(self._bounds), f32)
            nodes, ordered = build(bounds, max_prims, split_method)
            fs.nodes = nodes
            fs.prims = np.ascontiguousarray(prims[ordered])
            fs.prim_bounds = bounds
            pmedia = [np.concatenate(self._pmedia)[ordered]]
        else:
            pmedia = [np.zeros((0, 2), np.int32)]
        if obj_tables:
            fs.n_top_nodes, fs.n_top_prims = len(fs.nodes), len(fs.prims)
            objs = np.zeros(len(obj_tables), OBJECT_DTYPE)
            all_nodes, all_prims = [fs.nodes], [fs.prims]
            noff, poff = len(fs.nodes), len(fs.prims)
            for k, (onodes, oprims, _, opm) in enumerate(obj_tables):
                objs[k] = (noff, len(onodes), poff, len(oprims))
                all_nodes.append(onodes); all_prims.append(oprims); pmedia.append(opm)
                noff += len(onodes); poff += len(oprims)
            fs.nodes = np.ascontiguousarray(np.concatenate(all_nodes))
            fs.prims = np.ascontiguousarray(np.concatenate(all_prims))
            fs.objects = objs
            inst = np.zeros(len(self._instances), INSTANCE_DTYPE)
            for k, (name, ctm) in enumerate(self._instances):
                inst[k]["prim_to_world"], inst[k]["world_to_prim"], inst[k]["object"] = ctm.m.reshape(-1), ctm.m_inv.reshape(-1), used[name]
            fs.instances = inst
        if self._media:
            fs.media = np.array(self._media, MEDIUM_DTYPE)
            fs.grids = list(self._grids)
            pm = np.concatenate(pmedia)
            if len(pm) and (pm >= 0).any():
                fs.prim_media = np.ascontiguousarray(pm.view(MEDIUM_INTERFACE_DTYPE).reshape(-1))
        return fs


# ---------------------------------------------------------------------------
# Camera / Film / Sampler / Integrator descriptions
# ---------------------------------------------------------------------------


def _filter_eval(name, radius, x, y, **kw):
    """Filters::evaluate (src/filters/*.rs) for the table build in Film::new."""
    rx, ry = f32(radius[0]), f32(radius[1])
    if name == "box":
        return f32(1)
    if name == "gaussian":  # gaussian.rs:16-33
        alpha = f32(kw.get("alpha", 2.0))
        ex, ey = f32(np.exp(-alpha * rx * rx)), f32(np.exp(-alpha * ry * ry))
        gx = max(f32(0), f32(np.exp(-alpha * x * x)) - ex)
        gy = max(f32(0), f32(np.exp(-alpha * y * y)) - ey)
        return f32(gx * gy)
    if name == "triangle":  # triangle.rs (filters)
        return f32(max(f32(0), rx - abs(x)) * max(f32(0), ry - abs(y)))
    if name == "mitchell":  # mitchell.rs:26-45, including its two slips (`6B * 30C`, `x * x` in the inner branch)
        B, Cc = f32(kw.get("B", 1.0 / 3.0)), f32(kw.get("C", 1.0 / 3.0))

        def m1d(v):
            v = f32(v)
            a = abs(f32(2) * v)
            if a > 1:
                return f32(((-B - f32(6) * Cc) * a * a * a + (f32(6) * B * f32(30) * Cc) * a * a + (f32(-12) * B - f32(48) * Cc) * a +
                            (f32(8) * B + f32(24) * Cc)) * f32(1.0 / 6.0))
            return f32(((f32(12) - f32(9) * B - f32(6) * Cc) * a * a * a + (f32(-18) + f32(12) * B + f32(6) * Cc) * v * v + (f32(6) - f32(2) * B)) *
                       f32(1.0 / 6.0))

        return f32(m1d(f32(x) * (f32(1) / rx)) * m1d(f32(y) * (f32(1) / ry)))
    if name == "sinc":  # sinc.rs:18-45: the window test is `y < radius -> 0`, so the table is zero inside the support (kept as is)
        tau = f32(kw.get("tau", 3.0))

        def sinc(v):
            v = abs(f32(v))
            if v < f32(1e-5):
                return f32(1)
            return f32(np.sin(f32(np.pi) * v)) / (f32(np.pi) * v)

        def wsinc(v, r):
            v = abs(f32(v))
            if v < r:
                return f32(0)
            return f32(sinc(v) * sinc(v / tau))

        return f32(wsinc(x, rx) * wsinc(y, ry))
    raise B200Error(f'Filter "{name}" unknown')  # api.rs:868-881 panics


FILTER_DEFAULT_RADIUS = {"box": (0.5, 0.5), "gaussian": (2.0, 2.0), "triangle": (2.0, 2.0), "mitchell": (2.0, 2.0), "sinc": (4.0, 4.0)}


class Film:
    """Film::new (film.rs:56-102): crop bounds, 16x16 filter table, sample bounds."""

    def __init__(self, xres, yres, filter="box", radius=None, crop=(0.0, 1.0, 0.0, 1.0), scale=1.0, max_sample_luminance=float("inf"), **fkw):
        self.full_resolution = (int(xres), int(yres))
        self.filter = filter
        self.radius = tuple(radius or FILTER_DEFAULT_RADIUS[filter])
        x0, x1, y0, y1 = crop
        self.crop, self.filter_params = tuple(float(v) for v in crop), dict(fkw)
        self.cropped_pixel_bounds = (int(math.ceil(f32(xres) * f32(x0))), int(math.ceil(f32(yres) * f32(y0))),
                                     int(math.ceil(f32(xres) * f32(x1))), int(math.ceil(f32(yres) * f32(y1))))
        self.scale = scale
        self.max_sample_luminance = max_sample_luminance
        tab = np.zeros(256, f32)
        for y in range(16):
            for x in range(16):
                px = (f32(x) + f32(0.5)) * f32(self.radius[0]) / f32(16)
                py = (f32(y) + f32(0.5)) * f32(self.radius[1]) / f32(16)
                tab[y * 16 + x] = _filter_eval(filter, self.radius, px, py, **fkw)
        self.filter_table = tab

    @property
    def sample_bounds(self):  # film.rs:104-111
        b = self.cropped_pixel_bounds
        rx, ry = f32(self.radius[0]), f32(self.radius[1])
        return (int(math.floor(f32(b[0]) + f32(0.5) - rx)), int(math.floor(f32(b[1]) + f32(0.5) - ry)),
                int(math.ceil(f32(b[2]) - f32(0.5) + rx)), int(math.ceil(f32(b[3]) - f32(0.5) + ry)))

    @property
    def width(self):
        return self.cropped_pixel_bounds[2] - self.cropped_pixel_bounds[0]

    @property
    def height(self):
        return self.cropped_pixel_bounds[3] - self.cropped_pixel_bounds[1]

    def desc(self):
        d = FilmDesc()
        d.full_resolution[:] = self.full_resolution
        d.cropped_pixel_bounds[:] = self.cropped_pixel_bounds
        d.filter_radius[:] = self.radius
        d.filter_table[:] = self.filter_table.tolist()
        d.scale, d.max_sample_luminance = self.scale, self.max_sample_luminance
        return d


class PerspectiveCamera:
    """PerspectiveCamera::new + create_perspective_camera (perspective.rs:40-86,298-357)."""

    def __init__(self, film, camera_to_world, fov=90.0, lensradius=0.0, focaldistance=1.0e30, shutteropen=0.0, shutterclose=1.0, screenwindow=None):
        xr, yr = film.full_resolution
        frame = f32(xr) / f32(yr)
        if screenwindow is not None:
            sx0, sx1, sy0, sy1 = (f32(v) for v in screenwindow)
        elif frame > 1:
            sx0, sx1, sy0, sy1 = -frame, frame, f32(-1), f32(1)
        else:
            sx0, sx1, sy0, sy1 = f32(-1), f32(1), f32(-1) / frame, f32(1) / frame
        c2s = Transform.perspective(fov, 1e-2, 1000.0)
        s2r = (Transform.scale(f32(xr), f32(yr), 1) * Transform.scale(f32(1) / (sx1 - sx0), f32(1) / (sy0 - sy1), 1) *
               Transform.translate((-sx0, -sy1, 0)))
        self.raster_to_camera = c2s.inverse() * s2r.inverse()
        self.camera_to_world = camera_to_world
        self.lens_radius, self.focal_distance = lensradius, focaldistance
        self.fov, self.screenwindow = fov, (None if screenwindow is None else tuple(float(v) for v in screenwindow))
        self.shutter_open, self.shutter_close = shutteropen, shutterclose

    def desc(self):
        d = CameraDesc()
        d.raster_to_camera[:] = self.raster_to_camera.m.reshape(-1).tolist()
        d.camera_to_world[:] = self.camera_to_world.m.reshape(-1).tolist()
        d.lens_radius, d.focal_distance = self.lens_radius, self.focal_distance
        d.shutter_open, d.shutter_close = self.shutter_open, self.shutter_close
        return d


class Sampler:
    KINDS = {"sobol": SAMPLER_SOBOL, "halton": SAMPLER_HALTON, "02sequence": SAMPLER_ZEROTWO, "lowdiscrepancy": SAMPLER_ZEROTWO}

    def __init__(self, name="halton", pixelsamples=16, dimensions=4):
        if name not in self.KINDS:
            raise B200Error(f'Sampler "{name}" is outside the hot path (sobol, halton, 02sequence)')
        self.kind, self.spp, self.dimensions = self.KINDS[name], int(pixelsamples), int(dimensions)
        if self.kind == SAMPLER_ZEROTWO and self.spp > 0:  # zerotwosequence.rs:33-36 rounds up; SobolSampler::new only warns (sobol.rs:35-40)
            self.spp = 1 << (self.spp - 1).bit_length()

    def desc(self, film):
        t = sampler_tables()
        d = SamplerDesc()
        d.kind, d.samples_per_pixel, d.n_sampled_dimensions = self.kind, self.spp, self.dimensions
        d.sample_bounds[:] = film.sample_bounds
        d.sobol_matrices32, d.vdc_matrices, d.vdc_matrices_inv = _ptr(t["sobol32"]), _ptr(t["vdc"]), _ptr(t["vdc_inv"])
        return d


class PathIntegrator:
    """PathIntegrator + create_path_integrator (src/integrators/path.rs:32-59,225-253)."""

    STRATEGY = {"uniform": LIGHTS_UNIFORM, "power": LIGHTS_POWER, "spatial": LIGHTS_SPATIAL}
    kind = INTEGRATOR_PATH
    name = "path"

    def __init__(self, camera, film, sampler, maxdepth=5, rrthreshold=1.0, lightsamplestrategy="spatial", pixelbounds=None):
        self.camera, self.film, self.sampler = camera, film, sampler
        self.max_depth, self.rr_threshold = int(maxdepth), float(rrthreshold)
        if lightsamplestrategy not in self.STRATEGY:
            lightsamplestrategy = "spatial"  # path.rs -> lightdistrib.rs:27-30
        self.light_sample_strategy = lightsamplestrategy
        sb = film.sample_bounds
        self.pixelbounds_param = pixelbounds
        if pixelbounds is not None:  # path.rs:233-246: (x0, x1, y0, y1) intersected with the sample bounds
            x0, x1, y0, y1 = pixelbounds
            sb = (max(sb[0], x0), max(sb[1], y0), min(sb[2], x1), min(sb[3], y1))
        self.pixel_bounds = sb

    def desc(self, tile_range=None, sample_range=None, paths_in_flight=0, flags=0, tile_interleave=None, tile_order=0):
        d = RenderDesc()
        d.tile_order = int(tile_order)  # 0: the reference's row-major tile numbering; S: S x S-tile super-tiles (pbrt_b200.h)
        d.camera, d.film, d.sampler = self.camera.desc(), self.film.desc(), self.sampler.desc(self.film)
        d.integrator.max_depth, d.integrator.rr_threshold = self.max_depth, self.rr_threshold
        d.integrator.pixel_bounds[:] = self.pixel_bounds
        d.integrator.light_sample_strategy = self.STRATEGY[self.light_sample_strategy]
        d.integrator.kind = self.kind
        d.integrator.camera_medium = int(getattr(self, "camera_medium", -1))
        if tile_range:
            d.tile_begin, d.tile_end = tile_range
        if sample_range:
            d.sample_begin, d.sample_end = sample_range
        d.paths_in_flight, d.flags = paths_in_flight, flags
        if tile_interleave:  # (group, mod, rem): static multi-GPU ownership of tile groups
            d.tile_group, d.tile_mod, d.tile_rem = tile_interleave
        return d

    def n_tiles(self):  # integrator.rs:274-279
        sb = self.film.sample_bounds
        return ((sb[2] - sb[0] + 15) // 16) * ((sb[3] - sb[1] + 15) // 16)

    def n_tile_positions(self, tile_order=0):
        """Length of the tile numbering `tile_order` (pbrt_b200_tile_positions): n_tiles() for 0, padded to whole super-tiles otherwise."""
        sb = self.film.sample_bounds
        ntx, nty = (sb[2] - sb[0] + 15) // 16, (sb[3] - sb[1] + 15) // 16
        if not tile_order:
            return ntx * nty
        S = int(tile_order)
        return ((ntx + S - 1) // S) * ((nty + S - 1) // S) * S * S

    def render(self, scene, **kw):
        """Integrator::render (integrator.rs:249-252) -> linear RGB image [h, w, 3]."""
        rgbw, stats = scene.render(self, **kw)
        return scene.film_resolve(rgbw, self.film.scale).reshape(self.film.height, self.film.width, 3), stats


class DirectLightingIntegrator(PathIntegrator):
    """DirectLightingIntegrator + create_directlighting_integrator (src/integrators/directlighting.rs:27-39,122-157)."""
    name = "directlighting"

    def __init__(self, camera, film, sampler, maxdepth=5, strategy="all", pixelbounds=None):
        super().__init__(camera, film, sampler, maxdepth=maxdepth, lightsamplestrategy="uniform", pixelbounds=pixelbounds)
        if strategy not in ("one", "all"):
            strategy = "all"  # directlighting.rs:149-152: unknown strategies fall back to "all" with a warning
        self.strategy = strategy
        self.kind = INTEGRATOR_DIRECT_ALL if strategy == "all" else INTEGRATOR_DIRECT_ONE


class VolPathIntegrator(PathIntegrator):
    """VolPathIntegrator + create_volpath_integrator (src/integrators/volpath.rs:36-80,224-262): the path integrator's parameters, plus
    the medium the camera sits in (Camera.medium = the outside medium current at the Camera directive: SceneBuilder.camera_medium())."""
    name = "volpath"
    kind = INTEGRATOR_VOLPATH

    def __init__(self, camera, film, sampler, maxdepth=5, rrthreshold=1.0, lightsamplestrategy="spatial", pixelbounds=None, camera_medium=-1):
        super().__init__(camera, film, sampler, maxdepth=maxdepth, rrthreshold=rrthreshold, lightsamplestrategy=lightsamplestrategy, pixelbounds=pixelbounds)
        self.camera_medium = int(camera_medium)


class BDPTIntegrator(PathIntegrator):
    """BDPTIntegrator + create_bdpt_integrator (src/integrators/bdpt.rs; pbrt-v3 integrators/bdpt.cpp:448-480): maxdepth, the light
    sample strategy (default "power"; "spatial" is looked up at the camera vertex) and pixelbounds.  Its light-tracing strategies splat
    onto a second film, so it renders through Scene.render_splat; render() resolves both films with splat_scale = 1 / spp."""
    name = "bdpt"
    kind = INTEGRATOR_BDPT

    def __init__(self, camera, film, sampler, maxdepth=5, lightsamplestrategy="power", pixelbounds=None, visualizestrategies=False,
                 visualizeweights=False):
        if visualizestrategies or visualizeweights:
            raise B200Error('Integrator "bdpt": visualizestrategies / visualizeweights are not rendered on the device')
        if int(maxdepth) < 0 or int(maxdepth) > BDPT_MAX_DEPTH:
            raise B200Error(f'Integrator "bdpt": maxdepth {int(maxdepth)} is outside [0, {BDPT_MAX_DEPTH}] (every subpath vertex is kept in device memory)')
        if lightsamplestrategy not in self.STRATEGY:
            raise B200Error(f'Integrator "bdpt": unknown lightsamplestrategy "{lightsamplestrategy}" (uniform, power, spatial)')
        super().__init__(camera, film, sampler, maxdepth=maxdepth, rrthreshold=1.0, lightsamplestrategy=lightsamplestrategy, pixelbounds=pixelbounds)

    def render(self, scene, **kw):
        """-> linear RGB image [h, w, 3] (Film::write_image(1 / spp)), stats."""
        rgbw, splat, stats = scene.render_splat(self, **kw)
        img = scene.film_resolve_splat(rgbw, splat, 1.0 / self.sampler.spp, self.film.scale)
        return img.reshape(self.film.height, self.film.width, 3), stats


class WhittedIntegrator(PathIntegrator):
    """WhittedIntegrator + create_whitted_integrator (src/integrators/whitted.rs:25-50,108-131)."""
    name = "whitted"
    kind = INTEGRATOR_WHITTED

    def __init__(self, camera, film, sampler, maxdepth=5, pixelbounds=None):
        super().__init__(camera, film, sampler, maxdepth=maxdepth, lightsamplestrategy="uniform", pixelbounds=pixelbounds)


class Scene:
    """Device-resident Scene (scene.rs:23-29): owns the opaque `pbrt_b200_scene*`."""

    def __init__(self, flat: FlatScene, device=0):
        self.lib = load_library()
        self.flat = flat
        self.device = device
        h = C.c_void_p()
        d = flat.desc()
        grids = flat.grid_table()
        _check(self.lib.pbrt_b200_scene_create_with_grids(C.byref(d), _ptr(grids), len(grids), device, C.byref(h)), "pbrt_b200_scene_create")
        self.handle = h

    def close(self):
        if getattr(self, "handle", None):
            self.lib.pbrt_b200_scene_destroy(self.handle)
            self.handle = None

    __del__ = close

    def world_bound(self):
        b = np.zeros(6, f32)
        _check(self.lib.pbrt_b200_scene_world_bound(self.handle, _ptr(b)), "pbrt_b200_scene_world_bound")
        return b

    def intersect(self, rays):
        """Scene::intersect over a batch of RAY_DTYPE rays -> HIT_DTYPE records (host buffers)."""
        rays = np.ascontiguousarray(rays, RAY_DTYPE)
        hits = np.zeros(len(rays), HIT_DTYPE)
        _check(self.lib.pbrt_b200_intersect(self.handle, _ptr(rays), len(rays), _ptr(hits)), "pbrt_b200_intersect")
        return hits

    def intersect_p(self, rays):
        rays = np.ascontiguousarray(rays, RAY_DTYPE)
        occ = np.zeros(len(rays), np.uint8)
        _check(self.lib.pbrt_b200_intersect_p(self.handle, _ptr(rays), len(rays), _ptr(occ)), "pbrt_b200_intersect_p")
        return occ.astype(bool)

    def intersect_dev(self, rays_ptr, n, hits_ptr, stream=None):
        _check(self.lib.pbrt_b200_intersect_dev(self.handle, rays_ptr, n, hits_ptr, stream), "pbrt_b200_intersect_dev")

    def intersect_p_dev(self, rays_ptr, n, occ_ptr, stream=None):
        _check(self.lib.pbrt_b200_intersect_p_dev(self.handle, rays_ptr, n, occ_ptr, stream), "pbrt_b200_intersect_p_dev")

    def light_distribution_lookup(self, points, strategy="spatial", lazy=False):
        """LightDistribution::lookup at `points` -> (voxel [n,3] int32, func [n,n_lights] f32)."""
        pts = np.ascontiguousarray(points, f32).reshape(-1, 3)
        nl = len(self.flat.lights) if self.flat.lights is not None else 0
        voxel = np.zeros((len(pts), 3), np.int32)
        func = np.zeros((len(pts), max(nl, 1)), f32)
        _check(self.lib.pbrt_b200_light_distribution_lookup(self.handle, PathIntegrator.STRATEGY[strategy], RENDER_LAZY_SPATIAL if lazy else 0, _ptr(pts),
                                                           C.c_uint64(len(pts)), _ptr(voxel), _ptr(func)), "pbrt_b200_light_distribution_lookup")
        return voxel, func[:, :nl]

    def render(self, integrator, rgbw=None, tile_range=None, sample_range=None, paths_in_flight=0, device_ptr=None, tile_interleave=None, flags=0,
               tile_order=0):
        film = integrator.film
        stats = RenderStats()
        if device_ptr is not None:
            d = integrator.desc(tile_range, sample_range, paths_in_flight, RENDER_KEEP_ON_DEVICE | flags, tile_interleave, tile_order)
            _check(self.lib.pbrt_b200_render(self.handle, C.byref(d), device_ptr, C.byref(stats)), "pbrt_b200_render")
            return None, stats
        if rgbw is None:  # fresh image: the library overwrites it (no zero fill, no read-modify-write on the host)
            rgbw = np.empty((film.height * film.width, 4), f32)
            flags |= RENDER_OVERWRITE
        d = integrator.desc(tile_range, sample_range, paths_in_flight, flags, tile_interleave, tile_order)
        _check(self.lib.pbrt_b200_render(self.handle, C.byref(d), _ptr(rgbw), C.byref(stats)), "pbrt_b200_render")
        return rgbw, stats

    def film_resolve(self, rgbw, scale=1.0):
        rgbw = np.ascontiguousarray(rgbw, f32).reshape(-1, 4)
        out = np.zeros((len(rgbw), 3), f32)
        _check(self.lib.pbrt_b200_film_resolve(_ptr(rgbw), len(rgbw), scale, _ptr(out)), "pbrt_b200_film_resolve")
        return out

    def render_splat(self, integrator, rgbw=None, splat=None, tile_range=None, sample_range=None, device_ptrs=None, tile_interleave=None, flags=0,
                     tile_order=0):
        """pbrt_b200_render_splat -> ({r,g,b,w} sums [npix, 4], splat RGB sums [npix, 3], stats).  Buffers passed in are added to;
        device_ptrs = (rgbw, splat) device pointers keeps both films on the device."""
        film = integrator.film
        stats = RenderStats()
        if device_ptrs is not None:
            d = integrator.desc(tile_range, sample_range, 0, RENDER_KEEP_ON_DEVICE | flags, tile_interleave, tile_order)
            _check(self.lib.pbrt_b200_render_splat(self.handle, C.byref(d), device_ptrs[0], device_ptrs[1], C.byref(stats)), "pbrt_b200_render_splat")
            return None, None, stats
        if rgbw is None and splat is None:  # fresh films: the library overwrites them
            rgbw = np.empty((film.height * film.width, 4), f32)
            splat = np.empty((film.height * film.width, 3), f32)
            flags |= RENDER_OVERWRITE
        elif rgbw is None or splat is None:
            raise B200Error("render_splat: pass both films or neither")
        d = integrator.desc(tile_range, sample_range, 0, flags, tile_interleave, tile_order)
        _check(self.lib.pbrt_b200_render_splat(self.handle, C.byref(d), _ptr(rgbw), _ptr(splat), C.byref(stats)), "pbrt_b200_render_splat")
        return rgbw, splat, stats

    def film_resolve_splat(self, rgbw, splat, splat_scale, scale=1.0):
        rgbw = np.ascontiguousarray(rgbw, f32).reshape(-1, 4)
        splat = np.ascontiguousarray(splat, f32).reshape(-1, 3)
        out = np.zeros((len(rgbw), 3), f32)
        _check(self.lib.pbrt_b200_film_resolve_splat(_ptr(rgbw), _ptr(splat), len(rgbw), splat_scale, scale, _ptr(out)), "pbrt_b200_film_resolve_splat")
        return out


def make_rays(o, d, t_max=np.inf, time=0.0):
    o, d = np.asarray(o, f32).reshape(-1, 3), np.asarray(d, f32).reshape(-1, 3)
    r = np.zeros(len(o), RAY_DTYPE)
    r["o"], r["d"], r["t_max"], r["time"] = o, d, t_max, time
    return r
