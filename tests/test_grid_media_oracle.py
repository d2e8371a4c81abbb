"""Heterogeneous (grid density) media: the oracle's GridDensityMedium restatement (oracle/oracle_grid.hpp), the host and scene-file
front end that build its tables, and the checks scene_create makes before anything reaches the device.  Runs without a GPU.

The reference has no test for grid.rs, so the restatement is pinned to closed forms: the trilinear field against numpy, Beer-Lambert
through an absorbing grid against numpy quadrature of that field, and the white furnace, which has radiance 1 whatever the field is.
"""
import ctypes as C
import importlib
import math
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest
from oracle import oracle_grid as G

f32 = np.float32
HEADER = Path(__file__).resolve().parent.parent / "include" / "pbrt_b200.h"


def _np_density(d, nx, ny, nz, p):
    """GridDensityMedium::density restated in numpy (float64): trilinear over voxel centres, 0 outside the grid."""
    g = np.asarray(d, np.float64).reshape(nz, ny, nx)
    s = np.asarray(p, np.float64) * np.array([nx, ny, nz]) - 0.5
    i = np.floor(s).astype(np.int64)
    t = s - i
    out = np.zeros(len(s))
    for dz in (0, 1):
        for dy in (0, 1):
            for dx in (0, 1):
                x, y, z = i[:, 0] + dx, i[:, 1] + dy, i[:, 2] + dz
                inside = (x >= 0) & (y >= 0) & (z >= 0) & (x < nx) & (y < ny) & (z < nz)
                v = np.where(inside, g[np.clip(z, 0, nz - 1), np.clip(y, 0, ny - 1), np.clip(x, 0, nx - 1)], 0.0)
                w = (t[:, 0] if dx else 1 - t[:, 0]) * (t[:, 1] if dy else 1 - t[:, 1]) * (t[:, 2] if dz else 1 - t[:, 2])
                out += w * v
    return out


def _grid_scene(pkg, density, nx, ny, nz, p0, p1, sigma_a, sigma_s, g=0.0):
    H = pkg.host
    b = H.SceneBuilder()
    b.make_named_medium("m", type="heterogeneous", sigma_a=sigma_a, sigma_s=sigma_s, g=g, density=density, nx=nx, ny=ny, nz=nz, p0=p0, p1=p1)
    b.medium_interface("m", "m")
    return b


def test_density_matches_numpy_trilinear(pkg, oracle):
    rng = np.random.default_rng(3)
    nx, ny, nz = 5, 4, 3
    d = rng.uniform(0.0, 2.0, nx * ny * nz).astype(f32)
    b = _grid_scene(pkg, d, nx, ny, nz, (0, 0, 0), (1, 1, 1), (1.0,) * 3, (0.0,) * 3)
    b.area_light_source("diffuse", L=(1.0, 1.0, 1.0))
    P, I = pkg.scenes.quad((-1, -1, 3), (1, -1, 3), (1, 1, 3), (-1, 1, 3))
    b.shape("trianglemesh", P=P, indices=I)
    flat = b.world_end()
    row = flat.grid_table()[0]
    inside = rng.uniform(0.0, 1.0, (200, 3))
    # voxel centres and voxel boundaries (where floor() switches cells), and points outside the box where the field fades to 0
    centres = (np.stack(np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij"), -1).reshape(-1, 3) + 0.5) / np.array([nx, ny, nz])
    bounds = np.stack(np.meshgrid(np.arange(nx + 1) / nx, np.arange(ny + 1) / ny, np.arange(nz + 1) / nz, indexing="ij"), -1).reshape(-1, 3)
    outside = np.concatenate([rng.uniform(-0.5, 0.0, (30, 3)), rng.uniform(1.0, 1.5, (30, 3)), [[-0.2, 0.5, 0.5], [0.5, 1.2, 0.5], [0.5, 0.5, 5.0]]])
    pts = np.concatenate([inside, centres, bounds, outside]).astype(f32)
    got = G.grid_density(row, pts)
    want = _np_density(d, nx, ny, nz, pts)
    assert np.allclose(got, want, rtol=1e-5, atol=1e-5)
    assert np.allclose(G.grid_density(row, centres.astype(f32)), d.reshape(nz, ny, nx).transpose(2, 1, 0).reshape(-1), rtol=1e-6)
    assert np.all(G.grid_density(row, np.array([[-0.2, 0.5, 0.5], [0.5, 0.5, 5.0]], f32)) == 0.0)


def _emitter_behind_grid(pkg, density, nx, ny, nz, sigma_a, dist=2.0, spp=1024, res=8, L=(2.0, 3.0, 4.0)):
    """Camera at the origin inside an absorbing grid medium spanning x, y in [-1, 1] and z in [0, dist], looking down +z at an
    emissive quad at z = dist."""
    H = pkg.host
    b = _grid_scene(pkg, density, nx, ny, nz, (-1.0, -1.0, 0.0), (1.0, 1.0, dist), sigma_a, (0.0,) * 3)
    b.area_light_source("diffuse", L=L, twosided=True)
    b.material("matte", Kd=0.0)
    P, I = pkg.scenes.quad((-50, -50, dist), (50, -50, dist), (50, 50, dist), (-50, 50, dist))
    b.shape("trianglemesh", P=P, indices=I)
    cam_medium = b.camera_medium()
    flat = b.world_end()
    film = H.Film(res, res, "box")
    cam = H.PerspectiveCamera(film, H.Transform.look_at((0, 0, 0), (0, 0, 1), (0, 1, 0)).inverse(), fov=2.0)
    return flat, H.VolPathIntegrator(cam, film, H.Sampler("sobol", spp), maxdepth=5, lightsamplestrategy="uniform", camera_medium=cam_medium)


def _optical_depth(density, nx, ny, nz, n=4001):
    # along the axis of the narrow camera: medium-space x = y = 0.5, z from 0 to 1 (the box spans z in [0, dist]: ds = dist dz)
    z = np.linspace(0.0, 1.0, n)
    pts = np.stack([np.full(n, 0.5), np.full(n, 0.5), z], -1)
    return np.trapezoid(_np_density(density, nx, ny, nz, pts), z)


@pytest.mark.parametrize("sigma_a,chromatic", [((0.6, 0.6, 0.6), False), ((0.6, 1.5, 0.1), True)])
def test_beer_lambert_through_an_absorbing_grid(pkg, oracle, sigma_a, chromatic):
    # sigma_s = 0: a sampled interaction has weight 0, so the emitter is seen with probability Tr = exp(-sigma_t * integral density ds).
    # A grid medium's sigma_t is the FIRST channel of sigma_a + sigma_s (the constructor's rule): the chromatic case attenuates every
    # channel by channel 0's coefficient.
    nx, ny, nz, dist = 3, 3, 6, 2.0
    z = (np.arange(nz) + 0.5) / nz
    d = np.repeat((0.4 + 1.2 * np.sin(np.pi * z) ** 2)[:, None], nx * ny, axis=1).reshape(-1).astype(f32)  # varies along the ray only
    if chromatic:
        with pytest.warns(UserWarning, match="spectrally uniform"):
            flat, integ = _emitter_behind_grid(pkg, d, nx, ny, nz, sigma_a, dist)
    else:
        flat, integ = _emitter_behind_grid(pkg, d, nx, ny, nz, sigma_a, dist)
    img, _ = G.render_image(flat, integ)
    tr = math.exp(-sigma_a[0] * dist * _optical_depth(d, nx, ny, nz))
    want = np.array([2.0, 3.0, 4.0]) * tr
    got = img.reshape(-1, 3).mean(0)
    # 8 x 8 x 1024 Bernoulli(Tr ~ 0.3) samples: sigma ~ 0.6 %
    assert np.allclose(got, want, rtol=0.03), (got, want, tr)


def _grid_furnace(pkg, density, nx, ny, nz, sigma_s, g, spp=512, maxdepth=90, res=6):
    H = pkg.host
    b = _grid_scene(pkg, density, nx, ny, nz, (-1.0, -1.0, -1.0), (1.0, 1.0, 1.0), (0.0,) * 3, (sigma_s,) * 3, g=g)
    b.area_light_source("diffuse", L=(1.0, 1.0, 1.0), twosided=True)
    b.material("matte", Kd=0.0)
    P, I = pkg.scenes.box_mesh((-1, -1, -1), (1, 1, 1))
    b.shape("trianglemesh", P=P, indices=I)
    cam_medium = b.camera_medium()
    flat = b.world_end()
    film = H.Film(res, res, "box")
    cam = H.PerspectiveCamera(film, H.Transform.look_at((0.1, -0.2, 0.05), (0.7, 0.3, 1.0), (0, 1, 0)).inverse(), fov=70.0)
    return flat, H.VolPathIntegrator(cam, film, H.Sampler("halton", spp), maxdepth=maxdepth, rrthreshold=0.0, lightsamplestrategy="uniform",
                                     camera_medium=cam_medium)


@pytest.mark.parametrize("g", [0.0, 0.6])
def test_white_furnace_with_a_scattering_grid(pkg, oracle, g):
    # a closed emitting cube (L = 1, black walls) filled with a non-absorbing grid medium: radiance 1 whatever the field, since delta
    # tracking, ratio tracking with roulette, phase sampling and MIS all have to agree for it
    nx, ny, nz = 5, 4, 6
    d = pkg.scenes.smoke_density(nx, ny, nz, seed=11) * f32(1.5)
    flat, integ = _grid_furnace(pkg, d, nx, ny, nz, 2.0, g)
    img, _ = G.render_image(flat, integ)
    got = img.reshape(-1, 3).mean(0)
    assert np.allclose(got, 1.0, atol=0.06), got


def test_flattening_of_a_parsed_heterogeneous_medium(pkg):
    H = pkg.host
    d = np.arange(2 * 3 * 4, dtype=f32) * f32(0.25)
    text = ('WorldBegin\nMakeNamedMedium "haze" "string type" "homogeneous" "rgb sigma_s" [0.1 0.1 0.1]\n'
            'AttributeBegin\nTranslate 1 2 3\nRotate 30 0 0 1\nScale 2 1 0.5\n'
            f'MakeNamedMedium "smoke" "string type" "heterogeneous" "integer nx" 2 "integer ny" 3 "integer nz" 4 "point p0" [-1 0 0.5] '
            f'"point p1" [1 2 1.5] "rgb sigma_a" [1 1 1] "rgb sigma_s" [2 2 2] "float scale" 0.5 "float density" [{" ".join(str(v) for v in d)}]\n'
            'AttributeEnd\nMediumInterface "smoke" "haze"\nShape "sphere"\nWorldEnd')
    flat = pkg.pbrt_parse_string(text).jobs[0].flat
    assert list(flat.media["grid"]) == [0, 1] and len(flat.grids) == 1
    assert np.allclose(flat.media[1]["sigma_a"], 0.5) and np.allclose(flat.media[1]["sigma_s"], 1.0)
    g = flat.grids[0]
    assert (g.nx, g.ny, g.nz) == (2, 3, 4) and np.array_equal(g.density, d)  # x fastest, as written
    want = (H.Transform.translate((1, 2, 3)) * H.Transform.rotate(30, (0, 0, 1)) * H.Transform.scale(2, 1, 0.5)
            * H.Transform.translate((-1, 0, 0.5)) * H.Transform.scale(2, 2, 1))
    assert np.array_equal(g.medium_to_world, want.m) and np.array_equal(g.world_to_medium, want.m_inv)
    row = flat.grid_table()[0]
    assert np.array_equal(row["medium_to_world"], want.m.reshape(-1)) and (row["nx"], row["ny"], row["nz"]) == (2, 3, 4)
    assert np.array_equal(np.ctypeslib.as_array(C.cast(int(row["density"]), C.POINTER(C.c_float)), (24,)), d)
    assert np.array_equal(flat.prim_media[0].tolist(), (1, 0))


def test_write_pbrt_round_trip(pkg, oracle, tmp_path):
    setup = pkg.scenes.smoke_box_scene(xres=16, yres=16, spp=2, camera_in_smoke=True)
    integ = setup.make_integrator()
    path = tmp_path / "smoke.pbrt"
    importlib.import_module("pbrt-rust_b200.scenefile").write_pbrt(path, setup.flat, integ)
    job = pkg.pbrt_parse(path).jobs[0]
    assert job.integrator.camera_medium == integ.camera_medium
    assert np.array_equal(job.flat.media, setup.flat.media) and np.array_equal(job.flat.prim_media, setup.flat.prim_media)
    assert len(job.flat.grids) == 1
    for a, b in zip(job.flat.grids, setup.flat.grids):
        assert np.array_equal(a.density, b.density) and np.array_equal(a.medium_to_world, b.medium_to_world)
        assert np.array_equal(a.world_to_medium, b.world_to_medium) and (a.nx, a.ny, a.nz) == (b.nx, b.ny, b.nz)
    a, _ = G.render(setup.flat, integ)
    b, _ = G.render(job.flat, job.integrator)
    assert np.array_equal(a, b)


def test_heterogeneous_refusals(pkg):
    # deliberate deviation from the reference (which logs an error and creates no medium): missing or miscounted density raises
    for text in ('WorldBegin\nMakeNamedMedium "m" "string type" "heterogeneous"\nWorldEnd',
                 'WorldBegin\nMakeNamedMedium "m" "string type" "heterogeneous" "integer nx" 2 "float density" [1 2 3]\nWorldEnd',
                 'WorldBegin\nMakeNamedMedium "m" "string type" "heterogeneous" "string preset" "Skin1" "float density" [1]\nWorldEnd'):
        with pytest.raises(pkg.B200Error):
            pkg.pbrt_parse_string(text)


def _create_with_grids(pkg, flat, grids):
    lib = pkg.load_library()
    d = flat.desc()
    h = C.c_void_p()
    rc = lib.pbrt_b200_scene_create_with_grids(C.byref(d), None if grids is None else grids.ctypes.data_as(C.c_void_p),
                                               0 if grids is None else len(grids), 0, C.byref(h))
    if h.value:
        lib.pbrt_b200_scene_destroy(h)
    return rc, lib.pbrt_b200_last_error().decode()


def test_scene_create_rejects_malformed_grid_tables(pkg):
    # each malformed table is refused with PBRT_B200_ERR_INVALID (1) before anything reaches a device -- also on a host without one
    setup = pkg.scenes.smoke_box_scene(xres=8, yres=8, spp=1)
    flat = setup.flat
    good = flat.grid_table()
    keep = [g.density for g in flat.grids]  # the rows point into these

    def bad(**kw):
        t = good.copy()
        for k, v in kw.items():
            t[0][k] = v
        return t

    nan = np.array(keep[0], f32)
    nan[5] = np.nan
    neg = np.array(keep[0], f32)
    neg[7] = -1.0
    inf_m = good.copy()
    inf_m[0]["world_to_medium"][3] = np.inf
    cases = {"no grid table": None, "null density": bad(density=0), "zero count": bad(nz=0), "overflowing count": bad(nx=1 << 31, ny=1 << 31, nz=4),
             "NaN density": bad(density=nan.ctypes.data), "negative density": bad(density=neg.ctypes.data), "non-finite matrix": inf_m}
    for what, grids in cases.items():
        rc, msg = _create_with_grids(pkg, flat, grids)
        assert rc == 1, (what, rc, msg)
    media = flat.media.copy()
    flat.media = media
    media[1]["grid"] = 2  # only one grid supplied
    rc, msg = _create_with_grids(pkg, flat, good)
    assert rc == 1 and "grid index" in msg, msg
    del keep, nan, neg


def test_density_grid_layout_matches_what_a_c_compiler_sees(pkg, tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    dt = pkg.host.DENSITY_GRID_DTYPE
    lines = ["#include <stdio.h>", "#include <stddef.h>", f'#include "{HEADER}"', "int main(void) {",
             'printf("size %zu\\n", sizeof(pbrt_b200_density_grid));']
    lines += [f'printf("{f} %zu\\n", offsetof(pbrt_b200_density_grid, {f}));' for f in dt.names]
    lines.append("return 0; }")
    (tmp_path / "grid.c").write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(tmp_path / "grid"), str(tmp_path / "grid.c")], check=True)
    out = dict(l.split() for l in subprocess.run([str(tmp_path / "grid")], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(out["size"]) == dt.itemsize == 152
    for f in dt.names:
        assert int(out[f]) == dt.fields[f][1], f


def test_tracking_hang_guard_ends_the_path(pkg, oracle):
    # one voxel a billion times denser than the rest: delta tracking takes steps of ~1e-9 and gives up after ORC_VOL_TRACK_CAP of them,
    # which ends the path before it reaches the emitter; without the guard the emitter would show through (Tr ~ exp(-1.2) here)
    nx, ny, nz = 3, 3, 4
    d = np.ones(nx * ny * nz, f32)
    d[-1] = 1e9
    flat, integ = _emitter_behind_grid(pkg, d, nx, ny, nz, (0.6,) * 3, spp=1, res=4)
    img, stats = G.render_image(flat, integ)
    assert stats["camera_rays"] == 16 and np.all(img == 0.0)
