"""Heterogeneous (grid density) media on the GPU (k_vol_mega_grid, csrc/mega.cu) against the CPU oracle (oracle/oracle_grid.hpp).

The gate of tests/test_gpu_volpath.py: image relMSE <= 1e-3, equal camera-ray counts, ray counts within 0.3 %.  Grid media add two
things to check: the transmittance loops draw from the sampler, so the device must draw in the reference's order (the sample-order
check below), and delta / ratio tracking must follow the reference's arithmetic (the closed forms and the Sobol' index-0 sample).
"""
import math

import numpy as np
import pytest
from oracle import oracle_grid as G
from test_grid_media_oracle import _emitter_behind_grid, _grid_furnace, _optical_depth

pytestmark = pytest.mark.gpu
REL_MSE_TOL = 1e-3
# Share of pixels of the camera-in-smoke box (sobol, 32 x 32, 4 spp) whose GPU radiance equals the oracle's to 1e-4 relative.
# Measured on a B200: 0.994 (the rest are paths with a logf / expf rounding difference at a tracking decision).  A build that draws the
# next direction and roulette before the shadow / MIS walks, as k_vol_mega does for homogeneous media, shifts every later dimension of
# every path that meets the grid: measured 0.000.
SAMPLE_ORDER_MIN_SHARE = 0.97


def _render(pkg, setup, integ, **kw):
    sc = pkg.Scene(setup.flat if hasattr(setup, "flat") else setup)
    try:
        return sc.render(integ, **kw)
    finally:
        sc.close()


def _compare(pkg, oracle, setup, integ=None, **render_kw):
    integ = integ or setup.make_integrator()
    got, st = _render(pkg, setup, integ, **render_kw)
    want, ost = G.render(setup.flat, integ, **render_kw)
    assert np.isfinite(got).all()
    assert np.array_equal(got[:, 3] > 0, want[:, 3] > 0)
    a, b = oracle.film_resolve(got, integ.film.scale), oracle.film_resolve(want, integ.film.scale)
    err = oracle.rel_mse(a, b)
    assert err <= REL_MSE_TOL, f"relMSE {err:.3e}"
    assert st.camera_rays == ost["camera_rays"]
    assert abs(int(st.intersection_tests) - ost["intersection_tests"]) <= 0.003 * ost["intersection_tests"] + 8
    return err, a, b


@pytest.mark.parametrize("sampler", ["sobol", "halton"])
@pytest.mark.parametrize("camera_in_smoke", [False, True])
def test_smoke_box_matches_the_oracle(pkg, oracle, gpu_lib, sampler, camera_in_smoke):
    setup = pkg.scenes.smoke_box_scene(xres=64, yres=64, spp=8, sampler=sampler, camera_in_smoke=camera_in_smoke)
    _, a, _ = _compare(pkg, oracle, setup)
    assert a.mean() > 0.05


def sample_order_agreement(pkg, oracle):
    setup = pkg.scenes.smoke_box_scene(xres=32, yres=32, spp=4, camera_in_smoke=True)
    integ = setup.make_integrator()
    got, _ = _render(pkg, setup, integ)
    want, _ = G.render(setup.flat, integ)
    a, b = oracle.film_resolve(got, 1.0).reshape(-1, 3), oracle.film_resolve(want, 1.0).reshape(-1, 3)
    ok = np.all(np.abs(a - b) <= 1e-4 * np.maximum(np.abs(b), 1e-3), axis=1)
    return float(ok.mean())


def test_sample_order_of_the_transmittance_loops(pkg, oracle, gpu_lib):
    # most pixels agree to rounding: their paths drew the same samples in the same order on both sides
    share = sample_order_agreement(pkg, oracle)
    assert share >= SAMPLE_ORDER_MIN_SHARE, share


def test_instanced_textured_spatial_deep_paths(pkg, oracle, gpu_lib):
    setup = pkg.scenes.smoke_box_scene(xres=48, yres=48, spp=8, maxdepth=40, instanced=True, textured=True)
    _compare(pkg, oracle, setup, integ=setup.make_integrator(strategy="spatial", rrthreshold=1.0))


def test_sobol_index_zero_through_a_zero_border(pkg, oracle, gpu_lib):
    # Sobol' sample 0 of the pixel at the sample-bounds origin has every dimension 0: its camera ray starts on the face of a grid whose
    # border voxels are empty, so every tracking step is 0 long and every density test fails until the sampler runs out of dimensions
    # (then every draw is 0.5 and the loop advances).  Both sides must walk that the same way.
    nx, ny, nz = 3, 3, 5
    d = np.ones((nz, ny, nx), np.float32)
    d[0] = 0.0
    flat, integ = _emitter_behind_grid(pkg, d.reshape(-1), nx, ny, nz, (0.8,) * 3, spp=4, res=4)
    kw = dict(sample_range=(0, 1))
    got, st = _render(pkg, flat, integ, **kw)
    want, ost = G.render(flat, integ, **kw)
    assert st.camera_rays == ost["camera_rays"] == 16
    assert np.allclose(got, want, rtol=1e-3, atol=1e-6), (got[:2], want[:2])


def test_grid_tile_and_sample_windows_add_up(pkg, oracle, gpu_lib):
    setup = pkg.scenes.smoke_box_scene(xres=48, yres=40, spp=8, camera_in_smoke=True)
    integ = setup.make_integrator()
    sc = pkg.Scene(setup.flat)
    full, st = sc.render(integ)
    acc = np.zeros_like(full)
    n = integ.n_tiles()
    rays = 0
    for tr in ((0, n // 2), (n // 2, n)):
        for sr in ((0, 3), (3, 8)):
            _, s = sc.render(integ, tile_range=tr, sample_range=sr, rgbw=acc)
            rays += s.camera_rays
    sc.close()
    assert rays == st.camera_rays
    assert np.allclose(acc, full, rtol=2e-5, atol=1e-6)
    _compare(pkg, oracle, setup, integ=integ, tile_range=(n // 2, n), sample_range=(3, 8))


@pytest.mark.parametrize("camera_in_smoke", [False, True])
@pytest.mark.parametrize("instanced", [False, True])
def test_all_zero_grid_renders_as_vacuum(pkg, oracle, gpu_lib, camera_in_smoke, instanced):
    # k_vol_mega_grid with an empty grid against k_vol_mega on the scene without the medium: the same sample stream and the same image.
    # With the boundary instanced, both scenes run the full-featured family (k_vol_mega<true>), so the five-phase trip must give exactly
    # the whole-vertex trip's ray counts; without, the vacuum scene runs k_vol_mega<false>, which differs from the full family by a few
    # paths (as between the instanced and plain fog box of test_gpu_volpath.py), so its counts get the oracle gate.
    zero = pkg.scenes.smoke_box_scene(xres=48, yres=48, spp=8, camera_in_smoke=camera_in_smoke, instanced=instanced,
                                      density=np.zeros(14 * 11 * 9, np.float32))
    none = pkg.scenes.smoke_box_scene(xres=48, yres=48, spp=8, camera_in_smoke=camera_in_smoke, instanced=instanced, smoke=False)
    a, sa = _render(pkg, zero, zero.make_integrator())
    b, sb = _render(pkg, none, none.make_integrator())
    assert sa.camera_rays == sb.camera_rays
    if instanced:
        assert sa.intersection_tests == sb.intersection_tests
    else:
        assert abs(int(sa.intersection_tests) - int(sb.intersection_tests)) <= 0.003 * int(sb.intersection_tests) + 8
    assert oracle.rel_mse(oracle.film_resolve(a, 1.0), oracle.film_resolve(b, 1.0)) <= 1e-5


def test_beer_lambert_and_furnace_closed_forms(pkg, oracle, gpu_lib):
    nx, ny, nz, dist = 3, 3, 6, 2.0
    z = (np.arange(nz) + 0.5) / nz
    d = np.repeat((0.4 + 1.2 * np.sin(np.pi * z) ** 2)[:, None], nx * ny, axis=1).reshape(-1).astype(np.float32)
    flat, integ = _emitter_behind_grid(pkg, d, nx, ny, nz, (0.6,) * 3, dist)
    got, _ = _render(pkg, flat, integ)
    img = oracle.film_resolve(got, 1.0).reshape(-1, 3).mean(0)
    want = np.array([2.0, 3.0, 4.0]) * math.exp(-0.6 * dist * _optical_depth(d, nx, ny, nz))
    assert np.allclose(img, want, rtol=0.03), (img, want)
    d = pkg.scenes.smoke_density(5, 4, 6, seed=11) * np.float32(1.5)
    flat, integ = _grid_furnace(pkg, d, 5, 4, 6, 2.0, 0.6)
    got, _ = _render(pkg, flat, integ)
    assert np.allclose(oracle.film_resolve(got, 1.0).reshape(-1, 3).mean(0), 1.0, atol=0.06)
