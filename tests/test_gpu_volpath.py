"""VolPathIntegrator on the GPU (k_vol_mega, csrc/mega.cu) against the CPU oracle (oracle/oracle_volpath.hpp).

Same gate as the surface path integrator: image relMSE <= 1e-3 (north_star), equal camera-ray counts, ray counts within
0.3 % (a path whose medium / Russian-roulette decision sits on a rounding boundary -- expf / logf differ by an ulp
between the two sides -- continues differently).  The scene puts every volume rule on the light paths: camera inside a
medium, medium-transition and non-transition surfaces, a material-less boundary (crossed by path, shadow and MIS rays),
an absorbing medium inside glass, delta and area lights.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
REL_MSE_TOL = 1e-3


def _compare(pkg, oracle, setup, integ=None, **render_kw):
    integ = integ or setup.make_integrator()
    sc = pkg.Scene(setup.flat)
    got, st = sc.render(integ, **render_kw)
    sc.close()
    want, ost = oracle.render(setup.flat, integ, **render_kw)
    assert np.isfinite(got).all()
    assert np.array_equal(got[:, 3] > 0, want[:, 3] > 0)
    a, b = oracle.film_resolve(got, integ.film.scale), oracle.film_resolve(want, integ.film.scale)
    err = oracle.rel_mse(a, b)
    assert err <= REL_MSE_TOL, f"relMSE {err:.3e}"
    assert st.camera_rays == ost["camera_rays"]
    assert abs(int(st.intersection_tests) - ost["intersection_tests"]) <= 0.003 * ost["intersection_tests"] + 8
    assert st.shadow_tests == 0 and ost["shadow_tests"] == 0  # volpath's visibility is Scene::intersect (light.rs:133), never intersect_p
    return err, a, b


@pytest.mark.parametrize("sampler", ["sobol", "halton"])
def test_fog_box_matches_the_oracle(pkg, oracle, gpu_lib, sampler):
    setup = pkg.scenes.fog_box_scene(xres=96, yres=96, spp=16, sampler=sampler)
    _, a, _ = _compare(pkg, oracle, setup)
    assert a.mean() > 0.1


def test_fog_box_camera_outside_the_medium(pkg, oracle, gpu_lib):
    _compare(pkg, oracle, pkg.scenes.fog_box_scene(xres=96, yres=96, spp=8, camera_in_fog=False))


def test_fog_box_with_the_boundary_in_an_object_instance(pkg, oracle, gpu_lib):
    # the material-less cube is an ObjectInstance: its GeometricPrimitives keep their MediumInterface (api.rs:1527), the
    # TransformedPrimitive has none -- and the image is the one of the un-instanced scene
    setup = pkg.scenes.fog_box_scene(xres=64, yres=64, spp=8, instanced=True)
    _, a, _ = _compare(pkg, oracle, setup)
    plain = pkg.scenes.fog_box_scene(xres=64, yres=64, spp=8)
    sc = pkg.Scene(plain.flat)
    got, _ = sc.render(plain.make_integrator())
    sc.close()
    assert oracle.rel_mse(a, oracle.film_resolve(got, 1.0)) <= 1e-6


def test_fog_box_spatial_strategy_deep_paths_and_roulette(pkg, oracle, gpu_lib):
    setup = pkg.scenes.fog_box_scene(xres=64, yres=64, spp=8, maxdepth=40)
    _compare(pkg, oracle, setup, integ=setup.make_integrator(strategy="spatial", rrthreshold=1.0))
    _compare(pkg, oracle, setup, integ=setup.make_integrator(strategy="power", rrthreshold=0.0, filt="gaussian"))


def test_volpath_tile_and_sample_windows_add_up(pkg, oracle, gpu_lib):
    setup = pkg.scenes.fog_box_scene(xres=64, yres=48, spp=8)
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
    assert np.allclose(acc, full, rtol=2e-5, atol=1e-6)  # same samples; only the order of the film's float additions differs
    want, _ = oracle.render(setup.flat, integ, tile_range=(n // 2, n), sample_range=(3, 8))
    sc = pkg.Scene(setup.flat)
    got, _ = sc.render(integ, tile_range=(n // 2, n), sample_range=(3, 8))
    sc.close()
    assert oracle.rel_mse(oracle.film_resolve(got, 1.0)[want[:, 3] > 0], oracle.film_resolve(want, 1.0)[want[:, 3] > 0]) <= REL_MSE_TOL


def test_volpath_without_media_matches_the_path_kernels(pkg, oracle, gpu_lib):
    # no media, no material-less surfaces: the megakernel and the wavefront path integrator render the same image
    setup = pkg.scenes.cornell_scene(xres=96, yres=96, spp=16)
    integ = setup.make_integrator()
    H = pkg.host
    vol = H.VolPathIntegrator(integ.camera, integ.film, integ.sampler, maxdepth=integ.max_depth, rrthreshold=integ.rr_threshold,
                              lightsamplestrategy=integ.light_sample_strategy)
    sc = pkg.Scene(setup.flat)
    a, _ = sc.render(integ)
    b, _ = sc.render(vol)
    sc.close()
    assert oracle.rel_mse(oracle.film_resolve(b, 1.0), oracle.film_resolve(a, 1.0)) <= 1e-5
    _compare(pkg, oracle, setup, integ=vol)


def test_beer_lambert_and_furnace_on_the_gpu(pkg, oracle, gpu_lib):
    import test_volpath_oracle as T
    flat, integ = T._emitter_behind_slab(pkg, (0.1, 0.5, 1.2), (0.0,) * 3, 1.5, spp=2048)
    sc = pkg.Scene(flat)
    img, _ = integ.render(sc)
    sc.close()
    assert np.allclose(img.reshape(-1, 3).mean(0), np.array([2.0, 3.0, 4.0]) * np.exp(-np.array([0.1, 0.5, 1.2]) * 1.5), rtol=0.03)
    flat, integ = T._furnace(pkg, (0.5, 1.0, 1.5), 0.7)
    sc = pkg.Scene(flat)
    img, _ = integ.render(sc)
    sc.close()
    assert np.allclose(img.reshape(-1, 3).mean(0), 1.0, atol=0.06)


def test_volpath_rejects_what_it_does_not_cover(pkg, gpu_lib):
    setup = pkg.scenes.fog_box_scene(xres=32, yres=32, spp=4, sampler="02sequence")
    sc = pkg.Scene(setup.flat)
    with pytest.raises(pkg.B200Error, match="sobol or halton"):
        sc.render(setup.make_integrator())
    integ = pkg.scenes.fog_box_scene(xres=32, yres=32, spp=4).make_integrator()
    integ.camera_medium = 7
    with pytest.raises(pkg.B200Error, match="camera_medium"):
        sc.render(integ)
    sc.close()
    bad = pkg.scenes.fog_box_scene(xres=32, yres=32, spp=4).flat
    bad.prim_media = bad.prim_media.copy()
    bad.prim_media["inside"][0] = 9
    with pytest.raises(pkg.B200Error, match="medium interface"):
        pkg.Scene(bad)
