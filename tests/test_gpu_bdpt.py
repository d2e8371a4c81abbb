"""BDPTIntegrator on the GPU (k_bdpt, csrc/bdpt.cu) against the CPU oracle (oracle/oracle_bdpt.hpp) on the same sample streams.

The gate of the volpath tests: image relMSE <= 1e-3 with the splat film resolved (splat_scale = 1 / spp), equal camera-ray counts,
closest-hit counts within 0.3 %.  Every visibility test of BDPT is a closest-hit walk (VisibilityTester::tr), so there are no any-hit rays.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
REL_MSE_TOL = 1e-3


@pytest.fixture(scope="module")
def obdpt():
    from oracle import oracle_bdpt
    oracle_bdpt.lib()
    return oracle_bdpt


def bdpt_of(pkg, integ, maxdepth=None, strategy="power", pixelbounds=None):
    return pkg.host.BDPTIntegrator(integ.camera, integ.film, integ.sampler, maxdepth=integ.max_depth if maxdepth is None else maxdepth,
                                   lightsamplestrategy=strategy, pixelbounds=pixelbounds)


def _compare(pkg, oracle, obdpt, flat, integ, **kw):
    sc = pkg.Scene(flat)
    rgbw, splat, st = sc.render_splat(integ, **kw)
    got = sc.film_resolve_splat(rgbw, splat, 1.0 / integ.sampler.spp, integ.film.scale)
    sc.close()
    wr, ws, ost = obdpt.render(flat, integ, **kw)
    want = obdpt.resolve(wr, ws, integ.sampler.spp, integ.film.scale)
    assert np.isfinite(got).all()
    err = oracle.rel_mse(got, want)
    assert err <= REL_MSE_TOL, f"relMSE {err:.3e}"
    assert st.camera_rays == ost["camera_rays"]
    assert abs(int(st.intersection_tests) - ost["intersection_tests"]) <= 0.003 * ost["intersection_tests"] + 8
    assert st.shadow_tests == 0
    return got, want, (rgbw, splat)


@pytest.mark.parametrize("sampler", ["sobol", "halton"])
def test_cornell_box_matches_the_oracle(pkg, oracle, obdpt, gpu_lib, sampler):
    setup = pkg.scenes.cornell_scene(xres=64, yres=64, spp=8, maxdepth=5, sampler=sampler)
    got, _, (_, splat) = _compare(pkg, oracle, obdpt, setup.flat, bdpt_of(pkg, setup.make_integrator()))
    assert got.mean() > 0.05 and np.abs(splat).sum() > 0  # light tracing reached the camera


def test_point_distant_and_infinite_lights_and_glass(pkg, oracle, obdpt, gpu_lib):
    # small_mixed_scene: quad area light, point, distant and constant infinite lights over matte / plastic / glass / mirror / metal
    setup = pkg.scenes.small_mixed_scene()
    for strategy in ("power", "uniform", "spatial"):
        _compare(pkg, oracle, obdpt, setup.flat, bdpt_of(pkg, setup.make_integrator(spp_=4, res=(64, 48)), strategy=strategy))


def test_mirror_and_glass_spheres_under_a_distant_light(pkg, oracle, obdpt, gpu_lib):
    setup = pkg.scenes.spheres_scene(xres=64, yres=64, spp=8)
    _compare(pkg, oracle, obdpt, setup.flat, bdpt_of(pkg, setup.make_integrator()))


def test_instancing(pkg, oracle, obdpt, gpu_lib):
    setup = pkg.scenes.instanced_scene(n_side=3)
    _compare(pkg, oracle, obdpt, setup.flat, bdpt_of(pkg, setup.make_integrator(spp_=4, res=(64, 48))))


@pytest.mark.parametrize("light", ["spot", "point", "sphere", "sphere_one_sided"])
def test_each_light_kind(pkg, oracle, obdpt, gpu_lib, light):
    setup = pkg.scenes.one_light_scene(light)
    got, _, (_, splat) = _compare(pkg, oracle, obdpt, setup.flat, bdpt_of(pkg, setup.make_integrator()))
    assert got.mean() > 0 and np.abs(splat).sum() > 0


def test_textured_materials_bump_maps_and_thin_lens(pkg, oracle, obdpt, gpu_lib):
    # every texture kind, uber and substrate, bump maps, a textured instance; the camera subpath's first vertex filters with the camera
    # ray's differentials.  Then the same scene through a thin lens (lensradius > 0: the lens branches of we / pdf_we / sample_wi).
    setup = pkg.scenes.textured_scene(xres=64, yres=48, spp=4, maxdepth=4)
    _compare(pkg, oracle, obdpt, setup.flat, bdpt_of(pkg, setup.make_integrator()))
    _compare(pkg, oracle, obdpt, setup.flat, bdpt_of(pkg, setup.make_integrator(lensradius=0.15)))


def test_crop_window_drops_splats_outside_it(pkg, oracle, obdpt, gpu_lib):
    setup = pkg.scenes.caustic_scene(xres=64, yres=64, spp=8, maxdepth=5)
    crop = (0.2, 0.7, 0.3, 0.9)
    integ = bdpt_of(pkg, setup.make_integrator(crop=crop))
    _, _, (_, splat) = _compare(pkg, oracle, obdpt, setup.flat, integ)
    w, h = integ.film.width, integ.film.height
    assert (w, h) == (32, 38) and splat.shape == (w * h, 3) and np.abs(splat).sum() > 0
    # the device and the oracle both drop splats that land outside the cropped bounds (Film::add_splat's InsideExclusive test)


def test_pixel_bounds(pkg, oracle, obdpt, gpu_lib):
    setup = pkg.scenes.cornell_scene(xres=64, yres=64, spp=4, maxdepth=4)
    _compare(pkg, oracle, obdpt, setup.flat, bdpt_of(pkg, setup.make_integrator(), pixelbounds=(8, 50, 4, 40)))


def test_tile_and_sample_windows_sum_to_the_full_render(pkg, oracle, obdpt, gpu_lib):
    setup = pkg.scenes.cornell_scene(xres=48, yres=48, spp=8, maxdepth=4)
    integ = bdpt_of(pkg, setup.make_integrator())
    sc = pkg.Scene(setup.flat)
    full_rgbw, full_splat, _ = sc.render_splat(integ)
    n = integ.n_tiles()
    rgbw = np.zeros_like(full_rgbw)
    splat = np.zeros_like(full_splat)
    for tr in ((0, n // 2), (n // 2, n)):
        for sr in ((0, 3), (3, 8)):
            sc.render_splat(integ, rgbw=rgbw, splat=splat, tile_range=tr, sample_range=sr)
    sc.close()
    np.testing.assert_allclose(rgbw, full_rgbw, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(splat, full_splat, rtol=1e-4, atol=1e-4)


def test_scene_file_end_to_end(pkg, oracle, obdpt, gpu_lib):
    text = """LookAt 0 0 5  0 0 0  0 1 0
Camera "perspective" "float fov" 40
Sampler "sobol" "integer pixelsamples" 8
Film "image" "integer xresolution" 48 "integer yresolution" 48
Integrator "bdpt" "integer maxdepth" 4
WorldBegin
AttributeBegin
  AreaLightSource "diffuse" "rgb L" [8 8 8]
  Shape "trianglemesh" "integer indices" [0 1 2 0 2 3] "point P" [-0.5 1.9 -0.5  0.5 1.9 -0.5  0.5 1.9 0.5  -0.5 1.9 0.5]
AttributeEnd
LightSource "spot" "point from" [0 1.5 3] "point to" [0 0 0] "float coneangle" 25 "rgb I" [6 6 6]
Material "matte" "rgb Kd" [0.6 0.6 0.6]
Shape "trianglemesh" "integer indices" [0 1 2 0 2 3] "point P" [-2 -1 -2  2 -1 -2  2 -1 2  -2 -1 2]
Material "plastic" "rgb Kd" [0.3 0.2 0.6] "float roughness" 0.2
Shape "trianglemesh" "integer indices" [0 1 2] "point P" [-1 -1 -1  1 -1 -1  0 1 -1]
WorldEnd
"""
    job = pkg.pbrt_parse_string(text).jobs[0]
    assert isinstance(job.integrator, pkg.host.BDPTIntegrator)
    img, st = job.render()
    _compare(pkg, oracle, obdpt, job.flat, job.integrator)
    assert img.shape == (48, 48, 3) and img.mean() > 0


def test_maxdepth_bound_and_refusals(pkg, gpu_lib):
    H = pkg.host
    setup = pkg.scenes.cornell_scene(xres=16, yres=16, spp=1, maxdepth=2)
    base = setup.make_integrator()
    sc = pkg.Scene(setup.flat)
    integ = bdpt_of(pkg, base, maxdepth=H.BDPT_MAX_DEPTH)
    sc.render_splat(integ)
    integ.max_depth = H.BDPT_MAX_DEPTH + 1  # past the bound: refused by the library before any allocation
    with pytest.raises(H.B200Error, match="maxdepth"):
        sc.render_splat(integ)
    with pytest.raises(H.B200Error, match="render_splat"):  # pbrt_b200_render with the BDPT kind names the splat entry point
        sc.render(bdpt_of(pkg, base))
    sc.close()


def test_caustic_scene_converges_to_the_path_integrator(pkg, oracle, gpu_lib):
    """Statistical: on the caustic scene BDPT at 256 spp and the path integrator at 1024 spp estimate the same image.  The tolerance is
    on the image mean, whose relative standard error at these sample counts is well under 1 % for both estimators."""
    setup = pkg.scenes.caustic_scene(xres=64, yres=64)
    path = setup.make_integrator(spp_=1024, maxdepth_=6)
    path.rr_threshold = 0.0
    sc = pkg.Scene(setup.flat)
    ip, _ = path.render(sc)
    ib, _ = bdpt_of(pkg, setup.make_integrator(spp_=256, maxdepth_=6)).render(sc)
    sc.close()
    assert abs(ib.mean() - ip.mean()) <= 0.03 * ip.mean()
