"""The path integrator at the limits of its sampler and film bookkeeping, against the CPU oracle.

Sobol' sample values reach the shade kernels three ways (path.cuh, PathSampler<false>): rows of the per-pixel and
per-sample tables, the pre-pass k_sample_block (Halton, and Sobol' dimensions the tables do not hold), and, past the
1024 dimensions of the generator matrices, the constant 0.5 (the oracle reads 0.5 there too; the reference panics).  The
three give bit-identical values, so renders in every mode take the same paths.  PBRT_B200_NO_SOBOL_TABLES turns the
tables off and PBRT_B200_SOBOL_TABLE_DIMS=N keeps only N dimensions in them; both are read by every render call.

The deep-path cases use a closed box of flat matte walls (Kd 0.8) lit by a small quad light whose own material is black,
with rrthreshold 0: a path ends only on the light or at maxdepth, and a matte bounce draws exactly 7 dimensions
(path_li in oracle/oracle_render.hpp: light choice 1, light 2, scattering 2, BSDF 2; no roulette draw).  The block a path
reads at bounce b therefore starts at dimension 5 + 7b.  Flat walls keep the two sides in lock-step: the next direction
depends on the normal and the sample only, never on where the incoming ray came from.
"""
import numpy as np
import pytest

gpu = pytest.mark.gpu
REL_MSE_TOL = 1e-3
ERR_INVALID = 1  # PBRT_B200_ERR_INVALID
STATS = ("camera_rays", "intersection_tests", "shadow_tests", "zero_radiance_paths")
SOBOL_DIMS, HALTON_DIMS = 1024, 1000  # NUM_SOBOL_DIMENSIONS, PRIME_TABLE_SIZE


def _dims_at(bounce):
    """First dimension of the 8-wide block a deep-box path reads when it shades at `bounce`."""
    return 5 + 7 * bounce


def deep_box(pkg, medium=False):
    """-> (flat, make(maxdepth, sampler, res, spp)).  `medium`: the box is filled with a thin homogeneous medium the camera sits in,
    and holds a material-less cube of a denser one (its boundary lowers volpath's bounce count at every crossing)."""
    H, S = pkg.host, pkg.scenes
    b = H.SceneBuilder()
    if medium:
        b.make_named_medium("haze", sigma_a=(0.02, 0.02, 0.03), sigma_s=(0.3, 0.3, 0.35), g=0.2)
        b.make_named_medium("dense", sigma_a=(0.1, 0.1, 0.1), sigma_s=(2.0, 2.2, 2.4), g=-0.3)
        b.medium_interface("haze", "haze")  # not a transition: rays keep their medium at the walls
    b.material("matte", Kd=(0.8, 0.8, 0.8))
    walls = (((-1, -1, -1), (1, -1, -1), (1, 1, -1), (-1, 1, -1)), ((-1, -1, 1), (-1, 1, 1), (1, 1, 1), (1, -1, 1)),
             ((-1, -1, -1), (-1, 1, -1), (-1, 1, 1), (-1, -1, 1)), ((1, -1, -1), (1, -1, 1), (1, 1, 1), (1, 1, -1)),
             ((-1, -1, -1), (-1, -1, 1), (1, -1, 1), (1, -1, -1)), ((-1, 1, -1), (1, 1, -1), (1, 1, 1), (-1, 1, 1)))
    for w in walls:
        P, I = S.quad(*w)
        b.shape("trianglemesh", P=P, indices=I)
    b.attribute_begin()
    b.area_light_source("diffuse", L=(40, 36, 30))
    b.material("matte", Kd=0.0)
    P, I = S.quad((-.15, -.15, .999), (-.15, .15, .999), (.15, .15, .999), (.15, -.15, .999))  # facing down
    b.shape("trianglemesh", P=P, indices=I)
    b.attribute_end()
    if medium:
        b.attribute_begin()
        b.medium_interface("dense", "haze")
        b.material("none")
        P, I = S.box_mesh((0.2, 0.1, -0.9), (0.7, 0.6, -0.4))
        b.shape("trianglemesh", P=P, indices=I)
        b.attribute_end()
    cam_medium = b.camera_medium() if medium else -1
    flat = b.world_end()
    w2c = H.Transform.look_at((0.0, -0.9, -0.2), (0.0, 1.0, 0.1), (0, 0, 1))

    def make(maxdepth, sampler="sobol", res=(32, 32), spp=4):
        film = H.Film(res[0], res[1], "box")
        cam = H.PerspectiveCamera(film, w2c.inverse(), fov=70.0)
        if medium:
            return H.VolPathIntegrator(cam, film, H.Sampler(sampler, spp), maxdepth=maxdepth, rrthreshold=0.0, lightsamplestrategy="power",
                                       camera_medium=cam_medium)
        return H.PathIntegrator(cam, film, H.Sampler(sampler, spp), maxdepth=maxdepth, rrthreshold=0.0, lightsamplestrategy="power")

    return flat, make


def _set_mode(monkeypatch, mode):
    """"full": tables as large as the budget allows; "none": no tables; an int N: the tables hold N dimensions."""
    monkeypatch.delenv("PBRT_B200_NO_SOBOL_TABLES", raising=False)
    monkeypatch.delenv("PBRT_B200_SOBOL_TABLE_DIMS", raising=False)
    if mode == "none":
        monkeypatch.setenv("PBRT_B200_NO_SOBOL_TABLES", "1")
    elif mode != "full":
        monkeypatch.setenv("PBRT_B200_SOBOL_TABLE_DIMS", str(int(mode)))


def _render(monkeypatch, sc, integ, mode="full", **kw):
    _set_mode(monkeypatch, mode)
    try:
        return sc.render(integ, **kw)
    finally:
        _set_mode(monkeypatch, "full")


def _stats(st):
    return {k: int(getattr(st, k)) for k in STATS}


def _check_oracle(oracle, integ, got, st, want, ost, ray_tol=0.002, image=True):
    """Ray budgets and image relMSE of one render against the oracle's render of the same samples."""
    assert np.isfinite(got).all()
    assert np.array_equal(got[:, 3] > 0, want[:, 3] > 0)
    assert st.camera_rays == ost["camera_rays"]
    assert abs(int(st.intersection_tests) - ost["intersection_tests"]) <= ray_tol * ost["intersection_tests"] + 8
    assert abs(int(st.shadow_tests) - ost["shadow_tests"]) <= ray_tol * ost["shadow_tests"] + 8
    if image:
        covered = want[:, 3] > 0
        a = oracle.film_resolve(got, integ.film.scale)[covered]
        b = oracle.film_resolve(want, integ.film.scale)[covered]
        err = oracle.rel_mse(a, b)
        assert err <= REL_MSE_TOL, f"relMSE {err:.3e}"


# ---------------------------------------------------------------------------------------------------------------------
# 1. the three Sobol' modes render the same image
# ---------------------------------------------------------------------------------------------------------------------
# 13, 21, 29, 45 = 5 + 8k: a table boundary on a block boundary of a path that draws 8 dimensions per bounce; 20 is off them
TABLE_CAPS = (13, 20, 21, 29, 45)
MODE_SCENES = {
    "cornell": (lambda S: S.cornell_scene(), dict(spp_=8, res=(48, 40))),  # gaussian filter: the sample bounds start at -2
    "mixed": (lambda S: S.small_mixed_scene(), dict(spp_=8, res=(64, 48))),
}
# At maxdepth 12 this small_mixed_scene image hangs on a few glass / metal paths that sit on a rounding boundary: moving the camera by
# 1e-6 changes the oracle's own image by relMSE 4.6e-2 (its ray counts by 9 of 61 511).  There the oracle check is the ray budget;
# the modes are still compared with each other exactly.
ORACLE_IMAGE_UNSTABLE = {("mixed", 12)}


@gpu
@pytest.mark.parametrize("maxdepth", [5, 12])
@pytest.mark.parametrize("scene", list(MODE_SCENES))
def test_sobol_table_modes_are_bit_identical(pkg, oracle, gpu_lib, monkeypatch, scene, maxdepth):
    make, kw = MODE_SCENES[scene]
    setup = make(pkg.scenes)
    integ = setup.make_integrator(maxdepth_=maxdepth, **kw)
    if scene == "cornell":
        assert integ.film.sample_bounds[:2] == (-2, -2)
    want, ost = oracle.render(setup.flat, integ)
    sc = pkg.Scene(setup.flat)
    try:
        image = (scene, maxdepth) not in ORACLE_IMAGE_UNSTABLE
        base, bst = _render(monkeypatch, sc, integ, "full")
        _check_oracle(oracle, integ, base, bst, want, ost, image=image)
        # capped and uncapped tables alternate on one scene: the cached pixel table is keyed by its row stride
        for mode in ("none",) + sum(((c, "full") for c in TABLE_CAPS), ()):
            got, st = _render(monkeypatch, sc, integ, mode)
            assert _stats(st) == _stats(bst), f"mode {mode}"
            assert np.allclose(got, base, rtol=2e-5, atol=2e-5), f"mode {mode}"
            _check_oracle(oracle, integ, got, st, want, ost, image=image)
    finally:
        sc.close()


@gpu
def test_sobol_table_modes_with_tile_and_sample_windows(pkg, oracle, gpu_lib, monkeypatch):
    """sample_range starting at 3: the per-sample table starts at sample 3 (vs_begin), and k_sample_block converts the slot's
    sample number to the Sobol' index of the pixel."""
    setup = pkg.scenes.cornell_scene()
    integ = setup.make_integrator(spp_=8, res=(64, 48), maxdepth_=12)
    n = integ.n_tiles()
    win = dict(tile_range=(n // 4, n - 1), sample_range=(3, 8))
    want, ost = oracle.render(setup.flat, integ, **win)
    sc = pkg.Scene(setup.flat)
    try:
        base, bst = _render(monkeypatch, sc, integ, "full", **win)
        _check_oracle(oracle, integ, base, bst, want, ost)
        for mode in ("none", 13, 20, 45):
            got, st = _render(monkeypatch, sc, integ, mode, **win)
            assert _stats(st) == _stats(bst), f"mode {mode}"
            assert np.allclose(got, base, rtol=2e-5, atol=2e-5), f"mode {mode}"
            _check_oracle(oracle, integ, got, st, want, ost)
    finally:
        sc.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2-4. deep paths across the sampler's dimension limits
# ---------------------------------------------------------------------------------------------------------------------
# full tables hold min(1024, 5 + 8 * maxdepth) dimensions: 1021 at 127, 1024 from 128 on.  The last bounce a path shades is
# maxdepth - 1; its block [5 + 7b, 5 + 7b + 8) fits in 1024 dimensions up to b = 144 and straddles dimension 1024 from b = 145
# (maxdepth 146) on.  At maxdepth 300 the deepest blocks lie past 1024, where both sides read 0.5.
SOBOL_DEPTHS = (127, 128, 145, 146, 147, 200, 300)
# Halton: the block at b = 141 (maxdepth 142) ends at dimension 999, the last one with a prime; b = 142 (maxdepth 143) starts at 999
# and straddles 1000; 144 and 200 go past it.
HALTON_DEPTHS = (142, 143, 144, 200)
# Ray budgets of the deep box against the oracle.  A path that leaves lock-step with the oracle (a rounding difference at the edge of
# the light or of a wall) goes on for about a hundred more bounces, so a handful of such paths move the count by tenths of a percent:
# the oracle against itself with the camera moved by 1e-6 / 1e-5: 0.10 % / 0.32 % at maxdepth 127; the device at 127 .. 300:
# 0.4 .. 0.9 %.  A wrong sample value past a limit changes every path that gets there (at maxdepth 300 about half of the budget).
DEEP_RAY_TOL = 0.02


def test_deep_box_block_boundaries():
    assert _dims_at(144) + 8 <= SOBOL_DIMS < _dims_at(145) + 8
    assert min(1024, 5 + 8 * 127) < SOBOL_DIMS == min(1024, 5 + 8 * 128)
    assert _dims_at(141) + 8 <= HALTON_DIMS and _dims_at(142) < HALTON_DIMS < _dims_at(142) + 8
    assert _dims_at(146) >= SOBOL_DIMS  # maxdepth 300: from bounce 146 on every dimension reads 0.5


@gpu
@pytest.mark.parametrize("maxdepth", SOBOL_DEPTHS)
def test_deep_paths_across_sobol_dimension_1024(pkg, oracle, gpu_lib, monkeypatch, maxdepth):
    flat, make = deep_box(pkg)
    integ = make(maxdepth)
    want, ost = oracle.render(flat, integ)
    sc = pkg.Scene(flat)
    try:
        base, bst = _render(monkeypatch, sc, integ, "full")
        _check_oracle(oracle, integ, base, bst, want, ost, ray_tol=DEEP_RAY_TOL)
        for mode in ("none", 64):
            got, st = _render(monkeypatch, sc, integ, mode)
            assert _stats(st) == _stats(bst), f"mode {mode}"
            assert np.allclose(got, base, rtol=2e-5, atol=2e-5), f"mode {mode}"
    finally:
        sc.close()


@gpu
@pytest.mark.parametrize("maxdepth", HALTON_DEPTHS)
def test_deep_paths_across_halton_prime_table(pkg, oracle, gpu_lib, maxdepth):
    flat, make = deep_box(pkg)
    integ = make(maxdepth, sampler="halton")
    want, ost = oracle.render(flat, integ)
    sc = pkg.Scene(flat)
    try:
        got, st = sc.render(integ)
    finally:
        sc.close()
    _check_oracle(oracle, integ, got, st, want, ost, ray_tol=DEEP_RAY_TOL)


VOL_VERTEX_CAP = 65536  # PB_VOL_VERTEX_CAP, mega.cu


@gpu
@pytest.mark.parametrize("sampler", ["sobol", "halton"])
def test_deep_volpath_direct_sampler(pkg, oracle, gpu_lib, sampler):
    """k_vol_mega's DirectSampler one dimension at a time past both tables' ends; boundary crossings lower the 16-bit bounce count."""
    flat, make = deep_box(pkg, medium=True)
    integ = make(160, sampler=sampler)
    want, ost = oracle.render(flat, integ)
    sc = pkg.Scene(flat)
    try:
        got, st = sc.render(integ)
    finally:
        sc.close()
    # volpath's visibility is Scene::intersect: no any-hit rays; a medium or roulette decision on a rounding boundary may differ
    _check_oracle(oracle, integ, got, st, want, ost, ray_tol=DEEP_RAY_TOL)
    # the megakernel's per-path vertex cap never cut a path short: the ray budget above matches the oracle's, which has no cap,
    # and no path came near the cap
    assert st.intersection_tests < VOL_VERTEX_CAP * st.camera_rays // 64


# ---------------------------------------------------------------------------------------------------------------------
# 5. negative and huge maxdepth
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("sampler", ["sobol", "halton", "02sequence"])
def test_negative_maxdepth_is_emission_only(pkg, oracle, gpu_lib, sampler):
    """path.rs compares the bounce count with a signed maxdepth: -1 ends every path at its first hit, as maxdepth 0 does."""
    setup = pkg.scenes.small_mixed_scene()
    neg = setup.make_integrator(spp_=4, res=(64, 48), maxdepth_=-1, sampler_=sampler)
    zero = setup.make_integrator(spp_=4, res=(64, 48), maxdepth_=0, sampler_=sampler)
    want, ost = oracle.render(setup.flat, neg)
    sc = pkg.Scene(setup.flat)
    try:
        a, sa = sc.render(neg)
        b, sb = sc.render(zero)
    finally:
        sc.close()
    _check_oracle(oracle, neg, a, sa, want, ost)
    assert _stats(sa) == _stats(sb)
    assert sa.intersection_tests == sa.camera_rays and sa.shadow_tests == 0
    assert np.allclose(a, b, rtol=2e-5, atol=2e-5)


@gpu
def test_negative_maxdepth_volpath(pkg, oracle, gpu_lib):
    setup = pkg.scenes.fog_box_scene(xres=48, yres=48, spp=4, maxdepth=-1)
    neg = setup.make_integrator()
    zero = pkg.scenes.fog_box_scene(xres=48, yres=48, spp=4, maxdepth=0).make_integrator()
    want, ost = oracle.render(setup.flat, neg)
    sc = pkg.Scene(setup.flat)
    try:
        a, sa = sc.render(neg)
        b, sb = sc.render(zero)
    finally:
        sc.close()
    _check_oracle(oracle, neg, a, sa, want, ost, ray_tol=0.003)
    assert _stats(sa) == _stats(sb)
    assert np.allclose(a, b, rtol=2e-5, atol=2e-5)


@gpu
def test_maxdepth_past_the_16_bit_bounce_counter_is_refused(pkg, oracle, gpu_lib):
    H = pkg.host
    setup = pkg.scenes.small_mixed_scene()
    fog = pkg.scenes.fog_box_scene(xres=16, yres=16, spp=1)
    for flat, integ in ((setup.flat, setup.make_integrator(spp_=1, res=(16, 16), maxdepth_=0xfff1)),
                        (fog.flat, fog.make_integrator(maxdepth_=0xfff1))):
        sc = pkg.Scene(flat)
        try:
            with pytest.raises(H.B200Error, match=rf"\(code {ERR_INVALID}\).*maxdepth"):
                sc.render(integ)
        finally:
            sc.close()
    # the largest accepted value renders what the oracle renders (paths end by roulette long before)
    cornell = pkg.scenes.cornell_scene()
    integ = cornell.make_integrator(spp_=4, res=(32, 24), maxdepth_=0xfff0)
    want, ost = oracle.render(cornell.flat, integ)
    sc = pkg.Scene(cornell.flat)
    try:
        got, st = sc.render(integ)
    finally:
        sc.close()
    _check_oracle(oracle, integ, got, st, want, ost)


# ---------------------------------------------------------------------------------------------------------------------
# 6. film sizes at the edges of the pixel packing and of sobol_interval_to_index
# ---------------------------------------------------------------------------------------------------------------------
def _film_setup(pkg, res, spp, screenwindow):
    """cornell_scene on a box-filtered film of `res` pixels; the screen window keeps the box in view at any aspect ratio.  (Its matte
    and plastic surfaces keep a 1-sample-per-pixel image stable: small_mixed_scene's glass moves by relMSE 1.5e-3 when the camera moves
    by 1e-6.)"""
    H = pkg.host
    setup = pkg.scenes.cornell_scene()
    base = setup.make_integrator(spp_=spp, res=res, maxdepth_=5, filt="box")
    cam = H.PerspectiveCamera(base.film, base.camera.camera_to_world, fov=40.0, screenwindow=screenwindow)
    return setup, H.PathIntegrator(cam, base.film, base.sampler, maxdepth=5, lightsamplestrategy="power")


@gpu
@pytest.mark.parametrize("mode", ["full", "none"])
def test_widest_film(pkg, oracle, gpu_lib, monkeypatch, mode):
    """65535 x 2: sample bounds 65535 wide, so m = 16 and the largest packed x, 65534, is shifted to bit 31."""
    setup, integ = _film_setup(pkg, (65535, 2), 1, (-1.0, 1.0, -1.0, 1.0))
    sb = integ.film.sample_bounds
    assert (sb[2] - sb[0], sb[3] - sb[1]) == (65535, 2)
    want, ost = oracle.render(setup.flat, integ)
    sc = pkg.Scene(setup.flat)
    try:
        got, st = _render(monkeypatch, sc, integ, mode)
    finally:
        sc.close()
    _check_oracle(oracle, integ, got, st, want, ost)


@gpu
def test_film_wider_than_the_pixel_packing_is_refused(pkg, gpu_lib):
    setup, integ = _film_setup(pkg, (65536, 1), 1, (-1.0, 1.0, -1.0, 1.0))
    sc = pkg.Scene(setup.flat)
    try:
        with pytest.raises(pkg.host.B200Error, match=rf"\(code {ERR_INVALID}\).*sample bounds"):
            sc.render(integ)
    finally:
        sc.close()


@gpu
@pytest.mark.parametrize("res", [(1, 1), (2, 1)])
def test_tiny_films(pkg, oracle, gpu_lib, res):
    """1 x 1: m = 0, no tables, and sobol_interval_to_index is 0 for every sample (as in the reference): all 16 samples are the
    path through the film's corner, which the screen window puts in the middle of the view.  2 x 1: m = 1."""
    setup, integ = _film_setup(pkg, res, 16, (0.0, 0.2, -0.2, 0.0))
    want, ost = oracle.render(setup.flat, integ)
    sc = pkg.Scene(setup.flat)
    try:
        got, st = sc.render(integ)
    finally:
        sc.close()
    _check_oracle(oracle, integ, got, st, want, ost)


# ---------------------------------------------------------------------------------------------------------------------
# 7. the deep scenes reach the regime they are meant to test (oracle only, no GPU)
# ---------------------------------------------------------------------------------------------------------------------
# calibrated on the oracle (measured: 144.7 rays per path at maxdepth 200, 58 % of the paths shade at bounce 145, 244.8 rays per
# volpath path at maxdepth 160)
DEEP_BOX_RAYS_PER_PATH_200 = 120
DEEP_BOX_SHADE_145_FRACTION = 0.4
DEEP_VOL_RAYS_PER_PATH_160 = 200


def test_deep_box_paths_are_deep(pkg, oracle):
    flat, make = deep_box(pkg)
    _, s145 = oracle.render(flat, make(145))
    _, s146 = oracle.render(flat, make(146))
    _, s200 = oracle.render(flat, make(200))
    cams = s200["camera_rays"]
    assert cams == 32 * 32 * 4
    assert s200["intersection_tests"] / cams >= DEEP_BOX_RAYS_PER_PATH_200
    # a path that shades at bounce 145 -- its block straddles dimension 1024 -- traces one more path ray at maxdepth 146
    assert s146["intersection_tests"] - s145["intersection_tests"] >= DEEP_BOX_SHADE_145_FRACTION * cams


def test_deep_volpath_box_paths_are_deep(pkg, oracle):
    flat, make = deep_box(pkg, medium=True)
    _, st = oracle.render(flat, make(160))
    assert st["intersection_tests"] / st["camera_rays"] >= DEEP_VOL_RAYS_PER_PATH_160
