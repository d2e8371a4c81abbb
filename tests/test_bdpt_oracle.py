"""The BDPT oracle (oracle/oracle_bdpt.hpp) against the path-integrator oracle, and the scene-file front end of `Integrator "bdpt"`.

Both oracles are seeded (Sobol'), so every test here is deterministic.  The path side runs with Russian roulette off (rrthreshold 0),
so both integrators estimate the same truncated sum over path depths <= maxdepth.
"""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def obdpt():
    from oracle import oracle_bdpt
    oracle_bdpt.lib()
    return oracle_bdpt


def _pair(pkg, setup, maxdepth, spp, strategy="power", res=(32, 32)):
    # box filter: with a wider filter the sample bounds exceed the image and pbrt-v3's splat scale 1 / spp over-weights light tracing
    # by (sample-bounds area / image area), a reference quirk the BDPT oracle keeps (DESIGN.md §4f)
    path = setup.make_integrator(spp_=spp, res=res, maxdepth_=maxdepth, filt="box")
    path.rr_threshold = 0.0
    bd = pkg.host.BDPTIntegrator(path.camera, path.film, path.sampler, maxdepth=maxdepth, lightsamplestrategy=strategy)
    return path, bd


K = 8       # sample windows: the spread of the K window estimates gives each estimator's standard error
BLOCK = 16  # per-block comparison (16 x 16 pixels): fine enough to catch a local error; coarse enough that a block sees enough of the
            # rare paths (a pure camera path reaching the small light after three bounces) for the window spread to estimate its error
NSIGMA = 5.0


def _blocks(img, w, h):
    img = np.asarray(img, np.float64).reshape(h, w, 3)
    return img.reshape(h // BLOCK, BLOCK, w // BLOCK, BLOCK, 3).mean(axis=(1, 3)).reshape(-1, 3)


def _windows(render_window, spp):
    """render_window(sample_range) -> per-block estimate; returns the K window estimates [K, nblocks, 3]."""
    step = spp // K
    return np.stack([render_window((k * step, (k + 1) * step)) for k in range(K)])


def _path_windows(oracle, flat, path, w, h):
    return _windows(lambda sr: _blocks(oracle.film_resolve(oracle.render(flat, path, sample_range=sr)[0], 1.0), w, h), path.sampler.spp)


def _assert_same(a, b, what):
    """a, b: [K, nblocks, 3] window estimates of two estimators of the same image.  Each block's difference of means must lie within
    NSIGMA standard errors of the difference (standard errors from the window spread, treating the two as independent, which over-
    estimates the error of correlated pairs), plus 1e-4 absolute for blocks that are black in both."""
    ma, mb = a.mean(axis=0), b.mean(axis=0)
    se = np.sqrt(a.var(axis=0, ddof=1) / K + b.var(axis=0, ddof=1) / K)
    bad = np.abs(ma - mb) > NSIGMA * se + 1e-4
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} block values differ, e.g. {ma[bad][:4]} vs {mb[bad][:4]} (se {se[bad][:4]})"


def _bdpt_strategy_windows(obdpt, flat, bd, w, h, weighted):
    n = obdpt.n_strategies(bd.max_depth)
    step = bd.sampler.spp // K

    def one(sr):
        films = np.zeros((n, w * h, 3), np.float32)
        obdpt.render(flat, bd, sample_range=sr, strategies=films, weighted=weighted)
        return np.stack([_blocks(f / step, w, h) for f in films])  # a strategy film holds sums; each pixel drew `step` samples
    return np.stack([one((k * step, (k + 1) * step)) for k in range(K)])  # [K, n, nblocks, 3]


@pytest.fixture(scope="module")
def cornell_depths(pkg, oracle, obdpt):
    """Cornell box (area light only, matte and plastic), 32 x 32, 64 spp: the path oracle's depth-d image minus its depth-(d-1) image
    for d <= 3, and BDPT's per-strategy films (unweighted and MIS-weighted) at maxdepth 3, all as K sample windows."""
    setup = pkg.scenes.cornell_scene(xres=32, yres=32, spp=64)
    paths = []
    for d in range(4):
        path, _ = _pair(pkg, setup, d, 64)
        paths.append(_path_windows(oracle, setup.flat, path, 32, 32))
    diff = [paths[0]] + [paths[d] - paths[d - 1] for d in range(1, 4)]  # maxdepth 0 still adds the first hit's emission
    _, bd = _pair(pkg, setup, 3, 64)
    un = _bdpt_strategy_windows(obdpt, setup.flat, bd, 32, 32, weighted=False)
    wt = _bdpt_strategy_windows(obdpt, setup.flat, bd, 32, 32, weighted=True)
    return diff, un, wt


def _strategies(d):
    return [(s, d + 2 - s) for s in range(0, d + 2) if not (s == 1 and d == 0)]


@pytest.mark.parametrize("depth", [0, 1, 2, 3])
def test_each_unweighted_strategy_estimates_the_depth_image(obdpt, cornell_depths, depth):
    diff, un, _ = cornell_depths
    for s, t in _strategies(depth):
        _assert_same(un[:, obdpt.strategy_index(s, t)], diff[depth], f"depth {depth} strategy s={s} t={t}")


@pytest.mark.parametrize("depth", [0, 1, 2, 3])
def test_weighted_strategies_of_a_depth_sum_to_the_depth_image(obdpt, cornell_depths, depth):
    # weights that do not sum to one over a depth's strategies bias this sum
    diff, _, wt = cornell_depths
    total = sum(wt[:, obdpt.strategy_index(s, t)] for s, t in _strategies(depth))
    _assert_same(total, diff[depth], f"depth {depth} weighted sum")


def _full_image_case(pkg, oracle, obdpt, setup, maxdepth, res=(32, 32)):
    path, bd = _pair(pkg, setup, maxdepth, 64, res=res)
    w, h = res
    a = _path_windows(oracle, setup.flat, path, w, h)

    def one(sr):
        rgbw, splat, st = obdpt.render(setup.flat, bd, sample_range=sr)
        return _blocks(obdpt.resolve(rgbw, splat, sr[1] - sr[0]), w, h)
    b = _windows(one, 64)
    _assert_same(b, a, f"{setup.name} maxdepth {maxdepth}")


@pytest.mark.parametrize("maxdepth", [0, 1, 3])
def test_bdpt_matches_the_path_integrator_on_the_cornell_box(pkg, oracle, obdpt, maxdepth):
    _full_image_case(pkg, oracle, obdpt, pkg.scenes.cornell_scene(xres=32, yres=32, spp=64), maxdepth)
    _, bd = _pair(pkg, pkg.scenes.cornell_scene(xres=32, yres=32, spp=64), maxdepth, 64)
    _, _, st = obdpt.render(pkg.scenes.cornell_scene(xres=32, yres=32, spp=64).flat, bd)
    assert st["camera_rays"] == 32 * 32 * 64


# The two-sided sphere light is an expected failure, kept as the reference has it (SURVEY §8 a-Q8, DESIGN.md §4f): the sphere's cone
# sample (Light::sample_li, the s = 1 strategy) leaves the sampled normal at zero, so that vertex counts as "not on a surface" and its
# pdf_le direction density is zero in MISWeight.  The s = 1 weights then do not sum to one with the others and BDPT renders the sphere's
# light about 5 % darker than the path integrator.  (Setting the normal from the sphere's centre makes the two agree.)
SPHERE_QUIRK = pytest.mark.xfail(strict=True, reason="sphere cone sample with n = 0 biases the s = 1 MIS weights (reference quirk)")


@pytest.mark.parametrize("light", ["spot", "point", pytest.param("sphere", marks=SPHERE_QUIRK)])
def test_bdpt_matches_the_path_integrator_under_each_light(pkg, oracle, obdpt, light):
    _full_image_case(pkg, oracle, obdpt, pkg.scenes.one_light_scene(light), 3)


def test_bdpt_matches_the_path_integrator_with_distant_infinite_lights_and_glass(pkg, oracle, obdpt):
    # small_mixed_scene: quad area light, point, distant and constant infinite lights over matte / plastic / glass / mirror / metal
    _full_image_case(pkg, oracle, obdpt, pkg.scenes.small_mixed_scene(), 3)


SCENE = """LookAt 0 0 5  0 0 0  0 1 0
Camera "perspective" "float fov" 40
Sampler "{sampler}" "integer pixelsamples" 4
Film "image" "integer xresolution" 16 "integer yresolution" 16
Integrator "bdpt" {params}
WorldBegin
{media}
AttributeBegin
  AreaLightSource "diffuse" "rgb L" [8 8 8]
  Shape "trianglemesh" "integer indices" [0 1 2 0 2 3] "point P" [-0.5 1.9 -0.5  0.5 1.9 -0.5  0.5 1.9 0.5  -0.5 1.9 0.5]
AttributeEnd
Material "matte"
Shape "trianglemesh" "integer indices" [0 1 2 0 2 3] "point P" [-2 -1 -2  2 -1 -2  2 -1 2  -2 -1 2]
WorldEnd
"""


def _parse(pkg, sampler="sobol", params="", media=""):
    return pkg.pbrt_parse_string(SCENE.format(sampler=sampler, params=params, media=media)).jobs[0]


def test_front_end_parses_bdpt(pkg):
    job = _parse(pkg, params='"integer maxdepth" 7 "string lightsamplestrategy" "spatial" "integer pixelbounds" [2 10 3 12]')
    integ = job.integrator
    assert isinstance(integ, pkg.host.BDPTIntegrator)
    assert integ.max_depth == 7 and integ.light_sample_strategy == "spatial" and tuple(integ.pixel_bounds) == (2, 3, 10, 12)
    d = integ.desc()
    assert d.integrator.kind == pkg.host.INTEGRATOR_BDPT
    assert _parse(pkg).integrator.light_sample_strategy == "power" and _parse(pkg).integrator.max_depth == 5


@pytest.mark.parametrize("kw", [dict(params='"bool visualizestrategies" "true"'), dict(params='"bool visualizeweights" "true"'),
                                dict(sampler="02sequence"), dict(params='"integer maxdepth" 65'),
                                dict(media='MakeNamedMedium "fog" "string type" "homogeneous"\nMediumInterface "" "fog"')])
def test_front_end_refusals(pkg, kw):
    with pytest.raises(pkg.host.B200Error):
        _parse(pkg, **kw)
