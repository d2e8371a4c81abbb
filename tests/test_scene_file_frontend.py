"""Scene-file front end (SURVEY.md §8 f2): `.pbrt` lexer / grammar, ParamSet, API state machine, plymesh.

The reference has no tests for its parser; parity is anchored on (1) its own spheres scene file, re-emitted directive for
directive as tests/golden/reference_spheres_scene.pbrt, (2) known answers that its code fixes — the copper RGB of metal.rs
through `from_sampled`, f32 literal rounding, the ParamSet lookup rules — and (3) the closed loop
scene -> .pbrt/.ply -> parser -> API -> byte-identical FlatScene and render descriptor.
"""
import importlib
import os
import warnings
from fractions import Fraction
from pathlib import Path

import numpy as np
import pytest

pkg = importlib.import_module("pbrt-rust_b200")
PP, PS, SP, SF, PLY = pkg.pbrtparser, pkg.paramset, pkg.spectrum, importlib.import_module("pbrt-rust_b200.scenefile"), pkg.plymesh
f32 = np.float32

FLAT_KEYS = ("nodes", "prims", "vertex_p", "vertex_n", "vertex_s", "vertex_uv", "tri_indices", "spheres", "materials", "lights", "objects", "instances")


def same_flat(a, b):
    for k in FLAT_KEYS:
        x, y = getattr(a, k), getattr(b, k)
        if (x is None) != (y is None) or (x is not None and x.tobytes() != y.tobytes()):
            return k
    if (a.n_top_nodes, a.n_top_prims) != (b.n_top_nodes, b.n_top_prims):
        return "n_top"
    return None


SPHERES = """
# the reference's src/scenes/spheres-differentials-texfilt.pbrt with the path integrator and a constant Kd
LookAt 2 2 5   0 -.4 0 0 1 0
Camera "perspective" "float fov" [30 ]
Film "image" "integer xresolution" [400 ] "integer yresolution" [400 ]
    "string filename" "spheres.exr"
Integrator "path" "integer maxdepth" [5]
Sampler "sobol" "integer pixelsamples" [64]
PixelFilter "box"
WorldBegin
LightSource "distant" "point from" [0 10 0 ] "point to" [0 0 0 ]
    "color L" [3.141593 3.141593 3.141593 ]
AttributeBegin
\tTranslate .25 0 0
\tMaterial "matte" "color Kd" [.5 .5 .5]
    Shape "trianglemesh"  "integer indices" [0 1 2 0 2 3 ]
\t"point P" [-100 -1 -100 400 -1 -100 400 -1 400 -100 -1 400 ]
AttributeEnd
Translate -1.3 0 0
Material "mirror"
Shape "sphere"
Translate 2.6 0 0
Material "glass"
Shape "sphere"
WorldEnd
"""


def test_lexer_tokens_and_comments():
    cmds = PP.parse_commands('# c\nTranslate 1 -2.5 .5e1 #tail\nShape "sphere" "float radius" 2 "string x" ["a" "b"]\nWorldEnd')
    assert cmds[0] == ("Translate", [1.0, -2.5, 5.0])
    assert cmds[1][0:2] == ("Shape", "sphere")
    ps = cmds[1][2]
    assert ps.find_one_float("radius", 1.0) == 2.0 and ps.strings["x"] == ["a", "b"]
    assert cmds[2] == ("WorldEnd",)


def test_lexer_keyword_prefixes_follow_lexer_rs():
    # lexer.rs matches keywords as prefixes in a fixed order: TransformBegin / TransformEnd before Transform
    cmds = PP.parse_commands("TransformBegin TransformEnd Transform [1 0 0 0 0 1 0 0 0 0 1 0 0 0 0 1] ActiveTransform StartTime")
    assert [c[0] for c in cmds] == ["TransformBegin", "TransformEnd", "Transform", "ActiveTransform"]
    assert cmds[3][1] == "StartTime"


def test_parse_errors():
    for bad in ("", "Shape", 'Shape "sphere" "float radius"', "LookAt 1 2 3", "Bogus 1 2", 'Shape "sphere" "float r" [1 "a"]', 'Shape "sphere" "float r" []',
                'Shape "sphere" "quux radius" 1'):
        with pytest.raises(pkg.B200Error):
            PP.parse_commands(bad)


def test_f32_literals_are_correctly_rounded():
    # Rust's str::parse::<f32> rounds the decimal once; going through f64 rounds twice.  16777217 = 2^24 + 1 sits exactly
    # between two f32 values; digits after it decide the direction, which a double cannot see.
    cases = ["16777217", "16777217.0000000001", "16777216.9999999999", "0.1", "1e-45", "3.4028235e38", "1.00000005960464477539062500001",
             "1.000000059604644775390625", "1.00000017881393432617187500", "-7.038531e-26"]
    got = PP.parse_f32(cases)
    for tok, g in zip(cases, got):
        exact = Fraction(tok)
        with np.errstate(over="ignore"):
            cands = [c for c in (g, np.nextafter(g, f32(np.inf)), np.nextafter(g, f32(-np.inf))) if np.isfinite(c)]
        errs = [abs(Fraction(float(c)) - exact) for c in cands]
        assert errs[0] == min(errs), tok
        if errs.count(errs[0]) > 1:  # tie -> even mantissa
            assert int(np.array(g, f32).view(np.uint32)) & 1 == 0, tok
    assert got[1] == f32(16777218.0) and got[2] == f32(16777216.0) and got[0] == f32(16777216.0)
    r = np.random.default_rng(5)
    x = (r.standard_normal(20000) * 10.0 ** r.integers(-30, 30, 20000)).astype(f32)
    toks = [SF._num(v) for v in x]
    assert PP.parse_f32(toks).tobytes() == x.tobytes()


def test_paramset_lookup_rules():
    ps = PS.ParamSet()
    ps.add("float a", np.array([1, 2], f32))
    ps.add("float b", np.array([3], f32))
    ps.add("integer n", np.array([7.9], f32))
    ps.add("bool t", ["true"])
    ps.add("point P", np.arange(7, dtype=f32))  # excess value dropped with a warning
    assert ps.find_one_float("a", 9.0) == 9.0  # find_one only matches single-valued items (paramset.rs:39-51)
    assert ps.find_one_float("b", 9.0) == 3.0 and list(ps.find_float("a")) == [1.0, 2.0]
    assert ps.find_one_int("n", 0) == 7 and ps.find_one_bool("t", False) is True
    assert ps.find_point3f("P").shape == (2, 3)
    ps.add("float b", np.array([4], f32))  # a second declaration replaces the first (erase_float)
    assert ps.find_one_float("b", 9.0) == 4.0
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        ps.report_unused()
    assert not any('"b"' in str(x.message) for x in w)


def test_spectrum_parameters_known_answers():
    # metal.rs:50-53 COPPER_N / COPPER_K through RGBSpectrum::from_sampled: the constants host.py has carried since the
    # first round were derived independently from the same tables
    n, k = SP.copper()
    assert np.allclose(n, pkg.host.COPPER_N, rtol=0, atol=1e-7) and np.allclose(k, pkg.host.COPPER_K, rtol=0, atol=1e-6)
    assert np.array_equal(SP.xyz_to_rgb((0, 0, 0)), np.zeros(3, f32))
    # a flat spectrum of 1 integrates to Y = sum(CIE_Y) * (830-360) / (CIE_Y_INTEGRAL * 471): slightly below 1
    flat = SP.from_sampled([300.0, 900.0], [1.0, 1.0])
    t = SP.cie_tables()
    y = 0.212671 * flat[0] + 0.715160 * flat[1] + 0.072169 * flat[2]
    assert abs(y - float(t["cie_y"].sum()) * 470.0 / (float(t["cie_y_integral"]) * 471.0)) < 1e-4
    ps = PS.ParamSet()
    ps.add("blackbody L", np.array([6500, 2], f32))
    bb = ps.find_one_spectrum("L", 0.0)
    assert bb.shape == (3,) and 1.5 < bb[1] < 2.0 and bb[0] > bb[1] * 0.95  # ~white at 6500 K, scaled by 2
    ps.add("xyz X", np.array([0.2, 0.3, 0.4], f32))
    assert np.array_equal(ps.find_one_spectrum("X", 0.0), SP.xyz_to_rgb((0.2, 0.3, 0.4)))
    ps.add("spectrum S", np.array([400, 0.5, 700, 0.5], f32))
    assert np.allclose(ps.find_one_spectrum("S", 0.0), 0.5 * flat, atol=1e-6)


def test_spheres_file_equals_the_api_built_scene():
    api = pkg.pbrt_parse_string(SPHERES)
    assert len(api.jobs) == 1 and not api.errors
    job, ref = api.jobs[0], pkg.scenes.spheres_scene()
    assert same_flat(job.flat, ref.flat) is None
    assert bytes(job.integrator.desc()) == bytes(ref.make_integrator().desc())
    assert job.filename == "spheres.exr"


@pytest.mark.parametrize("gen", ["spheres_scene", "cornell_scene", "small_mixed_scene", "instanced_scene", "many_lights_scene"])
def test_written_scene_files_parse_back_bit_identically(gen, tmp_path):
    setup = getattr(pkg.scenes, gen)()
    integ = setup.make_integrator()
    files = SF.write_pbrt(tmp_path / (gen + ".pbrt"), setup.flat, integ)
    api = pkg.pbrt_parse(files[0])
    assert not api.errors and len(api.jobs) == 1
    assert same_flat(api.jobs[0].flat, setup.flat) is None
    assert bytes(api.jobs[0].integrator.desc()) == bytes(integ.desc())


def test_directlighting_and_whitted_scene_files(tmp_path):
    setup = pkg.scenes.small_mixed_scene()
    base = setup.make_integrator()
    for integ in (pkg.host.WhittedIntegrator(base.camera, base.film, base.sampler, maxdepth=7),
                  pkg.host.DirectLightingIntegrator(base.camera, base.film, base.sampler, maxdepth=3, strategy="one"),
                  pkg.host.DirectLightingIntegrator(base.camera, base.film, base.sampler)):
        job = pkg.pbrt_parse(SF.write_pbrt(tmp_path / (integ.name + ".pbrt"), setup.flat, integ)[0]).jobs[0]
        assert type(job.integrator) is type(integ) and bytes(job.integrator.desc()) == bytes(integ.desc())
        assert same_flat(job.flat, setup.flat) is None
    # directlighting.rs:146-152: strategy defaults to "all"; area lights asking for several samples cannot cross the C ABI
    job = pkg.pbrt_parse_string('Integrator "directlighting"\nWorldBegin\nShape "sphere"\nWorldEnd').jobs[0]
    assert job.integrator.kind == pkg.host.INTEGRATOR_DIRECT_ALL and job.integrator.max_depth == 5
    # a light's "samples" travels in pbrt_b200_light.n_samples (diffuse.rs:184-185); multi-sample arrays need a global sampler
    tri = 'AreaLightSource "diffuse" "integer samples" [4]\nShape "trianglemesh" "integer indices" [0 1 2] "point P" [0 0 0 1 0 0 0 1 0]\nWorldEnd'
    job = pkg.pbrt_parse_string('Integrator "directlighting"\nWorldBegin\nLightSource "infinite" "integer nsamples" 2\n' + tri).jobs[0]
    assert job.flat.lights["n_samples"].tolist() == [2, 4]
    with pytest.raises(pkg.B200Error):
        pkg.pbrt_parse_string('Integrator "directlighting"\nSampler "02sequence"\nWorldBegin\n' + tri)


def test_inline_meshes_and_ply_meshes_agree(tmp_path):
    setup = pkg.scenes.small_mixed_scene()
    integ = setup.make_integrator(sampler_="02sequence", filt="gaussian")
    a = pkg.pbrt_parse(SF.write_pbrt(tmp_path / "ply.pbrt", setup.flat, integ, ply_min_vertices=8)[0]).jobs[0]
    b = pkg.pbrt_parse(SF.write_pbrt(tmp_path / "inline.pbrt", setup.flat, integ, ply_min_vertices=10 ** 9)[0]).jobs[0]
    assert same_flat(a.flat, setup.flat) is None and same_flat(b.flat, setup.flat) is None
    assert bytes(a.integrator.desc()) == bytes(integ.desc()) == bytes(b.integrator.desc())


@pytest.mark.parametrize("fmt", ["ascii", "binary_little_endian", "binary_big_endian"])
def test_plymesh_formats_and_quads(fmt, tmp_path):
    P, idx = pkg.scenes.box_mesh((-1, -1, -1), (1, 2, 3))
    N = np.tile(np.array([[0, 0, 1]], f32), (len(P), 1))
    PLY.write_ply(tmp_path / "m.ply", P, idx, N=N, fmt=fmt)
    m = PLY.read_ply(str(tmp_path / "m.ply"))
    assert m["P"].tobytes() == np.asarray(P, f32).tobytes() and m["indices"].tobytes() == np.asarray(idx, np.uint32).tobytes()
    assert m["N"].tobytes() == N.tobytes() and m["uv"] is None
    # a quad face splits into (0 1 2) (3 0 2), plymesh.rs:98-114; a pentagon is skipped
    (tmp_path / "q.ply").write_text("ply\nformat ascii 1.0\ncomment x\nelement vertex 5\nproperty float x\nproperty float y\nproperty float z\n"
                                    "property float u\nproperty float v\nelement face 3\nproperty list uchar int vertex_indices\nend_header\n"
                                    "0 0 0 0 0\n1 0 0 1 0\n1 1 0 1 1\n0 1 0 0 1\n.5 2 0 .5 1\n4 0 1 2 3\n5 0 1 2 3 4\n3 2 3 4\n")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        q = PLY.read_ply(str(tmp_path / "q.ply"))
    assert q["indices"].tolist() == [[0, 1, 2], [3, 0, 2], [2, 3, 4]] and q["uv"].shape == (5, 2)


def test_api_state_rules():
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        # options inside the world block and shapes outside it are ignored with an error (verify_options! / verify_world!)
        api = pkg.pbrt_parse_string('Shape "sphere"\nWorldBegin\nFilm "image" "integer xresolution" [8]\nShape "sphere"\nAttributeEnd\nWorldEnd')
        assert len(api.errors) == 3 and len(api.jobs[0].flat.spheres) == 1
        assert api.jobs[0].film.full_resolution == (1280, 720)  # film.rs:364-365 defaults
        # Camera registers its space as "name" (api.rs:1210), so CoordSysTransform "camera" finds nothing and keeps the CTM
        api = pkg.pbrt_parse_string('Translate 1 2 3\nCamera "perspective"\nWorldBegin\nCoordSysTransform "camera"\nShape "sphere"\n'
                                    'CoordSysTransform "name"\nShape "sphere"\nWorldEnd')
        sph = api.jobs[0].flat.spheres
        assert np.array_equal(sph[0]["object_to_world"].reshape(4, 4), np.eye(4, dtype=f32))
        assert np.array_equal(sph[1]["object_to_world"].reshape(4, 4)[:3, 3], np.array([-1, -2, -3], f32))
    # named materials, shape-level material overrides (get_materialfor_shape), constant textures
    api = pkg.pbrt_parse_string('WorldBegin\nTexture "g" "color" "constant" "rgb value" [.1 .2 .3]\n'
                                'MakeNamedMaterial "m" "string type" "plastic" "texture Kd" "g" "float roughness" .3\nNamedMaterial "m"\n'
                                'Shape "sphere"\nShape "sphere" "rgb Ks" [.9 .9 .9]\nWorldEnd')
    mats = api.jobs[0].flat.materials
    assert len(mats) == 2 and np.allclose(mats[0]["a"], [.1, .2, .3]) and np.allclose(mats[0]["b"], .25) and np.allclose(mats[1]["b"], .9)
    assert mats[0]["f0"] == f32(.3) and mats[1]["f0"] == f32(.3)


def test_out_of_scope_features_fail_loudly():
    for text in ('Integrator "sppm"\nWorldBegin\nWorldEnd', 'WorldBegin\nMaterial "disney"\nWorldEnd', 'WorldBegin\nShape "cylinder"\nWorldEnd',
                 'Camera "orthographic"\nWorldBegin\nWorldEnd',
                 'WorldBegin\nShape "trianglemesh" "integer indices" [0 1 2] "point P" [0 0 0 1 0 0 0 1 0] "texture alpha" "t"\nWorldEnd',
                 'WorldBegin\nLightSource "infinite" "string mapname" "env.exr"\nWorldEnd', 'Sampler "random"\nWorldBegin\nWorldEnd',
                 'WorldBegin\nMakeNamedMedium "m" "string type" "heterogeneous"\nWorldEnd',
                 'WorldBegin\nMakeNamedMedium "m" "string type" "homogeneous" "string preset" "Skin1"\nWorldEnd'):
        with pytest.raises(pkg.B200Error):
            pkg.pbrt_parse_string(text)


def test_textures_that_are_declared_but_unused_and_missing_image_maps(tmp_path):
    # a procedural texture nobody references is not an error (the reference's spheres scene declares one); an image map whose
    # file cannot be read is the constant grey texture of imagemap.rs:136-142, inverse-gamma-corrected for .png / .tga
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        job = pkg.pbrt_parse_string('WorldBegin\nTexture "c" "color" "checkerboard" "float uscale" 4\n'
                                    'Texture "a" "color" "imagemap" "string filename" "nope/lines.png" "float scale" 2\n'
                                    'Texture "b" "color" "imagemap" "string filename" "nope/lines.exr"\n'
                                    'Texture "f" "float" "imagemap" "string filename" "nope/r.tga"\n'
                                    'Material "matte" "texture Kd" "a"\nShape "sphere"\nMaterial "matte" "texture Kd" "b" "texture sigma" "f"\nShape "sphere"\nWorldEnd',
                                    search_dir=str(tmp_path)).jobs[0]
    m = job.flat.materials
    g = ((0.5 + 0.055) / 1.055) ** 2.4
    assert np.allclose(m[0]["a"], 2 * g, rtol=1e-6) and np.allclose(m[1]["a"], 0.5) and abs(m[1]["f0"] - g) < 1e-6
    # a file that exists but cannot be decoded is the same grey texel, kept as a 1x1 image map (imagemap.rs:136-142)
    (tmp_path / "real.png").write_bytes(b"\x89PNG\r\n")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        job = pkg.pbrt_parse_string('WorldBegin\nTexture "a" "color" "imagemap" "string filename" "real.png"\nMaterial "matte" "texture Kd" "a"\nShape "sphere"\nWorldEnd',
                                    search_dir=str(tmp_path)).jobs[0]
    assert len(job.flat.mipmaps) == 1 and job.flat.mipmaps[0]["width"] == 1 and job.flat.materials[0]["textured"] == 1
    assert np.allclose(job.flat.mipmap_objects[0].texels, g, rtol=1e-6)


def test_include_resolves_against_the_scene_directory(tmp_path):
    (tmp_path / "geo").mkdir()
    (tmp_path / "geo" / "inc.pbrt").write_text('Material "mirror"\nShape "sphere" "float radius" 2\n')
    (tmp_path / "main.pbrt").write_text('WorldBegin\nInclude "geo/inc.pbrt"\nWorldEnd\n')
    job = pkg.pbrt_parse(tmp_path / "main.pbrt").jobs[0]
    assert job.flat.spheres[0]["radius"] == 2.0 and job.flat.materials[0]["type"] == pkg.host.MAT_MIRROR


def test_reference_spheres_scene_file_parses():
    """The directives of the reference's src/scenes/spheres-differentials-texfilt.pbrt (directlighting "all", lowdiscrepancy sampler,
    missing image map -> grey); tests/test_gpu_recursive_integrators.py renders the same file on the GPU."""
    path = Path(__file__).parent / "golden" / "reference_spheres_scene.pbrt"
    cmds = PP.parse_commands(path.read_text())
    assert len(cmds) == 22 and cmds[-1] == ("WorldEnd",) and sum(c[0] == "WorldBegin" for c in cmds) == 1
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        job = pkg.pbrt_parse(path).jobs[0]
    assert job.integrator.kind == pkg.host.INTEGRATOR_DIRECT_ALL and len(job.flat.spheres) == 2 and job.flat.vertex_uv is not None
