"""`API` — the scene-description state machine of pbrt-rust (src/core/api.rs:899-1780) for the PathIntegrator
hot path, sitting between the `.pbrt` parser (pbrtparser.py) and the C ABI (host.py).

Same directives, same state rules (options block vs world block, attribute / transform stacks, named coordinate
systems, named materials, object instancing), same parameter names and defaults as the reference's `create_*`
functions.  `WorldEnd` does what `API::world_end` does up to the call of `Integrator::render`
(api.rs:1715-1747): it flattens the scene into the tables of `pbrt_b200_scene_desc`, builds the BVH through
`pbrt_b200_bvh_build` and assembles film / camera / sampler / integrator; the result is a `RenderJob` whose
`render(device)` runs the CUDA path.  Anything the device path does not implement (other integrators, shapes and
materials, alpha cut-outs, media presets, image-mapped infinite lights, non-perspective cameras) raises `B200Error` naming the
feature: there is no CPU fallback and no silent substitution.  Textures (every class of src/textures/, image maps through
MIPMap pyramids), bump maps, `uber` / `substrate`, homogeneous media and heterogeneous (grid density) media are on the device
path.  One deliberate deviation there: a heterogeneous medium without `density` values, or with
a count other than nx * ny * nz, raises `B200Error` where the reference logs an error and creates no medium.

Reference behaviours kept on purpose (each cited where it is implemented): `Camera` registers the camera space
under the name "name", not "camera" (api.rs:1210); `ActiveTransform` never restricts which transform a
directive edits (`for_active_transform!` ignores the bits, api.rs:941-953), so transforms are never animated;
`Transform` / `ConcatTransform` read their 16 numbers column-major (`from_col_slice`, api.rs:1014,1027); the
point light's translate(P.x, P.y, P.x) (point.rs:103); the mitchell / sinc filter formulas (host.py).
"""
from __future__ import annotations

import os
import warnings

import numpy as np

from . import host as H
from . import paramset as PS
from . import spectrum as S
from . import textures as TX
from .host import B200Error, Transform

f32 = np.float32

KNOWN_MATERIALS = ("matte", "plastic", "fourier", "disney", "mirror", "glass", "hair", "translucent", "metal", "substrate", "subsurface",
                   "kdsubsurface", "uber", "mix")  # api.rs:601-639
HOT_PATH_MATERIALS = ("matte", "plastic", "mirror", "glass", "metal", "uber", "substrate")
KNOWN_SHAPES = ("sphere", "cylinder", "disk", "cone", "paraboloid", "hyperboloid", "curve", "trianglemesh", "plymesh", "heightfield", "loopsubdiv",
                "nurbs")  # api.rs:562-585
KNOWN_INTEGRATORS = ("whitted", "directlighting", "path", "volpath", "bdpt", "mlt", "ambientocclusion", "sppm")  # api.rs:277-289


class RenderJob:
    """What `API::world_end` hands to `Integrator::render`: the flattened scene and the integrator."""

    def __init__(self, flat, integrator, filename, accelerator):
        self.flat, self.integrator, self.filename, self.accelerator = flat, integrator, filename, accelerator
        self.film, self.camera, self.sampler = integrator.film, integrator.camera, integrator.sampler

    def render(self, device=0, **kw):
        """Scene upload + `pbrt_b200_render` + film resolve -> (image [h, w, 3] linear RGB, stats)."""
        scene = H.Scene(self.flat, device=device)
        try:
            return self.integrator.render(scene, **kw)
        finally:
            scene.close()

    @staticmethod
    def write_image(path, image):
        """Film::write_image hands the resolved linear RGB image to an encoder chosen by extension (film.rs:217-264,
        imageio.rs:42-66).  Image encoders are outside this repo's scope (SURVEY.md §2): `.pfm` (the reference writes it too,
        imageio.rs) and `.npy` are written here; any other extension is replaced by `.pfm` and the path actually written is
        returned."""
        path = str(path)
        img = np.ascontiguousarray(image, np.float32)
        if path.lower().endswith(".npy"):
            np.save(path, img)
            return path
        if not path.lower().endswith(".pfm"):
            path = os.path.splitext(path)[0] + ".pfm"
        h, w = img.shape[:2]
        with open(path, "wb") as f:  # PFM: bottom-to-top scanlines, negative scale = little endian
            f.write(b"PF\n%d %d\n-1.0\n" % (w, h))
            f.write(img[::-1].astype("<f4").tobytes())
        return path


class _GraphicsState:
    def __init__(self):
        self.float_textures = {}
        self.spectrum_textures = {}
        self.named_materials = {}
        self.current_material = ("matte", PS.ParamSet())  # GraphicsState::new, api.rs:345-360: default matte
        self.area_light = ""
        self.area_light_params = PS.ParamSet()
        self.reverse_orientation = False
        self.current_inside_medium = self.current_outside_medium = ""  # api.rs:340-341

    def clone(self):
        g = _GraphicsState()
        g.float_textures, g.spectrum_textures, g.named_materials = dict(self.float_textures), dict(self.spectrum_textures), dict(self.named_materials)
        g.current_material, g.area_light, g.area_light_params = self.current_material, self.area_light, self.area_light_params
        g.reverse_orientation = self.reverse_orientation
        g.current_inside_medium, g.current_outside_medium = self.current_inside_medium, self.current_outside_medium
        return g


class API:
    def __init__(self, quick_render=False, image_file="", crop_window=((0.0, 1.0), (0.0, 1.0))):
        self.opts = {"quick_render": bool(quick_render), "image_file": image_file, "crop_window": crop_window}  # pbrt.rs Options
        self.jobs = []
        self.errors = []
        self._reset()

    # --- state -------------------------------------------------------------------------
    def _reset(self):
        self.state = "options"
        self.ctm = Transform()
        self.named_coordinate_system = {}
        self.pushed_graphics_states, self.pushed_transforms = [], []
        self.gs = _GraphicsState()
        self.builder = H.SceneBuilder()
        ro = self.ro = {}
        ro["transform_start_time"], ro["transform_end_time"] = 0.0, 1.0
        ro["filter"], ro["film"], ro["sampler"] = ("box", PS.ParamSet()), ("image", PS.ParamSet()), ("halton", PS.ParamSet())
        ro["accelerator"], ro["integrator"], ro["camera"] = ("bvh", PS.ParamSet()), ("path", PS.ParamSet()), ("perspective", PS.ParamSet())
        ro["camera_to_world"] = Transform()
        self.have_scattering_media = False
        self._max_light_samples = 1

    def _error(self, msg):  # the reference logs with `error!` and carries on
        self.errors.append(msg)
        warnings.warn(msg)

    def _verify_options(self, func):  # verify_options!, api.rs:923-930
        if self.state == "world":
            self._error(f'Options cannot be set inside world block; "{func}" not allowed. Ignoring')
            return False
        return True

    def _verify_world(self, func):  # verify_world!, api.rs:932-939
        if self.state == "options":
            self._error(f'Scene description must be inside world block; "{func}" not allowed. Ignoring')
            return False
        return True

    # --- transforms (api.rs:992-1131) ------------------------------------------------------
    def identity(self):
        self.ctm = Transform()

    def translate(self, dx, dy, dz):
        self.ctm = self.ctm * Transform.translate((dx, dy, dz))

    def rotate(self, angle, dx, dy, dz):
        self.ctm = self.ctm * Transform.rotate(angle, (dx, dy, dz))

    def scale(self, sx, sy, sz):
        self.ctm = self.ctm * Transform.scale(sx, sy, sz)

    def lookat(self, ex, ey, ez, lx, ly, lz, ux, uy, uz):
        self.ctm = self.ctm * Transform.look_at((ex, ey, ez), (lx, ly, lz), (ux, uy, uz))

    @staticmethod
    def _matrix(tr):
        tr = np.asarray(tr, f32)
        if tr.size != 16:
            raise B200Error(f"Transform / ConcatTransform need 16 numbers, got {tr.size}")  # assert_eq!(tr.len(), 16)
        return Transform(tr.reshape(4, 4).T.copy())  # Matrix4x4::from_col_slice

    def transform(self, tr):
        self.ctm = self._matrix(tr)

    def concat_transform(self, tr):
        self.ctm = self.ctm * self._matrix(tr)

    def coordinate_system(self, name):
        self.named_coordinate_system[name] = self.ctm

    def coord_sys_transform(self, name):
        if name in self.named_coordinate_system:
            self.ctm = self.named_coordinate_system[name]
        else:
            warnings.warn(f'Couldn\'t find named coordinate system "{name}"')

    def active_transform_all(self):  # api.rs:1098-1120 set bits that for_active_transform! never reads
        pass

    active_transform_endtime = active_transform_starttime = active_transform_all

    def transform_times(self, start, end):
        if self._verify_options("TransformTimes"):
            self.ro["transform_start_time"], self.ro["transform_end_time"] = start, end

    # --- options block (api.rs:1133-1216) ----------------------------------------------------
    def pixel_filter(self, name, params):
        if self._verify_options("PixelFilter"):
            self.ro["filter"] = (name, params)

    def film(self, ty, params):
        if self._verify_options("Film"):
            self.ro["film"] = (ty, params)

    def sampler(self, name, params):
        if self._verify_options("Sampler"):
            self.ro["sampler"] = (name, params)

    def accelerator(self, name, params):
        if self._verify_options("Accelerator"):
            self.ro["accelerator"] = (name, params)

    def integrator(self, name, params):
        if self._verify_options("Integrator"):
            self.ro["integrator"] = (name, params)

    def camera(self, name, params):
        if self._verify_options("Camera"):
            self.ro["camera"] = (name, params)
            self.ro["camera_to_world"] = self.ctm.inverse()
            self.named_coordinate_system["name"] = self.ro["camera_to_world"]  # sic, api.rs:1210 (pbrt-v3 says "camera")
            # the camera's medium is resolved in make_camera (api.rs:302-320) from the graphics state AT WorldEnd (RenderOptions::make_camera is
            # called from make_integrator), where the attribute stack is back at its outermost level

    def include(self, name):  # api.rs:1198-1201
        from . import pbrtparser

        pbrtparser.parse_file(os.path.abspath(PS.resolve_filename(name)), self)

    def make_named_medium(self, name, params):  # api.rs:1211-1241 + make_medium :706-760
        ty = params.find_one_string("type", "")
        if not ty:
            self._error('No parameter string "type" found in MakeNamedMedium')
            return
        if ty not in ("homogeneous", "heterogeneous"):
            warnings.warn(f'Medium "{ty}" unknown.')
            return
        preset = params.find_one_string("preset", "")
        if preset:
            raise B200Error("MakeNamedMedium presets (get_medium_scattering_properties) are outside the hot path: give sigma_a / sigma_s")
        scale = float(params.find_one_float("scale", 1.0))
        g = float(params.find_one_float("g", 0.0))
        siga = params.find_one_spectrum("sigma_a", np.array([0.0011, 0.0024, 0.014], f32))
        sigs = params.find_one_spectrum("sigma_s", np.array([2.55, 3.21, 3.77], f32))
        grid = {}
        if ty == "heterogeneous":  # GridDensityMedium; missing or miscounted density raises B200Error (SceneBuilder.make_named_medium)
            grid = {"density": params.find_float("density"), "nx": params.find_one_int("nx", 1), "ny": params.find_one_int("ny", 1),
                    "nz": params.find_one_int("nz", 1), "p0": params.find_one_point3f("p0", (0.0, 0.0, 0.0)),
                    "p1": params.find_one_point3f("p1", (1.0, 1.0, 1.0))}
        params.report_unused()
        self.builder.ctm = self.ctm  # a grid's medium_to_world starts from the CTM at MakeNamedMedium (api.rs make_medium)
        self.builder.make_named_medium(name, type=ty, sigma_a=siga, sigma_s=sigs, g=g, scale=scale, **grid)

    def _medium_names(self):  # create_medium_interface, api.rs:382-403: an undefined name is logged and stands for no medium
        out = []
        for n in (self.gs.current_inside_medium, self.gs.current_outside_medium):
            if n and n not in self.builder._media_index:
                self._error(f'Named medium "{n}" undefined')
                n = ""
            out.append(n)
        return tuple(out)

    def medium_interface(self, inside, outside):  # api.rs:1243-1258
        self.gs.current_inside_medium, self.gs.current_outside_medium = inside, outside
        self.have_scattering_media = True

    # --- world block -----------------------------------------------------------------------------
    def world_begin(self):  # api.rs:1255-1266
        if not self._verify_options("WorldBegin"):
            return
        self.state = "world"
        self.ctm = Transform()
        self.named_coordinate_system["world"] = self.ctm

    def attribute_begin(self):
        if self._verify_world("AttributeBegin"):
            self.pushed_graphics_states.append(self.gs.clone())
            self.pushed_transforms.append(self.ctm)

    def attribute_end(self):
        if not self._verify_world("AttributeEnd"):
            return
        if not self.pushed_graphics_states:
            self._error("Unmatched attribute_end() encountered. Ignoring it.")
            return
        self.gs = self.pushed_graphics_states.pop()
        self.ctm = self.pushed_transforms.pop()

    def transform_begin(self):
        if self._verify_world("TransformBegin"):
            self.pushed_transforms.append(self.ctm)

    def transform_end(self):
        if not self._verify_world("TransformEnd"):
            return
        if not self.pushed_transforms:
            self._error("Unmatched transform_end() encountered. Ignoring it.")
            return
        self.ctm = self.pushed_transforms.pop()

    def reverse_orientation(self):
        if self._verify_world("ReverseOrientation"):
            self.gs.reverse_orientation = not self.gs.reverse_orientation

    def texture(self, name, ty, texname, params):  # api.rs:1329-1389 + make_*_texture :656-704
        if not self._verify_world("Texture"):
            return
        tp = PS.TextureParams(params, params, self.gs.float_textures, self.gs.spectrum_textures)
        if ty not in ("float", "color", "spectrum"):
            self._error(f'Texture type "{ty}" unknown.')
            return
        table = self.gs.float_textures if ty == "float" else self.gs.spectrum_textures
        if name in table:
            warnings.warn(f'Texture "{name}" being redefined')
        tex = self._make_texture(ty == "float", texname, tp)
        if tex is not None:
            table[name] = tex
        params.looked_up.update((b, n) for b in params.BUCKETS for n in getattr(params, b))

    def _mapping2d(self, tp):  # get_mapping2d, texture.rs:433-463
        ty = tp.find_string("mapping", "uv")
        if ty == "uv":
            return TX.Mapping2D.uv(tp.find_float("uscale", 1.0), tp.find_float("vscale", 1.0), tp.find_float("udelta", 0.0), tp.find_float("vdelta", 0.0))
        if ty == "planar":
            return TX.Mapping2D.planar(tp.find_vector3f("v1", (1.0, 0.0, 0.0)), tp.find_vector3f("v2", (0.0, 1.0, 0.0)), tp.find_float("udelta", 0.0),
                                       tp.find_float("vdelta", 0.0))
        if ty == "spherical":
            return TX.Mapping2D.spherical(self.ctm.inverse())
        if ty == "cylindrical":
            return TX.Mapping2D.cylindrical(self.ctm.inverse())
        self._error(f'2D texture mapping "{ty}" unknown')
        return TX.Mapping2D.uv()

    def _make_texture(self, is_float, texname, tp):
        """make_float_texture / make_spectrum_texture, api.rs:656-704 -> constant (f32 scalar / RGB), textures.Tex, or None.
        Constant operands fold (same f32 arithmetic the per-hit evaluation would do)."""
        one = (lambda v: f32(v)) if is_float else (lambda v: np.full(3, v, f32))
        get = tp.get_floattexture if is_float else tp.get_spectrumtexture
        findv = tp.find_float if is_float else tp.find_spectrum
        t2w = self.ctm  # IdentityMapping3D::new(t2w) keeps tex-to-world AS world_to_texture (fbm.rs:29, checkerboard.rs:135); 2D mappings invert it
        if texname == "constant":  # textures/constant.rs:24-34
            return findv("value", 1.0)
        if texname == "scale":  # textures/scaled.rs:35-53
            a, b = get("tex1", 1.0), get("tex2", 1.0)
            if not TX.is_texture(a) and not TX.is_texture(b):
                return f32(a * b) if is_float else (a * b).astype(f32)
            return TX.Tex.scale(a, b)
        if texname == "mix":  # textures/mix.rs:37-52
            a, b, amt = get("tex1", 0.0), get("tex2", 1.0), tp.get_floattexture("amount", 0.5)
            if not any(TX.is_texture(x) for x in (a, b, amt)):
                r = np.asarray(a, f32) * f32(f32(1.0) - amt) + np.asarray(b, f32) * f32(amt)
                return f32(r) if is_float else r.astype(f32)
            return TX.Tex.mix(a, b, amt)
        if texname == "bilerp":  # textures/biler.rs:38-55
            m = self._mapping2d(tp)
            return TX.Tex.bilerp(m, findv("v00", 0.0), findv("v01", 1.0), findv("v10", 0.0), findv("v11", 1.0))
        if texname == "imagemap":  # textures/imagemap.rs:178-234
            m = self._mapping2d(tp)
            max_aniso, trilerp = tp.find_float("maxanisotropy", 8.0), tp.find_bool("trilinear", False)
            wrap = tp.find_string("wrap", "repeat")
            wrap = wrap if wrap in ("black", "clamp") else "repeat"
            scale = tp.find_float("scale", 1.0)
            fn = tp.find_filename("filename", "")
            gamma = tp.find_bool("gamma", fn.lower().endswith((".tga", ".png")))
            if not os.path.isfile(fn):
                # ImageTexture::get_texture, imagemap.rs:136-142: an image that cannot be read becomes a 1x1 grey (0.5) texture, converted
                # like any texel (:71-98).  Every lookup of a 1x1 pyramid returns that texel: the texture is folded into a constant
                warnings.warn(f'Creating a constant grey texture to replace "{fn}".')
                texel = TX.convert_texels(np.full((1, 1, 3), 0.5, f32), is_float, float(scale), gamma)[0, 0]
                return f32(texel[0]) if is_float else texel.astype(f32)
            mip = TX.image_mipmap(fn, is_float, trilerp, max_aniso, wrap, float(scale), gamma)
            return TX.Tex.imagemap(m, mip)
        if texname == "uv":  # textures/uv.rs:36-44
            return None if is_float else TX.Tex.uv(self._mapping2d(tp))
        if texname == "checkerboard":  # textures/checkerboard.rs:102-180 (the dimension is read from an INTEGER parameter called "mapping")
            dim = tp.find_int("mapping", 2)
            if dim not in (2, 3):
                self._error(f"{dim} dimensional checkerboard texture not supported")
                return None
            a, b = get("tex1", 1.0), get("tex2", 0.0)
            if dim == 3:
                return TX.Tex.checkerboard3d(t2w, a, b)
            m = self._mapping2d(tp)
            aa = tp.find_string("aamode", "none")
            if aa not in ("none", "closedform"):
                warnings.warn(f'Antialiasing mode "{aa}" not understood by Checkerboard2DTexture; using "closedform"')
                aa = "closedform"
            return TX.Tex.checkerboard(m, a, b, aa)
        if texname == "dots":  # textures/dots.rs:59-70: DotsTexture::new(map, inside, outside) fills (outside, inside) -- the two are swapped, kept
            m = self._mapping2d(tp)
            inside, outside = get("inside", 1.0), get("outside", 0.0)
            return TX.Tex.dots(m, outside=inside, inside=outside)
        if texname in ("fbm", "wrinkled"):  # textures/fbm.rs:30-44, wrinkled.rs:32-46
            octaves, omega = tp.find_int("octaves", 8), tp.find_float("roughness", 0.5)
            return (TX.Tex.fbm if texname == "fbm" else TX.Tex.wrinkled)(t2w, octaves, omega)
        if texname == "marble":  # textures/marble.rs:78-82
            if is_float:
                return None
            return TX.Tex.marble(t2w, tp.find_int("octaves", 8), tp.find_float("roughness", 0.5), tp.find_float("scale", 1.0), tp.find_float("variation", 0.2))
        if texname == "windy":  # textures/windy.rs:30-41
            return TX.Tex.windy(t2w)
        warnings.warn(f'{"Float" if is_float else "Spectrum"} texture "{texname}" unknown.')
        return None

    # --- materials (api.rs:595-654,1391-1460; src/materials/*.rs create_*) ----------------------------
    def _make_material(self, name, mp):
        """-> ("row", MATERIAL_DTYPE row) | None (no material).  Mirrors make_material + the create_* defaults."""
        if name == "" or name == "none":
            return None
        if name not in KNOWN_MATERIALS:
            warnings.warn(f'Material "{name}" unknown. Using "matte".')
            name = "matte"
        if name not in HOT_PATH_MATERIALS:
            raise B200Error(f'Material "{name}" is outside the device path (matte, plastic, mirror, glass, metal, uber, substrate; SURVEY.md §8 f3)')
        kw = {}

        def keep(v):  # a constant stays a number, a texture tree stays a tree
            return v if TX.is_texture(v) else (f32(v) if np.ndim(v) == 0 else v)

        if name == "matte":  # matte.rs:55-61
            kw["Kd"], kw["sigma"] = mp.get_spectrumtexture("Kd", 0.5), keep(mp.get_floattexture("sigma", 0.0))
        elif name == "plastic":  # plastic.rs:72-80
            kw["Kd"], kw["Ks"] = mp.get_spectrumtexture("Kd", 0.25), mp.get_spectrumtexture("Ks", 0.25)
            kw["roughness"] = keep(mp.get_floattexture("roughness", 0.1))
        elif name == "mirror":  # mirror.rs:44-49
            kw["Kr"] = mp.get_spectrumtexture("Kr", 0.9)
        elif name in ("glass", "uber"):  # glass.rs:95-108, uber.rs:114-128
            if name == "glass":
                kw["Kr"], kw["Kt"] = mp.get_spectrumtexture("Kr", 1.0), mp.get_spectrumtexture("Kt", 1.0)
            else:
                kw["Kd"], kw["Ks"] = mp.get_spectrumtexture("Kd", 0.25), mp.get_spectrumtexture("Ks", 0.25)
                kw["Kr"], kw["Kt"] = mp.get_spectrumtexture("Kr", 0.0), mp.get_spectrumtexture("Kt", 0.0)
                kw["roughness"] = keep(mp.get_floattexture("roughness", 0.1))
            if name == "glass":
                eta = mp.get_floattexture_ornull("eta")
                kw["eta"] = keep(eta) if eta is not None else keep(mp.get_floattexture("index", 1.5))
                kw["uroughness"], kw["vroughness"] = keep(mp.get_floattexture("uroughness", 0.0)), keep(mp.get_floattexture("vroughness", 0.0))
            else:
                for key in ("uroughness", "vroughness"):
                    v = mp.get_floattexture_ornull(key)
                    if v is not None:
                        kw[key] = keep(v)
                eta = mp.get_floattexture_ornull("eta")
                kw["eta"] = keep(eta) if eta is not None else keep(mp.get_floattexture("index", 1.5))
                kw["opacity"] = mp.get_spectrumtexture("opacity", 1.0)
        elif name == "metal":  # metal.rs:115-125
            cn, ck = S.copper()
            kw["eta"], kw["k"] = mp.get_spectrumtexture("eta", cn), mp.get_spectrumtexture("k", ck)
            kw["roughness"] = keep(mp.get_floattexture("roughness", 0.01))
            for key in ("uroughness", "vroughness"):
                v = mp.get_floattexture_ornull(key)
                if v is not None:
                    kw[key] = keep(v)
        elif name == "substrate":  # substrate.rs:64-71
            kw["Kd"], kw["Ks"] = mp.get_spectrumtexture("Kd", 0.5), mp.get_spectrumtexture("Ks", 0.5)
            kw["uroughness"], kw["vroughness"] = keep(mp.get_floattexture("uroughness", 0.1)), keep(mp.get_floattexture("vroughness", 0.1))
        bump = mp.get_floattexture_ornull("bumpmap")
        if bump is not None:
            kw["bumpmap"] = bump
        if name in ("plastic", "glass", "metal", "uber", "substrate"):
            kw["remaproughness"] = mp.find_bool("remaproughness", True)
        mp.report_unused()
        return H.SceneBuilder._mat_row(name, **kw)

    def material(self, name, params):
        if not self._verify_world("Material"):
            return
        mp = PS.TextureParams(params, PS.ParamSet(), self.gs.float_textures, self.gs.spectrum_textures)
        self.gs.current_material = (name, params, self._make_material(name, mp))

    def make_named_material(self, name, params):
        if not self._verify_world("MakeNamedMaterial"):
            return
        mp = PS.TextureParams(params, PS.ParamSet(), self.gs.float_textures, self.gs.spectrum_textures)
        mat_name = mp.find_string("type", "")
        if not mat_name:
            self._error('No parameter string "type" found in MakeNamedMaterial')
        row = self._make_material(mat_name, mp)
        if name in self.gs.named_materials:
            warnings.warn(f'Named Material "{name}" redefined.')
        self.gs.named_materials[name] = (mat_name, params, row)

    def named_material(self, name):
        if not self._verify_world("NamedMaterial"):
            return
        if name in self.gs.named_materials:
            self.gs.current_material = self.gs.named_materials[name]
        else:
            self._error(f'NamedMaterial "{name}" unknown')

    def _material_for_shape(self, params):  # GraphicsState::get_materialfor_shape, api.rs:363-380
        cur = self.gs.current_material
        if len(cur) == 2:  # the default matte, created lazily
            cur = self.gs.current_material = (cur[0], cur[1], self._make_material(cur[0], PS.TextureParams(cur[1], PS.ParamSet(), {}, {})))
        if _shape_may_set_material_parameters(params):
            mp = PS.TextureParams(params, cur[1], self.gs.float_textures, self.gs.spectrum_textures)
            return self._make_material(cur[0], mp)
        return cur[2]

    # --- lights (api.rs:764-805,1462-1491) ---------------------------------------------------------
    def light_source(self, name, params):
        if not self._verify_world("LightSource"):
            return
        b = self.builder
        b.ctm = self.ctm
        one = f32(1.0)
        if name == "point":  # point.rs:97-106
            b.light_source("point", I=params.find_one_spectrum("I", one), scale=params.find_one_spectrum("scale", one),
                           **{"from": params.find_one_point3f("from", (0, 0, 0))})
        elif name == "spot":  # spot.rs:119-146
            b.light_source("spot", I=params.find_one_spectrum("I", one), scale=params.find_one_spectrum("scale", one),
                           coneangle=params.find_one_float("coneangle", 30.0), conedeltaangle=params.find_one_float("conedeltaangle", 5.0),
                           to=params.find_one_point3f("to", (0, 0, 1)), **{"from": params.find_one_point3f("from", (0, 0, 0))})
        elif name == "distant":  # distant.rs:122-132
            b.light_source("distant", L=params.find_one_spectrum("L", one), scale=params.find_one_spectrum("scale", one),
                           to=params.find_one_point3f("to", (0, 0, 1)), **{"from": params.find_one_point3f("from", (0, 0, 0))})
        elif name in ("infinite", "exinfinite"):  # infinite.rs:243-262
            if params.find_one_filename("mapname", ""):
                raise B200Error("image-mapped infinite lights are outside the device path (constant-radiance infinite lights only)")
            ns = params.find_one_int("samples", params.find_one_int("nsamples", 1))  # infinite.rs:249-250
            if self.opts["quick_render"]:
                ns = max(1, ns // 4)
            self._max_light_samples = max(self._max_light_samples, ns)
            b.light_source("infinite", L=params.find_one_spectrum("L", one), scale=params.find_one_spectrum("scale", one), samples=ns)
        elif name in ("goniometric", "projection"):
            raise B200Error(f'LightSource "{name}" is outside the hot path (point, spot, distant, infinite, diffuse area)')
        else:
            warnings.warn(f'Light "{name}" unknown.')
            self._error(f'LightSource: light type "{name}" unknown.')
        params.report_unused()

    def area_lightsource(self, name, params):
        if self._verify_world("AreaLightSource"):
            self.gs.area_light, self.gs.area_light_params = name, params

    # --- shapes (api.rs:552-593,1493-1619) -----------------------------------------------------------
    def shape(self, name, params):
        if not self._verify_world("Shape"):
            return
        if name not in KNOWN_SHAPES:
            warnings.warn(f'Shape "{name}" unknown.')
            return
        b = self.builder
        b.ctm, b.reverse_orientation = self.ctm, self.gs.reverse_orientation
        b._medium_names = self._medium_names()
        kw = self._shape_arguments(name, params)
        if kw is None:
            return  # make_shapes returned no shape: nothing else happens (api.rs:1518-1520)
        b._material = self._material_for_shape(params)
        params.report_unused()
        b._area_light = None
        if self.gs.area_light:
            ap = self.gs.area_light_params
            if self.gs.area_light in ("area", "diffuse"):  # diffuse.rs:178-196
                L = (ap.find_one_spectrum("L", f32(1.0)) * ap.find_one_spectrum("scale", f32(1.0))).astype(f32)
                ns = ap.find_one_int("samples", ap.find_one_int("nsamples", 1))  # diffuse.rs:184-190
                if self.opts["quick_render"]:
                    ns = max(1, ns // 4)
                self._max_light_samples = max(self._max_light_samples, ns)
                two = ap.find_one_bool("twosided", False)
                if b._cur_object is not None:
                    warnings.warn("Area lights not supported with object instancing")  # api.rs:1604-1606: the light is dropped
                else:
                    b._area_light = (L, two, max(ns, 1))
            else:
                warnings.warn(f'Area light "{self.gs.area_light}" unknown.')
        b.shape("trianglemesh" if name == "plymesh" else name, **kw)

    def _shape_arguments(self, name, params):
        if name == "sphere":  # sphere.rs:424-433
            radius = params.find_one_float("radius", 1.0)
            zmin, zmax = params.find_one_float("zmin", -radius), params.find_one_float("zmax", radius)
            phimax = params.find_one_float("phimax", 360.0)
            if zmin > -radius or zmax < radius or phimax < 360.0:
                raise B200Error("partial spheres (zmin / zmax / phimax) are outside the hot path")
            return {"radius": float(radius)}
        if name == "trianglemesh":  # triangle.rs:657-760
            vi, P = params.find_int("indices"), params.find_point3f("P")
            uv = params.find_point2f("uv")
            if uv is None:
                uv = params.find_point2f("st")
            if uv is None:
                fuv = params.find_float("uv")
                if fuv is None:
                    fuv = params.find_float("st")
                if fuv is not None:
                    uv = np.asarray(fuv, f32)[: 2 * (len(fuv) // 2)].reshape(-1, 2)
            if vi is None or len(vi) == 0:
                self._error('Vertex indices "indices" not provided with triangle mesh shape')
                return None
            if P is None or len(P) == 0:
                self._error('Vertex positions "P" not provided with triangle mesh shape')
                return None
            if uv is not None and len(uv):
                if len(uv) < len(P):
                    raise B200Error(f'Not enough "uv"s for triangle mesh: expected {len(P)}, found {len(uv)} (the reference would index past the array)')
                if len(uv) > len(P):
                    warnings.warn(f'More "uv"s provided than will be used for triangle mesh. ({len(P)} expected, {len(uv)} found)')
                    uv = uv[: len(P)]
            else:
                uv = None
            Sv, N = params.find_vector3f("S"), params.find_normal3f("N")
            if Sv is not None and len(Sv) != len(P):
                self._error('Number of "S"s for triangle mesh must match "P"s')
                Sv = None
            if N is not None and len(N) != len(P):
                self._error('Number of "N"s for triangle mesh must match "P"s')
                N = None
            if vi.min() < 0 or vi.max() >= len(P):
                self._error(f'trianglemesh has out of-bounds vertex index ({len(P)} "P" values were given)')
                return None
            self._reject_alpha(params)
            return {"P": P, "indices": np.asarray(vi[: 3 * (len(vi) // 3)], np.uint32), "N": N, "S": Sv, "uv": uv}
        if name == "plymesh":  # plymesh.rs:17-167
            from .plymesh import read_ply

            filename = params.find_one_filename("filename", "")
            mesh = read_ply(filename)
            if mesh is None:
                return None
            self._reject_alpha(params)
            return mesh
        raise B200Error(f'Shape "{name}" is outside the hot path (trianglemesh, plymesh, sphere)')

    def _reject_alpha(self, params):
        for key in ("alpha", "shadowalpha"):
            if params.find_texture(key, "") or params.find_one_float(key, 1.0) == 0.0:
                raise B200Error(f'"{key}" cut-out textures are outside the device path')

    # --- object instancing (api.rs:1630-1713) -------------------------------------------------------
    def object_begin(self, name):
        if not self._verify_world("ObjectBegin"):
            return
        self.attribute_begin()
        self.builder.object_begin(name)

    def object_end(self):
        if not self._verify_world("ObjectEnd"):
            return
        if self.builder._cur_object is None:
            self._error("ObjectEnd called outside of instance definition")
        else:
            self.builder.object_end()
        self.attribute_end()

    def object_instance(self, name):
        if not self._verify_world("ObjectInstance"):
            return
        b = self.builder
        if b._cur_object is not None:
            self._error("ObjectInstance can't be called inside instance definition")
            return
        if name not in b._objects:
            self._error(f'Unable to find instance named "{name}"')
            return
        b.ctm = self.ctm
        b.object_instance(name)

    # --- WorldEnd (api.rs:244-326,1715-1780) ----------------------------------------------------------
    def world_end(self):
        if not self._verify_world("WorldEnd"):
            return
        for _ in self.pushed_graphics_states:
            warnings.warn("Missing end to attribute_begin()")
        job = self._make_job()
        self.jobs.append(job)
        self._reset()
        return job

    def _make_film(self):
        fname, fp = self.ro["filter"]
        if fname not in H.FILTER_DEFAULT_RADIUS:
            raise B200Error(f'Filter "{fname}" unknown')  # make_filter panics, api.rs:868-881
        dx, dy = H.FILTER_DEFAULT_RADIUS[fname]
        radius = (float(fp.find_one_float("xwidth", dx)), float(fp.find_one_float("ywidth", dy)))
        fkw = {}
        if fname == "gaussian":
            fkw["alpha"] = fp.find_one_float("alpha", 2.0)
        elif fname == "mitchell":
            fkw["B"], fkw["C"] = fp.find_one_float("B", 1.0 / 3.0), fp.find_one_float("C", 1.0 / 3.0)
        elif fname == "sinc":
            fkw["tau"] = fp.find_one_float("tau", 3.0)
        fp.report_unused()
        name, p = self.ro["film"]
        if name != "image":
            raise B200Error(f'Film "{name}" unknown.')  # the reference then fails with "Unable to create film."
        filename = self.opts["image_file"] or p.find_one_string("filename", "pbrt.exr")  # film.rs:347-362
        xres, yres = p.find_one_int("xresolution", 1280), p.find_one_int("yresolution", 720)
        if self.opts["quick_render"]:
            xres, yres = max(1, xres // 4), max(1, yres // 4)
        cr = p.find_float("cropwindow")
        clamp01 = lambda v: min(max(f32(v), f32(0)), f32(1))
        if cr is not None and len(cr) == 4:
            crop = (clamp01(min(cr[0], cr[1])), clamp01(max(cr[0], cr[1])), clamp01(min(cr[2], cr[3])), clamp01(max(cr[2], cr[3])))
        else:
            if cr is not None:
                self._error(f'{len(cr)} values supplied for "cropwindow". Expected 4.')
            cw = self.opts["crop_window"]
            crop = (clamp01(cw[0][0]), clamp01(cw[0][1]), clamp01(cw[1][0]), clamp01(cw[1][1]))
        scale = float(p.find_one_float("scale", 1.0))
        p.find_one_float("diagonal", 35.0)
        msl = float(p.find_one_float("maxsampleluminance", np.inf))
        p.report_unused()
        return H.Film(xres, yres, filter=fname, radius=radius, crop=crop, scale=scale, max_sample_luminance=msl, **fkw), filename

    def _make_camera(self, film):
        name, p = self.ro["camera"]
        if name != "perspective":
            if name in ("orthographic", "realistic", "environment"):
                raise B200Error(f'Camera "{name}" is outside the hot path (perspective)')
            raise B200Error(f'Camera "{name}" unknown')  # "Unable to create camera"
        so, sc = p.find_one_float("shutteropen", 0.0), p.find_one_float("shutterclose", 1.0)  # perspective.rs:298-357
        if sc < so:
            warnings.warn(f"Shutter close time [{sc}] < shutter open [{so}]. Swapping time.")
            so, sc = sc, so
        lensradius, focaldistance = p.find_one_float("lensradius", 0.0), p.find_one_float("focaldistance", 1.0e30)
        frame = p.find_one_float("frameaspectratio", f32(film.full_resolution[0]) / f32(film.full_resolution[1]))
        if frame > 1:
            screen = [-frame, frame, f32(-1), f32(1)]
        else:
            screen = [f32(-1), f32(1), f32(-1) / frame, f32(1) / frame]
        sw = p.find_float("screenwindow")
        if sw is not None:
            if len(sw) == 4:
                screen = [f32(v) for v in sw]
            else:
                self._error('"screenwindow" should have four values')
        fov, halffov = p.find_one_float("fov", 90.0), p.find_one_float("halffov", -1.0)
        if halffov > 0.5:
            fov = f32(2.0) * halffov
        p.report_unused()
        return H.PerspectiveCamera(film, self.ro["camera_to_world"], fov=fov, lensradius=float(lensradius), focaldistance=float(focaldistance),
                                   shutteropen=float(so), shutterclose=float(sc), screenwindow=screen)

    def _make_sampler(self):
        name, p = self.ro["sampler"]
        if name not in H.Sampler.KINDS:
            if name in ("maxmindist", "random", "stratified"):
                raise B200Error(f'Sampler "{name}" is outside the hot path (sobol, halton, 02sequence / lowdiscrepancy)')
            raise B200Error(f'Sampler "{name}" unknown.')  # "Unable to create sampler."
        nsamp = p.find_one_int("pixelsamples", 16)
        if self.opts["quick_render"]:
            nsamp = 1
        dims = 4
        if name in ("02sequence", "lowdiscrepancy"):
            dims = p.find_one_int("dimensions", 4)
        if name == "halton" and p.find_one_bool("samplepixelcenter", False):
            raise B200Error('HaltonSampler "samplepixelcenter" is outside the hot path')
        p.report_unused()
        return H.Sampler(name, pixelsamples=nsamp, dimensions=dims)

    def _make_job(self):
        film, filename = self._make_film()
        camera = self._make_camera(film)
        sampler = self._make_sampler()
        name, p = self.ro["integrator"]
        if name not in ("path", "directlighting", "whitted", "volpath", "bdpt"):
            if name in KNOWN_INTEGRATORS:
                raise B200Error(f'Integrator "{name}" is outside the device path ("path", "volpath", "bdpt", "directlighting", "whitted")')
            raise B200Error(f'Integrator "{name}" unknown.')
        maxdepth = p.find_one_int("maxdepth", 5)  # path.rs:225-253, directlighting.rs:125, whitted.rs:111
        pb = p.find_int("pixelbounds")
        pixelbounds = None
        if pb is not None:
            if len(pb) != 4:
                self._error(f'Expected four values for "pixelbounds" parameter. Got {len(pb)}.')
            else:
                pixelbounds = tuple(int(v) for v in pb)
        if name == "path":
            rr = float(p.find_one_float("rrthreshold", 1.0))
            strategy = p.find_one_string("lightsamplestrategy", "spatial")
            integ = H.PathIntegrator(camera, film, sampler, maxdepth=maxdepth, rrthreshold=rr, lightsamplestrategy=strategy, pixelbounds=pixelbounds)
        elif name == "volpath":  # volpath.rs:224-262; Camera.medium = the outside medium of the graphics state make_camera sees (api.rs:256)
            rr = float(p.find_one_float("rrthreshold", 1.0))
            strategy = p.find_one_string("lightsamplestrategy", "spatial")
            self.builder._medium_names = self._medium_names()
            cam_medium = self.builder.camera_medium()
            integ = H.VolPathIntegrator(camera, film, sampler, maxdepth=maxdepth, rrthreshold=rr, lightsamplestrategy=strategy, pixelbounds=pixelbounds,
                                        camera_medium=cam_medium)
        elif name == "bdpt":  # bdpt.rs / pbrt-v3 CreateBDPTIntegrator (bdpt.cpp:448-480)
            if sampler.kind == H.SAMPLER_ZEROTWO:
                raise B200Error('Integrator "bdpt" needs the sobol or halton sampler on the device path (as volpath does)')
            vs, vw = p.find_one_bool("visualizestrategies", False), p.find_one_bool("visualizeweights", False)
            if vs or vw:
                raise B200Error('Integrator "bdpt": visualizestrategies / visualizeweights are not rendered on the device')
            strategy = p.find_one_string("lightsamplestrategy", "power")
            integ = H.BDPTIntegrator(camera, film, sampler, maxdepth=maxdepth, lightsamplestrategy=strategy, pixelbounds=pixelbounds)
        elif name == "directlighting":  # directlighting.rs:146-156
            st = p.find_one_string("strategy", "all")
            if st not in ("one", "all"):
                warnings.warn(f'Strategy "{st}" for direct lighting unknown. Using "all".')
                st = "all"
            if st == "all" and self._max_light_samples != 1 and sampler.kind == H.SAMPLER_ZEROTWO:
                raise B200Error('directlighting "all" with lights asking for more than one sample needs the sobol or halton sampler on the device path '
                                "(the 02sequence sample arrays are built for one element per pixel sample)")
            integ = H.DirectLightingIntegrator(camera, film, sampler, maxdepth=maxdepth, strategy=st, pixelbounds=pixelbounds)
        else:
            integ = H.WhittedIntegrator(camera, film, sampler, maxdepth=maxdepth, pixelbounds=pixelbounds)
        p.report_unused()
        if pixelbounds is not None and (integ.pixel_bounds[2] <= integ.pixel_bounds[0] or integ.pixel_bounds[3] <= integ.pixel_bounds[1]):
            self._error('Degenerate "pixelbounds" specified.')
        aname, ap = self.ro["accelerator"]  # make_accelerator, api.rs:807-819 + bvh.rs:913-930
        if aname == "kdtree":
            raise B200Error('Accelerator "kdtree" is outside the hot path ("bvh")')
        if aname != "bvh":
            warnings.warn(f'Accelerator "{aname}" unknown. Using BVH.')
        split = ap.find_one_string("splitmethod", "sah")
        if split == "hlbvh":
            raise B200Error('BVH splitmethod "hlbvh" is not mirrored by pbrt_b200_bvh_build (sah, middle, equal)')
        if split not in H.SPLIT:
            warnings.warn(f'BVH split method "{split}" unknown.  Using "sah".')
            split = "sah"
        max_prims = ap.find_one_int("maxnodeprims", 4)
        ap.report_unused()
        flat = self.builder.world_end(max_prims=max_prims, split_method=split)
        if name == "bdpt":
            self.builder._medium_names = self._medium_names()
            if len(flat.media) or self.builder.camera_medium() >= 0:
                raise B200Error('Integrator "bdpt" renders surfaces only: the scene has participating media (use "volpath")')
        if self.have_scattering_media and name not in ("volpath", "bdpt"):
            warnings.warn(f'Scene has scattering media but "{name}" integrator doesn\'t support volume scattering.')
        return RenderJob(flat, integ, filename, (split, max_prims))


def _shape_may_set_material_parameters(ps):  # api.rs:1782-1817
    if any(n not in ("alpha", "shadowalpha") for n in ps.textures):
        return True
    if any(len(v) == 1 and n not in ("filename", "type", "scheme") for n, v in ps.strings.items()):
        return True
    for bucket in ("bools", "ints", "point2fs", "vector2fs", "point3fs", "vector3fs", "normals", "spectra"):
        if any(len(v) == 1 for v in getattr(ps, bucket).values()):
            return True
    return False
