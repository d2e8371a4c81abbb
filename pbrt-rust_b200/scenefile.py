"""Write a scene back out as a `.pbrt` file (+ binary `.ply` meshes): the inverse of pbrtparser.py.

`SceneBuilder` logs every directive it executes; `write_pbrt` serialises that log and the integrator's film /
camera / sampler / filter / accelerator settings with the reference's directive and parameter names, so that

    scene.pbrt --pbrtparser--> API --> FlatScene      ==      the FlatScene the generator built directly

holds byte for byte (tests/test_scene_file_frontend.py).  Every number is written as the shortest decimal that
reads back to the same f32.  This is also how the synthetic benchmark scenes (scenes.py S1..S5) become files
that the reference binary itself could render.
"""
from __future__ import annotations

import os

import numpy as np

from . import host as H
from . import textures as T
from .plymesh import write_ply

f32 = np.float32
_SAMPLER_NAMES = {H.SAMPLER_SOBOL: "sobol", H.SAMPLER_HALTON: "halton", H.SAMPLER_ZEROTWO: "02sequence"}
_RGB_KEYS = {"Kd", "Ks", "Kr", "Kt", "k", "I", "L", "scale"}


def _num(x):
    x = f32(x)
    if not np.isfinite(x):
        raise ValueError("non-finite numbers have no .pbrt spelling")
    return np.format_float_positional(x, unique=True, trim="-") if 1e-5 <= abs(x) < 1e9 or x == 0 else np.format_float_scientific(x, unique=True, trim="-")


def _nums(a):
    return " ".join(_num(v) for v in np.asarray(a, f32).reshape(-1))


def _rgb(v):
    v = np.full(3, v, f32) if np.isscalar(v) else np.asarray(v, f32)
    return _nums(v)


def _params(kind, name, kw):
    """kwargs of SceneBuilder.material / light_source / area_light_source -> typed parameter list."""
    out = []
    for k, v in kw.items():
        if v is None:
            continue
        if T.is_texture(v):
            raise H.B200Error(f'write_pbrt: parameter "{k}" of {kind} "{name}" is a texture tree built through the Python API; the writer emits '
                              "constants only (textured scenes come from scene files, not the other way round)")
        if isinstance(v, (bool, np.bool_)):
            out.append(f'"bool {k}" ["{"true" if v else "false"}"]')
        elif k in ("from", "to"):
            out.append(f'"point {k}" [{_nums(v)}]')
        elif k == "scale" and kind == "MakeNamedMedium":
            out.append(f'"float scale" [{_num(v)}]')
        elif kind == "MakeNamedMedium" and k in ("nx", "ny", "nz"):
            out.append(f'"integer {k}" [{int(v)}]')
        elif kind == "MakeNamedMedium" and k in ("p0", "p1"):
            out.append(f'"point {k}" [{_nums(v)}]')
        elif kind == "MakeNamedMedium" and k == "density":
            out.append(f'"float density" [{_nums(v)}]')
        elif k in _RGB_KEYS or k in ("sigma_a", "sigma_s") or (k == "eta" and name == "metal"):
            out.append(f'"rgb {k}" [{_rgb(v)}]')
        elif k == "samples":
            out.append(f'"integer samples" [{int(v)}]')
        elif isinstance(v, str):
            out.append(f'"string {k}" "{v}"')
        else:
            out.append(f'"float {k}" [{_num(v)}]')
    return " ".join(out)


def write_pbrt(path, flat, integrator, ply_min_vertices=64):
    """`flat` = FlatScene from SceneBuilder.world_end (carries the directive log); returns the list of files written."""
    path = str(path)
    base, d = os.path.splitext(os.path.basename(path))[0], os.path.dirname(os.path.abspath(path))
    film, cam, samp = integrator.film, integrator.camera, integrator.sampler
    L, files, n_ply = [], [path], 0
    c2w = cam.camera_to_world
    look = getattr(getattr(c2w, "inverse_of", None), "lookat_args", None)
    if look is not None:
        L.append("LookAt " + "  ".join(_nums(v) for v in look))
    else:  # world->camera matrix, column-major as `Transform` reads it (api.rs:1014)
        L.append(f"Transform [{_nums(c2w.m_inv.T)}]")
    cp = [f'"float fov" [{_num(cam.fov)}]']
    if cam.lens_radius:
        cp.append(f'"float lensradius" [{_num(cam.lens_radius)}] "float focaldistance" [{_num(cam.focal_distance)}]')
    if (cam.shutter_open, cam.shutter_close) != (0.0, 1.0):
        cp.append(f'"float shutteropen" [{_num(cam.shutter_open)}] "float shutterclose" [{_num(cam.shutter_close)}]')
    if cam.screenwindow is not None:
        cp.append(f'"float screenwindow" [{_nums(cam.screenwindow)}]')
    L.append('Camera "perspective" ' + " ".join(cp))
    fp = [f'"integer xresolution" [{film.full_resolution[0]}] "integer yresolution" [{film.full_resolution[1]}]']
    if tuple(film.crop) != (0.0, 1.0, 0.0, 1.0):
        fp.append(f'"float cropwindow" [{_nums(film.crop)}]')
    if film.scale != 1.0:
        fp.append(f'"float scale" [{_num(film.scale)}]')
    if np.isfinite(film.max_sample_luminance):
        fp.append(f'"float maxsampleluminance" [{_num(film.max_sample_luminance)}]')
    L.append('Film "image" ' + " ".join(fp))
    flt = [f'"float xwidth" [{_num(film.radius[0])}] "float ywidth" [{_num(film.radius[1])}]']
    flt += [f'"float {k}" [{_num(v)}]' for k, v in film.filter_params.items()]
    L.append(f'PixelFilter "{film.filter}" ' + " ".join(flt))
    sp = f'"integer pixelsamples" [{samp.spp}]'
    if samp.kind == H.SAMPLER_ZEROTWO:
        sp += f' "integer dimensions" [{samp.dimensions}]'
    L.append(f'Sampler "{_SAMPLER_NAMES[samp.kind]}" {sp}')
    ip = [f'"integer maxdepth" [{integrator.max_depth}]']
    if integrator.name in ("path", "volpath"):
        ip += [f'"float rrthreshold" [{_num(integrator.rr_threshold)}]', f'"string lightsamplestrategy" "{integrator.light_sample_strategy}"']
    elif integrator.name == "directlighting":
        ip.append(f'"string strategy" "{integrator.strategy}"')
    if integrator.pixelbounds_param is not None:
        ip.append('"integer pixelbounds" [%d %d %d %d]' % tuple(integrator.pixelbounds_param))
    L.append(f'Integrator "{integrator.name}" ' + " ".join(ip))
    split, max_prims = getattr(flat, "accelerator", ("sah", 4))
    L.append(f'Accelerator "bvh" "string splitmethod" "{split}" "integer maxnodeprims" [{max_prims}]')
    L.append("WorldBegin")
    ind = 0
    for e in flat.source_log:
        k = e[0]
        if k in ("AttributeEnd", "ObjectEnd"):
            ind -= 1
        pad = "  " * ind
        if k in ("AttributeBegin", "AttributeEnd", "ObjectEnd", "Identity"):
            L.append(pad + k)
        elif k in ("ObjectBegin", "ObjectInstance"):
            L.append(f'{pad}{k} "{e[1]}"')
        elif k in ("Translate", "Scale", "Rotate"):
            L.append(f"{pad}{k} {_nums(e[1:])}")
        elif k == "ConcatTransform":
            L.append(f"{pad}ConcatTransform [{_nums(e[1].m.T)}]")
        elif k == "MakeNamedMedium":
            L.append(f'{pad}MakeNamedMedium "{e[1]}" {_params(k, e[1], e[2])}'.rstrip())
        elif k == "MediumInterface":
            L.append(f'{pad}MediumInterface "{e[1]}" "{e[2]}"')
        elif k in ("Material", "LightSource", "AreaLightSource"):
            L.append(f'{pad}{k} "{e[1]}" {_params(k, e[1], e[2])}'.rstrip())
        elif k == "Shape":
            name, kw = e[1], e[2]
            if name == "sphere":
                L.append(f'{pad}Shape "sphere" "float radius" [{_num(kw.get("radius", 1.0))}]')
            else:
                P = np.asarray(kw["P"], f32).reshape(-1, 3)
                idx = np.asarray(kw["indices"]).reshape(-1, 3)
                N, Sv, uv = kw.get("N"), kw.get("S"), kw.get("uv")
                if len(P) >= ply_min_vertices and Sv is None:
                    n_ply += 1
                    rel = f"{base}_mesh{n_ply:04d}.ply"
                    write_ply(os.path.join(d, rel), P, idx, N=N, uv=uv)
                    files.append(os.path.join(d, rel))
                    L.append(f'{pad}Shape "plymesh" "string filename" "{rel}"')
                else:
                    s = f'{pad}Shape "trianglemesh" "integer indices" [{" ".join(str(int(i)) for i in idx.reshape(-1))}] "point P" [{_nums(P)}]'
                    if N is not None:
                        s += f' "normal N" [{_nums(N)}]'
                    if Sv is not None:
                        s += f' "vector S" [{_nums(Sv)}]'
                    if uv is not None:
                        s += f' "float uv" [{_nums(uv)}]'
                    L.append(s)
        else:
            raise H.B200Error(f"scenefile: cannot serialise {k}")
        if k in ("AttributeBegin", "ObjectBegin"):
            ind += 1
    cam_medium = int(getattr(integrator, "camera_medium", -1))
    if integrator.name == "volpath":
        # Camera.medium is the OUTSIDE medium of the graphics state at WorldEnd (api.rs:1736-1739 -> make_camera): state it last
        names = [e[1] for e in flat.source_log if e[0] == "MakeNamedMedium"]
        L.append(f'MediumInterface "" "{names[cam_medium] if cam_medium >= 0 else ""}"')
    L.append("WorldEnd")
    with open(path, "w") as f:
        f.write("\n".join(L) + "\n")
    return files
