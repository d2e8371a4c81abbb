"""Deterministic synthetic scenes and ray batches (SURVEY.md s8(d): S1..S5, B-cam/B-diff/B-shadow).

Each generator drives the SceneBuilder exactly as a .pbrt file would drive pbrt-rust's
API, and returns (FlatScene, integrator factory).  All randomness is PCG32 (the
reference's RNG, src/core/rng.rs) from the stated seeds.
"""
from __future__ import annotations

import math

import numpy as np

from . import host as H

f32 = np.float32
ONE_MINUS_EPSILON = f32(float.fromhex("0x1.fffffep-1"))  # src/core/rng.rs:4


# ---------------------------------------------------------------------------
# PCG32 (src/core/rng.rs:25-76), vectorised over streams when needed
# ---------------------------------------------------------------------------
class PCG32:
    MULT = 0x5851F42D4C957F2D

    def __init__(self, seq=None):
        self.state, self.inc = 0x853C49E6748FEA9B, 0xDA3E39CB94B95BDB
        if seq is not None:
            self.set_sequence(seq)

    def set_sequence(self, seq):  # rng.rs:33-39
        self.state = 0
        self.inc = ((seq << 1) | 1) & 0xFFFFFFFFFFFFFFFF
        self.uniform_u32()
        self.state = (self.state + 0x853C49E6748FEA9B) & 0xFFFFFFFFFFFFFFFF
        self.uniform_u32()

    def uniform_u32(self):  # rng.rs:41-49
        old = self.state
        self.state = (old * self.MULT + self.inc) & 0xFFFFFFFFFFFFFFFF
        xs = (((old >> 18) ^ old) >> 27) & 0xFFFFFFFF
        rot = old >> 59
        return ((xs >> rot) | (xs << ((-rot) & 31))) & 0xFFFFFFFF

    def uniform_float(self):  # rng.rs:66-68
        return min(ONE_MINUS_EPSILON, f32(f32(self.uniform_u32()) * f32(2.3283064365386963e-10)))

    def floats(self, n):
        """n floats from this stream (vectorised LCG jump-free loop in numpy uint64)."""
        out = np.empty(n, np.uint32)
        st, inc, mult = np.uint64(self.state), np.uint64(self.inc), np.uint64(self.MULT)
        with np.errstate(over="ignore"):
            for i in range(n):
                old = st
                st = old * mult + inc
                xs = np.uint32(((old >> np.uint64(18)) ^ old) >> np.uint64(27))
                rot = np.uint32(old >> np.uint64(59))
                out[i] = (xs >> rot) | (xs << ((np.uint32(32) - rot) & np.uint32(31)))
        self.state = int(st)
        return np.minimum(ONE_MINUS_EPSILON, out.astype(f32) * f32(2.3283064365386963e-10))


def _hash_floats(n, seed):
    """Counter-based PCG-style hash -> n floats in [0,1): one independent PCG32 stream
    per element (sequence index = element index, seed folded into the state), first
    output.  Used where millions of values are needed (vertex displacement, ray batches)."""
    idx = np.arange(n, dtype=np.uint64)
    mult = np.uint64(PCG32.MULT)
    with np.errstate(over="ignore"):
        inc = (idx << np.uint64(1)) | np.uint64(1)
        st = np.zeros(n, np.uint64)
        st = st * mult + inc
        st = st + np.uint64(0x853C49E6748FEA9B) + np.uint64(seed) * np.uint64(0x9E3779B97F4A7C15)
        st = st * mult + inc
        old = st
        xs = (((old >> np.uint64(18)) ^ old) >> np.uint64(27)).astype(np.uint32)
        rot = (old >> np.uint64(59)).astype(np.uint32)
        out = (xs >> rot) | (xs << ((np.uint32(32) - rot) & np.uint32(31)))
    return np.minimum(ONE_MINUS_EPSILON, out.astype(f32) * f32(2.3283064365386963e-10))


# ---------------------------------------------------------------------------
# geometry helpers
# ---------------------------------------------------------------------------
def quad(p0, p1, p2, p3):
    """Two triangles (0,1,2),(0,2,3) like the reference's scene files (spheres-differentials-texfilt.pbrt:26)."""
    return np.array([p0, p1, p2, p3], f32), np.array([[0, 1, 2], [0, 2, 3]], np.uint32)


def box_mesh(lo, hi):
    x0, y0, z0 = lo
    x1, y1, z1 = hi
    P = np.array([[x0, y0, z0], [x1, y0, z0], [x1, y1, z0], [x0, y1, z0], [x0, y0, z1], [x1, y0, z1], [x1, y1, z1], [x0, y1, z1]], f32)
    I = np.array([[0, 2, 1], [0, 3, 2], [4, 5, 6], [4, 6, 7], [0, 1, 5], [0, 5, 4], [2, 3, 7], [2, 7, 6], [1, 2, 6], [1, 6, 5], [0, 4, 7], [0, 7, 3]], np.uint32)
    return P, I


def _value_noise(p, seed):
    """Trilinear value noise on the integer lattice, lattice values from _hash3."""
    pi = np.floor(p).astype(np.int64)
    pf = (p - pi).astype(f32)
    w = pf * pf * (f32(3) - f32(2) * pf)

    def lat(dx, dy, dz):
        x, y, z = pi[:, 0] + dx, pi[:, 1] + dy, pi[:, 2] + dz
        h = (x * 73856093) ^ (y * 19349663) ^ (z * 83492791) ^ (seed * 2654435761)
        h = (h & 0xFFFFFFFF).astype(np.uint64)
        h = (h ^ (h >> np.uint64(15))) * np.uint64(0x2C1B3C6D) & np.uint64(0xFFFFFFFF)
        h = (h ^ (h >> np.uint64(12))) * np.uint64(0x297A2D39) & np.uint64(0xFFFFFFFF)
        h = h ^ (h >> np.uint64(15))
        return (h.astype(np.float64) / 4294967296.0).astype(f32)

    c = [[[lat(i, j, k) for k in (0, 1)] for j in (0, 1)] for i in (0, 1)]
    wx, wy, wz = w[:, 0], w[:, 1], w[:, 2]
    x00 = c[0][0][0] * (1 - wx) + c[1][0][0] * wx
    x10 = c[0][1][0] * (1 - wx) + c[1][1][0] * wx
    x01 = c[0][0][1] * (1 - wx) + c[1][0][1] * wx
    x11 = c[0][1][1] * (1 - wx) + c[1][1][1] * wx
    y0 = x00 * (1 - wy) + x10 * wy
    y1 = x01 * (1 - wy) + x11 * wy
    return (y0 * (1 - wz) + y1 * wz).astype(f32)


def fbm(p, seed=1234, octaves=5):
    s = np.zeros(len(p), f32)
    amp, freq = f32(0.5), f32(1.0)
    for o in range(octaves):
        s += amp * (_value_noise(p * freq, seed + o) * f32(2) - f32(1))
        amp *= f32(0.5)
        freq *= f32(2.0)
    return s


def displaced_sphere(nlong, nlat, radius=1.0, amplitude=0.1, seed=1234, freq=4.0):
    """UV sphere with nlong x nlat quads (2 triangles each, shared vertices; the pole rows
    are degenerate-free triangle fans), displaced along the normal by amplitude*fbm.
    Returns P, indices, N (per-vertex normals of the displaced surface)."""
    th = (np.arange(nlat + 1, dtype=np.float64) / nlat) * math.pi
    ph = (np.arange(nlong, dtype=np.float64) / nlong) * 2.0 * math.pi
    T, Ph = np.meshgrid(th, ph, indexing="ij")
    d = np.stack([np.sin(T) * np.cos(Ph), np.sin(T) * np.sin(Ph), np.cos(T)], axis=-1).reshape(-1, 3)
    disp = fbm((d * freq).astype(f32) + f32(17.0), seed=seed)
    r = (radius + amplitude * disp.astype(np.float64))[:, None]
    P = (d * r).astype(f32)
    # collapse pole rows to single positions (keeps the mesh watertight)
    P[:nlong] = P[0]
    P[nlat * nlong:] = P[nlat * nlong]
    i = np.arange(nlat)[:, None]
    j = np.arange(nlong)[None, :]
    a = (i * nlong + j).reshape(-1)
    b = (i * nlong + (j + 1) % nlong).reshape(-1)
    c = ((i + 1) * nlong + j).reshape(-1)
    dd = ((i + 1) * nlong + (j + 1) % nlong).reshape(-1)
    I = np.concatenate([np.stack([a, c, dd], 1), np.stack([a, dd, b], 1)]).astype(np.uint32)
    # interleave so that the two triangles of a quad are adjacent
    nq = nlat * nlong
    I = np.stack([I[:nq], I[nq:]], axis=1).reshape(-1, 3)
    # area-weighted vertex normals
    p0, p1, p2 = (P[I[:, k]].astype(np.float64) for k in range(3))
    fn = np.cross(p1 - p0, p2 - p0)
    N = np.zeros((len(P), 3), np.float64)
    for k in range(3):
        np.add.at(N, I[:, k], fn)
    ln = np.linalg.norm(N, axis=1, keepdims=True)
    N = np.where(ln > 0, N / np.maximum(ln, 1e-30), d)
    return P, I, N.astype(f32)


# ---------------------------------------------------------------------------
# scenes
# ---------------------------------------------------------------------------
class SceneSetup:
    def __init__(self, name, flat, make_integrator, description):
        self.name, self.flat, self.make_integrator, self.description = name, flat, make_integrator, description


def spheres_scene(xres=400, yres=400, spp=64, maxdepth=5, sampler="sobol"):
    """S1 / config C1: the reference's spheres scene (src/scenes/spheres-differentials-texfilt.pbrt:1-37)
    as a path-traced scene: mirror + glass sphere over a matte ground quad, distant light."""
    b = H.SceneBuilder()
    cam_w2c = H.Transform.look_at((2, 2, 5), (0, -0.4, 0), (0, 1, 0))
    b.light_source("distant", **{"from": (0, 10, 0), "to": (0, 0, 0), "L": (3.141593, 3.141593, 3.141593)})
    b.attribute_begin()
    b.translate(0.25, 0, 0)
    b.material("matte", Kd=0.5)
    P, I = quad((-100, -1, -100), (400, -1, -100), (400, -1, 400), (-100, -1, 400))
    b.shape("trianglemesh", P=P, indices=I)
    b.attribute_end()
    b.translate(-1.3, 0, 0)
    b.material("mirror")
    b.shape("sphere", radius=1.0)
    b.translate(2.6, 0, 0)
    b.material("glass")
    b.shape("sphere", radius=1.0)
    flat = b.world_end()

    def make(spp_=spp, res=(xres, yres), maxdepth_=maxdepth, sampler_=sampler, strategy="spatial"):
        film = H.Film(res[0], res[1], "box")
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=30.0)
        return H.PathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy)

    return SceneSetup("S1-spheres", flat, make, "two spheres (mirror, glass) + ground quad, distant light, path maxdepth 5")


def cornell_scene(xres=1024, yres=1024, spp=256, maxdepth=8, sampler="sobol"):
    """S2 / config C2: Cornell box, diffuse quad area light (2 triangles => 2 lights), matte walls,
    two plastic boxes, lightsamplestrategy "power", gaussian 2x2 filter."""
    b = H.SceneBuilder()
    cam_w2c = H.Transform.look_at((278, 273, -800), (278, 273, 0), (0, 1, 0))
    white, red, green = (0.73, 0.73, 0.73), (0.65, 0.05, 0.05), (0.12, 0.45, 0.15)
    S = 555.0

    def wall(col, *pts):
        b.material("matte", Kd=col)
        P, I = quad(*pts)
        b.shape("trianglemesh", P=P, indices=I)

    wall(white, (0, 0, 0), (S, 0, 0), (S, 0, S), (0, 0, S))       # floor
    wall(white, (0, S, 0), (0, S, S), (S, S, S), (S, S, 0))       # ceiling
    wall(white, (0, 0, S), (S, 0, S), (S, S, S), (0, S, S))       # back
    wall(green, (0, 0, 0), (0, 0, S), (0, S, S), (0, S, 0))       # right (x=0)
    wall(red, (S, 0, 0), (S, S, 0), (S, S, S), (S, 0, S))         # left (x=S)
    b.attribute_begin()
    b.area_light_source("diffuse", L=(17, 12, 4))
    b.material("matte", Kd=0.0)
    P, I = quad((213, S - 0.1, 227), (343, S - 0.1, 227), (343, S - 0.1, 332), (213, S - 0.1, 332))
    b.shape("trianglemesh", P=P, indices=I)
    b.attribute_end()
    for (lo, hi, ang, tr) in (((0, 0, 0), (165, 165, 165), -18.0, (130, 0.05, 65)), ((0, 0, 0), (165, 330, 165), 15.0, (265, 0.05, 295))):
        b.attribute_begin()
        b.translate(*tr)
        b.rotate(ang, 0, 1, 0)
        b.material("plastic", Kd=(0.5, 0.5, 0.5), Ks=(0.25, 0.25, 0.25), roughness=0.1)
        P, I = box_mesh(lo, hi)
        b.shape("trianglemesh", P=P, indices=I)
        b.attribute_end()
    flat = b.world_end()

    def make(spp_=spp, res=(xres, yres), maxdepth_=maxdepth, sampler_=sampler, strategy="power", filt="gaussian"):
        film = H.Film(res[0], res[1], filt)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=40.0)
        return H.PathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy)

    return SceneSetup("S2-cornell", flat, make, "Cornell box, quad area light (2 triangle lights), matte + plastic, power light sampling")


def caustic_scene(xres=256, yres=256, spp=64, maxdepth=8, sampler="sobol"):
    """A caustic under a small light: a glass sphere on a matte floor in front of a matte back wall, lit by a small quad area
    light above and behind it.  Most of the light that reaches the floor under the sphere went through the glass, the case in which
    the path integrator converges slowly and the bdpt integrator's light subpaths help."""
    b = H.SceneBuilder()
    cam_w2c = H.Transform.look_at((0, 2.2, 5.5), (0, 0.4, 0), (0, 1, 0))
    b.material("matte", Kd=(0.7, 0.7, 0.7))
    P, I = quad((-4, 0, -4), (4, 0, -4), (4, 0, 4), (-4, 0, 4))
    b.shape("trianglemesh", P=P, indices=I)
    P, I = quad((-4, 0, -2), (-4, 4, -2), (4, 4, -2), (4, 0, -2))
    b.shape("trianglemesh", P=P, indices=I)
    b.attribute_begin()
    b.area_light_source("diffuse", L=(120, 110, 95))
    b.material("matte", Kd=0.0)
    P, I = quad((-0.2, 3.0, -0.6), (-0.2, 3.0, -0.2), (0.2, 3.0, -0.2), (0.2, 3.0, -0.6))
    b.shape("trianglemesh", P=P, indices=I)
    b.attribute_end()
    b.attribute_begin()
    b.translate(0, 0.8, 0)
    b.material("glass")
    b.shape("sphere", radius=0.8)
    b.attribute_end()
    flat = b.world_end()

    def make(spp_=spp, res=(xres, yres), maxdepth_=maxdepth, sampler_=sampler, strategy="power", filt="box", crop=(0.0, 1.0, 0.0, 1.0)):
        film = H.Film(res[0], res[1], filt, crop=crop)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=40.0)
        return H.PathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy)

    return SceneSetup("caustic", flat, make, "glass sphere on a matte floor under a small quad area light (caustic)")


def one_light_scene(light="spot", xres=48, yres=48, spp=16, maxdepth=4, sampler="sobol"):
    """A matte floor and back wall with a plastic box, lit by ONE light of kind `light`: "spot", "point", "sphere" (a two-sided sphere
    area light) or "sphere_one_sided" (one-sided: the reference's cone sample leaves the sampled normal at zero, so it emits through
    BSDF-sampled rays and light subpaths but not through light sampling).  For checking each light's sampling functions alone."""
    b = H.SceneBuilder()
    cam_w2c = H.Transform.look_at((0, 1.6, 5.0), (0, 0.6, 0), (0, 1, 0))
    b.material("matte", Kd=(0.6, 0.6, 0.6))
    P, I = quad((-4, 0, -4), (4, 0, -4), (4, 0, 4), (-4, 0, 4))
    b.shape("trianglemesh", P=P, indices=I)
    P, I = quad((-4, 0, -1.5), (-4, 4, -1.5), (4, 4, -1.5), (4, 0, -1.5))
    b.shape("trianglemesh", P=P, indices=I)
    b.material("plastic", Kd=(0.2, 0.4, 0.7), Ks=0.3, roughness=0.1)
    P, I = box_mesh((-0.9, 0.0, -0.6), (-0.1, 0.8, 0.2))
    b.shape("trianglemesh", P=P, indices=I)
    if light == "spot":
        b.light_source("spot", **{"from": (0.5, 2.8, 1.5), "to": (0.0, 0.0, -0.5), "coneangle": 35.0, "conedelta": 10.0, "I": (12, 11, 10)})
    elif light == "point":
        b.light_source("point", **{"from": (0.5, 2.5, 1.0), "I": (8, 8, 8)})
    else:
        b.attribute_begin()
        b.translate(0.8, 2.2, 0.6)
        b.area_light_source("diffuse", L=(6, 6, 5.5), twosided=(light == "sphere"))
        b.material("matte", Kd=0.0)
        b.shape("sphere", radius=0.3)
        b.attribute_end()
    flat = b.world_end()

    def make(spp_=spp, res=(xres, yres), maxdepth_=maxdepth, sampler_=sampler, strategy="power", filt="box"):
        film = H.Film(res[0], res[1], filt)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=45.0)
        return H.PathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy)

    return SceneSetup(f"one-light-{light}", flat, make, f"floor, wall and box under one {light} light")


def displaced_sphere_scene(nlong=1024, nlat=512, xres=1920, yres=1080, spp=512, maxdepth=5, sampler="sobol"):
    """S3 / config C3: nlong*nlat*2 triangles (1 048 576 at the defaults) on a displaced sphere with
    per-vertex normals, half plastic / half copper metal by octant parity, ground quad, one quad
    area light + one point light."""
    b = H.SceneBuilder()
    cam_w2c = H.Transform.look_at((0.0, -3.6, 1.4), (0, 0, 0.05), (0, 0, 1))
    P, I, N = displaced_sphere(nlong, nlat, 1.0, 0.1, 1234)
    cen = (P[I[:, 0]] + P[I[:, 1]] + P[I[:, 2]]) / f32(3)
    octant_parity = ((cen[:, 0] > 0).astype(int) + (cen[:, 1] > 0).astype(int) + (cen[:, 2] > 0).astype(int)) % 2
    for par, (mat, kw) in enumerate((("plastic", dict(Kd=(0.25, 0.25, 0.25), Ks=(0.25, 0.25, 0.25), roughness=0.1)), ("metal", dict(roughness=0.01)))):
        b.material(mat, **kw)
        b.shape("trianglemesh", P=P, indices=I[octant_parity == par], N=N)
    b.material("matte", Kd=(0.4, 0.4, 0.4))
    Pq, Iq = quad((-30, -30, -1.15), (30, -30, -1.15), (30, 30, -1.15), (-30, 30, -1.15))
    b.shape("trianglemesh", P=Pq, indices=Iq)
    b.attribute_begin()
    b.area_light_source("diffuse", L=(30, 30, 30))
    b.material("matte", Kd=0.0)
    Pl, Il = quad((-1.5, -1.5, 4.0), (-1.5, 1.5, 4.0), (1.5, 1.5, 4.0), (1.5, -1.5, 4.0))
    b.shape("trianglemesh", P=Pl, indices=Il)
    b.attribute_end()
    # positioned with the CTM: the reference's `from` handling has the (P.x, P.y, P.x) quirk (point.rs:103)
    b.attribute_begin()
    b.translate(3.0, -4.0, 3.0)
    b.light_source("point", I=(20, 18, 15))
    b.attribute_end()
    flat = b.world_end()

    def make(spp_=spp, res=(xres, yres), maxdepth_=maxdepth, sampler_=sampler, strategy="power", filt="box"):
        film = H.Film(res[0], res[1], filt)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=35.0)
        return H.PathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy)

    ntri = len(I) + 4
    return SceneSetup(f"S3-displaced-sphere-{ntri}", flat, make,
                      f"{ntri}-triangle displaced sphere (plastic/metal) + ground + quad area light + point light")


def glass_knot_scene(nu=2048, nv=512, xres=1024, yres=1024, spp=2048, maxdepth=32, sampler="sobol"):
    """S5 / config C5 stand-in: glass (eta 1.5) torus knot tube of nu*nv*2 triangles on a matte ground
    under a small bright quad light."""
    b = H.SceneBuilder()
    cam_w2c = H.Transform.look_at((0.0, -7.5, 4.5), (0, 0, 0.6), (0, 0, 1))
    u = np.arange(nu, dtype=np.float64) / nu * 2 * math.pi
    p, q = 2, 3
    rr = 2.0 + np.cos(q * u)
    c = np.stack([rr * np.cos(p * u), rr * np.sin(p * u), -np.sin(q * u) * 1.0 + 1.6], axis=1) * np.array([0.8, 0.8, 0.8])
    t = np.roll(c, -1, axis=0) - np.roll(c, 1, axis=0)
    t /= np.linalg.norm(t, axis=1, keepdims=True)
    up = np.array([0.0, 0.0, 1.0])
    n1 = np.cross(t, up)
    n1 /= np.linalg.norm(n1, axis=1, keepdims=True)
    n2 = np.cross(t, n1)
    v = np.arange(nv, dtype=np.float64) / nv * 2 * math.pi
    ring = np.cos(v)[None, :, None] * n1[:, None, :] + np.sin(v)[None, :, None] * n2[:, None, :]
    base = (c[:, None, :] + 0.32 * ring).reshape(-1, 3)
    disp = fbm((base * 3.0).astype(f32), seed=77).astype(np.float64)[:, None]
    P = (base + 0.03 * disp * ring.reshape(-1, 3)).astype(f32)
    i = np.arange(nu)[:, None]
    j = np.arange(nv)[None, :]
    a = (i * nv + j).reshape(-1)
    bb = (((i + 1) % nu) * nv + j).reshape(-1)
    cc = (i * nv + (j + 1) % nv).reshape(-1)
    dd = (((i + 1) % nu) * nv + (j + 1) % nv).reshape(-1)
    I = np.stack([np.stack([a, bb, dd], 1), np.stack([a, dd, cc], 1)], axis=1).reshape(-1, 3).astype(np.uint32)
    b.material("glass", index=1.5)
    b.shape("trianglemesh", P=P, indices=I)
    b.material("matte", Kd=(0.5, 0.5, 0.5))
    Pq, Iq = quad((-30, -30, 0), (30, -30, 0), (30, 30, 0), (-30, 30, 0))
    b.shape("trianglemesh", P=Pq, indices=Iq)
    b.attribute_begin()
    b.area_light_source("diffuse", L=(400, 400, 400))
    b.material("matte", Kd=0.0)
    Pl, Il = quad((-0.4, -0.4, 9.0), (-0.4, 0.4, 9.0), (0.4, 0.4, 9.0), (0.4, -0.4, 9.0))
    b.shape("trianglemesh", P=Pl, indices=Il)
    b.attribute_end()
    flat = b.world_end()

    def make(spp_=spp, res=(xres, yres), maxdepth_=maxdepth, sampler_=sampler, strategy="power", filt="box"):
        film = H.Film(res[0], res[1], filt)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=40.0)
        return H.PathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, rrthreshold=1.0, lightsamplestrategy=strategy)

    return SceneSetup(f"S5-glass-knot-{len(I) + 4}", flat, make, "glass torus knot, caustic light, maxdepth 32")


def fog_box_scene(xres=128, yres=128, spp=16, maxdepth=5, sampler="sobol", camera_in_fog=True, instanced=False):
    """Participating media for the volpath integrator (SURVEY.md s8 f4): a closed box of matte walls filled with a thin homogeneous medium
    ("haze", the camera sits in it), a dense forward-scattering medium ("smoke", g = 0.6) inside a material-less cube (a pure medium
    boundary, Material "none"), a glass sphere whose inside is a coloured absorbing medium ("dye"), a mirror quad, one quad area light and
    one point light.  Every medium-transition rule of primitive.rs:134-140 and both transmittance loops (VisibilityTester::tr through the
    material-less cube, Scene::intersect_tr) are on the light paths of this scene.  `instanced`: the smoke cube is an ObjectInstance."""
    b = H.SceneBuilder()
    cam_w2c = H.Transform.look_at((0.0, -3.4, 1.0), (0.0, 0.0, 0.9), (0, 0, 1))
    b.make_named_medium("haze", sigma_a=(0.01, 0.012, 0.02), sigma_s=(0.12, 0.12, 0.14), g=0.1, scale=1.0)
    b.make_named_medium("smoke", sigma_a=(0.3, 0.3, 0.3), sigma_s=(2.5, 2.6, 2.8), g=0.6, scale=1.5)
    b.make_named_medium("dye", sigma_a=(0.2, 1.5, 2.5), sigma_s=(0.05, 0.05, 0.05), g=0.0)
    outer = "haze" if camera_in_fog else ""
    b.medium_interface("", outer)  # the outermost state: what Camera.medium resolves to at WorldEnd

    def wall(col, *pts, mat="matte", **kw):
        b.material(mat, **({"Kd": col} if mat == "matte" else kw))
        P, I = quad(*pts)
        b.shape("trianglemesh", P=P, indices=I)

    # the floor is created under the outermost state (inside "", outside haze): a transition -- rays leaving on its normal side (+z) are in the haze
    wall((0.7, 0.7, 0.7), (-2, -4, 0), (2, -4, 0), (2, 2, 0), (-2, 2, 0))        # floor (normal +z)
    b.attribute_begin()
    b.medium_interface(outer, outer)  # both sides the same medium: NOT a transition, the ray keeps its medium (primitive.rs:138)
    wall((0.7, 0.7, 0.7), (-2, -4, 2.5), (-2, 2, 2.5), (2, 2, 2.5), (2, -4, 2.5))  # ceiling
    wall((0.7, 0.7, 0.7), (-2, 2, 0), (2, 2, 0), (2, 2, 2.5), (-2, 2, 2.5))      # back
    wall((0.6, 0.1, 0.1), (-2, -4, 0), (-2, 2, 0), (-2, 2, 2.5), (-2, -4, 2.5))  # left
    wall((0.1, 0.5, 0.15), (2, -4, 0), (2, -4, 2.5), (2, 2, 2.5), (2, 2, 0))     # right
    wall((0.7, 0.7, 0.7), (-2, -4, 0), (-2, -4, 2.5), (2, -4, 2.5), (2, -4, 0))  # behind the camera
    wall(None, (-1.9, 1.2, 0.4), (-1.2, 1.95, 0.4), (-1.2, 1.95, 1.9), (-1.9, 1.2, 1.9), mat="mirror", Kr=0.9)
    b.attribute_end()
    b.attribute_begin()
    b.medium_interface(outer, outer)
    b.area_light_source("diffuse", L=(14, 13, 11))
    b.material("matte", Kd=0.0)
    P, I = quad((-0.5, -0.5, 2.49), (-0.5, 0.5, 2.49), (0.5, 0.5, 2.49), (0.5, -0.5, 2.49))
    b.shape("trianglemesh", P=P, indices=I)
    b.attribute_end()
    b.light_source("point", **{"from": (1.4, -1.5, 1.4), "I": (3.0, 3.0, 3.5)})
    # dense smoke inside a material-less cube
    b.attribute_begin()
    b.medium_interface("smoke", outer)
    b.material("none")
    P, I = box_mesh((-1.2, -0.2, 0.05), (-0.2, 0.8, 1.05))
    if instanced:
        b.object_begin("smokebox")
        b.shape("trianglemesh", P=P, indices=I)
        b.object_end()
        b.object_instance("smokebox")
    else:
        b.shape("trianglemesh", P=P, indices=I)
    b.attribute_end()
    # glass sphere filled with dye
    b.attribute_begin()
    b.medium_interface("dye", outer)
    b.material("glass", index=1.5)
    b.translate(0.8, 0.1, 0.55)
    b.shape("sphere", radius=0.5)
    b.attribute_end()
    cam_medium = b.camera_medium()
    flat = b.world_end()

    def make(spp_=spp, res=(xres, yres), maxdepth_=maxdepth, sampler_=sampler, strategy="uniform", filt="box", rrthreshold=1.0, integrator="volpath"):
        film = H.Film(res[0], res[1], filt)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=55.0)
        if integrator == "path":
            return H.PathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy, rrthreshold=rrthreshold)
        return H.VolPathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy, rrthreshold=rrthreshold,
                                   camera_medium=cam_medium)

    return SceneSetup("V1-fog-box", flat, make, "matte box in haze, smoke cube (material-less boundary), dye-filled glass sphere, mirror; volpath")


def smoke_density(nx=14, ny=11, nz=9, seed=7):
    """A seeded smoke field for GridDensityMedium, density[(z * ny + y) * nx + x]: fbm noise shaped into a blob, an empty (zero) border
    of one voxel on every face and two empty spherical pockets inside."""
    z, y, x = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    p = np.stack([(x + 0.5) / nx, (y + 0.5) / ny, (z + 0.5) / nz], -1).reshape(-1, 3).astype(f32)
    r = np.linalg.norm((p - f32(0.5)) * np.array([1.0, 1.1, 1.3], f32), axis=1)
    d = np.clip(f32(1.6) * (f32(0.55) - r) + f32(0.9) * fbm(p * f32(3.0), seed=seed, octaves=3), 0.0, None).astype(f32) * f32(4.0)
    for c, rad in (((0.35, 0.45, 0.5), 0.16), ((0.65, 0.6, 0.4), 0.12)):
        d[np.linalg.norm(p - np.array(c, f32), axis=1) < rad] = 0.0
    d = d.reshape(nz, ny, nx)
    d[0, :, :] = d[-1, :, :] = d[:, 0, :] = d[:, -1, :] = d[:, :, 0] = d[:, :, -1] = 0.0
    return np.ascontiguousarray(d.reshape(-1), f32)


def smoke_box_scene(xres=128, yres=128, spp=16, maxdepth=5, sampler="sobol", camera_in_smoke=False, instanced=False, textured=False, density=None,
                    seed=7, smoke=True):
    """Heterogeneous media for the volpath integrator: the room of fog_box_scene (matte walls, a thin homogeneous "haze", a mirror, one
    quad area light, one point light) with a GridDensityMedium "smoke" (grid.rs) of 14 x 11 x 9 voxels from smoke_density(seed).  The
    grid's box is rotated and scaled non-uniformly (CTM x Translate(p0) x Scale(p1 - p0), with p0 / p1 not the unit box), and its
    material-less boundary mesh -- made under the same transformation -- reaches past the grid box on its -x side and cuts the box off
    on its +x side.  `camera_in_smoke`: the camera sits inside the boundary, in the smoke (Camera.medium = smoke).  `instanced`: the
    boundary is an ObjectInstance.  `textured`: the back wall is a checkerboard-textured matte.  `density`: replaces the field (same
    14 x 11 x 9 layout), e.g. all zeros.  `smoke=False`: the same scene with vacuum inside the boundary instead of the grid medium."""
    nx, ny, nz = 14, 11, 9
    dens = smoke_density(nx, ny, nz, seed) if density is None else np.asarray(density, f32)
    b = H.SceneBuilder()
    b.make_named_medium("haze", sigma_a=(0.01, 0.012, 0.02), sigma_s=(0.12, 0.12, 0.14), g=0.1)
    b.medium_interface("", "haze")

    def wall(col, *pts, mat="matte", **kw):
        b.material(mat, **({"Kd": col} if mat == "matte" else kw))
        P, I = quad(*pts)
        b.shape("trianglemesh", P=P, indices=I)

    wall((0.7, 0.7, 0.7), (-2, -4, 0), (2, -4, 0), (2, 2, 0), (-2, 2, 0))        # floor: a transition into the haze
    b.attribute_begin()
    b.medium_interface("haze", "haze")
    wall((0.7, 0.7, 0.7), (-2, -4, 2.5), (-2, 2, 2.5), (2, 2, 2.5), (2, -4, 2.5))  # ceiling
    if textured:
        from . import textures as T
        b.material("matte", Kd=T.Tex.checkerboard(T.Mapping2D.planar((0.8, 0, 0), (0, 0, 0.8), 0.1, 0.2), np.array([0.8, 0.8, 0.8], f32),
                                                  np.array([0.2, 0.3, 0.6], f32), "none"))
        P, I = quad((-2, 2, 0), (2, 2, 0), (2, 2, 2.5), (-2, 2, 2.5))
        b.shape("trianglemesh", P=P, indices=I)
    else:
        wall((0.7, 0.7, 0.7), (-2, 2, 0), (2, 2, 0), (2, 2, 2.5), (-2, 2, 2.5))      # back
    wall((0.6, 0.1, 0.1), (-2, -4, 0), (-2, 2, 0), (-2, 2, 2.5), (-2, -4, 2.5))  # left
    wall((0.1, 0.5, 0.15), (2, -4, 0), (2, -4, 2.5), (2, 2, 2.5), (2, 2, 0))     # right
    wall((0.7, 0.7, 0.7), (-2, -4, 0), (-2, -4, 2.5), (2, -4, 2.5), (2, -4, 0))  # behind the camera
    wall(None, (1.9, 1.2, 0.4), (1.2, 1.95, 0.4), (1.2, 1.95, 1.9), (1.9, 1.2, 1.9), mat="mirror", Kr=0.9)
    b.attribute_end()
    b.attribute_begin()
    b.medium_interface("haze", "haze")
    b.area_light_source("diffuse", L=(14, 13, 11))
    b.material("matte", Kd=0.0)
    P, I = quad((-0.5, -0.5, 2.49), (-0.5, 0.5, 2.49), (0.5, 0.5, 2.49), (0.5, -0.5, 2.49))
    b.shape("trianglemesh", P=P, indices=I)
    b.attribute_end()
    b.light_source("point", **{"from": (1.4, -1.5, 1.4), "I": (3.0, 3.0, 3.5)})
    b.attribute_begin()
    b.translate(-0.8, -0.6, 0.15)
    b.rotate(25.0, 0, 0, 1)
    b.rotate(-10.0, 1, 0, 0)
    b.scale(1.5, 1.3, 1.7)
    if smoke:
        b.make_named_medium("smoke", type="heterogeneous", sigma_a=(0.5, 0.25, 0.125), sigma_s=(2.0, 2.25, 2.375), g=0.5, scale=1.0,
                            density=dens, nx=nx, ny=ny, nz=nz, p0=(-0.1, 0.0, 0.05), p1=(1.0, 1.0, 0.95))
    ctm = b.ctm
    b.medium_interface("smoke" if smoke else "", "haze")
    b.material("none")
    P, I = box_mesh((-0.3, -0.05, 0.0), (0.85, 1.08, 1.0))
    if instanced:
        b.object_begin("smokebox")
        b.shape("trianglemesh", P=P, indices=I)
        b.object_end()
        b.object_instance("smokebox")
    else:
        b.shape("trianglemesh", P=P, indices=I)
    b.attribute_end()
    if camera_in_smoke:
        eye = (ctm.m @ np.array([0.3, 0.15, 0.5, 1.0], f32))[:3]
        cam_w2c = H.Transform.look_at(tuple(eye), (0.6, 1.9, 1.1), (0, 0, 1))
        b.medium_interface("", "smoke" if smoke else "")
    else:
        cam_w2c = H.Transform.look_at((0.0, -3.4, 1.0), (0.0, 0.0, 0.9), (0, 0, 1))
    cam_medium = b.camera_medium()
    flat = b.world_end()

    def make(spp_=spp, res=(xres, yres), maxdepth_=maxdepth, sampler_=sampler, strategy="uniform", filt="box", rrthreshold=1.0, pixelbounds=None):
        film = H.Film(res[0], res[1], filt)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=55.0)
        return H.VolPathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy, rrthreshold=rrthreshold,
                                   camera_medium=cam_medium, pixelbounds=pixelbounds)

    return SceneSetup("V2-smoke-box", flat, make, "grid-density smoke (rotated, non-uniformly scaled, clipped boundary) in a hazy room; volpath")


def _test_image(w=96, h=64, channels=3):
    """A small deterministic image (NOT a power of two: MIPMap::new resamples it): stripes, a ramp and a few bright texels."""
    y, x = np.mgrid[0:h, 0:w]
    img = np.zeros((h, w, 3), f32)
    img[..., 0] = 0.15 + 0.6 * ((x // 6) % 2)
    img[..., 1] = 0.1 + 0.8 * (y / f32(h - 1))
    img[..., 2] = 0.25 + 0.5 * (((x + y) // 9) % 2)
    img[(x % 17 == 3) & (y % 11 == 5)] = (2.5, 2.0, 1.5)
    return img if channels == 3 else img.mean(axis=2, keepdims=True).astype(f32)


def textured_scene(xres=160, yres=120, spp=8, maxdepth=5, sampler="sobol", instanced=True):
    """SURVEY.md s8 f3 in one scene: every texture kind (image maps with EWA and trilinear filtering under the three wrap modes, 2D / 3D
    checkerboards, dots, fbm, wrinkled, marble, windy, uv, bilerp, scale, mix), every mapping (uv, planar, spherical, cylindrical, 3D),
    float and spectrum textures as parameters of all seven materials (incl. uber with an opacity texture and substrate), bump maps on a
    sphere and on a triangle mesh with per-vertex normals, and a textured object instance.  Rendered by the path, volpath, whitted and
    directlighting integrators (ray differentials through the mirror and the glass sphere only exist under the latter two)."""
    from . import textures as T
    Tex, M2 = T.Tex, T.Mapping2D
    b = H.SceneBuilder()
    cam_w2c = H.Transform.look_at((0.3, 2.4, 6.2), (0.0, 0.6, 0.0), (0, 1, 0))
    rgb_img = T.MipMap(_test_image(), do_trilinear=False, max_anisotropy=8.0, wrap="repeat")
    tri_img = T.MipMap(_test_image(64, 64), do_trilinear=True, wrap="clamp")
    flt_img = T.MipMap(_test_image(40, 24, channels=1), do_trilinear=False, max_anisotropy=4.0, wrap="black")

    def tex3(sc):
        # noise() takes `floor(x) as usize` (texture.rs:332-334): a negative coordinate saturates to cell 0 with a negative offset and the
        # quintic weights explode (mirrored, tests/test_oracle_textures.py) -- so the scene keeps its 3D textures in the positive octant
        return H.Transform.translate((40.0, 40.0, 40.0)) * H.Transform.scale(sc, sc, sc)

    b.light_source("point", **{"from": (-3.0, 4.5, 3.0), "I": (30.0, 28.0, 26.0)})
    b.light_source("distant", **{"from": (2, 6, 4), "to": (0, 0, 0), "L": (1.2, 1.2, 1.3)})
    b.attribute_begin()
    b.area_light_source("diffuse", L=(9, 9, 8))
    b.material("matte", Kd=0.0)
    P, I = quad((1.0, 4.0, -1.0), (2.2, 4.0, -1.0), (2.2, 4.0, 0.2), (1.0, 4.0, 0.2))
    b.shape("trianglemesh", P=P, indices=I)
    b.attribute_end()
    # ground: EWA-filtered image map through the mesh's uv ("st"), scaled so that it minifies towards the horizon
    P, I = quad((-12, 0, -14), (12, 0, -14), (12, 0, 8), (-12, 0, 8))
    uvq = np.array([[0, 0], [1, 0], [1, 1], [0, 1]], f32)
    b.material("matte", Kd=Tex.imagemap(M2.uv(12.0, 11.0, 0.25, 0.1), rgb_img), sigma=Tex.mix(0.0, 40.0, Tex.fbm(tex3(0.7), 4, 0.6)))
    b.shape("trianglemesh", P=P, indices=I, uv=uvq)
    # back wall: closed-form antialiased checkerboard (planar mapping) of marble and a constant
    P, I = quad((-7, 0, -6), (7, 0, -6), (7, 6, -6), (-7, 6, -6))
    marble = Tex.marble(tex3(1.5), 6, 0.5, 1.2, 0.3)
    b.material("matte", Kd=Tex.checkerboard(M2.planar((0.8, 0, 0), (0, 0.8, 0), 0.1, 0.2), marble, np.array([0.15, 0.3, 0.55], f32), "closedform"))
    b.shape("trianglemesh", P=P, indices=I)
    # plastic sphere: uv checkerboard as Kd, dots as roughness, wrinkled bump map
    b.attribute_begin()
    b.translate(-2.3, 1.0, 0.2)
    b.material("plastic", Kd=Tex.checkerboard(M2.uv(10.0, 6.0), np.array([0.8, 0.2, 0.15], f32), Tex.uv(M2.uv(3.0, 3.0)), "none"),
               Ks=0.3, roughness=Tex.dots(M2.uv(14.0, 9.0), outside=0.05, inside=0.4), bumpmap=Tex.scale(Tex.wrinkled(tex3(3.0), 5, 0.55), 0.05))
    b.shape("sphere", radius=1.0)
    b.attribute_end()
    # uber sphere: opacity from a 3D checkerboard (partly see-through), Kd spherical image map, Kr / Kt constants
    b.attribute_begin()
    b.translate(0.0, 0.9, 1.6)
    b.material("uber", Kd=Tex.imagemap(M2.spherical(H.Transform.translate((0.0, 0.9, 1.6)).inverse()), tri_img), Ks=0.2, Kr=0.15, Kt=0.1,
               opacity=Tex.checkerboard3d(tex3(2.5), np.array([1.0, 1.0, 1.0], f32), np.array([0.25, 0.35, 0.3], f32)), roughness=0.08, index=1.4)
    b.shape("sphere", radius=0.9)
    b.attribute_end()
    # substrate on a triangle mesh with per-vertex normals and uvs: trilinear image map as Kd, float image map as bump
    Pm, Im, Nm = displaced_sphere(40, 20, radius=0.9, amplitude=0.05)[:3]
    th = np.arctan2(Pm[:, 2], Pm[:, 0]).astype(f32)
    uvm = np.stack([(th / f32(2 * np.pi) + f32(0.5)), np.clip(Pm[:, 1] / f32(1.9) + f32(0.5), 0, 1)], axis=1).astype(f32)
    b.attribute_begin()
    b.translate(2.4, 1.0, 0.3)
    b.material("substrate", Kd=Tex.imagemap(M2.uv(3.0, 2.0), tri_img), Ks=np.array([0.05, 0.06, 0.05], f32), uroughness=0.1,
               vroughness=Tex.mix(0.02, 0.3, Tex.imagemap(M2.uv(2.0, 2.0), flt_img)), bumpmap=Tex.scale(Tex.imagemap(M2.uv(4.0, 4.0, 0.1, 0.0), flt_img), 0.08))
    b.shape("trianglemesh", P=Pm, indices=Im, N=Nm, uv=uvm)
    b.attribute_end()
    # glass sphere with a bilerp tint on Kt; a mirror quad whose Kr is a windy spectrum texture; a metal box with a textured roughness
    b.attribute_begin()
    b.translate(-0.9, 0.55, 3.2)
    b.material("glass", Kr=1.0, Kt=Tex.bilerp(M2.uv(), (1.0, 0.9, 0.8), (0.8, 1.0, 0.85), (0.85, 0.85, 1.0), (1.0, 1.0, 1.0)), index=1.5)
    b.shape("sphere", radius=0.55)
    b.attribute_end()
    P, I = quad((3.2, 0.0, -3.5), (6.0, 0.0, -1.0), (6.0, 3.0, -1.0), (3.2, 3.0, -3.5))
    b.material("mirror", Kr=Tex.mix(0.55, 0.95, Tex.windy(tex3(0.8))))
    b.shape("trianglemesh", P=P, indices=I)
    P, I = box_mesh((-5.5, 0.0, -3.0), (-4.0, 1.6, -1.5))
    b.material("metal", roughness=Tex.checkerboard(M2.cylindrical(H.Transform.translate((-4.75, 0.0, -2.25)).inverse()), 0.01, 0.25, "none"))
    b.shape("trianglemesh", P=P, indices=I)
    # a textured object, instanced twice (the second one rotated and scaled)
    Pb, Ib = box_mesh((-0.4, 0.0, -0.4), (0.4, 0.8, 0.4))
    crate = Tex.scale(Tex.imagemap(M2.planar((1.1, 0, 0), (0, 1.1, 0.4)), rgb_img), np.array([0.9, 0.8, 0.7], f32))
    if instanced:
        b.object_begin("crate")
        b.material("matte", Kd=crate)
        b.shape("trianglemesh", P=Pb, indices=Ib)
        b.object_end()
        for k, (tx, tz, rot, sc) in enumerate(((1.2, 3.4, 25.0, 1.0), (3.6, 2.4, -40.0, 1.3))):
            b.attribute_begin()
            b.translate(tx, 0.0, tz)
            b.rotate(rot, 0, 1, 0)
            b.scale(sc, sc, sc)
            b.object_instance("crate")
            b.attribute_end()
    else:
        b.attribute_begin()
        b.translate(1.2, 0.0, 3.4)
        b.material("matte", Kd=crate)
        b.shape("trianglemesh", P=Pb, indices=Ib)
        b.attribute_end()
    flat = b.world_end()
    flat.keepalive = (rgb_img, tri_img, flt_img)

    def make(spp_=spp, res=(xres, yres), maxdepth_=maxdepth, sampler_=sampler, strategy="power", integrator="path", filt="box", lensradius=0.0):
        film = H.Film(res[0], res[1], filt)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=42.0, lensradius=lensradius, focaldistance=6.5)
        smp = H.Sampler(sampler_, spp_)
        if integrator == "path":
            return H.PathIntegrator(cam, film, smp, maxdepth=maxdepth_, lightsamplestrategy=strategy)
        if integrator == "volpath":
            return H.VolPathIntegrator(cam, film, smp, maxdepth=maxdepth_, lightsamplestrategy=strategy)
        if integrator == "whitted":
            return H.WhittedIntegrator(cam, film, smp, maxdepth=maxdepth_)
        return H.DirectLightingIntegrator(cam, film, smp, maxdepth=maxdepth_, strategy=integrator.split(":")[1] if ":" in integrator else "all")

    return SceneSetup("T1-textures", flat, make, "every texture kind / mapping / textured material, bump maps, a textured instance")


def small_mixed_scene(n=24, seed=5):
    """Test-sized scene touching every material/light/shape kind on the hot path."""
    b = H.SceneBuilder()
    cam_w2c = H.Transform.look_at((0.0, -5.0, 2.0), (0, 0, 0.3), (0, 0, 1))
    P, I, N = displaced_sphere(n, n // 2, 0.8, 0.08, seed)
    mats = [("matte", dict(Kd=(0.6, 0.3, 0.2), sigma=20.0)), ("plastic", dict(Kd=(0.2, 0.3, 0.6), Ks=0.3, roughness=0.05)),
            ("metal", dict(roughness=0.05)), ("glass", dict(index=1.5)), ("mirror", dict(Kr=0.8)), ("glass", dict(uroughness=0.1, vroughness=0.1))]
    for k, (m, kw) in enumerate(mats):
        b.attribute_begin()
        b.translate(-3.0 + 1.2 * k, 0.3 * (k % 2), 0.0)
        b.material(m, **kw)
        if k % 2 == 0:
            b.shape("trianglemesh", P=P, indices=I, N=N)
        else:
            b.shape("trianglemesh", P=P, indices=I)
        b.attribute_end()
    b.attribute_begin()
    b.translate(0, 1.8, 0.2)
    b.material("glass")
    b.shape("sphere", radius=0.7)
    b.attribute_end()
    b.material("matte", Kd=(0.5, 0.5, 0.5))
    Pq, Iq = quad((-10, -10, -0.9), (10, -10, -0.9), (10, 10, -0.9), (-10, 10, -0.9))
    b.shape("trianglemesh", P=Pq, indices=Iq)
    b.attribute_begin()
    b.area_light_source("diffuse", L=(25, 25, 22))
    Pl, Il = quad((-1, -1, 4.0), (-1, 1, 4.0), (1, 1, 4.0), (1, -1, 4.0))
    b.shape("trianglemesh", P=Pl, indices=Il)
    b.attribute_end()
    b.attribute_begin()
    b.translate(-3.0, -3.0, 3.0)
    b.light_source("point", I=(8, 8, 8))
    b.attribute_end()
    b.light_source("distant", **{"from": (1, -1, 2), "to": (0, 0, 0), "L": (0.6, 0.6, 0.7)})
    b.light_source("infinite", L=(0.15, 0.18, 0.25))
    flat = b.world_end()

    def make(spp_=16, res=(96, 64), maxdepth_=5, sampler_="sobol", strategy="power", filt="gaussian"):
        film = H.Film(res[0], res[1], filt)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=45.0)
        return H.PathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy)

    return SceneSetup("mixed-small", flat, make, "all hot-path materials/lights/shapes at test size")


def sphere_lights_scene(enclosing=True, tessellated=False):
    """Sphere area lights (Sphere::sample_interaction / pdf_wi, sphere.rs:313-395): a small two-sided sphere light seen from
    outside (cone sampling), a one-sided one (the reference's cone branch leaves the sampled normal at zero, so it only emits
    through BSDF-sampled rays and camera hits), and -- `enclosing` -- a large two-sided sphere light around the whole scene
    (every shading point is inside it: uniform-area branch).  `tessellated`: the small two-sided light as a 64x32 triangle
    mesh with the same emission instead (cross-check: same image in expectation)."""
    b = H.SceneBuilder()
    cam_w2c = H.Transform.look_at((0.0, -6.0, 2.5), (0, 0, 0.6), (0, 0, 1))
    b.material("matte", Kd=(0.5, 0.5, 0.5))
    Pq, Iq = quad((-8, -8, 0), (8, -8, 0), (8, 8, 0), (-8, 8, 0))
    b.shape("trianglemesh", P=Pq, indices=Iq)
    b.attribute_begin()
    b.translate(-1.2, 0.5, 0.7)
    b.material("plastic", Kd=(0.2, 0.4, 0.7), Ks=0.3, roughness=0.1)
    b.shape("sphere", radius=0.7)
    b.attribute_end()
    b.attribute_begin()
    b.translate(1.3, 0.2, 0.6)
    b.material("metal", roughness=0.08)
    P, I, N = displaced_sphere(24, 12, 0.6, 0.05, 3)
    b.shape("trianglemesh", P=P, indices=I, N=N)
    b.attribute_end()
    b.attribute_begin()  # two-sided sphere light, outside case
    b.translate(0.0, 0.5, 2.6)
    b.area_light_source("diffuse", L=(14, 13, 11), twosided=True)
    b.material("matte", Kd=0.0)
    if tessellated:
        Pt, It, _ = displaced_sphere(64, 32, 0.35, 0.0, 1)
        b.shape("trianglemesh", P=Pt, indices=It)
    else:
        b.shape("sphere", radius=0.35)
    b.attribute_end()
    b.attribute_begin()  # one-sided sphere light
    b.translate(-2.5, -1.0, 1.6)
    b.area_light_source("diffuse", L=(3, 6, 9))
    b.material("matte", Kd=0.0)
    b.shape("sphere", radius=0.3)
    b.attribute_end()
    if enclosing:
        b.attribute_begin()
        b.area_light_source("diffuse", L=(0.12, 0.14, 0.2), twosided=True)
        b.material("matte", Kd=0.0)
        b.shape("sphere", radius=30.0)
        b.attribute_end()
    flat = b.world_end()

    def make(spp_=16, res=(96, 64), maxdepth_=5, sampler_="sobol", strategy="power", filt="box"):
        film = H.Film(res[0], res[1], filt)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=42.0)
        return H.PathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy)

    return SceneSetup("sphere-lights", flat, make, "sphere area lights: cone-sampled, one-sided, enclosing")


def _plant_mesh(n_blades=10, seg=6, seed=17):
    """A small procedural 'plant': n_blades curved two-sided blades of 2*seg triangles each, fanned around the z axis."""
    rng = PCG32(seed)
    u = rng.floats(4 * n_blades)
    P, I = [], []
    for b in range(n_blades):
        ang = 2 * math.pi * (b + 0.5 * float(u[4 * b])) / n_blades
        lean, height, width = 0.3 + 0.5 * float(u[4 * b + 1]), 0.7 + 0.6 * float(u[4 * b + 2]), 0.05 + 0.05 * float(u[4 * b + 3])
        ca, sa = math.cos(ang), math.sin(ang)
        base = len(P)
        for k in range(seg + 1):
            t = k / seg
            r, z, w = lean * t * t, height * t, width * (1 - 0.9 * t)
            cx, cy = r * ca, r * sa
            P.append((cx - w * sa, cy + w * ca, z)); P.append((cx + w * sa, cy - w * ca, z))
        for k in range(seg):
            a = base + 2 * k
            I.append((a, a + 1, a + 3)); I.append((a, a + 3, a + 2))
    return np.array(P, f32), np.array(I, np.uint32)


def instanced_scene(n_side=6, baked=False, seed=99):
    """Object instancing at test size (config C4's structure): a 'plant' object (its own BVH), a one-sphere object (a
    single primitive: no accelerator, api.rs:1691) and a one-triangle object, instanced n_side^2 times with translations,
    rotations, non-uniform and mirroring scales over a ground quad.  `baked=True` builds the SAME geometry as ordinary
    world-space meshes instead of instances (for cross-checking the instancing code against the plain path)."""
    b = H.SceneBuilder()
    cam_w2c = H.Transform.look_at((0.0, -7.5, 4.0), (0, 0, 0.4), (0, 0, 1))
    Pp, Ip = _plant_mesh()
    Ptri, Itri = np.array([(-0.3, 0, 0), (0.3, 0, 0), (0, 0.1, 0.8)], f32), np.array([(0, 1, 2)], np.uint32)
    mats = {"plant": ("plastic", dict(Kd=(0.15, 0.45, 0.12), Ks=0.2, roughness=0.2)), "ball": ("metal", dict(roughness=0.05)),
            "shard": ("matte", dict(Kd=(0.7, 0.3, 0.2)))}

    def define(name):
        m, kw = mats[name]
        b.material(m, **kw)
        if name == "plant":
            b.shape("trianglemesh", P=Pp, indices=Ip)
        elif name == "ball":
            b.translate(0, 0, 0.35)
            b.shape("sphere", radius=0.35)
        else:
            b.shape("trianglemesh", P=Ptri, indices=Itri)

    if not baked:
        for name in mats:
            b.object_begin(name)
            define(name)
            b.object_end()
    b.material("matte", Kd=(0.5, 0.5, 0.45))
    Pq, Iq = quad((-12, -12, 0), (12, -12, 0), (12, 12, 0), (-12, 12, 0))
    b.shape("trianglemesh", P=Pq, indices=Iq)
    rng = PCG32(seed)
    u = rng.floats(6 * n_side * n_side)
    names = list(mats)
    for j in range(n_side):
        for i in range(n_side):
            k = 6 * (j * n_side + i)
            b.attribute_begin()
            b.translate(-4.5 + 9.0 * (i + 0.5 + 0.6 * (float(u[k]) - 0.5)) / n_side, -3.0 + 9.0 * (j + 0.5 + 0.6 * (float(u[k + 1]) - 0.5)) / n_side, 0.0)
            b.rotate(360.0 * float(u[k + 2]), 0, 0, 1)
            sx = 0.6 + 0.9 * float(u[k + 3])
            b.scale(sx, sx * (1.0 if (i + j) % 3 else 1.4), (0.7 + 0.8 * float(u[k + 4])) * (-1.0 if (i * 7 + j) % 5 == 0 else 1.0))
            if (i * 7 + j) % 5 == 0:
                b.translate(0, 0, -1.2)  # mirrored in z: lift it back above the ground
            name = names[(i + 2 * j) % 3] if (i + j) % 4 else "plant"
            if baked:
                define(name)
            else:
                b.object_instance(name)
            b.attribute_end()
    b.attribute_begin()
    b.area_light_source("diffuse", L=(30, 30, 27))
    Pl, Il = quad((-1.5, -1.5, 6.0), (-1.5, 1.5, 6.0), (1.5, 1.5, 6.0), (1.5, -1.5, 6.0))
    b.shape("trianglemesh", P=Pl, indices=Il)
    b.attribute_end()
    b.attribute_begin()
    b.translate(4.0, -4.0, 3.0)
    b.light_source("point", I=(10, 10, 12))
    b.attribute_end()
    flat = b.world_end()

    def make(spp_=16, res=(128, 96), maxdepth_=5, sampler_="sobol", strategy="power", filt="box"):
        film = H.Film(res[0], res[1], filt)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=50.0)
        return H.PathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy)

    return SceneSetup("instanced-small", flat, make, f"{n_side * n_side} object instances (plant BVH / single sphere / single triangle) on a ground quad")


def foliage_field_scene(n_instances=2000, n_blades=250, seg=20, n_point=9800, n_quads=100, field=100.0, xres=3840, yres=2160, spp=64, maxdepth=5, sampler="sobol",
                        seed=99):
    """S4 / config C4 (SURVEY.md s8(d)): `n_instances` instances (PCG32 placement on a field x field area, random yaw and
    scale) of ONE procedural plant of 2 * n_blades * seg triangles (default 10 000 => 20 M instanced triangles), lit by
    `n_point` point lights on a jittered grid plus `n_quads` small quad area lights (2 triangle lights each), power light
    sampling.  Instanced geometry is stored once (~1 MB); the top-level BVH holds the instances, the ground and the lights."""
    b = H.SceneBuilder()
    half = 0.5 * field
    cam_w2c = H.Transform.look_at((0.0, -0.62 * field, 0.16 * field), (0, -0.1 * field, 0.0), (0, 0, 1))
    Pp, Ip = _plant_mesh(n_blades=n_blades, seg=seg, seed=17)
    b.object_begin("plant")
    b.material("plastic", Kd=(0.12, 0.4, 0.1), Ks=(0.15, 0.15, 0.15), roughness=0.2)
    b.shape("trianglemesh", P=Pp, indices=Ip)
    b.object_end()
    b.material("matte", Kd=(0.35, 0.3, 0.22))
    Pq, Iq = quad((-half * 1.5, -half * 1.5, 0), (half * 1.5, -half * 1.5, 0), (half * 1.5, half * 1.5, 0), (-half * 1.5, half * 1.5, 0))
    b.shape("trianglemesh", P=Pq, indices=Iq)
    rng = PCG32(seed)
    u = rng.floats(4 * n_instances + 7 * n_point + 8 * n_quads)
    k = 0
    side = max(1, int(math.ceil(math.sqrt(n_instances))))
    for i in range(n_instances):
        gx, gy = i % side, i // side
        b.attribute_begin()
        b.translate(-half + field * (gx + float(u[k])) / side, -half + field * (gy + float(u[k + 1])) / side, 0.0)
        b.rotate(360.0 * float(u[k + 2]), 0, 0, 1)
        sc = (0.8 + 1.2 * float(u[k + 3])) * field / side * 0.9
        b.scale(sc, sc, sc)
        b.object_instance("plant")
        b.attribute_end()
        k += 4
    lside = max(1, int(math.ceil(math.sqrt(max(n_point, 1)))))
    for i in range(n_point):
        gx, gy = i % lside, i // lside
        b.attribute_begin()
        b.translate(-half + field * (gx + float(u[k])) / lside, -half + field * (gy + float(u[k + 1])) / lside, field * (0.05 + 0.05 * float(u[k + 2])))
        c = field * field / max(n_point, 1) * (0.05 + 0.4 * float(u[k + 3]) ** 2)
        b.light_source("point", I=(c * (0.7 + 0.3 * float(u[k + 4])), c * (0.7 + 0.3 * float(u[k + 5])), c * (0.6 + 0.4 * float(u[k + 6]))))
        b.attribute_end()
        k += 7
    for i in range(n_quads):
        cx, cy, cz = -half + field * float(u[k]), -half + field * float(u[k + 1]), field * (0.06 + 0.04 * float(u[k + 2]))
        hs = field * (0.004 + 0.006 * float(u[k + 3]))
        b.attribute_begin()
        e = field * field / max(n_quads, 1) * 0.02 / (hs * hs)
        b.area_light_source("diffuse", L=(e * (0.7 + 0.3 * float(u[k + 4])), e * (0.7 + 0.3 * float(u[k + 5])), e * (0.6 + 0.4 * float(u[k + 6]))))
        Pl, Il = quad((cx - hs, cy - hs, cz), (cx - hs, cy + hs, cz), (cx + hs, cy + hs, cz), (cx + hs, cy - hs, cz))
        b.shape("trianglemesh", P=Pl, indices=Il)
        b.attribute_end()
        k += 8
    flat = b.world_end()

    def make(spp_=spp, res=(xres, yres), maxdepth_=maxdepth, sampler_=sampler, strategy="power", filt="box"):
        film = H.Film(res[0], res[1], filt)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=45.0)
        return H.PathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy)

    ntri = 2 * n_blades * seg
    return SceneSetup("S4-foliage", flat, make, f"{n_instances} instances x {ntri} triangles = {n_instances * ntri} instanced triangles, "
                      f"{n_point} point + {2 * n_quads} triangle area lights, power light sampling")


def many_lights_scene(grid=6, n_quads=6, seed=99):
    """Room lit by many small lights (a test-sized stand-in for config C4's light population): grid x grid point lights
    under the ceiling, a few spot lights and small quad area lights (2 triangle lights each).  With this many lights of
    very different reach the three `lightsamplestrategy` choices give visibly different sampling distributions."""
    b = H.SceneBuilder()
    cam_w2c = H.Transform.look_at((0.0, -9.5, 3.0), (0, 0, 1.5), (0, 0, 1))
    rng = PCG32(seed)
    u = rng.floats(8 * (grid * grid + n_quads + 8))
    k = 0
    b.material("matte", Kd=(0.55, 0.55, 0.5))
    for pts in (((-10, -10, 0), (10, -10, 0), (10, 10, 0), (-10, 10, 0)), ((-10, 10, 0), (10, 10, 0), (10, 10, 6), (-10, 10, 6)),
                ((-10, -10, 0), (-10, 10, 0), (-10, 10, 6), (-10, -10, 6)), ((10, -10, 0), (10, -10, 6), (10, 10, 6), (10, 10, 0))):
        Pq, Iq = quad(*pts)
        b.shape("trianglemesh", P=Pq, indices=Iq)
    P, I, N = displaced_sphere(24, 12, 0.9, 0.08, 3)
    for j, (m, kw) in enumerate((("plastic", dict(Kd=(0.6, 0.2, 0.2), Ks=0.3, roughness=0.1)), ("metal", dict(roughness=0.08)), ("matte", dict(Kd=(0.2, 0.5, 0.7))))):
        b.attribute_begin()
        b.translate(-4.0 + 4.0 * j, 1.0 - 1.5 * (j % 2), 0.95)
        b.material(m, **kw)
        b.shape("trianglemesh", P=P, indices=I, N=N)
        b.attribute_end()
    for gy in range(grid):
        for gx in range(grid):
            b.attribute_begin()
            b.translate(-8.5 + 17.0 * (gx + float(u[k])) / grid, -8.5 + 17.0 * (gy + float(u[k + 1])) / grid, 4.0 + 1.5 * float(u[k + 2]))
            c = 0.3 + 2.5 * float(u[k + 3]) ** 3
            b.light_source("point", I=(c * (0.6 + 0.4 * float(u[k + 4])), c * (0.6 + 0.4 * float(u[k + 5])), c * (0.6 + 0.4 * float(u[k + 6]))))
            b.attribute_end()
            k += 8
    for j in range(4):
        x, y = -6.0 + 4.0 * j, -6.0 + 3.0 * (j % 2)
        b.light_source("spot", **{"from": (x, y, 5.5), "to": (x + 1.0, y + 2.0, 0.0), "I": (30, 28, 22), "coneangle": 25.0, "conedeltaangle": 8.0})
    for j in range(n_quads):
        cx, cy, cz = -8.0 + 16.0 * float(u[k]), -8.0 + 16.0 * float(u[k + 1]), 5.0 + 0.8 * float(u[k + 2])
        hs = 0.15 + 0.2 * float(u[k + 3])
        b.attribute_begin()
        b.area_light_source("diffuse", L=(20 + 40 * float(u[k + 4]), 20 + 30 * float(u[k + 5]), 15 + 30 * float(u[k + 6])))
        Pl, Il = quad((cx - hs, cy - hs, cz), (cx - hs, cy + hs, cz), (cx + hs, cy + hs, cz), (cx + hs, cy - hs, cz))
        b.shape("trianglemesh", P=Pl, indices=Il)
        b.attribute_end()
        k += 8
    flat = b.world_end()

    def make(spp_=16, res=(128, 72), maxdepth_=5, sampler_="sobol", strategy="spatial", filt="box"):
        film = H.Film(res[0], res[1], filt)
        cam = H.PerspectiveCamera(film, cam_w2c.inverse(), fov=55.0)
        return H.PathIntegrator(cam, film, H.Sampler(sampler_, spp_), maxdepth=maxdepth_, lightsamplestrategy=strategy)

    return SceneSetup("many-lights", flat, make, f"{grid * grid} point + 4 spot + {2 * n_quads} triangle area lights in a room")


# ---------------------------------------------------------------------------
# ray batches (SURVEY.md s8(d))
# ---------------------------------------------------------------------------
def rays_diffuse(flat, n, seed=7):
    """B-diff: origins uniform in the world bound, directions uniform on the sphere."""
    wb = flat.world_bound
    u = _hash_floats(5 * n, seed).reshape(5, n)
    lo, hi = wb[:3], wb[3:]
    o = lo[None, :] + (hi - lo)[None, :] * u[:3].T
    z = f32(1) - f32(2) * u[3]
    r = np.sqrt(np.maximum(f32(0), f32(1) - z * z)).astype(f32)
    phi = f32(2 * math.pi) * u[4]
    d = np.stack([r * np.cos(phi), r * np.sin(phi), z], axis=1).astype(f32)
    return H.make_rays(o.astype(f32), d)


def rays_shadow(flat, n, seed=11):
    """B-shadow: segments between random points on random triangles (t_max = 1 - 1e-4, like
    Interaction::spawn_rayto_interaction, interaction.rs:46-52)."""
    nt = len(flat.tri_indices)
    u = _hash_floats(8 * n, seed).reshape(8, n)

    def pts(ua, ub, uc):
        t = np.minimum((ua * nt).astype(np.int64), nt - 1)
        idx = flat.tri_indices[t]
        su = np.sqrt(ub)
        b0, b1 = 1 - su, uc * su
        p = (flat.vertex_p[idx[:, 0]] * b0[:, None] + flat.vertex_p[idx[:, 1]] * b1[:, None] + flat.vertex_p[idx[:, 2]] * (1 - b0 - b1)[:, None])
        return p.astype(f32)

    a, bpt = pts(u[0], u[1], u[2]), pts(u[3], u[4], u[5])
    d = bpt - a
    keep = (d * d).sum(1) > 0
    return H.make_rays(a[keep], d[keep], t_max=f32(1.0) - f32(1e-4))


def rays_camera(integ, sample=0, max_rays=None):
    """B-cam: pinhole camera rays through pixel centres (host-side, for batch tests only)."""
    film, cam = integ.film, integ.camera
    x0, y0, x1, y1 = film.cropped_pixel_bounds
    xs, ys = np.meshgrid(np.arange(x0, x1, dtype=f32) + f32(0.5), np.arange(y0, y1, dtype=f32) + f32(0.5))
    pf = np.stack([xs.reshape(-1), ys.reshape(-1), np.zeros(xs.size, f32)], axis=1)
    if max_rays:
        pf = pf[:: max(1, len(pf) // max_rays)]
    pc = cam.raster_to_camera.points(pf)
    d = pc * (f32(1) / np.sqrt((pc * pc).sum(1, dtype=f32)))[:, None]
    o = cam.camera_to_world.points(np.zeros((len(d), 3), f32))
    return H.make_rays(o, cam.camera_to_world.vectors(d))


def rays_surface(flat, n, seed=23, tri_lo=0, tri_hi=None):
    """B-surf: incoherent secondary-like rays: origins on random triangles (offset along the face normal),
    directions uniform in the hemisphere about that normal, t_max = inf.  Representative of bounce >= 1 path rays."""
    idxs = flat.tri_indices[tri_lo:tri_hi]
    nt = len(idxs)
    u = _hash_floats(6 * n, seed).reshape(6, n)
    t = np.minimum((u[0] * nt).astype(np.int64), nt - 1)
    idx = idxs[t]
    p0, p1, p2 = flat.vertex_p[idx[:, 0]], flat.vertex_p[idx[:, 1]], flat.vertex_p[idx[:, 2]]
    su = np.sqrt(u[1])
    b0, b1 = 1 - su, u[2] * su
    p = p0 * b0[:, None] + p1 * b1[:, None] + p2 * (1 - b0 - b1)[:, None]
    nrm = np.cross(p1 - p0, p2 - p0)
    ln = np.linalg.norm(nrm, axis=1, keepdims=True)
    keep = ln[:, 0] > 0
    nrm = nrm / np.maximum(ln, 1e-30)
    z = f32(1) - f32(2) * u[3]
    r = np.sqrt(np.maximum(f32(0), f32(1) - z * z))
    phi = f32(2 * math.pi) * u[4]
    d = np.stack([r * np.cos(phi), r * np.sin(phi), z], axis=1)
    flip = (d * nrm).sum(1) < 0
    d[flip] = -d[flip]
    o = p + nrm * f32(1e-4)
    return H.make_rays(o[keep].astype(f32), d[keep].astype(f32))
