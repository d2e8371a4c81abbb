"""Packet traversal (trace.cuh: trav_run_packet) returns exactly what the per-lane walk returns.

A warp whose 32 rays share an octant walks the BVH as one packet: one stack, one depth-first walk over the union of the nodes
its lanes need, each lane testing its own boxes and triangles against its own t_max.  The path integrator uses it for its
coherent queues by default (camera rays of a wave's first iteration, their shadow rays); PBRT_B200_PACKET_TRAVERSAL=0 turns it
off, and =2 also routes the batch entry points (intersect_dev / intersect_p_dev) through it.  Both are read per call, so one
scene object renders and traces in both modes here.

Chunks whose rays do not share an octant, or have a zero direction component, fall back to the per-lane walk: the batches
below contain both on purpose (warps across the image's centre row and column, zeroed direction components, a ragged tail).
"""
import numpy as np
import pytest

gpu = pytest.mark.gpu
STATS = ("camera_rays", "intersection_tests", "shadow_tests", "zero_radiance_paths")
KNOB = "PBRT_B200_PACKET_TRAVERSAL"


def _scene(pkg, name):
    S = pkg.scenes
    if name == "s3small":
        return S.displaced_sphere_scene(256, 128), (480, 270)
    return S.cornell_scene(), (64, 48)


def _set_knob(monkeypatch, mode):
    if mode is None:
        monkeypatch.delenv(KNOB, raising=False)
    else:
        monkeypatch.setenv(KNOB, str(mode))


def _camera_rays_item_order(pkg, integ, spp=32, seed=3, stride=1):
    """Jittered pinhole camera rays, `spp` consecutive samples per pixel (the renderer's item order: a warp = 32 samples of a pixel),
    over every `stride`-th pixel of the film; plus 16 + 16 samples on either side of the film's centre column and centre row, which
    put the octant change inside one warp."""
    H = pkg.host
    film, cam = integ.film, integ.camera
    x0, y0, x1, y1 = film.cropped_pixel_bounds
    xs, ys = np.meshgrid(np.arange(x0, x1, stride, dtype=np.float32), np.arange(y0, y1, stride, dtype=np.float32))
    px, py = np.repeat(xs.reshape(-1), spp), np.repeat(ys.reshape(-1), spp)
    rng = np.random.default_rng(seed)
    jit = rng.random((len(px), 2), dtype=np.float32)
    pf = [np.stack([px + jit[:, 0], py + jit[:, 1]], axis=1)]
    cx, cy = np.float32(0.5 * (film.full_resolution[0])), np.float32(0.5 * (film.full_resolution[1]))
    for y in np.arange(y0, y1, max(1, stride), dtype=np.float32):  # across the centre column
        off = np.concatenate([-rng.random(16, dtype=np.float32), rng.random(16, dtype=np.float32)])
        pf.append(np.stack([cx + off, np.full(32, y + np.float32(0.5), np.float32)], axis=1))
    for x in np.arange(x0, x1, max(1, stride), dtype=np.float32):  # across the centre row
        off = np.concatenate([-rng.random(16, dtype=np.float32), rng.random(16, dtype=np.float32)])
        pf.append(np.stack([np.full(32, x + np.float32(0.5), np.float32), cy + off], axis=1))
    pf = np.concatenate(pf).astype(np.float32)
    pf = np.concatenate([pf, np.zeros((len(pf), 1), np.float32)], axis=1)
    pc = cam.raster_to_camera.points(pf)
    d = pc * (np.float32(1) / np.sqrt((pc * pc).sum(1, dtype=np.float32)))[:, None]
    o = cam.camera_to_world.points(np.zeros((len(d), 3), np.float32))
    return H.make_rays(o, cam.camera_to_world.vectors(d).astype(np.float32))


def _with_zero_components(rays):
    """A copy in which some whole warps and some single lanes have a zero direction component (the NaN-exact walk)."""
    z = rays.copy()
    n = len(z) // 32 * 32
    z["d"][0:n:7 * 32, 0] = 0.0  # one lane in every 7th warp
    for w in range(3, n // 32, 11):  # whole warps, one axis each
        z["d"][32 * w:32 * w + 32, w % 3] = -0.0 if w % 2 else 0.0
    return z


def _mixed_octant_warps(rays):
    s = np.signbit(rays["d"][: len(rays) // 32 * 32]).reshape(-1, 32, 3)
    return int((s.any(axis=1) & ~s.all(axis=1)).any(axis=1).sum())


def _trace_both(monkeypatch, sc, rays, shadow):
    out = {}
    for mode in (0, 2):
        _set_knob(monkeypatch, mode)
        out[mode] = (sc.intersect(rays), sc.intersect_p(shadow))
    _set_knob(monkeypatch, None)
    return out


@gpu
@pytest.mark.parametrize("scene", ["s3small", "cornell"])
def test_camera_batches_match_per_lane_walk(pkg, gpu_lib, monkeypatch, scene):
    setup, res = _scene(pkg, scene)
    integ = setup.make_integrator(spp_=4, res=res)
    rays = _camera_rays_item_order(pkg, integ, stride=1 if scene == "cornell" else 3)
    assert _mixed_octant_warps(rays) > 0
    rays = np.concatenate([rays, _with_zero_components(rays[: 32 * 200])])[:-7]  # ragged tail: the last warp is partial
    # any-hit: the camera rays cut short (t_max = 0.6 x the closest hit's t is occluded only by something nearer), plus full-length
    sc = pkg.Scene(setup.flat)
    try:
        _set_knob(monkeypatch, 0)
        t = sc.intersect(rays)["t"]
        shadow = rays.copy()
        shadow["t_max"] = np.where(np.isfinite(t), t * np.float32(0.6), np.float32(1e30)).astype(np.float32)
        shadow = np.concatenate([shadow, rays])
        got = _trace_both(monkeypatch, sc, rays, shadow)
    finally:
        _set_knob(monkeypatch, None)
        sc.close()
    (h0, o0), (h2, o2) = got[0], got[2]
    assert h0.tobytes() == h2.tobytes(), f"{(h0 != h2).sum()} hit records differ"
    assert o0.tobytes() == o2.tobytes(), f"{(o0 != o2).sum()} any-hit flags differ"
    assert (h0["prim"] != np.iinfo(h0["prim"].dtype).max).any() and o0.any() and not o0.all()


@gpu
def test_camera_batch_matches_oracle(pkg, oracle, gpu_lib, monkeypatch):
    """Third arm on a small case: packet walk, per-lane walk and the CPU oracle agree bit for bit."""
    setup, _ = _scene(pkg, "cornell")
    integ = setup.make_integrator(spp_=4, res=(24, 18))
    rays = _camera_rays_item_order(pkg, integ)
    rays = np.concatenate([rays, _with_zero_components(rays[: 32 * 64])])
    shadow = rays.copy()
    shadow["t_max"] = np.float32(2.0)
    sc = pkg.Scene(setup.flat)
    try:
        got = _trace_both(monkeypatch, sc, rays, shadow)
    finally:
        sc.close()
    want, _ = oracle.intersect(setup.flat, rays)
    occ_want, _ = oracle.intersect_p(setup.flat, shadow)
    for mode in (0, 2):
        hits, occ = got[mode]
        assert hits.tobytes() == want.tobytes(), f"mode {mode}"
        assert np.array_equal(occ, occ_want), f"mode {mode}"


@gpu
@pytest.mark.parametrize("scene,spp", [("s3small", 4), ("s3small", 32), ("cornell", 4)])
def test_renders_match_per_lane_walk(pkg, gpu_lib, monkeypatch, scene, spp):
    setup, res = _scene(pkg, scene)
    integ = setup.make_integrator(spp_=spp, res=res)
    sc = pkg.Scene(setup.flat)
    try:
        out = {}
        for mode in (0, 2, None):
            _set_knob(monkeypatch, mode)
            out[mode] = sc.render(integ)
    finally:
        _set_knob(monkeypatch, None)
        sc.close()
    base, bst = out[0]
    assert np.isfinite(base).all() and (base[:, 3] > 0).any()
    for mode in (2, None):
        img, st = out[mode]
        assert {k: int(getattr(st, k)) for k in STATS} == {k: int(getattr(bst, k)) for k in STATS}, f"mode {mode}"
        # films: the same samples, summed by atomics in a different order
        assert np.allclose(img, base, rtol=2e-5, atol=2e-5), f"mode {mode}"
