"""A/B timing of the batch traversal kernels on the three ray populations of a path-traced frame of S3:
tile-ordered camera rays, bounce-1 rays (cosine-ish hemisphere about the hit normal) and shadow rays toward the
area light.  Run once per library build (csrc/Makefile: make NAME=<name>):  PBRT_B200_LIB=pbrt-rust_b200/libpbrt_b200_<name>.so python tools/trace_ab3.py
Prints Mrays/s per (tune, batch) and a CRC of the results so builds can be compared for bit-equality."""
import importlib, sys, ctypes as C, math, os, zlib
sys.path.insert(0, '.')
import numpy as np
import torch
P = importlib.import_module("pbrt-rust_b200")
S, H = P.scenes, P.host
setup = S.displaced_sphere_scene()
flat = setup.flat
sc = P.Scene(flat)
lib = P.load_library()
lib.pbrt_b200_debug_tune.argtypes = [C.c_int, C.c_int]
cam = S.rays_camera(setup.make_integrator())
W, Hh = 1920, 1080
ids = np.arange(W * Hh).reshape(Hh, W)
pad = np.full(((Hh + 15) // 16 * 16, W), -1); pad[:Hh] = ids
tiles = pad.reshape(-1, 16, W // 16, 16).transpose(0, 2, 1, 3).reshape(-1)
cam = cam[tiles[tiles >= 0]]
hits = sc.intersect(cam)
ok = hits["prim"] != H.NO_HIT
hc, hh = cam[ok], hits[ok]
p = hc["o"] + hc["d"] * hh["t"][:, None]
slot_of = np.zeros(len(flat.prims), np.int64); slot_of[flat.prims["creation_index"]] = np.arange(len(flat.prims))
tri = flat.prims["shape_index"][slot_of[hh["prim"]]]
idx = flat.tri_indices[tri]
p0, p1, p2 = flat.vertex_p[idx[:, 0]], flat.vertex_p[idx[:, 1]], flat.vertex_p[idx[:, 2]]
n = np.cross(p1 - p0, p2 - p0); n /= np.maximum(np.linalg.norm(n, axis=1, keepdims=True), 1e-30)
n[(n * hc["d"]).sum(1) > 0] *= -1
u = S._hash_floats(2 * len(p), 5).reshape(2, -1)
z = 1 - 2 * u[0]; r = np.sqrt(np.maximum(0, 1 - z * z)); phi = 2 * math.pi * u[1]
d = np.stack([r * np.cos(phi), r * np.sin(phi), z], 1).astype(np.float32)
d[(d * n).sum(1) < 0] *= -1
o1 = (p + n * 1e-4).astype(np.float32)
b1 = H.make_rays(o1, d)
# shadow rays to random points of the area light (first emissive triangle pair)
li = flat.lights[flat.lights["type"] == 3]
lt = flat.tri_indices[li["shape_index"][0]]
lp = flat.vertex_p[lt]
uu = S._hash_floats(2 * len(p), 9).reshape(2, -1)
su = np.sqrt(uu[0]); b0 = 1 - su; bb1 = uu[1] * su
tgt = (lp[0][None] * b0[:, None] + lp[1][None] * bb1[:, None] + lp[2][None] * (1 - b0 - bb1)[:, None]).astype(np.float32)
sh = H.make_rays(o1, tgt - o1, t_max=np.float32(1.0) - np.float32(1e-4))
batches = {"cam": cam, "bounce1": b1, "shadow": sh}
print("lib", os.environ.get("PBRT_B200_LIB", "default"), {k: len(v) for k, v in batches.items()}, flush=True)

def run(rays, anyhit, reps=10):
    m = len(rays)
    dr = torch.from_numpy(np.ascontiguousarray(rays).view(np.float32).reshape(-1, 8)).cuda()
    dh = torch.empty((m, 4), dtype=torch.int32, device='cuda') if not anyhit else torch.empty(m, dtype=torch.uint8, device='cuda')
    f = sc.intersect_p_dev if anyhit else sc.intersect_dev
    for _ in range(3): f(dr.data_ptr(), m, dh.data_ptr())
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): f(dr.data_ptr(), m, dh.data_ptr())
    e1.record(); torch.cuda.synchronize()
    out = dh.cpu().numpy()
    if os.environ.get("AB_DUMP"):  # hit records of this build, for a record-by-record comparison between two builds
        run.n = getattr(run, "n", 0) + 1
        if run.n <= 4: np.save(f"{os.environ['AB_DUMP']}_{run.n}_{len(rays)}_{int(anyhit)}.npy", out)  # cam, bounce1, shadow, shadow-any of the first config
    return m / (e0.elapsed_time(e1) / reps) / 1e3, zlib.crc32(out.tobytes())

configs = [(f"refill<{rb} interior_min {im}", {1: rb, 4: im}) for rb in (24,) for im in (0, 4, 8, 12, 16, 20, 24)]
configs += [(f"refill<{rb} interior_min {im}", {1: rb, 4: im}) for rb in (16, 28) for im in (0, 12)]
if os.environ.get("AB_QUICK"):
    configs = [("default (refill<24 interior_min 16)", {1: 24, 4: 16})] * int(os.environ["AB_QUICK"])
for name, tune in configs:
    for k, v in {0: 0, 1: 24, 2: 32, 3: 0, 4: 0, **tune}.items(): lib.pbrt_b200_debug_tune(k, v)
    out = []
    for bn, rays in batches.items():
        mr, crc = run(rays, False)
        out.append(f"{bn} {mr:7.1f} ({crc:08x})")
    mr, crc = run(sh, True)
    out.append(f"shadow-any {mr:7.1f} ({crc:08x})")
    print(f"{name:32s}", " | ".join(out), flush=True)
