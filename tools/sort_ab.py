"""Ray-ordering experiment (same batches as trace_ab3.py): how much do octant binning / Morton sorting of the ray
queue buy on the three ray populations of a path-traced frame of S3:
tile-ordered camera rays, bounce-1 rays (cosine-ish hemisphere about the hit normal) and shadow rays toward the
area light.  Run once per library build (csrc/Makefile: make NAME=<name>):  PBRT_B200_LIB=pbrt-rust_b200/libpbrt_b200_<name>.so python tools/sort_ab.py
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
    return m / (e0.elapsed_time(e1) / reps) / 1e3, zlib.crc32(dh.cpu().numpy().tobytes())


def octant(r):
    d = r["d"]
    return (d[:, 0] < 0).astype(np.int64) | ((d[:, 1] < 0).astype(np.int64) << 1) | ((d[:, 2] < 0).astype(np.int64) << 2)

def morton(r, bits=10):
    wb = np.asarray(flat.world_bound).reshape(-1)
    q = np.clip(((r["o"] - wb[:3]) / (wb[3:] - wb[:3]) * (1 << bits)).astype(np.int64), 0, (1 << bits) - 1)
    def spread(v):
        out = np.zeros_like(v)
        for b in range(bits): out |= ((v >> b) & 1) << (3 * b)
        return out
    return spread(q[:, 0]) | (spread(q[:, 1]) << 1) | (spread(q[:, 2]) << 2)

rng = np.random.default_rng(1)
for bn, rays in batches.items():
    anyhit = False
    orders = {"queue order": np.arange(len(rays)), "shuffled": rng.permutation(len(rays)), "octant (stable)": np.argsort(octant(rays), kind="stable"),
              "octant+morton": np.lexsort((morton(rays), octant(rays))), "morton": np.argsort(morton(rays), kind="stable"),
              "octant within 64k blocks": np.concatenate([np.argsort(octant(rays[i:i + 65536]), kind="stable") + i for i in range(0, len(rays), 65536)])}
    for on, perm in orders.items():
        mr, _ = run(rays[perm], False)
        line = f"{bn:8s} {on:26s} closest {mr:7.1f} Mrays/s"
        if bn == "shadow":
            mr2, _ = run(rays[perm], True)
            line += f"   any-hit {mr2:7.1f} Mrays/s"
        print(line, flush=True)
