"""Volpath throughput with grid media: the smoke box (scenes.smoke_box_scene, k_vol_mega_grid) and the fog box (scenes.fog_box_scene,
k_vol_mega) at 1024 x 1024, maxdepth 5, on one GPU, plus the CPU oracle on all host threads for scale.

    python tools/grid_media_bench.py [--spp 16] [--reps 3] [--parent-tree path/to/other/checkout]

With --parent-tree, the fog box also runs from that checkout (another commit with its library built, e.g. the parent of a change),
alternating with this tree, so the homogeneous path of the two can be compared in one call.  The other tree runs with its own Python
package: a library alone (csrc/Makefile NAME=x, PBRT_B200_LIB) only fits the host code of the commit it was built from.  Every measurement runs in a
process of its own; the card's name and power limit are read in the same call.  Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent

CHILD = r"""
import importlib, json, sys, time
sys.path.insert(0, {root!r})
S = importlib.import_module("pbrt-rust_b200.scenes")
H = importlib.import_module("pbrt-rust_b200.host")
kind, res, spp, device = {kind!r}, {res}, {spp}, {device}
if kind == "oracle":
    sys.path.insert(0, {root!r} + "/oracle")
    import oracle as O
    setup = S.smoke_box_scene(xres=res, yres=res, spp=spp)
    integ = setup.make_integrator()
    t = time.perf_counter(); _, st = O.render(setup.flat, integ); dt = time.perf_counter() - t
    print(json.dumps({{"seconds": dt, "samples": res * res * spp, "rays": st["intersection_tests"]}}))
else:
    setup = (S.smoke_box_scene if kind == "smoke" else S.fog_box_scene)(xres=res, yres=res, spp=spp)
    integ = setup.make_integrator()
    sc = H.Scene(setup.flat, device=device)
    sc.render(integ)  # warm-up: module load, buffers
    _, st = sc.render(integ)
    print(json.dumps({{"seconds": st.device_ms / 1e3, "samples": res * res * spp, "rays": int(st.intersection_tests),
                      "camera_rays": int(st.camera_rays)}}))
    sc.close()
"""


def child(kind, res, spp, device=0, root=ROOT):
    p = subprocess.run([sys.executable, "-c", CHILD.format(root=str(root), kind=kind, res=res, spp=spp, device=device)], capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError(f"{kind} run in {root} failed:\n{p.stderr}")
    out = p.stdout
    r = json.loads(out.strip().splitlines()[-1])
    r["samples_per_s"] = r["samples"] / r["seconds"]
    r["mrays_per_s"] = r["rays"] / r["seconds"] / 1e6
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=1024)
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--oracle-res", type=int, default=256)
    ap.add_argument("--oracle-spp", type=int, default=4)
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "-i", str(a.device), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, check=True).stdout.strip()
    runs = {"smoke": [], "fog": [], "fog_parent": []}
    for _ in range(a.reps):  # alternate the arms so that drift of a shared machine falls on all of them alike
        runs["smoke"].append(child("smoke", a.res, a.spp, a.device))
        runs["fog"].append(child("fog", a.res, a.spp, a.device))
        if a.parent_tree:
            runs["fog_parent"].append(child("fog", a.res, a.spp, a.device, Path(a.parent_tree).resolve()))
    t = time.perf_counter()
    orc = child("oracle", a.oracle_res, a.oracle_spp)
    orc["threads"] = os.cpu_count()
    result = {"card": card, "res": a.res, "spp": a.spp, "maxdepth": 5, "oracle_wall_s": time.perf_counter() - t, "oracle_smoke_box": orc}
    for k, v in runs.items():
        if v:
            result[k] = {"samples_per_s": [r["samples_per_s"] for r in v], "mrays_per_s": [r["mrays_per_s"] for r in v],
                         "camera_rays": v[0].get("camera_rays")}
    print(json.dumps(result))


if __name__ == "__main__":
    main()
