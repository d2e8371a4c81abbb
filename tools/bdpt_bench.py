"""Throughput and convergence of the bdpt integrator on one GPU (DESIGN.md §4f).

    python tools/bdpt_bench.py [--res 1024] [--spp 4] [--out result.json]

Prints one JSON object:
  - `cornell`, `caustic`: BDPT camera samples/s (device time from the library's CUDA events, median of three renders after a warm-up) on the
    Cornell box and on the caustic scene at res^2, maxdepth 5;
  - `oracle`: the CPU oracle's BDPT samples/s on this host's threads (caustic scene, 128^2 x 4 spp);
  - `equal_time`: on the caustic scene at 256^2, relMSE against a reference of 2048 path-integrator samples per pixel drawn from sample
    numbers the two estimates do not use, for BDPT and for the path integrator given the same device time;
  - `gpu`: card name, power limit and maximum SM clock, read in the same run.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import importlib  # noqa: E402

pkg = importlib.import_module("pbrt-rust_b200")
H = pkg.host


def bdpt_of(integ, maxdepth=5):
    return H.BDPTIntegrator(integ.camera, integ.film, integ.sampler, maxdepth=maxdepth)


def rate(sc, integ, reps=3):
    sc.render_splat(integ)
    ms = []
    for _ in range(reps):
        _, _, st = sc.render_splat(integ)
        ms.append(st.device_ms)
    return st.camera_rays / (float(np.median(ms)) * 1e-3)


def resolve(sc, rgbw, splat, n):
    return sc.film_resolve_splat(rgbw, splat, 1.0 / n, 1.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=1024)
    ap.add_argument("--spp", type=int, default=4)
    ap.add_argument("--out")
    a = ap.parse_args()
    out = {}
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out["gpu"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"
    for name, make in (("cornell", pkg.scenes.cornell_scene), ("caustic", pkg.scenes.caustic_scene)):
        setup = make(xres=a.res, yres=a.res, spp=a.spp)
        sc = H.Scene(setup.flat)
        out[name] = {"samples_per_s": rate(sc, bdpt_of(setup.make_integrator(spp_=a.spp, maxdepth_=5, filt="box"))), "res": a.res, "spp": a.spp}
        sc.close()
    from oracle import oracle_bdpt as OB
    setup = pkg.scenes.caustic_scene(xres=128, yres=128, spp=4)
    integ = bdpt_of(setup.make_integrator(spp_=4, maxdepth_=5))
    t0 = time.perf_counter()
    _, _, st = OB.render(setup.flat, integ)
    out["oracle"] = {"samples_per_s": st["camera_rays"] / (time.perf_counter() - t0), "threads": __import__("os").cpu_count()}
    # equal device time on the caustic scene
    R, NB, NREF = 256, 64, 2048
    setup = pkg.scenes.caustic_scene(xres=R, yres=R)
    sc = H.Scene(setup.flat)
    big = setup.make_integrator(spp_=NB * 64 + NREF, maxdepth_=5)
    ref, _ = sc.render(big, sample_range=(NB * 64, NB * 64 + NREF))
    ref = sc.film_resolve(ref)
    bd = bdpt_of(big)
    rgbw, splat, st = sc.render_splat(bd, sample_range=(0, NB))
    t_bdpt = st.device_ms
    img_b = resolve(sc, rgbw, splat, NB)
    # the path integrator's device time for NB samples, then as many samples as fit in BDPT's time
    _, stp = sc.render(big, sample_range=(0, NB))
    n_path = int(min(NB * 64, max(1, round(NB * t_bdpt / stp.device_ms))))
    rgbw_p, stp = sc.render(big, sample_range=(0, n_path))
    img_p = sc.film_resolve(rgbw_p)
    sc.close()

    def rel_mse(a_, b_):
        return float(np.mean((a_ - b_) ** 2 / (b_ ** 2 + 1e-2)))
    out["equal_time"] = {"res": R, "bdpt_spp": NB, "bdpt_ms": t_bdpt, "path_spp": n_path, "path_ms": stp.device_ms, "reference_path_spp": NREF,
                         "relmse_bdpt": rel_mse(img_b, ref), "relmse_path": rel_mse(img_p, ref)}
    s = json.dumps(out)
    print(s)
    if a.out:
        Path(a.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
