#!/usr/bin/env python3
"""bench.py -- PathIntegrator hot path on B200: samples/s (camera samples per second) and Mrays/s.

Workload (BASELINE.json configs[2], the configuration the target is quoted on): the synthetic
1 048 580-triangle displaced sphere (S3), SAH BVH, plastic+metal, 1920x1080, Sobol, path maxdepth 5.
One step = one pass of the wavefront path tracer over a batch of `--spp` camera samples per pixel of
the full frame (default 16; the 512-spp render of the config is 32 such batches with distinct Sobol
sample indices; `--spp 512` renders it in one step).  Under torchrun every rank owns an interleaved
set of 16x16 tiles (groups of 8) of the same frame and the step covers `spp * N` samples per pixel,
so per-GPU work is fixed ("weak"); the films are summed to rank 0 with one NCCL reduce per step.

  value  = samples of all ranks / device time of K steps, scene + film resident in HBM
  e2e    = same metric through the host-buffer C ABI: pbrt_b200_scene_create (scene tables H2D) +
           pbrt_b200_render + film D2H + destroy, per step
  --impl reference : the CPU restatement of pbrt-rust (oracle/) on all host threads, bounded sample
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "samples/sec (camera samples per second, PathIntegrator)"
UNIT = "samples/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--spp", type=int, default=64, help="camera samples per pixel per step and per GPU")
    ap.add_argument("--scene", default="s3", choices=["s3", "cornell", "spheres", "s3small", "s4", "s5", "t1"])
    ap.add_argument("--paths-in-flight", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--tiles", default="static", choices=["static", "dynamic"],
                    help="N > 1: static interleaved tile groups, or dynamic stealing of super-tile ranges from the shared-memory work counter")
    ap.add_argument("--ref-spp", type=int, default=8, help="--impl reference: samples per pixel per step (bounded sample of the GPU arm's step)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the film of the last timed step to DIR/*.npy (float32; a seeded pixel sample when the film exceeds 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_MAX_PIXELS = 1 << 21  # 32 MB of float32 RGBW (+ 16 MB of float64 pixel indices when sampled): under 64 MB in all


def dump_outputs(out_dir, rgbw, width, height):
    """The film accumulator (per pixel: filter-weighted R, G, B and the filter weight sum) that the render call handed back for the last
    timed step.  Films above DUMP_MAX_PIXELS are written as a fixed, seeded sample of pixels, with their row-major indices."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    rgbw = np.asarray(rgbw, np.float32).reshape(height * width, 4)
    if len(rgbw) <= DUMP_MAX_PIXELS:
        np.save(out / "film_rgbw.npy", rgbw.reshape(height, width, 4))
        return
    idx = np.sort(np.random.default_rng(0).choice(len(rgbw), DUMP_MAX_PIXELS, replace=False))
    np.save(out / "film_rgbw_sample.npy", rgbw[idx])
    np.save(out / "film_pixel_index.npy", idx.astype(np.float64))


def make_setup(pkg, name):
    S = pkg.scenes
    if name == "s3":
        return S.displaced_sphere_scene(), dict(), "S3: 1,048,580-triangle displaced sphere, SAH BVH (maxnodeprims 4), plastic+metal, quad area light + point light, 1920x1080, Sobol, maxdepth 5, power light sampling"
    if name == "s3small":
        return S.displaced_sphere_scene(256, 128), dict(res=(480, 270)), "S3-small (65k triangles, 480x270) -- smoke/profiling only"
    if name == "s4":
        return S.foliage_field_scene(), dict(), "S4: 2000 instances x 10,000-triangle plant (20M instanced triangles), 9800 point + 200 triangle area lights, power light sampling, 3840x2160, Sobol, maxdepth 5"
    if name == "s5":
        return S.glass_knot_scene(nu=4096, nv=640), dict(), "S5: 5,242,884-triangle glass torus-knot mesh, maxdepth 32, Russian roulette, 1024x1024, Sobol"
    if name == "t1":
        return S.textured_scene(xres=1920, yres=1080), dict(), ("T1: the textured test scene (every texture kind and mapping, EWA / trilinear image maps, bump maps, uber + substrate, "
                                                                 "a textured instance), 1920x1080, Sobol, maxdepth 5 -- SURVEY s8 f3, not a BASELINE config")
    if name == "cornell":
        return S.cornell_scene(), dict(), "S2: Cornell box 1024x1024, maxdepth 8, gaussian filter"
    return S.spheres_scene(), dict(), "S1: two spheres 400x400, maxdepth 5"


def bench_config(desc, spp, world, pif, tiles="static"):
    """`config` of the JSON line.  Both arms print the SAME dict (the reference arm runs on the GPU arm's config; what its bounded
    per-step sample is goes into its `cpu_baseline.sample`)."""
    how = ("tiles interleaved across ranks in groups of 8" if tiles == "static" or world == 1 else
           "ranks claim ranges of 8x8-tile super-tiles from a shared-memory work counter (guided self-scheduling)")
    return {"workload": desc, "step": f"{spp} spp per GPU over the full frame ({spp * world} spp per step in total), {how}",
            "l2": "no explicit flush: per-step working set (2^27 path slots x ~270 B state + 700 MB scene and sampler tables + 33 MB film) exceeds the 126 MB L2",
            "paths_in_flight": pif or 1 << 27, "film_reduce": "NCCL reduce(sum) to rank 0 per step" if world > 1 else "none"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            p = [x.strip() for x in l.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_baseline(pkg, setup, integ_kw, seconds, threads=0):
    """Oracle (CPU restatement) on a bounded sample of the same workload: whole frame, spp chosen for ~`seconds`."""
    from oracle import oracle as O
    nth = threads or (os.cpu_count() or 1)
    integ = setup.make_integrator(spp_=64, **integ_kw)
    film = integ.film
    npx = film.width * film.height
    t0 = time.time()
    _, st = O.render(setup.flat, integ, nthreads=nth, sample_range=(0, 1))
    dt = time.time() - t0
    samples, spent, s = st["camera_rays"], dt, 1
    agg = dict(st)
    while spent < seconds * 0.6 and s < 64:
        n = int(min(64 - s, max(1, (seconds - spent) / max(dt, 1e-3))))
        t0 = time.time()
        _, st = O.render(setup.flat, integ, nthreads=nth, sample_range=(s, s + n))
        spent += time.time() - t0
        samples += st["camera_rays"]
        for k in agg:
            agg[k] += st[k]
        s += n
    rays = agg["intersection_tests"] + agg["shadow_tests"]
    return {"value": samples / spent, "unit": UNIT, "cores": nth, "kind": "port",
            "sample": f"full {film.width}x{film.height} frame, sample indices [0,{s}) = {samples} camera samples in {spent:.1f} s on {nth} threads",
            "mrays_per_s": rays / spent / 1e6,
            "nodes_per_closest_ray": agg["closest_nodes"] / max(agg["closest_rays"], 1), "prims_per_closest_ray": agg["closest_prims"] / max(agg["closest_rays"], 1),
            "nodes_per_shadow_ray": agg["any_nodes"] / max(agg["any_rays"], 1), "prims_per_shadow_ray": agg["any_prims"] / max(agg["any_rays"], 1),
            "rays_per_sample": rays / max(samples, 1)}


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version line to stdout when
    NCCL_DEBUG=VERSION is set on the box), so fd 1 is pointed at stderr for the run and the JSON line goes to the saved fd."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    args = parse()
    out_stream = _claim_stdout()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    pkg = importlib.import_module("pbrt-rust_b200")

    if args.impl == "reference":
        # The reference's own CPU implementation of the path on all host threads.  pbrt-rust cannot be built here (nightly Rust +
        # LALRPOP + ~40 crates, no network), so this is the oracle port.  The scene is built WITHOUT the product library (the
        # accelerator comes from the oracle's BVH builder), and nothing below touches CUDA.
        if rank != 0:
            return 0
        from oracle import oracle as O
        pkg.host.DEFAULT_BVH_BUILDER = O.bvh_build
        setup, kw, desc = make_setup(pkg, args.scene)
        nth = os.cpu_count() or 1
        # each step = a bounded sample of the GPU arm's step: the same full frame, `ref_spp` of its sample indices in ONE oracle
        # call (one call per spp cost ~25 % in per-call set-up in round 1 and made the two CPU legs disagree)
        ref_spp = max(1, args.ref_spp)
        nst = args.steps + args.warmup
        integ = setup.make_integrator(spp_=max(64, ref_spp * nst), **kw)
        film = integ.film
        for w in range(args.warmup):
            O.render(setup.flat, integ, nthreads=nth, sample_range=(w * ref_spp, (w + 1) * ref_spp))
        t0 = time.time()
        samples = 0
        for k in range(args.steps):
            b = (args.warmup + k) * ref_spp
            rgbw, st = O.render(setup.flat, integ, nthreads=nth, sample_range=(b, b + ref_spp))
            samples += st["camera_rays"]
        dt = time.time() - t0
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, rgbw, film.width, film.height)
        v = samples / dt
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": bench_config(desc, args.spp, args.gpus, args.paths_in_flight, args.tiles),
                          "cpu_baseline": {"value": v, "unit": UNIT, "cores": nth, "kind": "port",
                                           "sample": f"{args.steps} steps, each {ref_spp} of the step's {args.spp} spp over the full {film.width}x{film.height} frame in one "
                                                     f"call = {samples} camera samples in {dt:.1f} s on {nth} threads (CPU oracle: the Rust reference cannot be built here)"},
                          "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), file=out_stream, flush=True)
        return 0

    import torch
    import torch.distributed as dist

    lib = pkg.load_library()
    if lib.pbrt_b200_device_count() <= 0:
        raise SystemExit("bench.py: no CUDA device visible; the CUDA library has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    setup, kw, desc = make_setup(pkg, args.scene)
    spp_step = args.spp * world
    nsteps_total = args.steps + args.warmup
    integ = setup.make_integrator(spp_=spp_step * nsteps_total, **kw)
    film = integ.film
    npix = film.width * film.height
    scene = pkg.Scene(setup.flat, device=local)
    film_t = torch.zeros((npix, 4), dtype=torch.float32, device="cuda")
    interleave = (8, world, rank) if world > 1 else None
    D = importlib.import_module("pbrt-rust_b200.distributed")
    dynamic = world > 1 and args.tiles == "dynamic"
    queue = D.open_shared_queue(pkg.host, integ, dist=dist, min_chunk_tiles=64) if dynamic else None
    frames = [0]

    class Acc:  # the stats of a step = the sum over the render calls (claims) the rank made for it
        FIELDS = ("camera_rays", "intersection_tests", "shadow_tests", "kernel_launches", "trace_closest_ms", "trace_any_ms", "device_ms", "shade_ms")

        def __init__(self):
            for f in self.FIELDS:
                setattr(self, f, 0)
            self.claims = 0

        def add(self, st):
            for f in self.FIELDS:
                setattr(self, f, getattr(self, f) + getattr(st, f))
            self.claims += 1

    def render_step(sc, k):
        """This rank's share of step k into film_t (zeroed), then the film reduce; static or dynamic tile assignment."""
        acc = Acc()
        sr = (k * spp_step, (k + 1) * spp_step)
        film_t.zero_()
        if dynamic:
            def render_tiles(tile_range, il, sample_range, tile_order):
                _, st = sc.render(integ, sample_range=sample_range, device_ptr=film_t.data_ptr(), tile_range=tile_range, tile_interleave=il, tile_order=tile_order,
                                  paths_in_flight=args.paths_in_flight)
                acc.add(st)
            D.render_distributed(render_tiles, film_t, integ, dist=dist, dynamic=True, queue=queue, sample_range=sr, frame=frames[0])
            frames[0] += 1
        else:
            _, st = sc.render(integ, sample_range=sr, device_ptr=film_t.data_ptr(), tile_interleave=interleave, paths_in_flight=args.paths_in_flight)
            acc.add(st)
            if world > 1:
                dist.reduce(film_t, dst=0, op=dist.ReduceOp.SUM)
        return acc

    def step(k):
        return render_step(scene, k)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for w in range(args.warmup):
        step(w)
    sync()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tot = dict(camera=0, closest=0, shadow=0, launches=0, trace_closest_ms=0.0, trace_any_ms=0.0, device_ms=0.0, shade_ms=0.0, claims=0)
    e0.record()
    for k in range(args.steps):
        st = step(args.warmup + k)
        tot["camera"] += st.camera_rays; tot["closest"] += st.intersection_tests; tot["shadow"] += st.shadow_tests
        tot["launches"] += st.kernel_launches; tot["trace_closest_ms"] += st.trace_closest_ms; tot["trace_any_ms"] += st.trace_any_ms
        tot["device_ms"] += st.device_ms; tot["shade_ms"] += st.shade_ms; tot["claims"] += st.claims
    e1.record()
    sync()
    ms = e0.elapsed_time(e1)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # film_t holds the last timed step (summed over ranks); the e2e leg below reuses it
        dump_outputs(args.dump_outputs, film_t.cpu().numpy(), film.width, film.height)
    vals = torch.tensor([ms, tot["camera"], tot["closest"], tot["shadow"], tot["launches"]], dtype=torch.float64, device="cuda")
    if world > 1:
        mx = vals.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = vals.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms, camera, closest, shadow, launches = mx[0].item(), sm[1].item(), sm[2].item(), sm[3].item(), sm[4].item()
    else:
        camera, closest, shadow, launches = tot["camera"], tot["closest"], tot["shadow"], tot["launches"]
    value = camera / (ms * 1e-3)
    per_rank = None
    if world > 1:  # what each rank did inside the timed region: wall (CUDA events), busy (sum of its render calls), closest-hit kernel, claims
        mine = torch.tensor([e0.elapsed_time(e1), tot["device_ms"], tot["trace_closest_ms"], tot["camera"], tot["claims"]], dtype=torch.float64, device="cuda")
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        rows = [r.tolist() for r in allr]
        busy = [r[1] for r in rows]
        per_rank = {"wall_ms": [r[0] for r in rows], "render_ms": busy, "trace_closest_ms": [r[2] for r in rows], "camera_samples": [int(r[3]) for r in rows],
                    "render_calls": [int(r[4]) for r in rows], "imbalance": (max(busy) - min(busy)) / max(max(busy), 1e-9)}

    # ---- e2e: host buffers through the C ABI, scene upload + render + film download per step
    e2e = None
    if not args.no_e2e:
        host_film = np.zeros((npix, 4), np.float32)
        scene_bytes = sum(a.nbytes for a in (setup.flat.nodes, setup.flat.prims, setup.flat.vertex_p, setup.flat.tri_indices, setup.flat.materials, setup.flat.lights)
                          if a is not None) + sum(a.nbytes for a in (setup.flat.vertex_n, setup.flat.vertex_uv, setup.flat.vertex_s) if a is not None)
        n_e2e = max(1, min(args.steps, 4))
        pinned_film = torch.empty((npix, 4), dtype=torch.float32).pin_memory() if world > 1 else None
        # the step's inputs live in PINNED host memory (the bench contract's wording): the scene tables are copied once, outside the timed
        # region, into page-locked buffers, and the film comes back into one; pbrt_b200_scene_create's cudaMemcpyAsync calls then run at
        # PCIe speed instead of through the runtime's pageable staging
        keep = []

        def pinned(a):
            if a is None or a.nbytes == 0:
                return a
            t = torch.empty(a.nbytes, dtype=torch.uint8).pin_memory()
            keep.append(t)
            v = t.numpy().view(a.dtype).reshape(a.shape)
            v[...] = a
            return v

        import copy
        flat_e2e = copy.copy(setup.flat)
        for name in ("nodes", "prims", "vertex_p", "vertex_n", "vertex_s", "vertex_uv", "tri_indices", "spheres", "materials", "lights", "objects", "instances", "media", "prim_media"):
            setattr(flat_e2e, name, pinned(getattr(flat_e2e, name)))
        host_film = pinned(host_film)

        def e2e_step(k):
            sc2 = pkg.Scene(flat_e2e, device=local)  # host scene tables -> HBM
            if world == 1:
                _, st = sc2.render(integ, rgbw=host_film, sample_range=(k * spp_step, (k + 1) * spp_step), paths_in_flight=args.paths_in_flight,
                                   flags=pkg.host.RENDER_OVERWRITE)  # render + film D2H into the caller's host buffer
            else:  # every rank renders its tiles; films summed to rank 0 over NCCL; rank 0 reads the image back
                st = render_step(sc2, k)
                if rank == 0:
                    pinned_film.copy_(film_t, non_blocking=False)
            sc2.close()
            return st.camera_rays

        e2e_step(0)  # untimed warm-up (fills the library's memory pool, as the W warm-up steps do for the device-resident arm)
        sync()
        t0 = time.perf_counter()
        cam = 0
        for k in range(n_e2e):
            cam += e2e_step(k)
        sync()
        dt = time.perf_counter() - t0
        ev = torch.tensor([dt, cam], dtype=torch.float64, device="cuda")
        if world > 1:
            mx = ev.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            sm = ev.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            dt, cam = mx[0].item(), sm[1].item()
        e2e = {"value": cam / dt, "unit": UNIT, "h2d_bytes_per_step": int(scene_bytes), "d2h_bytes_per_step": int(host_film.nbytes),
               "note": f"{n_e2e} steps after 1 warm-up; each = pbrt_b200_scene_create (host scene tables in pinned host memory -> HBM) + render"
                       + (" + NCCL film reduce to rank 0" if world > 1 else "") + " + film download to host + scene destroy; host wall clock"}

    # ---- Mrays/s on fixed ray batches through the batch C ABI (BASELINE.json metric (i); SURVEY.md s8(d) B-diff / B-shadow)
    ray_batches = None
    if rank == 0 and world == 1 and args.scene in ("s3", "s3small"):
        S = pkg.scenes
        ray_batches = {}
        for bname, rays, anyhit in (("B-diff closest-hit", S.rays_diffuse(setup.flat, 4_000_000, seed=7), False),
                                    ("B-surf closest-hit", S.rays_surface(setup.flat, 4_000_000, seed=23), False),
                                    ("B-shadow any-hit", S.rays_shadow(setup.flat, 4_000_000, seed=11), True)):
            m = len(rays)
            dr = torch.from_numpy(np.ascontiguousarray(rays).view(np.float32).reshape(-1, 8)).cuda()
            dh = torch.empty(m, dtype=torch.uint8, device="cuda") if anyhit else torch.empty((m, 4), dtype=torch.int32, device="cuda")
            f = scene.intersect_p_dev if anyhit else scene.intersect_dev
            for _ in range(3):
                f(dr.data_ptr(), m, dh.data_ptr())
            torch.cuda.synchronize()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            for _ in range(10):
                f(dr.data_ptr(), m, dh.data_ptr())
            b1.record(); torch.cuda.synchronize()
            ray_batches[bname] = {"rays": m, "mrays_per_s": m / (b0.elapsed_time(b1) / 10) / 1e3}

    if rank == 0:
        peaks = {}
        pk = ROOT / "MEASURED_PEAKS.json"
        if pk.exists():
            peaks = json.loads(pk.read_text())
        peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            cpu = cpu_baseline(pkg, setup, kw, args.cpu_seconds)
        # algorithmic bytes per closest-hit ray on the REFERENCE algorithm's data (SURVEY.md s8(d)):
        # 32 B per LinearBVHNode tested + 48 B per triangle tested + 32 B ray in + 16 B hit out
        prof = {}
        pj = ROOT / "profiles" / "roofline_inputs.json"
        if pj.exists():
            prof = json.loads(pj.read_text())
        npr = (cpu or prof).get("nodes_per_closest_ray")
        ppr = (cpu or prof).get("prims_per_closest_ray")
        roofline = None
        if npr is not None and tot["trace_closest_ms"] > 0:
            bytes_per_ray = 32.0 * npr + 48.0 * ppr + 48.0
            ach = tot["closest"] * bytes_per_ray / (tot["trace_closest_ms"] * 1e-3) / 1e9
            cap = prof.get("trace_closest", {})  # ncu --set full of one k_trace_closest launch of THIS build (tools/profile_pass.sh)
            traffic, t_ms, t_rays = cap.get("dram_bytes"), cap.get("ms"), cap.get("rays")
            roofline = {"bound": "hbm", "kernel": "k_trace_closest (+k_trace_mis): closest-hit BVH traversal", "achieved": ach, "peak": peak, "unit": "GB/s",
                        "frac": ach / peak, "peak_source": peak_src, "traffic": traffic,
                        "traffic_launch": {"rays": t_rays, "ms": t_ms, "algorithmic_bytes": None if t_rays is None else t_rays * bytes_per_ray,
                                           "source": prof.get("source")},
                        # what actually bounds the kernel (the algorithmic GB/s above is mostly L1 / L2 re-use of the tree top): the same
                        # capture's real DRAM share of the HBM peak, warp-issue utilisation and SIMD efficiency
                        "dram_frac": None if not (traffic and t_ms) else traffic / (t_ms * 1e-3) / 1e9 / peak,
                        "issue_active": cap.get("issue_active_pct"), "lanes_per_inst": cap.get("lanes_per_inst"),
                        "occupancy_pct": cap.get("occupancy_pct"), "l1_hit_pct": cap.get("l1_hit_pct"), "l2_hit_pct": cap.get("l2_hit_pct"),
                        "limiter": "latency of dependent node / leaf / stack fetches at ~44 % occupancy; real DRAM traffic is a small fraction of the algorithmic bytes",
                        "algorithmic_bytes_per_ray": bytes_per_ray, "nodes_per_ray": npr, "prims_per_ray": ppr,
                        "closest_rays_rank0": tot["closest"], "kernel_ms_rank0": tot["trace_closest_ms"],
                        "share_of_step": tot["trace_closest_ms"] / max(tot["device_ms"], 1e-9)}
            if tot["shade_ms"] > 0:
                # shade phase (k_classify + k_shade<material>): every closest-hit ray ends in one shaded (or escaped) vertex.  Algorithmic
                # bytes per vertex (DESIGN.md s4): 84 B path state in + 48 B leaf record + 48 B normals + 24 B prim row + 32 B sample-table
                # row + 48 B material = 284 B read; 32 B ray + 32 B L/beta + 48 B shadow ray + contribution + 4 B dim + 12 B queues = 128 B written
                shade_bpp = 412.0
                sc = prof.get("shade", {})
                sh_ach = tot["closest"] * shade_bpp / (tot["shade_ms"] * 1e-3) / 1e9
                roofline["shade"] = {"bound": "hbm", "kernel": "k_classify + k_shade<matte|plastic|metal|...>", "achieved": sh_ach, "peak": peak, "unit": "GB/s",
                                     "frac": sh_ach / peak, "algorithmic_bytes_per_vertex": shade_bpp, "vertices_rank0": tot["closest"], "kernel_ms_rank0": tot["shade_ms"],
                                     "share_of_step": tot["shade_ms"] / max(tot["device_ms"], 1e-9), "traffic": sc.get("dram_bytes"),
                                     "traffic_launch": {"ms": sc.get("ms"), "kernel": sc.get("kernel")}, "issue_active": sc.get("issue_active_pct"),
                                     "lanes_per_inst": sc.get("lanes_per_inst"), "occupancy_pct": sc.get("occupancy_pct")}
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": bench_config(desc, args.spp, world, args.paths_in_flight, args.tiles),
               "mrays_per_s": (closest + shadow) / (ms * 1e-3) / 1e6, "rays_per_sample": (closest + shadow) / max(camera, 1),
               "ray_batches": ray_batches, "per_rank": per_rank, "clocks": clk, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
               "kernel_ms": {"trace_closest": tot["trace_closest_ms"], "trace_shadow": tot["trace_any_ms"], "shade": tot["shade_ms"], "wavefront_total": tot["device_ms"]}}
        print(json.dumps(out), file=out_stream, flush=True)
    scene.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
