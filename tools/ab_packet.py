"""A/B of the packet traversal in one process on one GPU: S3 at 1920x1080, 64-spp steps (bench.py's flagship workload).

The arms are values of PBRT_B200_PACKET_TRAVERSAL, which pbrt_b200_render reads per call ("off": 0, the per-lane walk
everywhere; "on": unset, the default).  Arms alternate step by step and render the same sample ranges; each arm's film and
ray counts are checked against the first arm's.  Prints per-arm medians of the step time and of the traversal kernels' times.
PBRT_B200_LIB selects another build of the library (csrc/Makefile: make NAME=<name>)."""
import importlib
import os
import statistics
import sys

sys.path.insert(0, ".")
import numpy as np
import torch

P = importlib.import_module("pbrt-rust_b200")
ARMS = [("off", "0"), ("on", None)]
ROUNDS, SPP = int(os.environ.get("AB_ROUNDS", "6")), 64

setup = P.scenes.displaced_sphere_scene()
integ = setup.make_integrator(spp_=SPP * (ROUNDS + 2))
sc = P.Scene(setup.flat)
film = torch.zeros((integ.film.width * integ.film.height, 4), dtype=torch.float32, device="cuda")
print(torch.cuda.get_device_name(0), os.environ.get("PBRT_B200_LIB", "default library"), flush=True)


def step(knob, k):
    if knob is None:
        os.environ.pop("PBRT_B200_PACKET_TRAVERSAL", None)
    else:
        os.environ["PBRT_B200_PACKET_TRAVERSAL"] = knob
    film.zero_()
    _, st = sc.render(integ, sample_range=(k * SPP, (k + 1) * SPP), device_ptr=film.data_ptr())
    torch.cuda.synchronize()
    return st


ref = None
for name, knob in ARMS:  # warm-up, and the outputs of samples [0, 64)
    st = step(knob, 0)
    img, rays = film.cpu().numpy(), (st.camera_rays, st.intersection_tests, st.shadow_tests, st.zero_radiance_paths)
    ref = ref or (img, rays)
    same = rays == ref[1] and np.allclose(img, ref[0], rtol=2e-5, atol=2e-5)
    print(f"{name:4s} rays {rays} {'same as ' + ARMS[0][0] if same else 'DIFFERENT'}", flush=True)
res = {name: [] for name, _ in ARMS}
for r in range(ROUNDS):
    for name, knob in (ARMS if r % 2 == 0 else ARMS[::-1]):
        st = step(knob, 1 + r)
        res[name].append((st.device_ms, st.trace_closest_ms, st.trace_any_ms, st.shade_ms))
base = statistics.median(x[0] for x in res[ARMS[0][0]])
for name, _ in ARMS:
    m = [statistics.median(x[i] for x in res[name]) for i in range(4)]
    print(f"{name:4s} step {m[0]:7.2f} ms ({base / m[0] - 1:+6.1%})  closest+mis {m[1]:6.2f}  shadow {m[2]:6.2f}  shade {m[3]:6.2f}  "
          f"steps {[round(x[0], 1) for x in res[name]]}", flush=True)
if os.environ.get("AB_PROFILE"):  # one step per arm under torch.profiler: the traversal launches of the first iterations, in order
    from torch.profiler import ProfilerActivity, profile
    for name, knob in ARMS:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step(knob, 1)
        ks = sorted((e.time_range.start, e.name, e.time_range.elapsed_us()) for e in prof.events() if "k_trace" in e.name)
        print(f"{name:4s} " + "  ".join(f"{n.split('(')[0].replace('void pb::', '')} {us / 1e3:.2f}" for _, n, us in ks[:6]), flush=True)
sc.close()
