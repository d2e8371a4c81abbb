// Wavefront path tracer: SamplerIntegrator::render driving PathIntegrator::li
// (core/integrator.rs:81-403, integrators/path.rs:79-222) split into kernels:
//
//   raygen         get_camera_sample + generate_ray (samplers on device)             K1
//   trace_closest  BVHAccel::intersect for path rays, classify hit by material       K2 + K4
//   shade<mat>     emission, BSDF assembly, light pick + light sample (shadow ray),  K5 + K6
//                  MIS BSDF sample (MIS ray), BSDF sample for the next bounce, RR
//   trace_any      BVHAccel::intersect_p for shadow rays, adds the light-sample term K3
//   trace_mis      closest hit for the BSDF-sampled MIS ray, adds the BSDF-sample term K7
//   finish         radiance sanity rule + FilmTile::add_sample                       K8
//
// All queues live in HBM as index arrays; every kernel is a persistent grid-stride loop over
// a queue whose length is read from device memory, so a whole wave runs without host syncs.
//
// The kernels are compiled in three translation units, by the arithmetic they need (csrc/Makefile); device code that more than
// one unit uses is in path.cuh and recursive.cuh:
//   render.cu  (this file; --fmad=false, IEEE division / square root): ray generation, traversal, classification, film, light
//              tables, the sampler pre-pass and tables, the recursive integrators' shadow / MIS kernels, and the host side --
//              everything whose arithmetic is pinned bit for bit against the oracle;
//   shade.cu   (--use_fast_math): k_shade / k_rec_shade and their launchers;
//   mega.cu    (the flags of this file): the one-kernel forms k_zt_mega / k_vol_mega and their launchers.
#include <cuda_runtime.h>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <utility>
#include <vector>

#include "pool.h"
#include "path.cuh"
#include "recursive.cuh"

// Refill threshold of the wavefront trace kernels (lanes whose ray has finished are refilled once fewer than this many are still
// traversing).  Swept at 64 spp with runtime knobs (gpurun_out/r2q_tune.log): 16 -> 132.4 ms per step, 20 -> 133.2, 24 -> 134.7, 28 -> 136.5,
// 32 -> 141.0; interior_min 16 stays the best of 0 / 8 / 12 / 16 / 20 / 24.  (Compile-time constants: the runtime knobs cost 3 %.)
#define PB_WF_REFILL_BELOW 16

using namespace pb;

namespace pb {

// Start of a render call: every path slot is free and carries no sample.
__global__ void __launch_bounds__(256) k_init_slots(RenderDev R, uint32_t count) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        R.q_dead[1][i] = i;
        R.pixel[i] = PB_NO_SAMPLE;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) R.cnt->n_dead = count;
}


// ---------------------------------------------------------------------------
// K2: closest-hit for path rays (persistent ray queue), K4: compaction by material
// ---------------------------------------------------------------------------
struct PathClosestJob {
    RenderDev* R; const uint32_t* q;
    PB_D bool load(uint32_t i, f3* o, f3* d, float* t_max) const {
        uint32_t id = q[i];
        float4 a = R->ray[2 * id], b = R->ray[2 * id + 1];
        *o = f3(a.x, a.y, a.z); *d = f3(b.x, b.y, b.z); *t_max = a.w;
        return true;
    }
    PB_D void store(uint32_t i, const TravRay& r) const { store_closest_hit(*R, q[i], r); }
};

template <bool INST>
__global__ void __launch_bounds__(PB_TRACE_BLOCK) k_trace_closest(RenderDev R, int parity) {
    PathClosestJob job{&R, R.q_path[parity]};
    trace_queue<false, INST, PB_SH_STACK>(R.scene, job, R.cnt->n_path, &R.cnt->fetch_path, TraceTune{PB_WF_REFILL_BELOW, PB_FETCH_CHUNK, PB_INTERIOR_MIN});
}
// Packet mode (trace.cuh: trace_queue_packet) for the camera rays of a wave's first iteration, scenes without instances.  A kernel of
// its own: inside k_trace_closest<false> the packet walk took the per-lane kernel from 72 to 96 registers.  Left to itself ptxas gives
// this one 96 registers (5 CTAs of 128 threads per SM); measured on S3 (B200, 64-spp step against 114.6-114.8 ms per-lane,
// profiles/r03_packet_traversal.md): 5 CTAs 113.2 ms, 7 CTAs (71 registers) 111.4 ms, 8 CTAs (64 registers, 24 B of spills) 110.8 ms.
#define PB_TRACE_MINB_PACKET 8
__global__ void __launch_bounds__(PB_TRACE_BLOCK, PB_TRACE_MINB_PACKET) k_trace_closest_packet(RenderDev R, int parity) {
    PathClosestJob job{&R, R.q_path[parity]};
    trace_queue_packet<false, PB_SH_STACK>(R.scene, job, R.cnt->n_path, &R.cnt->fetch_path);
}
// Min resident CTAs per SM of the INSTANCED closest-hit / any-hit kernels (explicit specialisations: the plain kernels keep the compiler's
// own choice, 72 registers; note that __launch_bounds__(n, 1) is NOT "no constraint" -- it lets ptxas take 126 registers there).  Left to
// itself ptxas gives the two-level walk 96 / 80 registers = 5 / 6 CTAs of 128 threads; on S4 (gpurun_out/r2_s4_minb.log, 4-spp 4K step):
// default 303.9 ms, 6 CTAs (80 regs, closest only) 288.8, 7 CTAs (72 regs, both, 6-92 B of spills) 285.2, 8 CTAs (64 regs) 309.6.
#define PB_TRACE_MINB_INST 7
#define PB_TRACE_MINB_INST_ANY 7
template <>
__global__ void __launch_bounds__(PB_TRACE_BLOCK, PB_TRACE_MINB_INST) k_trace_closest<true>(RenderDev R, int parity) {
    PathClosestJob job{&R, R.q_path[parity]};
    trace_queue<false, true, PB_SH_STACK>(R.scene, job, R.cnt->n_path, &R.cnt->fetch_path, TraceTune{PB_WF_REFILL_BELOW, PB_FETCH_CHUNK, PB_INTERIOR_MIN});
}

// sort/compact-by-material.  Lanes of the same bin form a group (match.any) and the groups of the CTA's eight warps are
// added up in shared memory: one atomicAdd per bin per 256 paths (the per-warp form waited on the atomic's round trip for 83 % of
// its stall samples, profiles/r02_ncu_classify.md), queue order = path-queue order within a CTA's span.
__global__ void __launch_bounds__(256) k_classify(RenderDev R, int parity) {
    const uint32_t n = R.cnt->n_path;
    const uint32_t* q = R.q_path[parity];
    const uint32_t nround = (n + 255u) & ~255u;  // CTA-uniform trip count (barriers inside)
    __shared__ uint32_t s_cnt[8][Q_COUNT], s_base[Q_COUNT];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nround; i += gridDim.x * blockDim.x) {
        bool valid = i < n;
        uint32_t id = valid ? q[i] : 0u;
        int bin = valid ? (int)R.hit_bin[id] : -1;
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (lane < Q_COUNT) s_cnt[warp][lane] = 0;
        __syncwarp();
        if (valid && (int)lane == __ffs(peers) - 1) s_cnt[warp][bin] = (uint32_t)__popc(peers);
        __syncthreads();
        if (threadIdx.x < Q_COUNT) {
            uint32_t sum = 0;
            for (int w = 0; w < 8; ++w) { const uint32_t c = s_cnt[w][threadIdx.x]; s_cnt[w][threadIdx.x] = sum; sum += c; }
            s_base[threadIdx.x] = sum ? atomicAdd(&R.cnt->n_mat[threadIdx.x], sum) : 0u;
        }
        __syncthreads();
        if (valid) R.q_mat[bin][s_base[bin] + s_cnt[warp][bin] + __popc(peers & ((1u << lane) - 1u))] = id;
        __syncthreads();
    }
}


// ---------------------------------------------------------------------------
// SpatialLightDistribution
// ---------------------------------------------------------------------------
// compute_dsitribution, lightdistrib.rs:152-228: one CTA per voxel; thread j owns lights j, j+blockDim, ... and walks the
// 128 Halton points in order (same accumulation order as the reference); the sum / floor / cdf passes that the reference
// does sequentially are done by one thread so the f32 roundings match.
template <bool SPH>
__global__ void __launch_bounds__(128) k_spatial_build(RenderDev R, int eager, uint32_t n_eager) {
    const SpatialDev& S = R.sp;
    const uint32_t n = eager ? n_eager : S.counters[0];
    const uint32_t nl = R.n_lights;
    __shared__ float s_min;
    for (uint32_t e = blockIdx.x; e < n; e += gridDim.x) {
        uint32_t voxel, slot;
        if (eager) { voxel = e; slot = e; } else { uint2 vs = S.build_list[e]; voxel = vs.x; slot = vs.y; }
        int px = (int)(voxel % (uint32_t)S.nvox[0]), py = (int)((voxel / (uint32_t)S.nvox[0]) % (uint32_t)S.nvox[1]), pz = (int)(voxel / ((uint32_t)S.nvox[0] * (uint32_t)S.nvox[1]));
        const float* wb = R.scene.root_box;
        float lo[3], hi[3];
        const int pi[3] = {px, py, pz};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            float t0 = (float)pi[k] / (float)S.nvox[k], t1 = (float)(pi[k] + 1) / (float)S.nvox[k];
            float a = wb[k] * (1.0f - t0) + wb[3 + k] * t0, b = wb[k] * (1.0f - t1) + wb[3 + k] * t1;  // pbrt::lerp
            lo[k] = fminf(a, b); hi[k] = fmaxf(a, b);
        }
        float* func = S.func + (size_t)slot * nl;
        float* cdf = S.cdf + (size_t)slot * (nl + 1);
        for (uint32_t j = threadIdx.x; j < nl; j += blockDim.x) {
            float contrib = 0.0f;
            for (int i = 0; i < 128; ++i) {
                const float* h = S.halton + 5 * i;
                f3 po(lo[0] * (1.0f - h[0]) + hi[0] * h[0], lo[1] * (1.0f - h[1]) + hi[1] * h[1], lo[2] * (1.0f - h[2]) + hi[2] * h[2]);
                LightSample ls;
                ls.pdf = 0.0f; ls.Li = rgb(0.0f);
                light_sample_li<SPH>(R, j, po, make_float2(h[3], h[4]), ls);
                if (ls.pdf > 0.0f) contrib += lum(ls.Li) / ls.pdf;
            }
            func[j] = contrib;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            float sum = 0.0f;
            for (uint32_t j = 0; j < nl; ++j) sum += func[j];
            float avg = sum / (128.0f * (float)nl);
            s_min = avg > 0.0f ? 0.001f * avg : 1.0f;
        }
        __syncthreads();
        const float mc = s_min;
        for (uint32_t j = threadIdx.x; j < nl; j += blockDim.x) func[j] = fmaxf(func[j], mc);
        __syncthreads();
        if (threadIdx.x == 0) {  // Distribution1D::new, sampling.rs:13-33
            float c = 0.0f;
            cdf[0] = 0.0f;
            for (uint32_t j = 1; j <= nl; ++j) { c = c + func[j - 1] / (float)nl; cdf[j] = c; }
            S.func_int[slot] = c;
            s_min = c;
        }
        __syncthreads();
        const float fi = s_min;
        for (uint32_t j = 1 + threadIdx.x; j <= nl; j += blockDim.x) cdf[j] = (fi == 0.0f) ? (float)j / (float)nl : cdf[j] / fi;
        __syncthreads();
        if (threadIdx.x == 0) { __threadfence(); S.slot[voxel] = (int)slot; }
    }
}

// lazy mode: claim the voxels of this iteration's hits (the ones the shade kernels are about to look up)
__global__ void __launch_bounds__(256) k_spatial_mark(RenderDev R, int parity) {
    const uint32_t n = R.cnt->n_path;
    const uint32_t* q = R.q_path[parity];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint32_t id = q[i];
        if (R.hit_bin[id] == Q_MISS) continue;
        float4 ra = R.ray[2 * id], rb = R.ray[2 * id + 1];
        uint4 h = R.hit[id];
        uint32_t fl;
        const uint32_t hinst = R.scene.n_instances ? R.hit_inst[id] : PBRT_B200_NO_HIT;
        Surf si = surface_at_hit<true>(R.scene, hinst, h.x, f3(ra.x, ra.y, ra.z), f3(rb.x, rb.y, rb.z), __uint_as_float(h.y), __uint_as_float(h.z), __uint_as_float(h.w),
                                 R.hit_b2[id], &fl);
        int v = spatial_voxel(R, si.p);
        R.sp_voxel[id] = v;
        if (R.sp.slot[v] != -1) continue;
        if (atomicCAS(R.sp.slot + v, -1, -2) == -1) {
            uint32_t sl = atomicAdd(R.sp.counters + 1, 1u);
            if (sl < R.sp.capacity) R.sp.build_list[atomicAdd(R.sp.counters, 1u)] = make_uint2((uint32_t)v, sl);
            else atomicExch(R.sp.counters + 2, 1u);
        }
    }
}
__global__ void k_spatial_reset(SpatialDev S) { S.counters[0] = 0; }
// batch LightDistribution::lookup for caller-supplied points (pbrt_b200_light_distribution_lookup)
__global__ void __launch_bounds__(256) k_spatial_mark_points(RenderDev R, const float* pts, uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        int v = spatial_voxel(R, f3(pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]));
        if (R.sp.slot[v] != -1) continue;
        if (atomicCAS(R.sp.slot + v, -1, -2) == -1) {
            uint32_t sl = atomicAdd(R.sp.counters + 1, 1u);
            if (sl < R.sp.capacity) R.sp.build_list[atomicAdd(R.sp.counters, 1u)] = make_uint2((uint32_t)v, sl);
            else atomicExch(R.sp.counters + 2, 1u);
        }
    }
}
__global__ void __launch_bounds__(256) k_light_distrib_gather(RenderDev R, const float* pts, uint32_t n, int* voxel_out, float* func_out) {
    const uint32_t nl = R.n_lights;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float* func = R.ld_func;
        int vx = -1, vy = -1, vz = -1;
        if (R.sp.enabled) {
            int v = spatial_voxel(R, f3(pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]));
            vx = v % R.sp.nvox[0]; vy = (v / R.sp.nvox[0]) % R.sp.nvox[1]; vz = v / (R.sp.nvox[0] * R.sp.nvox[1]);
            int sl = R.sp.slot[v];
            func = sl >= 0 ? R.sp.func + (size_t)sl * nl : nullptr;
        }
        voxel_out[3 * i] = vx; voxel_out[3 * i + 1] = vy; voxel_out[3 * i + 2] = vz;
        for (uint32_t j = 0; j < nl; ++j) func_out[(size_t)i * nl + j] = func ? func[j] : -1.0f;
    }
}


// ---------------------------------------------------------------------------
// sampler pre-pass and Sobol' table builders
// ---------------------------------------------------------------------------
// The eight dimensions a hit path is about to consume, for paths the Sobol' tables do not serve (see PathSampler<false>):
// Halton (scrambled radical inverses), and Sobol' dimensions past the tables (deep paths when the table size was capped).
// Keeps the radical-inverse loops and the Sobol' bit walk out of the shade kernels (1 900 of the matte kernel's 9 950 SASS
// instructions were Halton code that a Sobol' render never runs, DESIGN.md s5).
__global__ void __launch_bounds__(256) k_sample_block(RenderDev R, int parity) {
    const uint32_t n = R.cnt->n_path;
    const uint32_t* q = R.q_path[parity];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t id = q[i];
        if (R.hit_bin[id] == Q_MISS) continue;
        SampleCursor c;
        c.dim = R.s_dim[id];
        if (sobol_tab_covers(R.sampler, c.dim)) continue;
        const uint32_t pxy = R.pixel[id];
        c.px = (int)(pxy & 0xffffu) + R.sampler.sb[0]; c.py = (int)(pxy >> 16) + R.sampler.sb[1];
        c.index = R.s_index[id];
        if (R.sampler.vdims)  // table mode: the slot holds the sample number
            c.index = sobol_interval_to_index(R.sampler, (uint32_t)R.sampler.log2_resolution, c.index, (int)(pxy & 0xffffu), (int)(pxy >> 16));
        SampleBlock b;
        sample_block(R.sampler, c, b);
        R.u8[2 * id] = make_float4(b.u[0], b.u[1], b.u[2], b.u[3]);
        R.u8[2 * id + 1] = make_float4(b.u[4], b.u[5], b.u[6], b.u[7]);
    }
}

// XOR of the generator-matrix columns of dimensions d0..d0+3 over the set bits of `a` (sobol_sample_float's inner loop)
PB_D uint4 sobol_bits4(const uint32_t* sobol_t, unsigned long long a, uint32_t d0) {
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    a &= (1ull << 52) - 1ull;  // SOBOL_MATRIX_SIZE columns; the reference indexes past the table (panics) beyond that
    while (a != 0) {
        const int bit = __ffsll((long long)a) - 1;
        a &= a - 1;
        const uint4 m = __ldg(reinterpret_cast<const uint4*>(sobol_t + (uint32_t)bit * 1024u + d0));
        v.x ^= m.x; v.y ^= m.y; v.z ^= m.z; v.w ^= m.w;
    }
    return v;
}
// vp[pixel][d]: one thread per (pixel, 4 dimensions), dimensions fastest so that a warp writes contiguous rows
__global__ void __launch_bounds__(256) k_sobol_table_pixels(SamplerDev S, uint32_t* vp, uint32_t npix) {
    const uint32_t groups = S.vstride / 4u;
    const unsigned long long total = (unsigned long long)npix * groups;
    const unsigned long long* VI = S.vdc_inv + (S.log2_resolution - 1) * 52;
    for (unsigned long long t = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; t < total; t += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t pix = (uint32_t)(t / groups), g = (uint32_t)(t % groups);
        const uint32_t px = pix % S.sbw, py = pix / S.sbw;
        unsigned long long b = ((unsigned long long)px << S.log2_resolution) | (unsigned long long)py, ip = 0;
        for (int c = 0; b != 0; b >>= 1, ++c)
            if (b & 1) ip ^= __ldg(VI + c);
        reinterpret_cast<uint4*>(vp)[t] = sobol_bits4(S.sobol_t, ip, 4u * g);
    }
}
// vs[s - s_begin][d]
__global__ void __launch_bounds__(256) k_sobol_table_samples(SamplerDev S, uint32_t* vs, uint32_t s_begin, uint32_t n_samples) {
    const uint32_t groups = S.vstride / 4u;
    const unsigned long long total = (unsigned long long)n_samples * groups;
    const uint32_t m = (uint32_t)S.log2_resolution;
    const unsigned long long* V = S.vdc + (m - 1) * 52;
    const unsigned long long* VI = S.vdc_inv + (m - 1) * 52;
    for (unsigned long long t = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; t < total; t += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long frame = s_begin + (uint32_t)(t / groups);
        const uint32_t g = (uint32_t)(t % groups);
        unsigned long long delta = 0, is = frame << (2u * m);
        unsigned long long f = frame;
        for (int c = 0; f != 0; f >>= 1, ++c)
            if (f & 1) delta ^= __ldg(V + c);
        for (int c = 0; delta != 0; delta >>= 1, ++c)
            if (delta & 1) is ^= __ldg(VI + c);
        reinterpret_cast<uint4*>(vs)[t] = sobol_bits4(S.sobol_t, is, 4u * g);
    }
}


// ---------------------------------------------------------------------------
// K3: shadow rays (VisibilityTester::unoccluded, core/light.rs:120-123)
// ---------------------------------------------------------------------------
struct ShadowJob {
    RenderDev* R;
    PB_D bool load(uint32_t i, f3* o, f3* d, float* t_max) const {
        uint32_t id = R->q_shadow[i];
        float4 a = R->sh_ray[2 * id], b = R->sh_ray[2 * id + 1];
        *o = f3(a.x, a.y, a.z); *d = f3(b.x, b.y, b.z); *t_max = a.w;
        return true;
    }
    PB_D void store(uint32_t i, const TravRay& r) const {
        if (r.found) return;
        shadow_unoccluded(*R, R->q_shadow[i]);
    }
};
template <bool INST>
__global__ void __launch_bounds__(PB_TRACE_BLOCK) k_trace_shadow(RenderDev R) {
    ShadowJob job{&R};
    trace_queue<true, INST, PB_SH_STACK>(R.scene, job, R.cnt->n_shadow, &R.cnt->fetch_shadow, TraceTune{PB_WF_REFILL_BELOW, PB_FETCH_CHUNK, PB_INTERIOR_MIN});
}
template <>
__global__ void __launch_bounds__(PB_TRACE_BLOCK, PB_TRACE_MINB_INST_ANY) k_trace_shadow<true>(RenderDev R) {
    ShadowJob job{&R};
    trace_queue<true, true, PB_SH_STACK>(R.scene, job, R.cnt->n_shadow, &R.cnt->fetch_shadow, TraceTune{PB_WF_REFILL_BELOW, PB_FETCH_CHUNK, PB_INTERIOR_MIN});
}

// ---------------------------------------------------------------------------
// K7: MIS rays (estimate_direct's BSDF-sampled branch, integrator.rs:205-234)
// ---------------------------------------------------------------------------
template <bool INST>
struct MisJob {
    RenderDev* R;
    PB_D bool load(uint32_t i, f3* o, f3* d, float* t_max) const {
        uint32_t id = R->q_mis[i];
        float4 a = R->mis_ray[2 * id], b = R->mis_ray[2 * id + 1];
        *o = f3(a.x, a.y, a.z); *d = f3(b.x, b.y, b.z); *t_max = a.w;
        return true;
    }
    PB_D void store(uint32_t i, const TravRay& r) const { mis_resolve<INST>(*R, R->q_mis[i], r); }
};
template <bool INST>
__global__ void __launch_bounds__(PB_TRACE_BLOCK) k_trace_mis(RenderDev R) {
    MisJob<INST> job{&R};
    trace_queue<false, INST, PB_SH_STACK>(R.scene, job, R.cnt->n_mis, &R.cnt->fetch_mis, TraceTune{PB_WF_REFILL_BELOW, PB_FETCH_CHUNK, PB_INTERIOR_MIN});
}

// ---------------------------------------------------------------------------
// recursive integrators (recursive.cuh): the shadow and MIS entries of k_rec_shade
// ---------------------------------------------------------------------------
struct RecShadowJob {
    RenderDev* R;
    PB_D bool load(uint32_t e, f3* o, f3* d, float* t_max) const {
        float4 a = R->rec.e_sh_ray[2 * e], b = R->rec.e_sh_ray[2 * e + 1];
        *o = f3(a.x, a.y, a.z); *d = f3(b.x, b.y, b.z); *t_max = a.w;
        return true;
    }
    PB_D void store(uint32_t e, const TravRay& r) const {
        if (r.found) return;
        float4 c = R->rec.e_sh_contrib[e];
        rec_atomic_add(R->L_eta, __float_as_uint(c.w), rgb(c.x, c.y, c.z));
    }
};
template <bool INST>
__global__ void __launch_bounds__(PB_TRACE_BLOCK) k_rec_shadow(RenderDev R) {
    RecShadowJob job{&R};
    trace_queue<true, INST, PB_SH_STACK>(R.scene, job, R.cnt->n_shadow, &R.cnt->fetch_shadow);
}

template <bool INST>
struct RecMisJob {
    RenderDev* R;
    PB_D bool load(uint32_t e, f3* o, f3* d, float* t_max) const {
        float4 a = R->rec.e_mis_ray[2 * e], b = R->rec.e_mis_ray[2 * e + 1];
        *o = f3(a.x, a.y, a.z); *d = f3(b.x, b.y, b.z); *t_max = a.w;
        return true;
    }
    PB_D void store(uint32_t e, const TravRay& r) const {  // integrator.rs:205-234, as MisJob::store
        float4 c = R->rec.e_mis_contrib[e];
        uint32_t ln = __float_as_uint(c.w);
        rgb li(0.0f);
        if (r.found) {
            const pbrt_b200_prim pr = R->scene.prims[r.hit.slot];
            if (pr.area_light == (int)ln) {
                uint32_t fl;
                Surf ls = surface_at_hit<INST>(R->scene, r.hit.inst, r.hit.slot, r.o, r.d, r.hit.t, r.hit.b0, r.hit.b1, r.hit.b2, &fl);
                const pbrt_b200_light& al = R->scene.lights[ln];
                if (al.two_sided || dot(ls.n, -r.d) > 0.0f) li = rgb3(al.L);
            }
        } else {
            const pbrt_b200_light& l = R->scene.lights[ln];
            if (l.type == PBRT_B200_LIGHT_INFINITE) li = rgb3(l.L);
        }
        if (!is_black(li)) rec_atomic_add(R->L_eta, R->rec.e_mis_slot[e], rgb(c.x * li.r, c.y * li.g, c.z * li.b));
    }
};
template <bool INST>
__global__ void __launch_bounds__(PB_TRACE_BLOCK) k_rec_mis(RenderDev R) {
    RecMisJob<INST> job{&R};
    trace_queue<false, INST, PB_SH_STACK>(R.scene, job, R.cnt->n_mis, &R.cnt->fetch_mis);
}

// ---------------------------------------------------------------------------
// K8: finished paths -> film
// ---------------------------------------------------------------------------
// K8 + K1 fused ("path regeneration"): a finished path adds its sample to the film, then its slot is handed the next
// camera sample of the call, so every iteration traces a full complement of rays instead of the dwindling tail of one wave.
__global__ void __launch_bounds__(256) k_finish_regen(RenderDev R, int parity, unsigned long long total_items) {
    const uint32_t n = R.cnt->n_dead;
    // every thread of a CTA runs the same number of iterations: the appends below are aggregated per CTA (two barriers per iteration)
    const uint32_t nround = (n + 255u) & ~255u;
    const unsigned long long cursor = R.cnt->item_cursor;  // advanced by k_iter_end
    const unsigned long long remaining = total_items > cursor ? total_items - cursor : 0ull;
    const uint32_t* q = R.q_dead[parity];
    __shared__ uint32_t s_cnt[8][2], s_base[2];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, below = (1u << lane) - 1u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nround; i += gridDim.x * blockDim.x) {
        bool valid = i < n, has_sample = false;
        rgb L(0.0f);
        float2 pf = make_float2(0.f, 0.f);
        uint32_t id = 0;
        if (valid) {
            id = q[i];
            has_sample = R.pixel[id] != PB_NO_SAMPLE;
        }
        if (has_sample) {
            float4 Le = R.L_eta[id];
            pf = R.pfilm[id];
            L = rgb(Le.x, Le.y, Le.z);
            // integrator.rs:350-368: NaN / negative / infinite luminance => black
            float y = lum(L);
            if (L.r != L.r || L.g != L.g || L.b != L.b) L = rgb(0.0f);
            else if (y < -1.0e-5f) L = rgb(0.0f);
            else if (isinf(y)) L = rgb(0.0f);
        }
        film_add_sample(R, pf, L, has_sample);
        bool regen = valid && (unsigned long long)i < remaining, ok = false;
        if (regen) ok = gen_camera_path(R, cursor + i, id);
        // Appends, aggregated per CTA: at the start of a wave every slot of the call regenerates (33 M camera paths on S3), and one
        // atomicAdd per WARP on the single counter n_next serialised at its L2 slice -- 56 % of the kernel's stall samples, 4.2 of the
        // 40 ms of a 16-spp step (profiles/r02_ncu_regen.md).  One atomic per 256 paths instead.
        const bool again = regen && !ok;
        const unsigned m = __ballot_sync(0xffffffffu, ok), m1 = __ballot_sync(0xffffffffu, again);
        if (lane == 0) { s_cnt[warp][0] = (uint32_t)__popc(m); s_cnt[warp][1] = (uint32_t)__popc(m1); }
        __syncthreads();
        if (threadIdx.x < 2) {
            uint32_t sum = 0;
            for (int w = 0; w < 8; ++w) { const uint32_t c = s_cnt[w][threadIdx.x]; s_cnt[w][threadIdx.x] = sum; sum += c; }
            uint32_t base = 0;
            if (sum) base = atomicAdd(threadIdx.x == 0 ? &R.cnt->n_next : &R.cnt->n_dead_next, sum);
            if (threadIdx.x == 0 && sum) atomicAdd(&R.cnt->camera_rays, (unsigned long long)sum);
            s_base[threadIdx.x] = base;
        }
        __syncthreads();
        if (ok) R.q_path[parity ^ 1][s_base[0] + s_cnt[warp][0] + __popc(m & below)] = id;
        if (again) R.q_dead[parity ^ 1][s_base[1] + s_cnt[warp][1] + __popc(m1 & below)] = id;
        __syncthreads();  // s_cnt / s_base are rewritten by the next iteration
    }
}

// ---------------------------------------------------------------------------
// (0,2)-sequence: tile-serial sample generation (zt_next_path, path.cuh)
// ---------------------------------------------------------------------------
// tile j of the call -> tile number, clipped bounds, generator (sampler.clone(seed = tile.y * ntiles.x + tile.x), integrator.rs:302-303)
__global__ void __launch_bounds__(128) k_zt_init(RenderDev R) {
    const uint32_t n = R.n_tiles_sel;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < ((n + 31u) & ~31u); j += gridDim.x * blockDim.x) {
        bool ok = false;
        if (j < n) {
            uint32_t t = R.tile_begin + ((j / R.tile_group) * R.tile_mod + R.tile_rem) * R.tile_group + (j % R.tile_group);
            ZtTile* tp = R.zt.tiles + j;
            R.pixel[j] = PB_NO_SAMPLE;
            int tx, ty;
            if (tile_xy(R, t, &tx, &ty) && t < R.tile_end) {
                int x0 = R.sampler.sb[0] + tx * 16, y0 = R.sampler.sb[1] + ty * 16;
                int x1 = min(x0 + 16, R.sampler.sb[2]), y1 = min(y0 + 16, R.sampler.sb[3]);
                tp->x0 = x0; tp->y0 = y0; tp->w = (uint32_t)max(x1 - x0, 0); tp->npix = tp->w * (uint32_t)max(y1 - y0, 0);
                tp->pixel_idx = 0; tp->sample_idx = 0; tp->cur1d = 0; tp->cur2d = 0;
                zt_set_sequence(*tp, (unsigned long long)((long long)ty * R.ntx + tx));
                ok = zt_next_path(R, j, true);
            }
        }
        unsigned m = __ballot_sync(0xffffffffu, ok);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(&R.cnt->camera_rays, (unsigned long long)__popc(m));
        queue_push(R.q_path[0], &R.cnt->n_next, j, ok);
    }
}
// finished paths -> film; their tile moves on to its next sample
__global__ void __launch_bounds__(128) k_finish_zt(RenderDev R, int parity) {
    const uint32_t n = R.cnt->n_dead;
    const uint32_t nround = (n + 31u) & ~31u;
    const uint32_t* q = R.q_dead[parity];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nround; i += gridDim.x * blockDim.x) {
        bool valid = i < n;
        rgb L(0.0f);
        float2 pf = make_float2(0.f, 0.f);
        uint32_t id = 0;
        if (valid) {
            id = q[i];
            float4 Le = R.L_eta[id];
            L = rgb(Le.x, Le.y, Le.z);
            pf = R.pfilm[id];
            float y = lum(L);  // integrator.rs:350-368
            if (L.r != L.r || L.g != L.g || L.b != L.b) L = rgb(0.0f);
            else if (y < -1.0e-5f) L = rgb(0.0f);
            else if (isinf(y)) L = rgb(0.0f);
        }
        film_add_sample(R, pf, L, valid);
        bool ok = valid && zt_next_path(R, id, false);
        unsigned m = __ballot_sync(0xffffffffu, ok);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(&R.cnt->camera_rays, (unsigned long long)__popc(m));
        queue_push(R.q_path[parity ^ 1], &R.cnt->n_next, id, ok);
    }
}

// single-thread bookkeeping between iterations: roll queue counters, accumulate stats
__global__ void k_iter_end(Counters* c, unsigned long long total_items) {
    c->closest_rays += (unsigned long long)c->n_path + c->n_mis;
    c->shadow_rays += c->n_shadow;
    unsigned long long remaining = total_items > c->item_cursor ? total_items - c->item_cursor : 0ull;
    c->item_cursor += remaining < (unsigned long long)c->n_dead ? remaining : (unsigned long long)c->n_dead;
    c->n_path = c->n_next;
    c->n_dead = c->n_dead_next;
    c->n_next = 0; c->n_shadow = 0; c->n_mis = 0; c->n_dead_next = 0;
    c->fetch_path = 0; c->fetch_shadow = 0; c->fetch_mis = 0;
    for (int k = 0; k < Q_COUNT; ++k) c->n_mat[k] = 0;
    c->iterations += 1;
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
struct RenderBuffers {  // all path-state arrays and queues sub-allocated from ONE pooled block (pool.h)
    void* block = nullptr;
    size_t block_bytes = 0;
    uint32_t capacity = 0;
    RenderDev dev;
    void* u8_block = nullptr;   // RenderDev::u8, allocated on first need (Halton, capped Sobol' tables)
    size_t u8_bytes = 0;
    void* diff_block = nullptr; // RenderDev::rdiff, allocated on first need (scenes with textured materials)
    size_t diff_bytes = 0;
    ~RenderBuffers() { pool_free(block, block_bytes); if (u8_block) pool_free(u8_block, u8_bytes); if (diff_block) pool_free(diff_block, diff_bytes); }
};

// Resources that depend only on the DEVICE, shared by every scene rendered on it and kept for the life of the process:
// sampler tables (the reference's compile-time constants), pinned progress ring, CUDA events.  Render calls on one device
// are serialised by `mu` (the reference calls Integrator::render from one thread, api.rs:1740-1747).
struct DeviceShared {
    std::mutex mu;
    // Halton tables (lowdiscrepancy.rs:359-378: permutations from the default-seeded RNG => a constant)
    uint16_t* perms = nullptr; uint32_t* primes = nullptr; uint32_t* prime_sums = nullptr; uint32_t n_halton_dims = 0;
    // Sobol tables copied to the device, keyed by a hash of the caller's arrays
    uint32_t* sobol32 = nullptr; uint32_t* sobol_t = nullptr; unsigned long long* vdc = nullptr; unsigned long long* vdc_inv = nullptr;
    unsigned long long sobol_hash = 0;
    float* filter_table = nullptr;
    // Sobol' sample tables (SamplerDev::vp / vs), pooled blocks; vp is rebuilt only when its key changes
    uint32_t* vp = nullptr; size_t vp_block = 0; unsigned long long vp_key[4] = {0, 0, 0, 0};
    uint32_t* vs = nullptr; size_t vs_block = 0;
    struct Progress { unsigned long long cursor; uint32_t n_path; uint32_t pad; };
    Progress* prog = nullptr;            // pinned, PB_PROG_RING entries
    std::vector<cudaEvent_t> events;     // pool, grown on demand
};
#define PB_PROG_RING 4
static DeviceShared* device_shared(int device) {
    static std::mutex m;
    static DeviceShared* tab[64] = {nullptr};
    std::lock_guard<std::mutex> g(m);
    if (device < 0 || device >= 64) device = 0;
    if (!tab[device]) tab[device] = new DeviceShared();  // never freed: outlives every scene; CUDA may be gone at exit
    return tab[device];
}

struct SceneRenderState {  // cached per scene: light tables + path-state buffers (pooled blocks)
    float* ld_func = nullptr; float* ld_cdf = nullptr; float ld_func_int = 0;
    InfDistrib* inf = nullptr; uint32_t* inf_list = nullptr; uint32_t n_inf = 0;
    int strategy = -1;
    std::vector<std::pair<void*, size_t>> light_blocks;  // pooled
    RenderBuffers* buffers = nullptr;
    std::vector<pbrt_b200_light> lights_host;
    bool lights_cached = false;
    // SpatialLightDistribution tables (persist across render calls of the scene: lazily built voxels stay built)
    SpatialDev sp = {};
    bool sp_eager_pending = false;
    DeviceShared* shared = nullptr;
    void release_light_blocks() {
        for (auto& b : light_blocks) pool_free(b.first, b.second);
        light_blocks.clear();
        ld_func = ld_cdf = nullptr; inf = nullptr; inf_list = nullptr;
        sp = SpatialDev{}; sp_eager_pending = false;
    }
};

void render_release_scene_state(pbrt_b200_scene* sc) {  // caller has synchronised the device
    SceneRenderState* st = reinterpret_cast<SceneRenderState*>(sc->light_distrib);
    if (!st) return;
    st->release_light_blocks();
    delete st->buffers;
    delete st;
    sc->light_distrib = nullptr;
}

}  // namespace pb

namespace {

// Distribution1D::new, core/sampling.rs:13-33
void make_distribution(const std::vector<float>& func, std::vector<float>& cdf, float* func_int) {
    size_t n = func.size();
    cdf.assign(n + 1, 0.0f);
    for (size_t i = 1; i < n + 1; ++i) cdf[i] = cdf[i - 1] + func[i - 1] / (float)n;
    *func_int = cdf[n];
    if (*func_int == 0.0f) { for (size_t i = 1; i < n + 1; ++i) cdf[i] = (float)i / (float)n; }
    else { for (size_t i = 1; i < n + 1; ++i) cdf[i] /= *func_int; }
}
Tiny1D make_tiny(float f0, float f1) {
    std::vector<float> cdf; float fi;
    make_distribution({f0, f1}, cdf, &fi);
    Tiny1D t; t.func[0] = f0; t.func[1] = f1; t.cdf[0] = cdf[0]; t.cdf[1] = cdf[1]; t.cdf[2] = cdf[2]; t.func_int = fi;
    return t;
}
float lum_host(const float* c) { return 0.212671f * c[0] + 0.715160f * c[1] + 0.072169f * c[2]; }

// PCG32 + shuffle for compute_radical_inverse_permutations (core/rng.rs:25-76, sampling.rs:178-186,
// lowdiscrepancy.rs:359-378)
struct Pcg32 {
    uint64_t state = 0x853c49e6748fea9bULL, inc = 0xda3e39cb94b95bdbULL;
    uint32_t next() {
        uint64_t old = state;
        state = old * 0x5851f42d4c957f2dULL + inc;
        uint32_t xs = (uint32_t)(((old >> 18) ^ old) >> 27), rot = (uint32_t)(old >> 59);
        return (xs >> rot) | (xs << ((~rot + 1u) & 31));
    }
    uint32_t bounded(uint32_t b) { uint32_t th = (~b + 1u) % b; for (;;) { uint32_t r = next(); if (r >= th) return r % b; } }
};

template <typename T> int pooled_alloc(std::vector<std::pair<void*, size_t>>& owner, T** d, size_t count) {
    size_t got = 0;
    *d = reinterpret_cast<T*>(pool_alloc(count * sizeof(T), &got));
    if (!*d) return fail(PBRT_B200_ERR_CUDA, "render: out of device memory");
    owner.push_back({*d, got});
    return PBRT_B200_OK;
}
template <typename T> int to_device(std::vector<std::pair<void*, size_t>>& owner, const std::vector<T>& h, T** d) {
    *d = nullptr;
    if (h.empty()) return PBRT_B200_OK;
    int rc = pooled_alloc(owner, d, h.size());
    if (rc) return rc;
    PB_CUDA_TRY(cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    return PBRT_B200_OK;
}
template <typename T> int to_device_once(const std::vector<T>& h, T** d) {  // device-shared tables: never freed (pool_alloc: trims the cache and retries)
    size_t got = 0;
    *d = reinterpret_cast<T*>(pool_alloc(h.size() * sizeof(T), &got));
    if (!*d) return fail(PBRT_B200_ERR_CUDA, "render: out of device memory for the sampler tables");
    PB_CUDA_TRY(cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    return PBRT_B200_OK;
}

// Scene-level light tables: create_light_sample_distribution (core/lightdistrib.rs:20-31) + infinite-light distributions.
int prepare_light_state(pbrt_b200_scene* sc, uint32_t strategy, uint32_t flags, SceneRenderState** out) {
    SceneRenderState* st = reinterpret_cast<SceneRenderState*>(sc->light_distrib);
    if (!st) { st = new SceneRenderState(); sc->light_distrib = st; }
    *out = st;
    int rc;
    if (!st->lights_cached) {  // lights live on the device; fetch them once per scene for the host-side distribution build
        st->lights_host.resize(sc->dev.n_lights);
        if (!st->lights_host.empty())
            PB_CUDA_TRY(cudaMemcpy(st->lights_host.data(), sc->dev.lights, st->lights_host.size() * sizeof(pbrt_b200_light), cudaMemcpyDeviceToHost));
        st->lights_cached = true;
    }
    const std::vector<pbrt_b200_light>& lights = st->lights_host;
    const size_t nl = lights.size();
    const int key = (int)strategy | ((flags & PBRT_B200_RENDER_LAZY_SPATIAL) ? 0x100 : 0);
    if (st->strategy != key) {
        if (st->strategy != -1) cudaDeviceSynchronize();
        st->release_light_blocks();
        // create_light_sample_distribution, core/lightdistrib.rs:20-31 ("spatial" is not built yet: DESIGN.md)
        std::vector<float> func(nl, 1.0f), cdf;
        const float wr = sc->dev.world_radius, PI = 3.14159265358979323846f;
        bool uniform = strategy == PBRT_B200_LIGHTS_UNIFORM || nl == 1;
        std::vector<InfDistrib> inf(nl);
        std::vector<uint32_t> inf_list;
        for (size_t i = 0; i < nl; ++i) {
            const pbrt_b200_light& l = lights[i];
            float p[3];
            for (int k = 0; k < 3; ++k) {
                switch (l.type) {  // Light::power
                    case PBRT_B200_LIGHT_POINT: p[k] = l.L[k] * 4.0f * PI; break;
                    case PBRT_B200_LIGHT_DISTANT: p[k] = l.L[k] * PI * wr * wr; break;
                    case PBRT_B200_LIGHT_SPOT: p[k] = l.L[k] * 2.0f * PI * (1.0f - 0.5f * (l.cos_falloff_start + l.cos_total_width)); break;
                    case PBRT_B200_LIGHT_DIFFUSE: p[k] = l.L[k] * l.area * PI; break;
                    default: p[k] = l.L[k] * wr * wr * PI; break;
                }
            }
            if (!uniform && strategy == PBRT_B200_LIGHTS_POWER) func[i] = lum_host(p);
            if (l.type == PBRT_B200_LIGHT_INFINITE) {
                inf_list.push_back((uint32_t)i);
                float y = lum_host(l.L);
                float s0 = sinf(PI * (0.0f + 0.5f) / 2.0f), s1 = sinf(PI * (1.0f + 0.5f) / 2.0f);
                inf[i].cond[0] = make_tiny(y * s0, y * s0);
                inf[i].cond[1] = make_tiny(y * s1, y * s1);
                inf[i].marg = make_tiny(inf[i].cond[0].func_int, inf[i].cond[1].func_int);
            }
        }
        // SpatialLightDistribution::new, lightdistrib.rs:113-150 (max_voxels = 64, lightdistrib.rs:26)
        if (!uniform && strategy == PBRT_B200_LIGHTS_SPATIAL && sc->n_nodes > 0) {
            SpatialDev& sp = st->sp;
            const float* wb = sc->dev.root_box;
            float diag[3] = {wb[3] - wb[0], wb[4] - wb[1], wb[5] - wb[2]};
            int me = (diag[0] > diag[1] && diag[0] > diag[2]) ? 0 : (diag[1] > diag[2] ? 1 : 2);  // bounds.rs:346-360
            float bmax = diag[me];
            size_t total = 1;
            for (int i = 0; i < 3; ++i) {
                float r = roundf(diag[i] / bmax * 64.0f);
                long long v = (r != r || r < 1.0f) ? 1 : (long long)r;  // `as usize` saturates, then max(1, .)
                sp.nvox[i] = (int)std::min<long long>(v, 1 << 20);
                total *= (size_t)sp.nvox[i];
            }
            if (total > (size_t)1 << 30) return fail(PBRT_B200_ERR_INVALID, "render: spatial light distribution grid too large");
            sp.enabled = 1;
            const bool force_lazy = (flags & PBRT_B200_RENDER_LAZY_SPATIAL) != 0;
            sp.lazy = (force_lazy || total * nl > ((size_t)1 << 25)) ? 1 : 0;
            size_t cap = sp.lazy ? std::min(total, std::max<size_t>(1024, ((size_t)1 << 28) / std::max<size_t>(nl, 1))) : total;
            sp.capacity = (uint32_t)cap;
            std::vector<float> hal(128 * 5);
            const unsigned bases[5] = {2, 3, 5, 7, 11};
            for (int i = 0; i < 128; ++i)
                for (int b = 0; b < 5; ++b) {  // radical_inverse, lowdiscrepancy.rs:398-414 / pbrt_macros lib.rs:92-110
                    if (b == 0) {
                        uint64_t n = (uint64_t)i, r = 0;
                        for (int k = 0; k < 64; ++k) { r = (r << 1) | (n & 1); n >>= 1; }
                        hal[5 * i] = (float)r * 5.421010862427522e-20f;
                    } else {
                        uint64_t base = bases[b], n = (uint64_t)i, rev = 0;
                        float inv_base = 1.0f / (float)base, inv_basen = 1.0f;
                        while (n != 0) { uint64_t next = n / base, digit = n - next * base; rev = rev * base + digit; inv_basen *= inv_base; n = next; }
                        hal[5 * i + b] = std::fmin((float)rev * inv_basen, 0.99999994f);
                    }
                }
            if ((rc = pooled_alloc(st->light_blocks, &sp.slot, total))) return rc;
            if ((rc = pooled_alloc(st->light_blocks, &sp.func, cap * nl))) return rc;
            if ((rc = pooled_alloc(st->light_blocks, &sp.cdf, cap * (nl + 1)))) return rc;
            if ((rc = pooled_alloc(st->light_blocks, &sp.func_int, cap))) return rc;
            if ((rc = pooled_alloc(st->light_blocks, &sp.build_list, cap))) return rc;
            if ((rc = pooled_alloc(st->light_blocks, &sp.counters, 4))) return rc;
            float* hal_dev = nullptr;
            if ((rc = pooled_alloc(st->light_blocks, &hal_dev, hal.size()))) return rc;
            PB_CUDA_TRY(cudaMemcpy(hal_dev, hal.data(), hal.size() * sizeof(float), cudaMemcpyHostToDevice));
            sp.halton = hal_dev;
            PB_CUDA_TRY(cudaMemset(sp.slot, 0xff, total * sizeof(int)));
            PB_CUDA_TRY(cudaMemset(sp.counters, 0, 4 * sizeof(uint32_t)));
            st->sp_eager_pending = !sp.lazy;
        }
        make_distribution(func, cdf, &st->ld_func_int);
        if ((rc = to_device(st->light_blocks, func, &st->ld_func))) return rc;
        if ((rc = to_device(st->light_blocks, cdf, &st->ld_cdf))) return rc;
        if ((rc = to_device(st->light_blocks, inf, &st->inf))) return rc;
        if ((rc = to_device(st->light_blocks, inf_list, &st->inf_list))) return rc;
        st->n_inf = (uint32_t)inf_list.size();
        st->strategy = key;
    }
    return PBRT_B200_OK;
}

int prepare_scene_state(pbrt_b200_scene* sc, const pbrt_b200_render_desc* rd, SceneRenderState** out) {
    SceneRenderState* st = nullptr;
    int rc = prepare_light_state(sc, rd->integrator.light_sample_strategy, rd->flags, &st);
    if (rc) return rc;
    DeviceShared* sh = device_shared(sc->device);
    st->shared = sh;
    if (rd->sampler.kind == PBRT_B200_SAMPLER_SOBOL) {
        if (!rd->sampler.sobol_matrices32 || !rd->sampler.vdc_matrices || !rd->sampler.vdc_matrices_inv)
            return fail(PBRT_B200_ERR_INVALID, "render: the Sobol sampler needs sobol_matrices32, vdc_matrices and vdc_matrices_inv");
        // FNV-1a over the caller's tables (~230 KB): the device copy is reused while the contents are the same
        unsigned long long h = 1469598103934665603ull;
        auto mix = [&](const void* p, size_t bytes) {
            const unsigned long long* w = reinterpret_cast<const unsigned long long*>(p);
            for (size_t i = 0; i < bytes / 8; ++i) { h ^= w[i]; h *= 1099511628211ull; }
        };
        mix(rd->sampler.sobol_matrices32, 1024 * 52 * 4); mix(rd->sampler.vdc_matrices, 25 * 52 * 8); mix(rd->sampler.vdc_matrices_inv, 26 * 52 * 8);
        if (h == 0) h = 1;
        if (sh->sobol_hash != h) {
            if (!sh->sobol32) {
                size_t got = 0;
                sh->sobol32 = reinterpret_cast<uint32_t*>(pool_alloc(1024 * 52 * 4, &got));
                sh->sobol_t = reinterpret_cast<uint32_t*>(pool_alloc(1024 * 52 * 4, &got));
                sh->vdc = reinterpret_cast<unsigned long long*>(pool_alloc(25 * 52 * 8, &got));
                sh->vdc_inv = reinterpret_cast<unsigned long long*>(pool_alloc(26 * 52 * 8, &got));
                if (!sh->sobol32 || !sh->sobol_t || !sh->vdc || !sh->vdc_inv) {
                    sh->sobol32 = nullptr;  // (the partial allocations stay with the process: 426 KB at most, once)
                    return fail(PBRT_B200_ERR_CUDA, "render: out of device memory for the Sobol' tables");
                }
            }
            PB_CUDA_TRY(cudaDeviceSynchronize());
            std::vector<uint32_t> tr(1024 * 52);
            for (int d = 0; d < 1024; ++d)
                for (int b = 0; b < 52; ++b) tr[b * 1024 + d] = rd->sampler.sobol_matrices32[d * 52 + b];
            PB_CUDA_TRY(cudaMemcpy(sh->sobol_t, tr.data(), tr.size() * 4, cudaMemcpyHostToDevice));
            PB_CUDA_TRY(cudaMemcpy(sh->sobol32, rd->sampler.sobol_matrices32, 1024 * 52 * 4, cudaMemcpyHostToDevice));
            PB_CUDA_TRY(cudaMemcpy(sh->vdc, rd->sampler.vdc_matrices, 25 * 52 * 8, cudaMemcpyHostToDevice));
            PB_CUDA_TRY(cudaMemcpy(sh->vdc_inv, rd->sampler.vdc_matrices_inv, 26 * 52 * 8, cudaMemcpyHostToDevice));
            sh->sobol_hash = h;
        }
    }
    if (rd->sampler.kind == PBRT_B200_SAMPLER_HALTON && !sh->perms) {
        const uint32_t N = 1000;  // PRIME_TABLE_SIZE, lowdiscrepancy.rs:9
        std::vector<uint32_t> primes, sums;
        for (uint32_t c = 2; primes.size() < N; ++c) {
            bool ok = true;
            for (uint32_t p : primes) { if (p * p > c) break; if (c % p == 0) { ok = false; break; } }
            if (ok) primes.push_back(c);
        }
        uint32_t total = 0;
        for (uint32_t p : primes) { sums.push_back(total); total += p; }
        std::vector<uint16_t> perms(total);
        Pcg32 rng;
        size_t off = 0;
        for (uint32_t i = 0; i < N; ++i) {
            for (uint32_t j = 0; j < primes[i]; ++j) perms[off + j] = (uint16_t)j;
            for (uint32_t k = 0; k < primes[i]; ++k) { uint32_t other = k + rng.bounded(primes[i] - k); std::swap(perms[off + k], perms[off + other]); }
            off += primes[i];
        }
        if ((rc = to_device_once(perms, &sh->perms))) return rc;
        if ((rc = to_device_once(primes, &sh->primes))) return rc;
        if ((rc = to_device_once(sums, &sh->prime_sums))) return rc;
        sh->n_halton_dims = N;
    }
    if (!sh->filter_table) {
        size_t got = 0;
        sh->filter_table = reinterpret_cast<float*>(pool_alloc(256 * sizeof(float), &got));
        if (!sh->filter_table) return fail(PBRT_B200_ERR_CUDA, "render: out of device memory for the filter table");
    }
    PB_CUDA_TRY(cudaMemcpyAsync(sh->filter_table, rd->film.filter_table, 256 * sizeof(float), cudaMemcpyHostToDevice, 0));
    if (!sh->prog) PB_CUDA_TRY(cudaMallocHost((void**)&sh->prog, PB_PROG_RING * sizeof(DeviceShared::Progress)));
    *out = st;
    return PBRT_B200_OK;
}

// *capacity_io: wanted slots in, slots obtained out.  When the path-state block does not fit (another scene, torch or NCCL
// holds the memory) the capacity is halved down to 2^20 slots before the call gives up: fewer paths in flight are slower
// (DESIGN.md s5), not wrong.
int ensure_buffers(SceneRenderState* st, uint32_t* capacity_io) {
    uint32_t capacity = *capacity_io;
    if (st->buffers && st->buffers->capacity >= capacity) return PBRT_B200_OK;
    if (st->buffers) cudaDeviceSynchronize();
    delete st->buffers;
    st->buffers = new RenderBuffers();
    RenderBuffers* rb = st->buffers;
    RenderDev& d = rb->dev;
    std::memset(&d, 0, sizeof d);
    // bytes per slot: ray 32, hit 16+4+4+1, L_eta 16, beta_st 16, pfilm 8, s_index 8, s_dim 4, pixel 4, sh_ray 32, sh_contrib 16, mis_ray 32,
    // mis_contrib 16, 6 + Q_COUNT index queues x 4
    const size_t per_slot = 32 + 16 + 4 + 4 + 1 + 16 + 16 + 8 + 8 + 4 + 4 + 32 + 16 + 32 + 16 + 4 * (6 + Q_COUNT) + 4;
    for (;;) {
        rb->block = pool_alloc(per_slot * capacity + 256 * 40 + sizeof(Counters), &rb->block_bytes);
        if (rb->block || capacity <= (1u << 20)) break;
        cudaGetLastError();
        capacity = ((capacity / 2u) + 255u) & ~255u;
    }
    *capacity_io = capacity;
    const size_t c = capacity;
    if (!rb->block) { delete st->buffers; st->buffers = nullptr; return fail(PBRT_B200_ERR_CUDA, "render: out of device memory for the path state"); }
    Arena A; A.base = reinterpret_cast<char*>(rb->block); A.size = rb->block_bytes;
    d.ray = A.take<float4>(2 * c); d.hit = A.take<uint4>(c); d.hit_b2 = A.take<float>(c); d.hit_inst = A.take<uint32_t>(c); d.hit_bin = A.take<uint8_t>(c); d.sp_voxel = A.take<int>(c);
    d.L_eta = A.take<float4>(c); d.beta_st = A.take<float4>(c); d.pfilm = A.take<float2>(c);
    d.s_index = A.take<unsigned long long>(c); d.s_dim = A.take<uint32_t>(c); d.pixel = A.take<uint32_t>(c);
    d.sh_ray = A.take<float4>(2 * c); d.sh_contrib = A.take<float4>(c); d.mis_ray = A.take<float4>(2 * c); d.mis_contrib = A.take<float4>(c);
    d.q_path[0] = A.take<uint32_t>(c); d.q_path[1] = A.take<uint32_t>(c); d.q_shadow = A.take<uint32_t>(c); d.q_mis = A.take<uint32_t>(c);
    d.q_dead[0] = A.take<uint32_t>(c); d.q_dead[1] = A.take<uint32_t>(c);
    for (int k = 0; k < Q_COUNT; ++k) d.q_mat[k] = A.take<uint32_t>(c);
    d.cnt = A.take<Counters>(1);
    if (!d.cnt) { delete st->buffers; st->buffers = nullptr; return fail(PBRT_B200_ERR_CUDA, "render: path-state arena too small (internal error)"); }
    rb->capacity = capacity;
    return PBRT_B200_OK;
}

long long ext_gcd(long long a, long long b, long long* x, long long* y) {  // halton.rs:19-27
    if (b == 0) { *x = 1; *y = 0; return a; }
    long long d = a / b, r1, r2;
    long long g = ext_gcd(b, a % b, &r1, &r2);
    *x = r2; *y = r1 - d * r2;
    return g;
}
long long mult_inverse(long long a, long long n) { long long x, y; ext_gcd(a, n, &x, &y); long long r = x - (x / n) * n; return r < 0 ? r + n : r; }

}  // namespace

namespace {
void launch_spatial_build(const RenderDev& R, uint32_t grid, cudaStream_t stream, int eager, uint32_t n_eager) {
    if (R.scene.n_sphere_lights) k_spatial_build<true><<<grid, 128, 0, stream>>>(R, eager, n_eager);
    else k_spatial_build<false><<<grid, 128, 0, stream>>>(R, eager, n_eager);
}
}  // namespace

extern "C" uint32_t pbrt_b200_tile_positions(int w, int h, uint32_t tile_order) {
    const uint32_t ntx = (uint32_t)((std::max(w, 0) + 15) / 16), nty = (uint32_t)((std::max(h, 0) + 15) / 16);
    if (tile_order == 0) return ntx * nty;
    return ((ntx + tile_order - 1) / tile_order) * ((nty + tile_order - 1) / tile_order) * tile_order * tile_order;
}

extern "C" int pbrt_b200_light_distribution_lookup(pbrt_b200_scene* sc, uint32_t strategy, uint32_t flags, const float* points, uint64_t n, int32_t* voxel_out,
                                                    float* func_out) {
    if (!sc || (n && (!points || !voxel_out || !func_out))) return fail(PBRT_B200_ERR_INVALID, "light_distribution_lookup: null argument");
    if (strategy > PBRT_B200_LIGHTS_SPATIAL) return fail(PBRT_B200_ERR_INVALID, "light_distribution_lookup: unknown strategy");
    if (n > 0x7fffffffull) return fail(PBRT_B200_ERR_INVALID, "light_distribution_lookup: batch too large");
    PB_CUDA_TRY(cudaSetDevice(sc->device));
    // the scene's light tables are shared with pbrt_b200_render: same per-device lock
    std::lock_guard<std::mutex> render_lock(device_shared(sc->device)->mu);
    SceneRenderState* st = nullptr;
    int rc = prepare_light_state(sc, strategy, flags, &st);
    if (rc) return rc;
    const uint32_t nl = sc->dev.n_lights;
    if (n == 0 || nl == 0) return PBRT_B200_OK;
    RenderDev R;
    std::memset(&R, 0, sizeof R);
    R.scene = sc->dev; R.n_lights = nl;
    R.ld_func = st->ld_func; R.ld_cdf = st->ld_cdf; R.ld_func_int = st->ld_func_int;
    R.inf_distrib = st->inf; R.infinite_lights = st->inf_list; R.n_infinite = st->n_inf;
    R.sp = st->sp;
    // one pooled scratch block: points, voxel coordinates, per-light values
    struct Scratch { void* p = nullptr; size_t n = 0; ~Scratch() { if (p) { cudaDeviceSynchronize(); pool_free(p, n); } } } scratch;
    const size_t need = Arena::padded(n * 3 * sizeof(float)) + Arena::padded(n * 3 * sizeof(int)) + Arena::padded(n * nl * sizeof(float)) + 1024;
    scratch.p = pool_alloc(need, &scratch.n);
    if (!scratch.p) return fail(PBRT_B200_ERR_CUDA, "light_distribution_lookup: out of device memory");
    Arena SA; SA.base = reinterpret_cast<char*>(scratch.p); SA.size = scratch.n;
    float* d_pts = SA.take<float>(n * 3); int* d_vox = SA.take<int>(n * 3); float* d_func = SA.take<float>(n * nl);
    if (!d_func) return fail(PBRT_B200_ERR_CUDA, "light_distribution_lookup: scratch arena too small (internal error)");
    PB_CUDA_TRY(cudaMemcpy(d_pts, points, n * 3 * sizeof(float), cudaMemcpyHostToDevice));
    if (R.sp.enabled) {
        if (st->sp_eager_pending) {
            const uint32_t nv = (uint32_t)R.sp.nvox[0] * (uint32_t)R.sp.nvox[1] * (uint32_t)R.sp.nvox[2];
            launch_spatial_build(R, std::min<uint32_t>(nv, 148u * 16u), 0, 1, nv);
            st->sp_eager_pending = false;
        } else if (R.sp.lazy) {
            k_spatial_mark_points<<<592, 256>>>(R, d_pts, (uint32_t)n);
            launch_spatial_build(R, 148 * 8, 0, 0, 0);
            k_spatial_reset<<<1, 1>>>(R.sp);
        }
    }
    k_light_distrib_gather<<<592, 256>>>(R, d_pts, (uint32_t)n, d_vox, d_func);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpy(voxel_out, d_vox, n * 3 * sizeof(int), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(func_out, d_func, n * nl * sizeof(float), cudaMemcpyDeviceToHost);
    PB_CUDA_TRY(e);
    return PBRT_B200_OK;
}

// Matrix4x4::inverse (Gauss-Jordan with full pivoting, transform.rs:78-145), row-major; the BDPT camera and spot lights need inverses
static void m4_inverse(const float* m, float* out) {
    int indxc[4] = {0, 0, 0, 0}, indxr[4] = {0, 0, 0, 0}, ipiv[4] = {0, 0, 0, 0};
    float a[4][4];
    for (int i = 0; i < 16; ++i) a[i / 4][i % 4] = m[i];
    for (int i = 0; i < 4; ++i) {
        int irow = 0, icol = 0;
        float big = 0.0f;
        for (int j = 0; j < 4; ++j)
            if (ipiv[j] != 1)
                for (int k = 0; k < 4; ++k)
                    if (ipiv[k] == 0 && std::fabs(a[j][k]) >= big) { big = std::fabs(a[j][k]); irow = j; icol = k; }
        ipiv[icol] += 1;
        if (irow != icol) for (int k = 0; k < 4; ++k) std::swap(a[irow][k], a[icol][k]);
        indxr[i] = irow; indxc[i] = icol;
        const float pivinv = 1.0f / a[icol][icol];
        a[icol][icol] = 1.0f;
        for (int j = 0; j < 4; ++j) a[icol][j] *= pivinv;
        for (int j = 0; j < 4; ++j)
            if (j != icol) {
                const float save = a[j][icol];
                a[j][icol] = 0.0f;
                for (int k = 0; k < 4; ++k) a[j][k] -= a[icol][k] * save;
            }
    }
    for (int i = 0; i < 4; ++i) {
        const int j = 3 - i;
        if (indxr[j] != indxc[j]) for (int k = 0; k < 4; ++k) std::swap(a[k][indxr[j]], a[k][indxc[j]]);
    }
    for (int i = 0; i < 16; ++i) out[i] = a[i / 4][i % 4];
}
static f3 m4_point_host(const float* M, f3 p) {  // Transform::transform_point (transform.rs:413-431)
    const float xp = p.x * M[0] + p.y * M[1] + p.z * M[2] + M[3], yp = p.x * M[4] + p.y * M[5] + p.z * M[6] + M[7];
    const float zp = p.x * M[8] + p.y * M[9] + p.z * M[10] + M[11], wp = p.x * M[12] + p.y * M[13] + p.z * M[14] + M[15];
    if (wp == 1.0f) return f3(xp, yp, zp);
    return f3(xp / wp, yp / wp, zp / wp);
}

// splat_out: the BDPT integrator's second film (pbrt_b200_render_splat); nullptr for pbrt_b200_render
static int render_impl(pbrt_b200_scene* sc, const pbrt_b200_render_desc* rd, float* rgbw_out, float* splat_out, pbrt_b200_render_stats* stats) {
    if (rd->sampler.kind > PBRT_B200_SAMPLER_ZEROTWO) return fail(PBRT_B200_ERR_UNSUPPORTED, "render: sampler outside the hot path (sobol, halton, 02sequence)");
    if (rd->sampler.samples_per_pixel == 0) return fail(PBRT_B200_ERR_INVALID, "render: samples_per_pixel is 0");
    const bool zt = rd->sampler.kind == PBRT_B200_SAMPLER_ZEROTWO;
    uint32_t spp_eff = rd->sampler.samples_per_pixel;
    if (zt) {  // ZeroTwoSequenceSampler::new rounds up to a power of two (zerotwosequence.rs:36-40)
        if (spp_eff > (1u << 20)) return fail(PBRT_B200_ERR_INVALID, "render: 02sequence pixelsamples too large");
        uint32_t v = 1; while (v < spp_eff) v <<= 1; spp_eff = v;
        if (rd->sampler.n_sampled_dimensions > 64) return fail(PBRT_B200_ERR_INVALID, "render: 02sequence dimensions too large");
    }
    if (rd->integrator.light_sample_strategy > PBRT_B200_LIGHTS_SPATIAL) return fail(PBRT_B200_ERR_INVALID, "render: unknown light_sample_strategy");
    const uint32_t ikind = rd->integrator.kind;
    if (ikind > PBRT_B200_INTEGRATOR_BDPT) return fail(PBRT_B200_ERR_INVALID, "render: unknown integrator kind");
    const bool bd = ikind == PBRT_B200_INTEGRATOR_BDPT;
    if (bd != (splat_out != nullptr))
        return fail(PBRT_B200_ERR_INVALID, bd ? "render: the bdpt integrator renders through pbrt_b200_render_splat (its light-tracing strategies need a splat film)"
                                              : "render_splat: only the bdpt integrator renders through pbrt_b200_render_splat");
    if (bd) {
        if (zt) return fail(PBRT_B200_ERR_UNSUPPORTED, "render: bdpt needs the sobol or halton sampler");
        if (sc->dev.n_media || rd->integrator.camera_medium >= 0)
            return fail(PBRT_B200_ERR_UNSUPPORTED, "render: bdpt renders surfaces only; scenes with participating media need volpath");
        if (rd->integrator.max_depth < 0 || rd->integrator.max_depth > PBRT_B200_BDPT_MAX_DEPTH) {
            char msg[160];
            snprintf(msg, sizeof msg, "render: bdpt maxdepth %d outside [0, %d] (every subpath vertex of a sample is kept in device memory)",
                     rd->integrator.max_depth, PBRT_B200_BDPT_MAX_DEPTH);
            return fail(PBRT_B200_ERR_UNSUPPORTED, msg);
        }
    }
    const bool vol = ikind == PBRT_B200_INTEGRATOR_VOLPATH;
    const bool path_like = ikind == PBRT_B200_INTEGRATOR_PATH || vol || bd;  // no recursion state
    if (vol) {
        if (zt) return fail(PBRT_B200_ERR_UNSUPPORTED, "render: volpath needs the sobol or halton sampler");
        if (rd->integrator.camera_medium < -1 || rd->integrator.camera_medium >= (int64_t)sc->dev.n_media)
            return fail(PBRT_B200_ERR_INVALID, "render: camera_medium out of range");
    }
    // the shade kernels keep the bounce count in 16 bits of the path state (volpath also counts down through material-less surfaces)
    if (path_like && rd->integrator.max_depth > 0xfff0) return fail(PBRT_B200_ERR_INVALID, "render: path / volpath maxdepth above 65520");
    if (!path_like && (rd->integrator.max_depth < 1 || rd->integrator.max_depth > 64))
        return fail(PBRT_B200_ERR_INVALID, "render: directlighting / whitted need 1 <= maxdepth <= 64");
    {   // path slots pack the pixel's offset in the sample bounds into 16 + 16 bits
        const int* b = rd->sampler.sample_bounds;
        if ((long long)b[2] - b[0] > 0xffff || (long long)b[3] - b[1] > 0xffff) {
            char msg[160];
            snprintf(msg, sizeof msg, "render: sample bounds [%d, %d) x [%d, %d) exceed 65535 pixels in x or y", b[0], b[2], b[1], b[3]);
            return fail(PBRT_B200_ERR_INVALID, msg);
        }
    }
    PB_CUDA_TRY(cudaSetDevice(sc->device));
    int rc;
    DeviceShared* sh = device_shared(sc->device);
    std::lock_guard<std::mutex> render_lock(sh->mu);
    const bool prof = getenv("PBRT_B200_PROFILE") != nullptr;
    auto t0 = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!prof) return;
        auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[pbrt_b200] render %-18s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    };
    SceneRenderState* st = nullptr;
    if ((rc = prepare_scene_state(sc, rd, &st))) return rc;
    lap("prepare");

    const int* sb = rd->sampler.sample_bounds;
    const int* crop = rd->film.cropped_pixel_bounds;
    const int W = crop[2] - crop[0], Hh = crop[3] - crop[1];
    if (W <= 0 || Hh <= 0) return fail(PBRT_B200_ERR_INVALID, "render: empty crop window");
    int ntx = (sb[2] - sb[0] + 15) / 16, nty = (sb[3] - sb[1] + 15) / 16;
    const uint32_t tile_order = rd->tile_order;
    if (tile_order > 64) return fail(PBRT_B200_ERR_INVALID, "render: tile_order (super-tile edge in tiles) must be <= 64");
    const uint32_t n_positions = pbrt_b200_tile_positions(sb[2] - sb[0], sb[3] - sb[1], tile_order);
    uint32_t tile_begin = rd->tile_begin, tile_end = rd->tile_end ? rd->tile_end : n_positions;
    uint32_t s_begin = rd->sample_begin, s_end = rd->sample_end ? rd->sample_end : spp_eff;
    if (tile_end > n_positions || tile_begin > tile_end || s_begin > s_end || s_end > spp_eff)
        return fail(PBRT_B200_ERR_INVALID, "render: tile/sample window out of range");
    uint32_t tile_group = rd->tile_group ? rd->tile_group : 1u, tile_mod = rd->tile_mod ? rd->tile_mod : 1u, tile_rem = rd->tile_rem;
    if (tile_rem >= tile_mod) return fail(PBRT_B200_ERR_INVALID, "render: tile_rem must be < tile_mod");
    // tiles owned by this call: whole groups g with g % tile_mod == tile_rem (the last one may be partial; raygen masks it)
    uint32_t n_groups = (tile_end - tile_begin + tile_group - 1) / tile_group;
    uint32_t n_owned_groups = n_groups > tile_rem ? (n_groups - tile_rem + tile_mod - 1) / tile_mod : 0;
    uint32_t n_tiles_sel = n_owned_groups * tile_group;
    unsigned long long total_items = (unsigned long long)n_tiles_sel * 256ull * (s_end - s_begin);

    // default 2^26 slots (~20 GB of path state on a 180 GB part): measured on S3, 2^21 -> 360 M samples/s, 2^23 -> 480, 2^24 -> 549,
    // 2^25 -> 600 (634 with this round's kernels), 2^26 -> 659, 2^27 -> 655 (fewer, fuller iterations; gpurun_out/ab18.log)
    // round 2 (samples innermost, faster streaming kernels): 2^26 -> 117.1 ms per 64-spp S3 step, 2^27 -> 115.0 ms (gpurun_out/r2r_refill.log): default 2^27
    // (~36 GB of path state; ensure_buffers halves it when that does not fit)
    uint32_t capacity = rd->paths_in_flight ? rd->paths_in_flight : (1u << 27);
    capacity = (capacity + 255u) & ~255u;
    if ((unsigned long long)capacity > total_items) capacity = (uint32_t)((total_items + 255ull) & ~255ull);
    if (zt) capacity = (n_tiles_sel + 255u) & ~255u;  // tile-serial: one path slot per tile (see ZtTile)
    // recursive integrators: per slot a stack of max_depth frames and up to `eps` shadow + MIS entries; keep that state <= 6 GB
    uint32_t rec_eps = path_like ? 0u : (ikind == PBRT_B200_INTEGRATOR_DIRECT_ONE ? 1u : std::max<uint32_t>(sc->dev.n_lights, 1u));
    uint32_t rec_multi = 0;
    if (ikind == PBRT_B200_INTEGRATOR_DIRECT_ALL) {  // one shadow + one MIS entry per light SAMPLE (uniform_sample_all_lights, integrator.rs:63-74)
        unsigned long long tot = 0;
        for (const pbrt_b200_light& l : st->lights_host) { tot += std::max<uint32_t>(l.n_samples, 1u); if (l.n_samples > 1) rec_multi = 1; }
        if (tot > (1ull << 20)) return fail(PBRT_B200_ERR_UNSUPPORTED, "render: too many light samples per surface for directlighting \"all\"");
        rec_eps = (uint32_t)std::max<unsigned long long>(tot, 1ull);
        if (rec_multi && zt) return fail(PBRT_B200_ERR_UNSUPPORTED, "render: directlighting \"all\" with multi-sample lights needs the sobol or halton sampler");
    }
    const size_t rec_per_slot = path_like ? 0 : 8 + (size_t)rd->integrator.max_depth * (sc->dev.material_ext ? 2 * (48 + 48) : 48) + (size_t)rec_eps * (48 + 52);
    if (rec_per_slot) {
        const unsigned long long fit = (6ull << 30) / rec_per_slot;
        if (fit < 256) return fail(PBRT_B200_ERR_UNSUPPORTED, "render: too many lights for one whitted / directlighting \"all\" surface evaluation");
        if (capacity > fit) capacity = (uint32_t)(fit & ~255ull);
    }
    // volpath / bdpt: one slot per thread of the megakernel's single resident wave
    int vol_grid = 0;
    if (bd) {
        int smc = 148;
        cudaDeviceGetAttribute(&smc, cudaDevAttrMultiProcessorCount, sc->device);
        const int per_sm = bdpt_blocks_per_sm(sc->dev.n_instances || sc->dev.n_sphere_lights || sc->dev.material_ext);
        const unsigned long long want = (total_items + (unsigned long long)PB_VOL_BLOCK - 1ull) / (unsigned long long)PB_VOL_BLOCK;
        vol_grid = (int)std::max<unsigned long long>(1ull, std::min<unsigned long long>((unsigned long long)smc * (unsigned long long)std::max(per_sm, 1), want));
        capacity = ((uint32_t)vol_grid * (uint32_t)PB_VOL_BLOCK + 255u) & ~255u;
    }
    if (vol) {
        int smc = 148, per_sm = 1;
        cudaDeviceGetAttribute(&smc, cudaDevAttrMultiProcessorCount, sc->device);
        per_sm = vol_mega_blocks_per_sm(sc->dev.n_instances || sc->dev.n_sphere_lights || sc->dev.material_ext, sc->grids != nullptr);
        const unsigned long long want = (total_items + (unsigned long long)PB_VOL_BLOCK - 1ull) / (unsigned long long)PB_VOL_BLOCK;
        vol_grid = (int)std::max<unsigned long long>(1ull, std::min<unsigned long long>((unsigned long long)smc * (unsigned long long)std::max(per_sm, 1), want));
        capacity = ((uint32_t)vol_grid * (uint32_t)PB_VOL_BLOCK + 255u) & ~255u;
    }
    if (capacity == 0) capacity = 256;
    if ((rc = ensure_buffers(st, &capacity))) return rc;
    if ((vol || bd) && capacity < (uint32_t)vol_grid * (uint32_t)PB_VOL_BLOCK) vol_grid = (int)(capacity / (uint32_t)PB_VOL_BLOCK);
    lap("buffers");
    RenderDev R = st->buffers->dev;
    R.capacity = capacity;
    R.scene = sc->dev;
    R.camera = rd->camera;
    // sampler
    SamplerDev& S = R.sampler;
    std::memset(&S, 0, sizeof S);
    S.kind = rd->sampler.kind; S.spp = rd->sampler.samples_per_pixel;
    for (int i = 0; i < 4; ++i) S.sb[i] = sb[i];
    {
        int v = std::max(sb[2] - sb[0], sb[3] - sb[1]);  // round_up_pow2_32 / log2_int, sobol.rs:43-46
        v--; v |= v >> 1; v |= v >> 2; v |= v >> 4; v |= v >> 8; v |= v >> 16; v++;
        S.resolution = v;
        S.log2_resolution = 0; while ((1 << S.log2_resolution) < v) S.log2_resolution++;
    }
    S.sobol32 = sh->sobol32; S.sobol_t = sh->sobol_t; S.vdc = sh->vdc; S.vdc_inv = sh->vdc_inv;
    {
        long long res[2] = {sb[2] - sb[0], sb[3] - sb[1]};
        for (int i = 0; i < 2; ++i) {
            long long base = i == 0 ? 2 : 3, scale = 1, e = 0;
            while (scale < std::min<long long>(res[i], 128)) { scale *= base; e += 1; }
            S.base_scales[i] = scale; S.base_exponents[i] = e;
        }
        S.sample_stride = (unsigned long long)(S.base_scales[0] * S.base_scales[1]);
        S.mult_inverse[0] = mult_inverse(S.base_scales[1], S.base_scales[0]);
        S.mult_inverse[1] = mult_inverse(S.base_scales[0], S.base_scales[1]);
    }
    S.perms = sh->perms; S.primes = sh->primes; S.prime_sums = sh->prime_sums; S.n_halton_dims = sh->n_halton_dims;
    // film
    for (int i = 0; i < 4; ++i) R.crop[i] = crop[i];
    R.filter_radius[0] = rd->film.filter_radius[0]; R.filter_radius[1] = rd->film.filter_radius[1];
    R.inv_filter_radius[0] = 1.0f / rd->film.filter_radius[0]; R.inv_filter_radius[1] = 1.0f / rd->film.filter_radius[1];
    R.max_sample_luminance = rd->film.max_sample_luminance;
    R.filter_table = sh->filter_table;
    // integrator
    // the kernels compare the bounce count unsigned; path.rs compares signed, so a negative maxdepth ends every path at its first hit
    R.max_depth = std::max(rd->integrator.max_depth, 0); R.rr_threshold = rd->integrator.rr_threshold;
    for (int i = 0; i < 4; ++i) R.pixel_bounds[i] = rd->integrator.pixel_bounds[i];
    R.ld_func = st->ld_func; R.ld_cdf = st->ld_cdf; R.ld_func_int = st->ld_func_int; R.n_lights = sc->dev.n_lights;
    R.inf_distrib = st->inf; R.infinite_lights = st->inf_list; R.n_infinite = st->n_inf;
    R.sp = st->sp;
    R.ntx = ntx; R.nty = nty;
    R.tile_begin = tile_begin; R.tile_end = tile_end; R.n_tiles_sel = n_tiles_sel; R.sample_begin = s_begin; R.n_samples_sel = s_end - s_begin;
    R.tile_group = tile_group; R.tile_mod = tile_mod; R.tile_rem = tile_rem;
    R.tile_order = tile_order; R.nstx = tile_order ? (uint32_t)((ntx + (int)tile_order - 1) / (int)tile_order) : 0u;

    // DirectLightingIntegrator::preprocess (directlighting.rs:61-76) with nsamples() == 1 for every light
    const uint32_t rec_n_arrays = ikind == PBRT_B200_INTEGRATOR_DIRECT_ALL ? (uint32_t)R.max_depth * R.n_lights * 2u : 0u;
    void* zt_block = nullptr; size_t zt_bytes = 0;
    RenderDev* zt_rdev = nullptr;  // R in device memory, for the out-of-line shade calls of k_zt_mega
    R.zt.n2d = rd->sampler.n_sampled_dimensions + rec_n_arrays;
    if (zt && n_tiles_sel > 0) {
        const size_t nd = rd->sampler.n_sampled_dimensions, per_tile = nd * spp_eff, per_tile2 = (size_t)R.zt.n2d * spp_eff;
        if (per_tile2 * n_tiles_sel * 8 > (8ull << 30)) return fail(PBRT_B200_ERR_UNSUPPORTED, "render: 02sequence sample arrays for directlighting \"all\" exceed 8 GB");
        const size_t need = Arena::padded(sizeof(ZtTile) * n_tiles_sel) + Arena::padded(4 * per_tile * n_tiles_sel) + Arena::padded(8 * per_tile2 * n_tiles_sel) + Arena::padded(sizeof(RenderDev)) + 1024;
        zt_block = pool_alloc(need, &zt_bytes);
        if (!zt_block) return fail(PBRT_B200_ERR_CUDA, "render: out of device memory for the 02sequence sample tables");
        Arena A; A.base = reinterpret_cast<char*>(zt_block); A.size = zt_bytes;
        R.zt.tiles = A.take<ZtTile>(n_tiles_sel); R.zt.s1d = A.take<float>(std::max<size_t>(per_tile * n_tiles_sel, 1)); R.zt.s2d = A.take<float2>(std::max<size_t>(per_tile2 * n_tiles_sel, 1));
        zt_rdev = A.take<RenderDev>(1);
        R.zt.spp = spp_eff; R.zt.ndims = (uint32_t)nd;
    }
    struct ZtRelease { void* p; size_t n; ~ZtRelease() { if (p) { cudaDeviceSynchronize(); pool_free(p, n); } } } zt_release{zt_block, zt_bytes};
    std::memset(&R.rec, 0, sizeof R.rec);
    void* rec_block = nullptr; size_t rec_bytes = 0;
    if (!path_like) {
        RecDev& rec = R.rec;
        rec.kind = ikind; rec.stack_depth = (uint32_t)R.max_depth; rec.entries_per_slot = rec_eps; rec.multi = rec_multi;
        if (ikind == PBRT_B200_INTEGRATOR_DIRECT_ALL) {
            rec.n_arrays = rec_n_arrays;
            if (rd->sampler.kind == PBRT_B200_SAMPLER_SOBOL && 5ull + 2ull * rec.n_arrays + 8ull > 1024ull)
                return fail(PBRT_B200_ERR_UNSUPPORTED, "render: directlighting \"all\" needs more Sobol' dimensions than the 1024 the tables hold (the reference panics)");
        }
        const size_t c = capacity, e = c * rec_eps;
        const bool textured = sc->dev.material_ext != nullptr;
        const size_t fr = textured ? 2 : 1;  // textured scenes: two candidate frames per stack level (uber's two specular transmission lobes)
        const size_t need = Arena::padded(4 * c) * 3 + Arena::padded(32 * c * rec.stack_depth * fr) + Arena::padded(16 * c * rec.stack_depth * fr) + Arena::padded(32 * e) * 2 +
                            Arena::padded(16 * e) * 2 + Arena::padded(4 * e) + (textured ? Arena::padded(48 * c * rec.stack_depth * fr) : 0) + 4096;
        rec_block = pool_alloc(need, &rec_bytes);
        if (!rec_block) return fail(PBRT_B200_ERR_CUDA, "render: out of device memory for the recursion state");
        Arena A; A.base = reinterpret_cast<char*>(rec_block); A.size = rec_bytes;
        rec.sp = A.take<uint32_t>(c); rec.arr = A.take<uint32_t>(c); rec.sample_num = A.take<uint32_t>(c);
        rec.st_ray = A.take<float4>(2 * c * rec.stack_depth * fr); rec.st_beta = A.take<float4>(c * rec.stack_depth * fr);
        rec.e_sh_ray = A.take<float4>(2 * e); rec.e_sh_contrib = A.take<float4>(e);
        rec.e_mis_ray = A.take<float4>(2 * e); rec.e_mis_contrib = A.take<float4>(e); rec.e_mis_slot = A.take<uint32_t>(e);
        if (textured) rec.st_diff = A.take<float4>(3 * c * rec.stack_depth * fr);
        if (!rec.e_mis_slot || (textured && !rec.st_diff)) { pool_free(rec_block, rec_bytes); return fail(PBRT_B200_ERR_CUDA, "render: recursion arena too small (internal error)"); }
    }
    ZtRelease rec_release{rec_block, rec_bytes};
    // film buffer: device pointer supplied, or a scratch film that is added back to the host buffer
    const size_t npix = (size_t)W * Hh;
    float4* film_dev = nullptr;
    bool own_film = !(rd->flags & PBRT_B200_RENDER_KEEP_ON_DEVICE);
    size_t film_block = 0;
    if (own_film) {
        film_dev = reinterpret_cast<float4*>(pool_alloc(npix * sizeof(float4), &film_block));
        if (!film_dev) return fail(PBRT_B200_ERR_CUDA, "render: out of device memory for the film");
    } else film_dev = reinterpret_cast<float4*>(rgbw_out);
    ZtRelease film_release{own_film ? film_dev : nullptr, film_block};  // every error return below gives the scratch film back (after a sync)
    if (own_film) PB_CUDA_TRY(cudaMemsetAsync(film_dev, 0, npix * sizeof(float4), 0));
    R.film = film_dev;

    int sm_count = 148;
    cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, sc->device);
    int trace_per_sm = 8;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&trace_per_sm, sc->dev.n_instances ? k_trace_closest<true> : k_trace_closest<false>, PB_TRACE_BLOCK, 0);
    int grid_trace = sm_count * (trace_per_sm > 0 ? trace_per_sm : 1);  // persistent: exactly one resident wave
    // ... of EACH kernel: the any-hit and MIS kernels have their own register allocation, hence their own number of resident CTAs
    int shadow_per_sm = trace_per_sm, mis_per_sm = trace_per_sm;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&shadow_per_sm, sc->dev.n_instances ? k_trace_shadow<true> : k_trace_shadow<false>, PB_TRACE_BLOCK, 0);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&mis_per_sm, sc->dev.n_instances ? k_trace_mis<true> : k_trace_mis<false>, PB_TRACE_BLOCK, 0);
    int grid_shadow = sm_count * (shadow_per_sm > 0 ? shadow_per_sm : 1), grid_mis = sm_count * (mis_per_sm > 0 ? mis_per_sm : 1);
    int packet_per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&packet_per_sm, k_trace_closest_packet, PB_TRACE_BLOCK, 0);
    const int grid_packet = sm_count * std::max(packet_per_sm, 1);
    // shade kernels keep 5 CTAs of 128 threads resident per SM (96-104 registers): 10 per SM = two full waves (8 left a
    // 3-CTA tail wave: -1.5 % on S3, gpurun_out/ab4.log)
    int grid_shade = sm_count * 20, grid_small = sm_count * 4;  // shade: 10 -> 20 CTAs per SM: 35.4 -> 35.2 ms per 16-spp S3 step (gpurun_out/r2o_grid.log)
    if (zt) {  // tile-serial: at most one path per tile in flight -- a few CTAs cover the queues
        const int need = (int)((capacity + 127u) / 128u);
        grid_trace = std::min(grid_trace, need); grid_shade = std::min(grid_shade, need); grid_small = std::min(grid_small, need);
        grid_shadow = std::min(grid_shadow, need); grid_mis = std::min(grid_mis, need);
    }

    // Packet traversal (trace.cuh: trace_queue_packet) for the closest-hit launch of a wave's first iteration: its queue holds the
    // wave's camera rays in item order, so an aligned run of 32 is 32 samples of one pixel (samples innermost).  The later closest-hit,
    // shadow and MIS queues lost with it on S3 (profiles/r03_packet_traversal.md) and keep the per-lane walk.
    // PBRT_B200_PACKET_TRAVERSAL=0, read per call, turns it off (A/B on one build).
    bool packet_camera = !zt;
    if (const char* e = getenv("PBRT_B200_PACKET_TRAVERSAL")) if (atoi(e) == 0) packet_camera = false;
    cudaStream_t stream = 0;
    // events come from the scene's pool: [0] start, [1] end, [2..2+PB_PROG_RING) progress copies, then timing marks
    size_t ev_used = 2 + PB_PROG_RING;
    auto pool_event = [&](size_t i) -> cudaEvent_t {
        while (sh->events.size() <= i) { cudaEvent_t e; cudaEventCreate(&e); sh->events.push_back(e); }
        return sh->events[i];
    };
    cudaEvent_t ev0 = pool_event(0), ev1 = pool_event(1);
    const size_t tev_base = ev_used;
    auto mark = [&]() { cudaEventRecord(pool_event(ev_used++), stream); };  // pairs around the trace kernels
    const bool timing = stats != nullptr && !zt;  // tile-serial mode runs ~10^5 tiny iterations: no per-phase events
    uint64_t launches = 0;
    // ---- Sobol' sample tables (sobol_tab_block) for the path integrator's global-sampler runs
    bool sample_prepass = !zt && !R.rec.kind && !vol && !bd;  // k_sample_block serves every path the tables do not
    R.u8 = nullptr;
    if (!zt && !R.rec.kind && !vol && !bd && S.kind == PBRT_B200_SAMPLER_SOBOL && S.log2_resolution > 0 && !getenv("PBRT_B200_NO_SOBOL_TABLES")) {
        const uint32_t sbw = (uint32_t)(sb[2] - sb[0]), sbh = (uint32_t)(sb[3] - sb[1]);
        // a path shading at bounce b < max_depth reads dimensions [s_dim, s_dim + 8) with s_dim <= 5 + 8b (camera 5, per bounce at most
        // light choice 1 + light 2 + scattering 2 + BSDF 2 + roulette 1): the tables serve every block iff they hold 5 + 8 * max_depth dimensions
        const unsigned long long dims_needed = 5ull + 8ull * (unsigned long long)R.max_depth;
        const uint32_t want = (uint32_t)std::min<unsigned long long>(1024ull, dims_needed);
        uint32_t vdims = want;
        const size_t budget = (size_t)4 << 30;  // the pixel table may take up to 4 GB; deeper dimensions then go through k_sample_block
        while (vdims > 13u && (size_t)sbw * sbh * ((vdims + 3u) & ~3u) * 4u > budget) vdims -= 8u;
        // test hook: fewer table dimensions, so that k_sample_block's table-index path runs on small films
        if (const char* e = getenv("PBRT_B200_SOBOL_TABLE_DIMS")) vdims = std::min<uint32_t>(vdims, (uint32_t)std::max(1, atoi(e)));
        const uint32_t vstride = (vdims + 3u) & ~3u;
        const size_t vp_need = (size_t)sbw * sbh * vstride * 4u;
        const size_t vs_need = (size_t)std::max<uint32_t>(s_end - s_begin, 1u) * vstride * 4u;
        if (vp_need <= budget && sbw <= 0xffffu && sbh <= 0xffffu) {
            SamplerDev T = S;
            T.vstride = vstride; T.sbw = sbw; T.vdims = vdims;
            const unsigned long long key[4] = {sh->sobol_hash, ((unsigned long long)sbw << 32) | sbh, ((unsigned long long)S.log2_resolution << 32) | vstride, 1ull};
            bool ok = true;
            if (std::memcmp(key, sh->vp_key, sizeof key) != 0 || !sh->vp) {
                if (sh->vp && sh->vp_block < vp_need) { pool_free(sh->vp, sh->vp_block); sh->vp = nullptr; }
                if (!sh->vp) sh->vp = reinterpret_cast<uint32_t*>(pool_alloc(vp_need, &sh->vp_block));
                if (sh->vp) {
                    k_sobol_table_pixels<<<148 * 8, 256, 0, stream>>>(T, sh->vp, sbw * sbh);
                    std::memcpy(sh->vp_key, key, sizeof key);
                } else { cudaGetLastError(); std::memset(sh->vp_key, 0, sizeof sh->vp_key); ok = false; }
            }
            if (ok && (!sh->vs || sh->vs_block < vs_need)) {
                if (sh->vs) pool_free(sh->vs, sh->vs_block);
                sh->vs = reinterpret_cast<uint32_t*>(pool_alloc(vs_need, &sh->vs_block));
                if (!sh->vs) { cudaGetLastError(); sh->vs_block = 0; ok = false; }
            }
            if (ok) {
                k_sobol_table_samples<<<64, 256, 0, stream>>>(T, sh->vs, s_begin, s_end - s_begin);
                S.vp = sh->vp; S.vs = sh->vs; S.vdims = vdims; S.vstride = vstride; S.sbw = sbw; S.vs_begin = s_begin;
                sample_prepass = dims_needed > vdims;  // paths past the tables' last block; beyond dimension 1024 too
            }
        }
    }
    if (sample_prepass) {
        RenderBuffers* rb = st->buffers;
        const size_t need = (size_t)capacity * 32u;
        if (rb->u8_block && rb->u8_bytes < need) { cudaDeviceSynchronize(); pool_free(rb->u8_block, rb->u8_bytes); rb->u8_block = nullptr; }
        if (!rb->u8_block) rb->u8_block = pool_alloc(need, &rb->u8_bytes);
        if (!rb->u8_block) return fail(PBRT_B200_ERR_CUDA, "render: out of device memory for the sample blocks");
        R.u8 = reinterpret_cast<float4*>(rb->u8_block);
    }
    R.rdiff = nullptr;
    R.tex_sort = nullptr;
    if (sc->dev.material_ext) {  // textured materials: every path slot carries its ray's differentials
        RenderBuffers* rb = st->buffers;
        const size_t sort_bytes = 8u * (size_t)sc->dev.n_materials;  // k_tex_count / k_tex_scan: counts (zero between iterations) + cursors
        const size_t need = (size_t)capacity * 48u + sort_bytes;
        if (rb->diff_block && rb->diff_bytes < need) { cudaDeviceSynchronize(); pool_free(rb->diff_block, rb->diff_bytes); rb->diff_block = nullptr; }
        if (!rb->diff_block) rb->diff_block = pool_alloc(need, &rb->diff_bytes);
        if (!rb->diff_block) return fail(PBRT_B200_ERR_CUDA, "render: out of device memory for the ray differentials");
        R.rdiff = reinterpret_cast<float4*>(rb->diff_block);
        R.tex_sort = reinterpret_cast<uint32_t*>(static_cast<char*>(rb->diff_block) + (size_t)capacity * 48u);
        PB_CUDA_TRY(cudaMemsetAsync(R.tex_sort, 0, sort_bytes, stream));
    }
    PB_CUDA_TRY(cudaMemsetAsync(R.cnt, 0, sizeof(Counters), stream));
    if (st->sp_eager_pending) {  // every voxel's distribution, once per scene
        const uint32_t nv = (uint32_t)R.sp.nvox[0] * (uint32_t)R.sp.nvox[1] * (uint32_t)R.sp.nvox[2];
        launch_spatial_build(R, std::min<uint32_t>(nv, (uint32_t)sm_count * 16u), stream, 1, nv);
        PB_CUDA_TRY(cudaGetLastError());
        st->sp_eager_pending = false;
    }
    if ((vol || bd) && R.sp.enabled && R.sp.lazy)
        return fail(PBRT_B200_ERR_UNSUPPORTED, "render: volpath / bdpt with lightsamplestrategy \"spatial\" needs the eagerly built voxel table (voxels x lights <= 2^25)");
    // bdpt: the splat film (device pointer supplied, or a scratch film added back to the host buffer) and the subpath vertices
    float* splat_dev = nullptr;
    size_t splat_block = 0, verts_block = 0, spot_block = 0;
    void* verts = nullptr;
    float* spot_dev = nullptr;
    if (bd) {
        if (own_film) {
            splat_dev = reinterpret_cast<float*>(pool_alloc(npix * 3 * sizeof(float), &splat_block));
            if (!splat_dev) return fail(PBRT_B200_ERR_CUDA, "render: out of device memory for the splat film");
            PB_CUDA_TRY(cudaMemsetAsync(splat_dev, 0, npix * 3 * sizeof(float), stream));
        } else splat_dev = splat_out;
        const size_t per_slot = (size_t)(2 * R.max_depth + 3) * bdpt_vertex_bytes();
        verts = pool_alloc(std::max<size_t>((size_t)capacity * per_slot, 256), &verts_block);
        if (!verts) { if (splat_block) pool_free(splat_dev, splat_block); return fail(PBRT_B200_ERR_CUDA, "render: out of device memory for the bdpt subpath vertices"); }
    }
    ZtRelease splat_release{splat_block ? splat_dev : nullptr, splat_block}, verts_release{verts, verts_block};
    BdptCam bcam;
    std::memset(&bcam, 0, sizeof bcam);
    if (bd) {  // PerspectiveCamera::new's image-plane area and the inverses of camera and spot-light matrices (pbrt-v3 perspective.cpp:55-62)
        const pbrt_b200_camera& cm = rd->camera;
        std::memcpy(bcam.c2w, cm.camera_to_world, sizeof bcam.c2w);
        m4_inverse(cm.camera_to_world, bcam.w2c);
        m4_inverse(cm.raster_to_camera, bcam.c2r);
        f3 pmin = m4_point_host(cm.raster_to_camera, f3(0.f, 0.f, 0.f));
        f3 pmax = m4_point_host(cm.raster_to_camera, f3((float)rd->film.full_resolution[0], (float)rd->film.full_resolution[1], 0.f));
        pmin = f3(pmin.x / pmin.z, pmin.y / pmin.z, pmin.z / pmin.z); pmax = f3(pmax.x / pmax.z, pmax.y / pmax.z, pmax.z / pmax.z);
        bcam.A = std::fabs((pmax.x - pmin.x) * (pmax.y - pmin.y));
        bcam.fwd = f3(cm.camera_to_world[2], cm.camera_to_world[6], cm.camera_to_world[10]);
        bcam.n_lens = f3(bcam.w2c[8], bcam.w2c[9], bcam.w2c[10]);
        bcam.lens_radius = cm.lens_radius; bcam.focal_distance = cm.focal_distance;
        for (int i = 0; i < 4; ++i) bcam.sb[i] = sb[i];
        std::vector<float> l2w(16 * std::max<size_t>(st->lights_host.size(), 1), 0.0f);
        for (size_t i = 0; i < st->lights_host.size(); ++i)
            if (st->lights_host[i].type == PBRT_B200_LIGHT_SPOT) m4_inverse(st->lights_host[i].world_to_light, l2w.data() + 16 * i);
        spot_dev = reinterpret_cast<float*>(pool_alloc(l2w.size() * sizeof(float), &spot_block));
        if (!spot_dev) return fail(PBRT_B200_ERR_CUDA, "render: out of device memory");
        PB_CUDA_TRY(cudaMemcpyAsync(spot_dev, l2w.data(), l2w.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
        bcam.spot_l2w = spot_dev;
    }
    ZtRelease spot_release{spot_dev, spot_block};
    PB_CUDA_TRY(cudaEventRecord(ev0, stream));
    if (bd) {
        if (total_items > 0) {
            launch_bdpt(R, bcam, verts, splat_dev, total_items, sc->dev.n_instances || sc->dev.n_sphere_lights || sc->dev.material_ext, vol_grid, stream);
            launches += 1;
            PB_CUDA_TRY(cudaGetLastError());
        }
    } else if (vol) {
        if (total_items > 0) {
            // R in device memory for the out-of-line shade calls (as k_zt_mega)
            size_t rdev_bytes = 0;
            RenderDev* rdev = reinterpret_cast<RenderDev*>(pool_alloc(sizeof(RenderDev), &rdev_bytes));
            if (!rdev) return fail(PBRT_B200_ERR_CUDA, "render: out of device memory");
            ZtRelease rdev_release{rdev, rdev_bytes};
            PB_CUDA_TRY(cudaMemcpyAsync(rdev, &R, sizeof(RenderDev), cudaMemcpyHostToDevice, stream));
            launch_vol_mega(R, rdev, total_items, rd->integrator.camera_medium, sc->dev.n_instances || sc->dev.n_sphere_lights || sc->dev.material_ext, sc->grids,
                            vol_grid, stream);
            launches += 1;
            PB_CUDA_TRY(cudaGetLastError());
            PB_CUDA_TRY(cudaStreamSynchronize(stream));  // rdev is released at the end of this block
        }
    } else if (zt ? n_tiles_sel > 0 : total_items > 0) {
        // Persistent wavefront: all `capacity` slots start free; each iteration traces every live path one segment,
        // shades, resolves shadow/MIS rays, then k_finish_regen retires finished paths and refills their slots.
        // The host never waits on the batch it has just submitted: after every batch of `poll` iterations the queue
        // state is copied to a pinned ring entry, and the host looks at the copy of the batch BEFORE the one in flight,
        // so the GPU always has work queued behind the running iteration (over-submitted iterations find empty queues).
        DeviceShared::Progress* prog = sh->prog;
        // Large queues run the call as back-to-back waves of `capacity` camera samples, each drained before the next starts:
        // slots then map to pixels in order, every per-slot array is read and written coalesced, and a wave's tail is a
        // few percent of its time.  (Measured on S3, 64 spp, 2^25 slots: refilling scattered dead slots from the middle of
        // the item stream -- the right policy for small queues, 263 -> 342 M samples/s at 2^21 -- runs at 532 M samples/s
        // against 619 M for drained waves: k_finish_regen's writes and the shade gathers lose their coalescing.)
        const bool drained_waves = !zt && capacity >= (1u << 22);
        unsigned long long iter = 0, batch = 0;
        const bool inst = sc->dev.n_instances != 0;                 // trace kernels: two-level walk
        const bool full = inst || sc->dev.n_sphere_lights != 0 || sc->dev.material_ext != nullptr;  // shade kernels: + instanced surfaces, sphere area lights, textures
        // (0,2)-sequence + PathIntegrator: the whole call is one kernel, a thread per tile (k_zt_mega, always the full-featured
        // family: one instantiation); the recursive integrators keep the wavefront tile-serial form
        const bool zt_mega = zt && !R.rec.kind;
        if (zt_mega) {
            PB_CUDA_TRY(cudaMemcpyAsync(zt_rdev, &R, sizeof(RenderDev), cudaMemcpyHostToDevice, stream));
            // tiles per warp, measured on B200 (gpurun_out/ab14.log): 625 tiles -> 2 lanes 7.1 M samples/s (1: 6.1, 4: 5.7); 8160 tiles ->
            // 8-16 lanes 11.2 M (1: 6.1, 32: 10.8); 32640 tiles -> 32 lanes 23.8 M (1: 6.5)
            uint32_t lanes = std::min<uint32_t>(32u, std::max<uint32_t>(1u, (n_tiles_sel + (uint32_t)sm_count * 4u - 1u) / ((uint32_t)sm_count * 4u)));
            const uint32_t nblk = (n_tiles_sel + lanes * PB_ZT_WARPS - 1) / (lanes * PB_ZT_WARPS);
            launch_zt_mega(R, zt_rdev, lanes, nblk, stream);
            launches += 1;
        }
        for (unsigned long long wave_begin = 0; !zt_mega && wave_begin < (zt ? 1ull : total_items);) {
        const unsigned long long wave_end = drained_waves ? std::min<unsigned long long>(wave_begin + capacity, total_items) : total_items;
        const unsigned long long loop_items = zt ? 0ull : wave_end;  // tile-serial mode: the queues themselves say when the tiles are done
        if (zt) {
            k_zt_init<<<grid_small, 128, 0, stream>>>(R);
            k_iter_end<<<1, 1, 0, stream>>>(R.cnt, 0ull);
            launches += 2;
        } else {
            k_init_slots<<<grid_small, 256, 0, stream>>>(R, capacity);
            k_finish_regen<<<grid_small, 256, 0, stream>>>(R, 1, wave_end);
            k_iter_end<<<1, 1, 0, stream>>>(R.cnt, wave_end);
            launches += 3;
        }
        int parity = 0;
        unsigned long long wave_iter = 0;  // iteration 0 traces the wave's camera rays
        const unsigned long long iter_cap = zt ? 256ull * spp_eff * (unsigned long long)(R.max_depth + 3) * 2ull + 4096
                                               : (total_items / capacity + 2) * (unsigned long long)(R.max_depth + 2 + 8) * 4ull *
                                                         (R.rec.kind ? 1ull << std::min(R.max_depth, 16) : 1ull) + 4096;  // recursive: a binary tree of rays
        const int poll = zt ? 32 : 4;  // tile-serial iterations are a few microseconds of work each
        bool done = false;
        while (!done) {
            for (int b = 0; b < poll; ++b) {
                if (timing) mark();
                if (inst) k_trace_closest<true><<<grid_trace, PB_TRACE_BLOCK, 0, stream>>>(R, parity);
                else if (packet_camera && wave_iter == 0) k_trace_closest_packet<<<grid_packet, PB_TRACE_BLOCK, 0, stream>>>(R, parity);
                else k_trace_closest<false><<<grid_trace, PB_TRACE_BLOCK, 0, stream>>>(R, parity);
                if (timing) mark();
                if (R.sp.enabled && R.sp.lazy) {
                    k_spatial_mark<<<grid_small, 256, 0, stream>>>(R, parity);
                    launch_spatial_build(R, (uint32_t)sm_count * 8u, stream, 0, 0);
                    k_spatial_reset<<<1, 1, 0, stream>>>(R.sp);
                    launches += 3;
                }
                if (R.rec.kind) {  // whitted / directlighting: one generic shade kernel, entry-indexed shadow and MIS rays
                    launch_rec_shade(R, parity, zt, full, stream);
                    if (timing) mark();
                    if (inst) k_rec_shadow<true><<<grid_trace, PB_TRACE_BLOCK, 0, stream>>>(R);
                    else k_rec_shadow<false><<<grid_trace, PB_TRACE_BLOCK, 0, stream>>>(R);
                    if (timing) mark();
                    if (inst) k_rec_mis<true><<<grid_trace, PB_TRACE_BLOCK, 0, stream>>>(R);
                    else k_rec_mis<false><<<grid_trace, PB_TRACE_BLOCK, 0, stream>>>(R);
                    if (timing) mark();
                } else {
                if (sample_prepass) { k_sample_block<<<grid_small, 256, 0, stream>>>(R, parity); launches += 1; }
                k_classify<<<grid_small, 256, 0, stream>>>(R, parity);
                launch_shade_kernels(R, parity, full, grid_small, grid_shade, stream);
                if (R.tex_sort) launches += 3;  // k_tex_count / k_tex_scan / k_tex_scatter
                if (timing) mark();
                if (inst) k_trace_shadow<true><<<grid_shadow, PB_TRACE_BLOCK, 0, stream>>>(R);
                else k_trace_shadow<false><<<grid_shadow, PB_TRACE_BLOCK, 0, stream>>>(R);
                if (timing) mark();
                if (inst) k_trace_mis<true><<<grid_mis, PB_TRACE_BLOCK, 0, stream>>>(R);
                else k_trace_mis<false><<<grid_mis, PB_TRACE_BLOCK, 0, stream>>>(R);
                if (timing) mark();
                }
                if (zt) k_finish_zt<<<grid_small, 128, 0, stream>>>(R, parity);
                else k_finish_regen<<<grid_small, 256, 0, stream>>>(R, parity, wave_end);
                k_iter_end<<<1, 1, 0, stream>>>(R.cnt, loop_items);
                if (timing) mark();
                launches += 13;
                parity ^= 1;
                iter++;
                wave_iter++;
            }
            // {item_cursor, n_path} of this batch -> ring entry, event marks the copy
            DeviceShared::Progress* pe = prog + (batch % PB_PROG_RING);
            cudaMemcpyAsync(&pe->cursor, &R.cnt->item_cursor, sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream);
            cudaMemcpyAsync(&pe->n_path, &R.cnt->n_path, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream);
            cudaEventRecord(pool_event(2 + batch % PB_PROG_RING), stream);
            if (batch >= 1) {  // wait for the PREVIOUS batch only
                unsigned long long pb = batch - 1;
                cudaError_t e = cudaEventSynchronize(pool_event(2 + pb % PB_PROG_RING));
                if (e != cudaSuccess) PB_CUDA_TRY(e);
                const DeviceShared::Progress* pp = prog + (pb % PB_PROG_RING);
                if (pp->cursor >= loop_items && pp->n_path == 0) done = true;
            }
            batch++;
            if (iter > iter_cap) return fail(PBRT_B200_ERR_CUDA, "render: path queue failed to drain");
        }
        wave_begin = zt ? 1ull : wave_end;
        }
    }
    PB_CUDA_TRY(cudaEventRecord(ev1, stream));
    PB_CUDA_TRY(cudaGetLastError());
    PB_CUDA_TRY(cudaStreamSynchronize(stream));
    lap("wavefront loop");
    if (R.sp.enabled) {
        uint32_t spc[4];
        PB_CUDA_TRY(cudaMemcpy(spc, R.sp.counters, sizeof spc, cudaMemcpyDeviceToHost));
        if (spc[2]) return fail(PBRT_B200_ERR_CUDA, "render: spatial light distribution slot table overflowed (more voxels touched than slots); the image is incomplete");
    }
    if (stats) {
        Counters c;
        PB_CUDA_TRY(cudaMemcpy(&c, R.cnt, sizeof c, cudaMemcpyDeviceToHost));
        std::memset(stats, 0, sizeof *stats);
        stats->camera_rays = c.camera_rays; stats->intersection_tests = c.closest_rays; stats->shadow_tests = c.shadow_rays;
        stats->zero_radiance_paths = c.zero_radiance; stats->kernel_launches = launches;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev0, ev1);
        stats->device_ms = ms;
        for (size_t k = tev_base; k + 5 < ev_used; k += 6) {
            float a = 0.f, b = 0.f, m = 0.f, shd = 0.f, fin = 0.f;
            cudaEventElapsedTime(&a, sh->events[k], sh->events[k + 1]);
            cudaEventElapsedTime(&shd, sh->events[k + 1], sh->events[k + 2]);
            cudaEventElapsedTime(&b, sh->events[k + 2], sh->events[k + 3]);
            cudaEventElapsedTime(&m, sh->events[k + 3], sh->events[k + 4]);
            cudaEventElapsedTime(&fin, sh->events[k + 4], sh->events[k + 5]);
            stats->trace_closest_ms += a + m; stats->trace_any_ms += b; stats->shade_ms += shd; stats->finish_ms += fin;
        }
        stats->iterations = c.iterations;
    }
    if (bd && own_film) {  // the splat film: same rules as the rgbw film
        std::vector<float> hs(npix * 3);
        PB_CUDA_TRY(cudaMemcpy(hs.data(), splat_dev, hs.size() * sizeof(float), cudaMemcpyDeviceToHost));
        if (rd->flags & PBRT_B200_RENDER_OVERWRITE) std::memcpy(splat_out, hs.data(), hs.size() * sizeof(float));
        else for (size_t i = 0; i < hs.size(); ++i) splat_out[i] += hs[i];
    }
    if (own_film) {
        // film tile merge (merge_film_tile, film.rs:142-161): device film -> pinned staging in chunks, each chunk added into
        // the caller's buffer while the next one is in flight
        size_t stage_bytes = 0;
        const size_t nfl = npix * 4, chunk = (size_t)1 << 20;  // floats per chunk (4 MB)
        if (rd->flags & PBRT_B200_RENDER_OVERWRITE) {
            // a page-locked destination takes the film in one DMA transfer, no staging and no host copy
            cudaPointerAttributes pa;
            if (cudaPointerGetAttributes(&pa, rgbw_out) == cudaSuccess && pa.type == cudaMemoryTypeHost) {
                PB_CUDA_TRY(cudaMemcpyAsync(rgbw_out, film_dev, nfl * sizeof(float), cudaMemcpyDeviceToHost, stream));
                PB_CUDA_TRY(cudaStreamSynchronize(stream));
                lap("film d2h (pinned)");
                return PBRT_B200_OK;
            }
            cudaGetLastError();  // (an unregistered host pointer reports cudaErrorInvalidValue on old drivers)
        }
        float* stage = reinterpret_cast<float*>(pool_alloc_host(std::min(nfl, 2 * chunk) * sizeof(float), &stage_bytes));
        if (!stage) return fail(PBRT_B200_ERR_CUDA, "render: out of pinned host memory");
        const float* src = reinterpret_cast<const float*>(film_dev);
        cudaEvent_t done[2] = {pool_event(0), pool_event(1)};
        const size_t nchunks = (nfl + chunk - 1) / chunk;
        cudaError_t e = cudaSuccess;
        for (size_t k = 0; k <= nchunks && e == cudaSuccess; ++k) {
            if (k < nchunks) {
                size_t o = k * chunk, m = std::min(chunk, nfl - o);
                e = cudaMemcpyAsync(stage + (k & 1) * chunk, src + o, m * sizeof(float), cudaMemcpyDeviceToHost, stream);
                if (e == cudaSuccess) e = cudaEventRecord(done[k & 1], stream);
            }
            if (k >= 1 && e == cudaSuccess) {
                size_t o = (k - 1) * chunk, m = std::min(chunk, nfl - o);
                e = cudaEventSynchronize(done[(k - 1) & 1]);
                const float* t = stage + ((k - 1) & 1) * chunk;
                float* dst = rgbw_out + o;
                if (rd->flags & PBRT_B200_RENDER_OVERWRITE) std::memcpy(dst, t, m * sizeof(float));
                else for (size_t i = 0; i < m; ++i) dst[i] += t[i];
            }
        }
        pool_free_host(stage, stage_bytes);
        PB_CUDA_TRY(e);
        lap("film d2h + merge");
    }
    return PBRT_B200_OK;
}

extern "C" int pbrt_b200_render(pbrt_b200_scene* sc, const pbrt_b200_render_desc* rd, float* rgbw_out, pbrt_b200_render_stats* stats) {
    if (!sc || !rd || !rgbw_out) return fail(PBRT_B200_ERR_INVALID, "render: null argument");
    return render_impl(sc, rd, rgbw_out, nullptr, stats);
}
extern "C" int pbrt_b200_render_splat(pbrt_b200_scene* sc, const pbrt_b200_render_desc* rd, float* rgbw_out, float* splat_out, pbrt_b200_render_stats* stats) {
    if (!sc || !rd || !rgbw_out || !splat_out) return fail(PBRT_B200_ERR_INVALID, "render_splat: null argument");
    return render_impl(sc, rd, rgbw_out, splat_out, stats);
}
