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
#include "scene.cuh"
#include "shading.cuh"
#include "trace.cuh"
#include "texture.cuh"
#include "util.cuh"

// Min resident CTAs per SM in __launch_bounds__, A/B-measured with tools/step_diag.py on S3: shade 5/6/8 CTAs (96/80/64 registers) and
// trace 6/8/10 CTAs are all within +-1% or slower than the compiler's default choice, so the shade kernels and the plain trace kernels
// set none.
#define PB_REC_BLOCK 384  /* threads per CTA of k_rec_shade (168 registers: one CTA per SM whose warps start every path together, see the kernel) */
#define PB_TEX_BLOCK 512  /* threads per CTA of k_shade<Q_TEX>: one CTA per SM whose warps start every path together (see k_shade) */

// This file is compiled THREE times (csrc/Makefile; mega.o -- the one-kernel forms -- is described where PB_MEGA_TU is defined below):
//   render.o  (PB_EXACT_TU = 1, --fmad=false, IEEE division / square root): ray generation, traversal, film, light tables, the
//             (0,2) megakernel and the host side -- everything whose arithmetic is pinned bit for bit against the oracle;
//   shade.o   (shade.cu defines PB_TU_SHADE and includes this file; --use_fast_math): only k_shade / k_rec_shade and their
//             launchers.  Shading is tolerance-parity by nature (libm differs from CUDA's transcendentals, SURVEY App. A.7):
//             there the ~200 IEEE divisions and square roots per path (8-10 SASS instructions each, with a slow-path call)
//             become MUFU.RCP / MUFU.RSQ sequences and a*b+c contracts to FFMA.
// Refill threshold of the wavefront trace kernels (lanes whose ray has finished are refilled once fewer than this many are still
// traversing).  Swept at 64 spp with runtime knobs (gpurun_out/r2q_tune.log): 16 -> 132.4 ms per step, 20 -> 133.2, 24 -> 134.7, 28 -> 136.5,
// 32 -> 141.0; interior_min 16 stays the best of 0 / 8 / 12 / 16 / 20 / 24.  (Compile-time constants: the runtime knobs cost 3 %.)
#define PB_WF_REFILL_BELOW 16
// Three translation units from this one source (csrc/Makefile): render.o (PB_EXACT_TU: everything but the kernels below, host side
// included), shade.o (PB_TU_SHADE, --use_fast_math: k_shade / k_rec_shade) and mega.o (PB_TU_MEGA, exact flags: the one-kernel forms
// k_zt_mega / k_vol_mega, whose out-of-line shade bodies are 2 minutes of ptxas on their own -- a separate unit compiles in parallel).
#if defined(PB_TU_SHADE)
#define PB_EXACT_TU 0
#define PB_MEGA_TU 0
#elif defined(PB_TU_MEGA)
#define PB_EXACT_TU 0
#define PB_MEGA_TU 1
#else
#define PB_EXACT_TU 1
#define PB_MEGA_TU 0
#endif
#define PB_SHADE_TU (!PB_EXACT_TU && !PB_MEGA_TU)
#define PB_ZT_WARPS 4u    /* warps per CTA of k_zt_mega (the host aims at ~4 warps per SM: one CTA), phases of a trip passed together */
#define PB_VOL_BLOCK 512  /* threads per CTA of k_vol_mega: the CTA's warps pass the phases of a trip together (barriers between them): see the kernel */

using namespace pb;

namespace pb {

enum { Q_MATTE = 0, Q_PLASTIC = 1, Q_MIRROR = 2, Q_GLASS = 3, Q_METAL = 4, Q_NOMAT = 5, Q_MISS = 6,
       Q_TEX = 7,  // `textured` material rows (texture.cuh): texture-valued parameters, bump maps, uber, substrate
       Q_COUNT = 8 };

struct Counters {
    uint32_t n_path;          // rays to trace this iteration
    uint32_t n_next;          // rays for the next iteration
    uint32_t n_shadow, n_mis;
    uint32_t n_dead;          // finished paths of this iteration (+ slots still waiting for a camera sample)
    uint32_t n_dead_next;     // slots re-queued because their item was outside the pixel bounds
    uint32_t n_mat[Q_COUNT];
    uint32_t fetch_path, fetch_shadow, fetch_mis;  // persistent ray-queue cursors (trace.cuh: trace_queue)
    uint32_t pad;
    unsigned long long camera_rays, closest_rays, shadow_rays, zero_radiance;
    unsigned long long item_cursor;  // next (sample, tile, pixel) item to hand to a free path slot
    unsigned long long iterations;
};

struct Tiny1D { float func[2], cdf[3], func_int; };  // Distribution1D with two entries
struct InfDistrib { Tiny1D cond[2], marg; };         // Distribution2D of a constant 1x1 env map (2x2 image)

struct SamplerDev {
    uint32_t kind, spp;
    int sb[4];
    // Sobol (samplers/sobol.rs:34-87)
    int resolution, log2_resolution;
    const uint32_t* sobol32;
    const uint32_t* sobol_t;  // transposed generator matrices [52 bits][1024 dims]: 8 consecutive dims of one bit are 32 contiguous bytes
    const unsigned long long* vdc;
    const unsigned long long* vdc_inv;
    // Halton (samplers/halton.rs:63-166)
    long long base_scales[2], base_exponents[2], mult_inverse[2];
    unsigned long long sample_stride;
    const uint16_t* perms;
    const uint32_t* primes;
    const uint32_t* prime_sums;
    uint32_t n_halton_dims;
    // Sobol' sample tables (see sobol_tab_block): value bits of dimension d for pixel p / sample number s, XORed at use
    const uint32_t* vp;     // [sample-bounds pixels][vstride]
    const uint32_t* vs;     // [samples of the call][vstride]
    uint32_t vdims;         // dimensions the tables cover; 0 = no tables (Halton, recursive integrators, 1x1 sample bounds)
    uint32_t vstride;       // row stride in words (multiple of 4: rows are 16-byte aligned)
    uint32_t sbw;           // sample-bounds width in pixels
    uint32_t vs_begin;      // sample number of row 0 of vs
};

// SpatialLightDistribution (core/lightdistrib.rs:105-340) on the device.  The reference fills a lock-free hash table of
// per-voxel Distribution1Ds on first touch; a voxel's distribution is a pure function of (scene, voxel), so here the
// table is dense (voxel -> slot) and slots are built either all up front ("eager", when voxels x lights is small) or
// per iteration for the voxels the current hits touch ("lazy": k_spatial_mark + k_spatial_build before the shade kernels).
struct SpatialDev {
    int enabled, lazy;
    int nvox[3];
    uint32_t capacity;      // slots allocated
    int* slot;              // [nvox total] -1 = not built, -2 = claimed (being built this iteration), >= 0 = slot
    float* func;            // [capacity][n_lights]   light_contrib after the min_contrib floor
    float* cdf;             // [capacity][n_lights+1]
    float* func_int;        // [capacity]
    uint2* build_list;      // {voxel, slot} pairs claimed this iteration
    uint32_t* counters;     // [0] build_count, [1] slot_count, [2] overflow / missing-voxel flag
    const float* halton;    // [128][5] radical_inverse(0..4, i)
};

// ZeroTwoSequenceSampler (src/samplers/zerotwosequence.rs:32-105 on the PixelSampler machinery, src/core/sampler.rs:185-253).
// The reference clones ONE sampler per 16x16 tile (seed = tile number, integrator.rs:302-303) and threads its PCG32 through
// every start_pixel() and every get_1d()/get_2d() beyond the precomputed dimensions of every path of the tile, in pixel /
// sample / bounce order: the random numbers a path sees depend on how many draws every earlier path of its tile made.  That
// stream cannot be reproduced with two paths of a tile in flight, so this sampler runs the wavefront "tile-serial": one
// path slot per tile, all tiles in parallel (8160 tiles at 1080p), each slot walking its tile's pixels and samples in
// the reference's order with the tile's generator state and sample tables in HBM.
struct ZtTile {
    unsigned long long state, inc;    // RNG (core/rng.rs:12-22)
    uint32_t pixel_idx, sample_idx;   // position in the tile's pixel loop (x fastest); current_pixel_sample_index
    uint32_t cur1d, cur2d;            // current_1d_dimension / current_2d_dimension
    int x0, y0;                       // tile bounds clipped to the sample bounds (integrator.rs:305-310)
    uint32_t w, npix;
};
struct ZtDev {
    ZtTile* tiles;
    float* s1d;      // [tile][dim][spp]   samples_1d
    float2* s2d;     // [tile][dim][spp]   samples_2d
    uint32_t spp;    // rounded up to a power of two (zerotwosequence.rs:36-40)
    uint32_t ndims;  // n_sampled_dimensions
    uint32_t n2d;    // rows of s2d per tile: ndims + the 2D sample arrays a DirectLightingIntegrator requested (one element per pixel sample:
                     // sobol_2d(1, spp) fills them right after the 2D dimensions, zerotwosequence.rs:67-71)
};

// State of the recursive integrators (recursive.cuh): per-slot stack of pending specular_transmit calls, sample-array
// cursor, and the per-iteration shadow / MIS entry arrays.  kind == 0 (path): nothing allocated.
struct RecDev {
    uint32_t kind;              // PBRT_B200_INTEGRATOR_*
    uint32_t stack_depth;       // frames per slot (= max_depth)
    uint32_t n_arrays;          // 2D sample arrays requested by DirectLightingIntegrator::preprocess ("all"): max_depth * n_lights * 2
    uint32_t multi;             // some light asks for more than one sample: array i then has lights[(i / 2) % n_lights].n_samples elements
    uint32_t* sample_num;       // [capacity] current_pixel_sample_index of the slot's camera sample (array element j = sample * n + k)
    uint32_t entries_per_slot;  // shadow (and MIS) rays one shaded surface can emit
    uint32_t* sp;               // [capacity] frames on the stack
    uint32_t* arr;              // [capacity] Sampler::array_2d_offset
    float4* st_ray;             // [capacity * stack_depth * 2] {o, valid}, {d, time}
    float4* st_beta;            // [capacity * stack_depth] {weight rgb, depth bits}
    float4* e_sh_ray;           // [capacity * entries_per_slot * 2]
    float4* e_sh_contrib;       // {rgb, slot bits}
    float4* e_mis_ray;
    float4* e_mis_contrib;      // {rgb factor, light index bits}
    uint32_t* e_mis_slot;
    float4* st_diff;            // [capacity * stack_depth * 3] ray differentials of the stacked rays (textured scenes only, else nullptr)
};

struct RenderDev {
    DevScene scene;
    pbrt_b200_camera camera;
    SamplerDev sampler;
    // film (core/film.rs)
    int crop[4];
    float filter_radius[2], inv_filter_radius[2];
    float max_sample_luminance;
    const float* filter_table;  // 256 floats
    float4* film;               // {r,g,b,w} per cropped pixel
    // integrator
    int max_depth;
    float rr_threshold;
    int pixel_bounds[4];
    // light distribution (core/lightdistrib.rs:20-83): uniform or power
    const float* ld_func;
    const float* ld_cdf;
    float ld_func_int;
    uint32_t n_lights;
    SpatialDev sp;
    ZtDev zt;
    RecDev rec;
    const InfDistrib* inf_distrib;     // indexed by light
    const uint32_t* infinite_lights;   // Scene.infinite_lights
    uint32_t n_infinite;
    // work decomposition (integrator.rs:274-279)
    int ntx, nty;
    uint32_t tile_begin, tile_end, n_tiles_sel, sample_begin, n_samples_sel;
    uint32_t tile_group, tile_mod, tile_rem;
    uint32_t tile_order, nstx;  // pbrt_b200_render_desc.tile_order; super-tile columns
    // path state, SoA over `capacity` slots
    uint32_t capacity;
    float4* ray;         // 2 x float4 per slot: {o, t_max}, {d, time}
    uint4* hit;          // {slot, t, b0, b1}
    float* hit_b2;
    uint32_t* hit_inst;  // instance of the hit (TransformedPrimitive) or PBRT_B200_NO_HIT; only touched when the scene has instances
    uint8_t* hit_bin;    // material bin of the hit (Q_*), written by trace_closest, consumed by classify
    float4* L_eta;       // {L.rgb, etascale}
    float4* beta_st;     // {beta.rgb, bits: bounces | specular_bounce << 16}
    float2* pfilm;
    unsigned long long* s_index;  // sampler: global sample index (Sobol / Halton)
    uint32_t* s_dim;              // sampler: next dimension
    uint32_t* pixel;              // x | y << 16 relative to sample bounds min
    float4* sh_ray;      // shadow ray (2 x float4)
    float4* sh_contrib;  // {rgb to add when unoccluded, -}
    float4* mis_ray;     // MIS ray (2 x float4)
    float4* mis_contrib; // {rgb factor (beta * f * |cos| * w / (scattpdf * lightselpdf)), light index bits}
    int* sp_voxel;       // lazy SpatialLightDistribution: the voxel k_spatial_mark claimed for the slot's hit.  The shade kernels (fast-math
                         // translation unit) would otherwise recompute the hit point with different roundings and, on a voxel boundary,
                         // look up a voxel nobody built
    uint32_t* tex_sort;  // textured scenes: {count[n_materials], cursor[n_materials]} of the per-iteration counting sort of the Q_TEX queue (k_tex_*)
    float4* rdiff;       // 3 x float4 per slot: RayDifferential of the slot's ray (texture.cuh store_diff), valid while PB_ST_HAS_DIFF is set in
                         // beta_st.w; nullptr unless the scene has textured materials
    float4* u8;          // 2 x float4 per slot: the next eight sample dimensions, written by k_sample_block when the Sobol' tables
                         // do not serve the path (Halton; dimensions beyond the tables); nullptr when that cannot happen
    uint32_t* q_path[2];
    uint32_t* q_shadow;
    uint32_t* q_mis;
    uint32_t* q_dead[2];
    uint32_t* q_mat[Q_COUNT];
    Counters* cnt;
};

// ---------------------------------------------------------------------------
// queue helpers: warp-aggregated append (one atomic per warp per queue)
// ---------------------------------------------------------------------------
PB_D void queue_push(uint32_t* q, uint32_t* counter, uint32_t value, bool pred) {
    unsigned mask = __ballot_sync(__activemask(), pred);
    if (!pred) return;
    int lane = threadIdx.x & 31;
    int leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(counter, (uint32_t)__popc(mask));
    base = __shfl_sync(mask, base, leader);
    q[base + __popc(mask & ((1u << lane) - 1))] = value;
}

// ---------------------------------------------------------------------------
// samplers on device
// ---------------------------------------------------------------------------
// core/lowdiscrepancy.rs:512-543
PB_D unsigned long long sobol_interval_to_index(const SamplerDev& S, uint32_t m, unsigned long long frame, int px, int py) {
    if (m == 0) return 0;
    uint32_t m2 = m << 1;
    unsigned long long index = frame << m2, delta = 0;
    const unsigned long long* V = S.vdc + (m - 1) * 52;
    for (int c = 0; frame != 0; frame >>= 1, ++c)
        if (frame & 1) delta ^= __ldg(V + c);
    unsigned long long b = ((unsigned long long)((uint32_t)px << m) | (unsigned long long)(long long)py) ^ delta;
    const unsigned long long* VI = S.vdc_inv + (m - 1) * 52;
    for (int c = 0; b != 0; b >>= 1, ++c)
        if (b & 1) index ^= __ldg(VI + c);
    return index;
}
// core/lowdiscrepancy.rs:549-569 + SobolSampler::sample_dimension (samplers/sobol.rs:69-87)
PB_D float sobol_dimension(const SamplerDev& S, unsigned long long a, uint32_t dim, int px, int py) {
    uint32_t v = 0;
    const uint32_t* M = S.sobol32 + dim * 52;
    for (; a != 0; a >>= 1, ++M)
        if (a & 1) v ^= __ldg(M);
    float s = fminf((float)v * 2.3283064365386963e-10f, PB_ONE_MINUS_EPSILON);
    if (dim == 0 || dim == 1) {
        s = s * (float)S.resolution + (float)S.sb[dim];
        s = clampf(s - (float)(dim == 0 ? px : py), 0.0f, PB_ONE_MINUS_EPSILON);
    }
    return s;
}
PB_D uint32_t reverse_bits32(uint32_t n) { return __brev(n); }  // lowdiscrepancy.rs:381-389
PB_D unsigned long long reverse_bits64(unsigned long long n) {
    return ((unsigned long long)__brev((uint32_t)n) << 32) | (unsigned long long)__brev((uint32_t)(n >> 32));
}
// radical_inverse / scrambled_radical_inverse, lowdiscrepancy.rs:398-414, 468-484
PB_D float radical_inverse(const SamplerDev& S, uint32_t base_index, unsigned long long n) {
    if (base_index == 0) return (float)reverse_bits64(n) * 5.421010862427522e-20f;  // 2^-64, no clamp
    unsigned long long base = __ldg(S.primes + base_index);
    float inv_base = 1.0f / (float)base, inv_basen = 1.0f;
    unsigned long long rev = 0;
    while (n != 0) {
        unsigned long long next = n / base, digit = n - next * base;
        rev = rev * base + digit;
        inv_basen *= inv_base;
        n = next;
    }
    return fminf((float)rev * inv_basen, PB_ONE_MINUS_EPSILON);
}
PB_D float scrambled_radical_inverse(const SamplerDev& S, uint32_t base_index, unsigned long long a) {
    unsigned long long base = __ldg(S.primes + base_index);
    const uint16_t* perm = S.perms + __ldg(S.prime_sums + base_index);
    float inv_base = 1.0f / (float)base, inv_basen = 1.0f;
    unsigned long long rev = 0;
    while (a != 0) {
        unsigned long long next = a / base, digit = a - next * base;
        rev = rev * base + (unsigned long long)__ldg(perm + digit);
        inv_basen *= inv_base;
        a = next;
    }
    float res = inv_basen * ((float)rev + inv_base * (float)__ldg(perm) / (1.0f - inv_base));
    return fminf(res, PB_ONE_MINUS_EPSILON);
}
PB_D long long mod_ll(long long a, long long b) { long long r = a - (a / b) * b; return r < 0 ? r + b : r; }
PB_D unsigned long long inverse_radical_inverse(unsigned long long base, unsigned long long inverse, unsigned long long nd) {
    unsigned long long index = 0;
    for (unsigned long long i = 0; i < nd; ++i) { unsigned long long digit = inverse % base; inverse /= base; index = index * base + digit; }
    return index;
}
// HaltonSampler::get_index_for_sample, halton.rs:124-152 (px,py are absolute pixel coordinates)
PB_D unsigned long long halton_index(const SamplerDev& S, unsigned long long sample, int px, int py) {
    unsigned long long off = 0;
    if (S.sample_stride > 1 && !(px == 0 && py == 0)) {  // pixel_for_offset starts at (0,0) in the reference
        long long pm0 = mod_ll(px, 128), pm1 = mod_ll(py, 128);
        off += inverse_radical_inverse(2, (unsigned long long)pm0, (unsigned long long)S.base_exponents[0]) *
               (S.sample_stride / (unsigned long long)S.base_scales[0]) * (unsigned long long)S.mult_inverse[0];
        off += inverse_radical_inverse(3, (unsigned long long)pm1, (unsigned long long)S.base_exponents[1]) *
               (S.sample_stride / (unsigned long long)S.base_scales[1]) * (unsigned long long)S.mult_inverse[1];
        off %= S.sample_stride;
    }
    return off + sample * S.sample_stride;
}
PB_D float halton_dimension(const SamplerDev& S, unsigned long long index, uint32_t dim) {
    if (dim == 0) return radical_inverse(S, 0, index >> (unsigned long long)S.base_exponents[0]);
    if (dim == 1) return radical_inverse(S, 1, index / (unsigned long long)S.base_scales[1]);
    return scrambled_radical_inverse(S, dim, index);
}

struct SampleCursor { unsigned long long index; uint32_t dim; int px, py; };  // absolute pixel
// Dimensions the tables hold: 1024 Sobol' matrices, PRIME_TABLE_SIZE primes.  The reference indexes past them and panics; here (and in the
// oracle) deeper dimensions read 0.5.
PB_D uint32_t sampler_dim_limit(const SamplerDev& S) { return S.kind == PBRT_B200_SAMPLER_SOBOL ? 1024u : S.n_halton_dims; }
PB_D float sample_dimension(const SamplerDev& S, const SampleCursor& c, uint32_t dim) {
    return S.kind == PBRT_B200_SAMPLER_SOBOL ? sobol_dimension(S, c.index, dim, c.px, c.py) : halton_dimension(S, c.index, dim);
}
// GlobalSampler::get_1d / get_2d, core/sampler.rs:322-353 (no sample arrays requested by the path integrator)
PB_D float get_1d(const SamplerDev& S, SampleCursor& c) { float r = sample_dimension(S, c, c.dim); c.dim += 1; return r; }
PB_D float2 get_2d(const SamplerDev& S, SampleCursor& c) {
    float y = sample_dimension(S, c, c.dim + 1);
    float x = sample_dimension(S, c, c.dim);
    c.dim += 2;
    return make_float2(x, y);
}

// Eight consecutive dimensions of one sample at once.  For Sobol' this walks the set bits of the
// index a single time and XORs 8 matrix columns per bit (sobol_sample_float, lowdiscrepancy.rs:549-569,
// evaluated for dims dim0..dim0+7 together); the values are bit-identical to the per-dimension loop.
struct SampleBlock { float u[8]; uint32_t used; };
PB_D void sample_block(const SamplerDev& S, const SampleCursor& c, SampleBlock& b) {
    b.used = 0;
    if (S.kind == PBRT_B200_SAMPLER_SOBOL && c.dim >= 2 && c.dim + 8 <= 1024) {
        uint32_t v[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
        unsigned long long a = c.index;
        while (a != 0) {
            int bit = __ffsll((long long)a) - 1;
            a &= a - 1;
            const uint32_t* row = S.sobol_t + (uint32_t)bit * 1024u + c.dim;
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] ^= __ldg(row + k);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) b.u[k] = fminf((float)v[k] * 2.3283064365386963e-10f, PB_ONE_MINUS_EPSILON);
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) b.u[k] = (c.dim + k < sampler_dim_limit(S)) ? sample_dimension(S, c, c.dim + k) : 0.5f;
    }
}
PB_D float block_pick(const SampleBlock& b, uint32_t k) {
    float r = b.u[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) r = (k == (uint32_t)i) ? b.u[i] : r;
    return r;
}
PB_D float get_1d(SampleBlock& b) { float r = block_pick(b, b.used); b.used += 1; return r; }
PB_D float2 get_2d(SampleBlock& b) {  // x from the lower dimension (sampler.rs:341-352)
    float2 r = make_float2(block_pick(b, b.used), block_pick(b, b.used + 1));
    b.used += 2;
    return r;
}

// Sobol' through tables.  sobol_interval_to_index and sobol_sample_float (lowdiscrepancy.rs:512-569) are linear over GF(2):
//   index(p, s) = Ip(p) ^ Is(s),  Ip = XOR of VdCInv columns over the bits of (p.x << m | p.y),
//                                 Is = (s << 2m) ^ XOR of VdCInv columns over the bits of delta(s)
//   bits_d(index) = XOR of generator-matrix columns of dimension d over the bits of index = bits_d(Ip) ^ bits_d(Is)
// so the 32 value bits of (pixel, sample, dimension) are vp[pixel][d] ^ vs[s][d]: two table rows replace the index
// computation and the ~15-step walk over the set bits of the index with 8 loads each (27 % of the shade kernels' stall
// samples, profiles/r01_ncu_full_s10.md).  XOR is associative and commutative: the bits, hence the floats, are identical.
// In table mode R.s_index[slot] holds the SAMPLE NUMBER, not the Sobol' index.
PB_D bool sobol_tab_covers(const SamplerDev& S, uint32_t dim) { return dim + 8u <= S.vdims; }
PB_D void sobol_tab_block(const SamplerDev& S, uint32_t pxy, uint32_t sample, uint32_t dim, float* u) {
    const uint32_t* a = S.vp + ((size_t)(pxy >> 16) * S.sbw + (pxy & 0xffffu)) * S.vstride + dim;
    const uint32_t* b = S.vs + (size_t)(sample - S.vs_begin) * S.vstride + dim;
    uint32_t va[8], vb[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { va[k] = __ldg(a + k); vb[k] = __ldg(b + k); }
#pragma unroll
    for (int k = 0; k < 8; ++k) u[k] = fminf((float)(va[k] ^ vb[k]) * 2.3283064365386963e-10f, PB_ONE_MINUS_EPSILON);
}

// ---- (0,2)-sequence sampler, tile-serial (see ZtTile)
PB_D uint32_t zt_u32(ZtTile& t) {  // RNG::uniform_int32, rng.rs:31-48
    unsigned long long old = t.state;
    t.state = old * 0x5851f42d4c957f2dULL + t.inc;
    uint32_t xs = (uint32_t)(((old >> 18) ^ old) >> 27), rot = (uint32_t)(old >> 59);
    return (xs >> rot) | (xs << ((~rot + 1u) & 31u));
}
PB_D uint32_t zt_bounded(ZtTile& t, uint32_t b) {  // uniform_int32_2, rng.rs:50-60
    uint32_t threshold = (~b + 1u) % b;
    for (;;) { uint32_t r = zt_u32(t); if (r >= threshold) return r % b; }
}
PB_D float zt_float(ZtTile& t) { return fminf(PB_ONE_MINUS_EPSILON, (float)zt_u32(t) * 2.3283064365386963e-10f); }  // rng.rs:62-64
PB_D void zt_set_sequence(ZtTile& t, unsigned long long seq) {  // rng.rs:66-74
    t.state = 0; t.inc = (seq << 1) | 1ull;
    zt_u32(t);
    t.state += 0x853c49e6748fea9bULL;
    zt_u32(t);
}
// ZeroTwoSequenceSampler::start_pixel (zerotwosequence.rs:54-66): van_der_corput / sobol_2d (lowdiscrepancy.rs:486-510) with
// one sample per pixel sample => gray-code points, one shuffle() of every 1-element block (a draw each), one shuffle of the lot
static __device__ __noinline__ void zt_start_pixel(ZtTile* tp, float* s1d, float2* s2d, uint32_t spp, uint32_t ndims, uint32_t n2d) {
    ZtTile t = *tp;
    for (uint32_t d = 0; d < ndims; ++d) {
        float* sm = s1d + (size_t)d * spp;
        uint32_t v = zt_u32(t);  // scramble
        for (uint32_t i = 0; i < spp; ++i) {  // gray_code_sample1d with CVAN_DER_CORPUT (identity, MSB first)
            sm[i] = fminf((float)v * 2.3283064365386963e-10f, PB_ONE_MINUS_EPSILON);
            v ^= 0x80000000u >> __ffs((int)(i + 1)) - 1;
        }
        for (uint32_t i = 0; i < spp; ++i) zt_u32(t);          // shuffle(&samples[i..], 1, 1): uniform_int32_2(1) = one draw (threshold 0), result 0
        for (uint32_t i = 0; i < spp; ++i) {                   // shuffle(samples, spp, 1), sampling.rs:178-186
            uint32_t other = i + zt_bounded(t, spp - i);
            float a = sm[i]; sm[i] = sm[other]; sm[other] = a;
        }
    }
    for (uint32_t d = 0; d < n2d; ++d) {  // the 2D dimensions, then the 2D sample arrays (no 1D arrays are ever requested)
        float2* sm = s2d + (size_t)d * spp;
        uint32_t v0 = zt_u32(t), v1 = zt_u32(t);
        for (uint32_t i = 0; i < spp; ++i) {  // gray_code_sample2d with CSOBOL[0], CSOBOL[1] (lowdiscrepancy.rs:203-217)
            sm[i] = make_float2(fminf((float)v0 * 2.3283064365386963e-10f, PB_ONE_MINUS_EPSILON), fminf((float)v1 * 2.3283064365386963e-10f, PB_ONE_MINUS_EPSILON));
            int k = __ffs((int)(i + 1)) - 1;
            v0 ^= 0x80000000u >> k;
            uint32_t c1 = 0x80000000u;  // CSOBOL[1][k]: c[0] = 2^31, c[j] = c[j-1] ^ (c[j-1] >> 1)
            for (int j = 0; j < k; ++j) c1 ^= c1 >> 1;
            v1 ^= c1;
        }
        for (uint32_t i = 0; i < spp; ++i) zt_u32(t);
        for (uint32_t i = 0; i < spp; ++i) {
            uint32_t other = i + zt_bounded(t, spp - i);
            float2 a = sm[i]; sm[i] = sm[other]; sm[other] = a;
        }
    }
    t.sample_idx = 0; t.cur1d = 0; t.cur2d = 0;
    *tp = t;
}
// PixelSampler get_1d / get_2d, sampler.rs:228-253 (beyond the precomputed dimensions: raw draws, y before x)
struct ZtCursor { ZtTile* t; const float* s1d; const float2* s2d; uint32_t spp, ndims, n2d; };
PB_D ZtCursor zt_cursor(const RenderDev& R, uint32_t tile_ordinal) {
    ZtCursor c;
    c.t = R.zt.tiles + tile_ordinal;
    c.s1d = R.zt.s1d + (size_t)tile_ordinal * R.zt.ndims * R.zt.spp;
    c.s2d = R.zt.s2d + (size_t)tile_ordinal * R.zt.n2d * R.zt.spp;
    c.spp = R.zt.spp; c.ndims = R.zt.ndims; c.n2d = R.zt.n2d;
    return c;
}
PB_D float get_1d(ZtCursor& c) {
    ZtTile& t = *c.t;
    if (t.cur1d < c.ndims) { float v = c.s1d[(size_t)t.cur1d * c.spp + t.sample_idx]; t.cur1d += 1; return v; }
    return zt_float(t);
}
PB_D float2 get_2d(ZtCursor& c) {
    ZtTile& t = *c.t;
    if (t.cur2d < c.ndims) { float2 v = c.s2d[(size_t)t.cur2d * c.spp + t.sample_idx]; t.cur2d += 1; return v; }
    float y = zt_float(t);
    float x = zt_float(t);
    return make_float2(x, y);
}

// The sampler interface the shade kernels are written against.  ZT = false: Sobol' / Halton, a pure function of
// (sample index, dimension) evaluated eight dimensions at a time; ZT = true: the tile's (0,2)-sequence state.
template <bool ZT> struct PathSampler;
template <> struct PathSampler<false> {
    SampleCursor c; SampleBlock sb;
    // The shade kernels carry no sampler arithmetic: either the Sobol' tables cover the block (two row reads), or the
    // pre-pass k_sample_block has left the eight values in R.u8 (Halton, Sobol' dimensions beyond the tables).
    uint32_t pxy;
    // Called first thing in shade_path: the slot's sampler state is loaded together with its ray and hit record, and the pixel's
    // table row (a random 32..64-byte span of a table far larger than L2) is requested from HBM right away -- by the time the
    // surface and the BSDF are set up it sits in L1, instead of being a third dependent DRAM round trip (queue -> state -> row)
    // in the middle of the kernel (27 % of the matte kernel's stall samples, profiles/r02_ncu_shade.md).
    PB_D void prefetch(const RenderDev& R, uint32_t id) {
        c.index = R.s_index[id]; c.dim = R.s_dim[id]; pxy = R.pixel[id];
        if (sobol_tab_covers(R.sampler, c.dim)) {
            const uint32_t* a = R.sampler.vp + ((size_t)(pxy >> 16) * R.sampler.sbw + (pxy & 0xffffu)) * R.sampler.vstride + c.dim;
            asm volatile("prefetch.global.L1 [%0];" ::"l"(a));
            asm volatile("prefetch.global.L1 [%0];" ::"l"(a + 7));
        }
    }
    PB_D void begin(const RenderDev& R, uint32_t id) {
        sb.used = 0;
        if (sobol_tab_covers(R.sampler, c.dim)) sobol_tab_block(R.sampler, pxy, (uint32_t)c.index, c.dim, sb.u);
        else {
            const float4 lo = R.u8[2 * id], hi = R.u8[2 * id + 1];
            sb.u[0] = lo.x; sb.u[1] = lo.y; sb.u[2] = lo.z; sb.u[3] = lo.w; sb.u[4] = hi.x; sb.u[5] = hi.y; sb.u[6] = hi.z; sb.u[7] = hi.w;
        }
    }
    PB_D float get_1d() { return pb::get_1d(sb); }
    PB_D float2 get_2d() { return pb::get_2d(sb); }
    PB_D void end(const RenderDev& R, uint32_t id) { R.s_dim[id] = c.dim + sb.used; }
};
template <> struct PathSampler<true> {
    ZtCursor z;
    PB_D void prefetch(const RenderDev&, uint32_t) {}
    PB_D void begin(const RenderDev& R, uint32_t id) { z = zt_cursor(R, id); }  // slot == tile ordinal
    PB_D float get_1d() { return pb::get_1d(z); }
    PB_D float2 get_2d() { return pb::get_2d(z); }
    PB_D void end(const RenderDev&, uint32_t) {}
};

// The volpath megakernel's sampler (k_vol_mega): GlobalSampler::get_1d / get_2d evaluated one dimension at a time, because the number
// of dimensions a path segment consumes depends on whether the ray travels in a medium (2 more) and on what it meets.
struct DirectSampler {
    SampleCursor c; const SamplerDev* S;
    PB_D void prefetch(const RenderDev& R, uint32_t id) {
        const uint32_t pxy = R.pixel[id];
        c.index = R.s_index[id]; c.dim = R.s_dim[id];
        c.px = (int)(pxy & 0xffffu) + R.sampler.sb[0]; c.py = (int)(pxy >> 16) + R.sampler.sb[1];
        S = &R.sampler;
    }
    PB_D void begin(const RenderDev&, uint32_t) {}
    PB_D float dim_value(uint32_t d) const { return d < sampler_dim_limit(*S) ? sample_dimension(*S, c, d) : 0.5f; }
    PB_D float get_1d() { float r = dim_value(c.dim); c.dim += 1; return r; }
    PB_D float2 get_2d() { float y = dim_value(c.dim + 1), x = dim_value(c.dim); c.dim += 2; return make_float2(x, y); }
    PB_D void end(const RenderDev& R, uint32_t id) { R.s_dim[id] = c.dim; }
};
template <bool ZT, bool VOL> struct SamplerSel { using type = PathSampler<ZT>; };
template <bool ZT> struct SamplerSel<ZT, true> { using type = DirectSampler; };

// Per-path state of the volpath integrator that the surface path integrator does not have (kept by the megakernel thread that owns
// the path): the medium the path ray travels in, and what the two transmittance loops of estimate_direct need to continue through
// material-less surfaces (VisibilityTester::tr, light.rs:125-150; Scene::intersect_tr, scene.rs:68-87).
struct VolState {
    int medium;            // Ray.medium of the path ray (-1: vacuum)
    int sh_medium;         // ... of the shadow ray's first segment
    int mis_medium;        // ... of the BSDF / phase-sampled ray's first segment
    f3 p1, p1_err, p1_n;   // VisibilityTester.p1: where the shadow segments are re-aimed
    f3 mi_p;               // the sampled MediumInteraction
};
// MediumInterface of an intersection (primitive.rs:134-140) and Interaction::get_medium_vec (interaction.rs:54-66)
struct VolInterface { int inside, outside; };
PB_D VolInterface vol_hit_interface(const DevScene& s, uint32_t slot, int ray_medium) {
    VolInterface mi{ray_medium, ray_medium};  // MediumInterface::new(ray.medium)
    if (s.prim_media) {
        const pbrt_b200_medium_interface pm = s.prim_media[slot];
        if (pm.inside != pm.outside) { mi.inside = pm.inside; mi.outside = pm.outside; }  // is_medium_transition
    }
    return mi;
}
PB_D int vol_medium_for(const VolInterface& mi, f3 n, f3 w) { return dot(w, n) > 0.0f ? mi.outside : mi.inside; }
// phase_hg and HenyeyGreenstein::sample_p, medium.rs:162-221
PB_D float phase_hg(float cos_theta, float g) {
    float denom = 1.0f + g * g + 2.0f * g * cos_theta;
    return PB_INV_4PI * (1.0f - g * g) / (denom * sqrtf(denom));
}
PB_D float hg_sample_p(float g, f3 wo, f3* wi, float2 u) {
    float cos_theta;
    if (fabsf(g) < 1.0e-3f) cos_theta = 1.0f - 2.0f * u.x;
    else {
        float sqr = (1.0f - g * g) / (1.0f + g - 2.0f * g * u.x);
        cos_theta = -(1.0f + g * g - sqr * sqr) / (2.0f * g);
    }
    float sin_theta = sqrtf(fmaxf(0.0f, 1.0f - cos_theta * cos_theta));
    float phi = 2.0f * PB_PI * u.y;
    f3 v1, v2;
    coordinate_system(wo, &v1, &v2);
    *wi = v1 * sin_theta * cosf(phi) + v2 * sin_theta * sinf(phi) + wo * cos_theta;  // spherical_direction_basis, geometry.rs:36-38
    return phase_hg(cos_theta, g);
}
PB_D rgb medium_sigma_t(const pbrt_b200_medium& m) { return rgb3(m.sigma_a) + rgb3(m.sigma_s); }
// HomogeneousMedium::tr, homogeneous.rs:30-33
PB_D rgb medium_tr(const pbrt_b200_medium& m, f3 d, float t_max) {
    const rgb st = medium_sigma_t(m);
    const float dist = fminf(t_max * len(d), PB_FLT_MAX);
    return rgb(expf(-st.r * dist), expf(-st.g * dist), expf(-st.b * dist));
}

// ---------------------------------------------------------------------------
// film: FilmTile::add_sample (core/film.rs:292-331) with warp-aggregated atomics
// ---------------------------------------------------------------------------
PB_D void film_atomic_add(float4* film, uint32_t pix, float4 v, bool active) {
    // lanes that target the same pixel are summed in-warp; one vector atomic per distinct pixel
    unsigned amask = __ballot_sync(__activemask(), active);
    if (!active) return;
    unsigned peers = __match_any_sync(amask, pix);
    int lane = threadIdx.x & 31;
    int leader = __ffs(peers) - 1;
    if (peers != (1u << lane)) {
        const int len = __popc(peers), rel = lane - leader;
        if ((peers >> leader) == (len == 32 ? 0xffffffffu : ((1u << len) - 1u))) {
            // a contiguous run of lanes (consecutive samples of one pixel: the common case with samples innermost): tree reduction,
            // every element reaches the run's first lane exactly once
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
                const float x = __shfl_down_sync(peers, v.x, off), y = __shfl_down_sync(peers, v.y, off), z = __shfl_down_sync(peers, v.z, off), w = __shfl_down_sync(peers, v.w, off);
                if (rel + off < len) { v.x += x; v.y += y; v.z += z; v.w += w; }
            }
        } else {
            // scattered peers (filters wider than a pixel): every peer publishes, the leader gathers
            float4 acc = v;
            unsigned rest = peers & ~(1u << leader);
            for (unsigned m = rest; m; m &= m - 1) {
                int src = __ffs(m) - 1;
                float x = __shfl_sync(peers, v.x, src), y = __shfl_sync(peers, v.y, src), z = __shfl_sync(peers, v.z, src), w = __shfl_sync(peers, v.w, src);
                if (lane == leader) { acc.x += x; acc.y += y; acc.z += z; acc.w += w; }
            }
            v = acc;
        }
    }
    if (lane == leader) atomicAdd(film + pix, v);
}

PB_D void film_add_sample(const RenderDev& R, float2 pfilm, rgb L, bool active) {
    // all lanes of the warp walk the same (maximal) footprint loop so the aggregation can use shuffles
    float rx = R.filter_radius[0], ry = R.filter_radius[1];
    int p0x = 0, p0y = 0, p1x = 0, p1y = 0;
    float dx = 0.f, dy = 0.f;
    if (active) {
        float ly = lum(L);
        if (ly > R.max_sample_luminance) L = L * rgb(R.max_sample_luminance / ly);
        dx = pfilm.x - 0.5f; dy = pfilm.y - 0.5f;
        p0x = max((int)ceilf(dx - rx), R.crop[0]); p0y = max((int)ceilf(dy - ry), R.crop[1]);
        p1x = min((int)floorf(dx + rx) + 1, R.crop[2]); p1y = min((int)floorf(dy + ry) + 1, R.crop[3]);
    }
    int nx = max(p1x - p0x, 0), ny = max(p1y - p0y, 0);
    unsigned amask = __activemask();
    int mx = nx, my = ny;
    for (int o = 16; o; o >>= 1) { mx = max(mx, __shfl_xor_sync(amask, mx, o)); my = max(my, __shfl_xor_sync(amask, my, o)); }
    const int width = R.crop[2] - R.crop[0];
    for (int j = 0; j < my; ++j)
        for (int i = 0; i < mx; ++i) {
            bool on = active && i < nx && j < ny;
            int x = p0x + i, y = p0y + j;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            uint32_t pix = 0;
            if (on) {
                float fx = fabsf(((float)x - dx) * R.inv_filter_radius[0] * 16.0f);
                float fy = fabsf(((float)y - dy) * R.inv_filter_radius[1] * 16.0f);
                int ix = min((int)floorf(fx), 15), iy = min((int)floorf(fy), 15);
                float fw = __ldg(R.filter_table + iy * 16 + ix);
                rgb c = L * rgb(1.0f) * rgb(fw);  // sample_weight = 1 (perspective.rs:141)
                v = make_float4(c.r, c.g, c.b, fw);
                pix = (uint32_t)((y - R.crop[1]) * width + (x - R.crop[0]));
            }
            film_atomic_add(R.film, pix, v, on);
        }
}

// ---------------------------------------------------------------------------
// K1: raygen
// ---------------------------------------------------------------------------
// PerspectiveCamera::generate_ray_differential (cameras/perspective.rs:120-179), main ray;
// Transform::transform_ray (core/transform.rs:543-577)
PB_D void generate_ray(const pbrt_b200_camera& c, float2 pfilm, float time_u, float2 plens, f3* o_out, f3* d_out, float* time_out) {
    f3 pc = xf_point(c.raster_to_camera, f3(pfilm.x, pfilm.y, 0.0f));
    f3 o(0.f, 0.f, 0.f), d = normalize(pc);
    if (c.lens_radius > 0.0f) {
        float2 pl = concentric_disk(plens);
        pl.x *= c.lens_radius; pl.y *= c.lens_radius;
        float ft = c.focal_distance / d.z;
        f3 pfocus = o + d * ft;
        o = f3(pl.x, pl.y, 0.0f);
        d = normalize(pfocus - o);
    }
    *time_out = c.shutter_open * (1.0f - time_u) + c.shutter_close * time_u;  // lerp, pbrt.rs:136-145
    f3 oerr;
    f3 ow = xf_point_err(c.camera_to_world, o, &oerr);
    f3 dw = xf_vector(c.camera_to_world, d);
    float l2 = len2(dw);
    if (l2 > 0.0f) {
        float dt = dot(vabs(dw), oerr) / l2;
        ow = ow + dw * dt;
    }
    *o_out = ow; *d_out = dw;
}

#define PB_ST_TWO_LOBES 0x40000u /* a stacked specular_transmit frame with two candidate lobes (recursive.cuh) */
#define PB_ST_HAS_DIFF 0x20000u /* beta_st.w: the slot's ray carries differentials (a camera ray, or a specular bounce of one under whitted / directlighting) */
// The differential half of PerspectiveCamera::generate_ray_differential (cameras/perspective.rs:144-176; dx_camera / dy_camera :64-70),
// then Ray::scale_differential(1 / sqrt(spp)) as the render loop applies it (integrator.rs:341, ray.rs:34-41).  o / d: the world ray.
// (inlined on purpose: an out-of-line call would take the address of the kernel parameter `R.camera`, and ptxas then copies the whole
// parameter block into a 1.3 KB local-memory frame in every thread of k_finish_regen -- textured scene or not)
PB_D void camera_differentials(const pbrt_b200_camera& c, float2 pfilm, float2 plens, f3 o, f3 d, uint32_t spp, float4* out, size_t slot) {
    const f3 pc = xf_point(c.raster_to_camera, f3(pfilm.x, pfilm.y, 0.0f));
    const f3 p2t = xf_point(c.raster_to_camera, f3(0.f, 0.f, 0.f));
    const f3 dxc = xf_point(c.raster_to_camera, f3(1.f, 0.f, 0.f)) - p2t, dyc = xf_point(c.raster_to_camera, f3(0.f, 1.f, 0.f)) - p2t;
    RayDiff r;
    r.has = true;
    if (c.lens_radius > 0.0f) {
        float2 pl = concentric_disk(plens);
        pl.x *= c.lens_radius; pl.y *= c.lens_radius;
        f3 dx = normalize(pc + dxc);
        float ft = c.focal_distance / dx.z;
        f3 pfocus = dx * ft;
        r.rxo = f3(pl.x, pl.y, 0.0f);
        r.rxd = normalize(pfocus - r.rxo);
        f3 dy = normalize(pc + dyc);
        ft = c.focal_distance / dy.z;
        pfocus = dy * ft;
        r.ryo = f3(pl.x, pl.y, 0.0f);
        r.ryd = normalize(pfocus - r.ryo);
    } else {
        r.rxo = r.ryo = f3(0.f, 0.f, 0.f);
        r.rxd = normalize(pc + dxc);
        r.ryd = normalize(pc + dyc);
    }
    r.rxo = xf_point(c.camera_to_world, r.rxo); r.ryo = xf_point(c.camera_to_world, r.ryo);
    r.rxd = xf_vector(c.camera_to_world, r.rxd); r.ryd = xf_vector(c.camera_to_world, r.ryd);
    const float sc = 1.0f / sqrtf((float)spp);
    r.rxo = o + (r.rxo - o) * sc; r.ryo = o + (r.ryo - o) * sc;
    r.rxd = d + (r.rxd - d) * sc; r.ryd = d + (r.ryd - d) * sc;
    store_diff(out, slot, r);
}

#define PB_NO_SAMPLE 0xffffffffu /* R.pixel[slot]: the slot carries no camera sample (nothing to add to the film) */

// Position t of the call's tile numbering (pbrt_b200_render_desc.tile_order) -> tile coordinates; false past the image edge.
PB_D bool tile_xy(const RenderDev& R, uint32_t t, int* tx, int* ty) {
    if (R.tile_order == 0) { *tx = (int)(t % (uint32_t)R.ntx); *ty = (int)(t / (uint32_t)R.ntx); return true; }
    const uint32_t S = R.tile_order, st = t / (S * S), w = t - st * (S * S);
    *tx = (int)((st % R.nstx) * S + w % S); *ty = (int)((st / R.nstx) * S + w / S);
    return *tx < R.ntx && *ty < R.nty;
}

// One camera sample into path slot `slot`.  Returns false when the item falls outside the sample/pixel bounds (partial edge
// tiles) -- the slot then stays free.  Item order: (tile, pixel-in-tile, sample) with the samples of the call
// INNERMOST, so the 32 lanes of a warp carry consecutive samples of ONE pixel (when the call has >= 32 of them): their camera
// rays walk the same nodes (one L1 wavefront per load instead of one per lane), hit the same few triangles, read the same pixel row
// of the sampler table, and their film contributions collapse into one atomic per warp.  The alternative (samples outermost:
// a warp = 32 neighbouring pixels of one sample) was round 1's order.  Every sample is an independent function of (pixel, sample
// number), so the image does not depend on the order (only the film's f32 summation order does).
PB_D bool gen_camera_path(const RenderDev& R, unsigned long long item, uint32_t slot) {
    uint32_t p, j, sample;  // pixel in tile; ordinal among the tiles this call owns; sample number
    {
        unsigned long long pp;  // tile-pixel ordinal
        if ((item >> 32) == 0) { const uint32_t i32 = (uint32_t)item, q = i32 / R.n_samples_sel; sample = i32 - q * R.n_samples_sel + R.sample_begin; pp = q; }
        else { pp = item / R.n_samples_sel; sample = (uint32_t)(item - pp * R.n_samples_sel) + R.sample_begin; }
        p = (uint32_t)(pp & 255u); j = (uint32_t)(pp >> 8);
    }
    const uint32_t jg = j / R.tile_group;
    uint32_t t = R.tile_begin + (jg * R.tile_mod + R.tile_rem) * R.tile_group + (j - jg * R.tile_group);
    int tx, ty;
    bool valid = tile_xy(R, t, &tx, &ty) && t < R.tile_end;
    int x = R.sampler.sb[0] + tx * 16 + (int)(p & 15u);
    int y = R.sampler.sb[1] + ty * 16 + (int)(p >> 4);
    valid = valid && x < R.sampler.sb[2] && y < R.sampler.sb[3] && x >= R.pixel_bounds[0] && x < R.pixel_bounds[2] && y >= R.pixel_bounds[1] &&
            y < R.pixel_bounds[3];
    if (!valid) { R.pixel[slot] = PB_NO_SAMPLE; return false; }
    SampleCursor c;
    c.px = x; c.py = y; c.dim = 0;
    // get_camera_sample, sampler.rs:170-180: dimensions 0..4
    float2 u, plens;
    float tu;
    if (R.sampler.vdims) {
        // Sobol' tables (sobol_tab_block): no index, no bit walk; the slot remembers the sample number
        const uint32_t* a = R.sampler.vp + ((size_t)(y - R.sampler.sb[1]) * R.sampler.sbw + (uint32_t)(x - R.sampler.sb[0])) * R.sampler.vstride;
        const uint32_t* b = R.sampler.vs + (size_t)(sample - R.sampler.vs_begin) * R.sampler.vstride;
        const uint4 a4 = __ldg(reinterpret_cast<const uint4*>(a)), b4 = __ldg(reinterpret_cast<const uint4*>(b));
        const uint32_t v[5] = {a4.x ^ b4.x, a4.y ^ b4.y, a4.z ^ b4.z, a4.w ^ b4.w, __ldg(a + 4) ^ __ldg(b + 4)};
        float f[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) f[k] = fminf((float)v[k] * 2.3283064365386963e-10f, PB_ONE_MINUS_EPSILON);
        f[0] = clampf(f[0] * (float)R.sampler.resolution + (float)R.sampler.sb[0] - (float)x, 0.0f, PB_ONE_MINUS_EPSILON);
        f[1] = clampf(f[1] * (float)R.sampler.resolution + (float)R.sampler.sb[1] - (float)y, 0.0f, PB_ONE_MINUS_EPSILON);
        u = make_float2(f[0], f[1]); tu = f[2]; plens = make_float2(f[3], f[4]);
        c.index = sample; c.dim = 5;
    } else if (R.sampler.kind == PBRT_B200_SAMPLER_SOBOL) {
        c.index = sobol_interval_to_index(R.sampler, (uint32_t)R.sampler.log2_resolution, sample, x - R.sampler.sb[0], y - R.sampler.sb[1]);
        // sobol_sample_float (lowdiscrepancy.rs:549-569) for the five dimensions in ONE walk over the set bits of the index,
        // reading 5 adjacent columns of the bit-transposed matrices; dims 0/1 then get SobolSampler::sample_dimension's
        // pixel remap (sobol.rs:69-87).  Same XOR sums as the per-dimension loops => identical values.
        uint32_t v[5] = {0u, 0u, 0u, 0u, 0u};
        unsigned long long a = c.index;
        while (a != 0) {
            int bit = __ffsll((long long)a) - 1;
            a &= a - 1;
            const uint32_t* row = R.sampler.sobol_t + (uint32_t)bit * 1024u;
#pragma unroll
            for (int k = 0; k < 5; ++k) v[k] ^= __ldg(row + k);
        }
        float f[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) f[k] = fminf((float)v[k] * 2.3283064365386963e-10f, PB_ONE_MINUS_EPSILON);
        f[0] = clampf(f[0] * (float)R.sampler.resolution + (float)R.sampler.sb[0] - (float)x, 0.0f, PB_ONE_MINUS_EPSILON);
        f[1] = clampf(f[1] * (float)R.sampler.resolution + (float)R.sampler.sb[1] - (float)y, 0.0f, PB_ONE_MINUS_EPSILON);
        u = make_float2(f[0], f[1]); tu = f[2]; plens = make_float2(f[3], f[4]);
        c.dim = 5;
    } else {
        c.index = halton_index(R.sampler, sample, x, y);
        u = get_2d(R.sampler, c);
        tu = get_1d(R.sampler, c);
        plens = get_2d(R.sampler, c);
    }
    float2 pfilm = make_float2((float)x + u.x, (float)y + u.y);
    f3 o, d;
    float time;
    generate_ray(R.camera, pfilm, tu, plens, &o, &d, &time);
    R.ray[2 * slot] = make_float4(o.x, o.y, o.z, PB_INF);
    R.ray[2 * slot + 1] = make_float4(d.x, d.y, d.z, time);
    R.L_eta[slot] = make_float4(0.f, 0.f, 0.f, 1.0f);
    R.beta_st[slot] = make_float4(1.f, 1.f, 1.f, __uint_as_float(R.rdiff ? PB_ST_HAS_DIFF : 0u));
    if (R.rdiff) camera_differentials(R.camera, pfilm, plens, o, d, R.sampler.spp, R.rdiff, slot);
    R.pfilm[slot] = pfilm;
    R.s_index[slot] = c.index;
    R.s_dim[slot] = c.dim;
    R.pixel[slot] = (uint32_t)(x - R.sampler.sb[0]) | ((uint32_t)(y - R.sampler.sb[1]) << 16);
    if (R.rec.kind) {  // start_next_sample resets the array offsets (sampler.rs:85-92)
        R.rec.sp[slot] = 0; R.rec.arr[slot] = 0;
        if (R.rec.multi) R.rec.sample_num[slot] = sample;
    }
    return true;
}

#if PB_EXACT_TU
// Start of a render call: every path slot is free and carries no sample.
__global__ void __launch_bounds__(256) k_init_slots(RenderDev R, uint32_t count) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        R.q_dead[1][i] = i;
        R.pixel[i] = PB_NO_SAMPLE;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) R.cnt->n_dead = count;
}
#endif  // PB_EXACT_TU


// ---------------------------------------------------------------------------
// K2: closest-hit for path rays (persistent ray queue), K4: compaction by material
// ---------------------------------------------------------------------------
// hit record + material bin of a path's closest-hit ray
PB_D int store_closest_hit(const RenderDev& R, uint32_t id, const TravRay& r) {
    R.hit[id] = make_uint4(r.hit.slot, __float_as_uint(r.hit.t), __float_as_uint(r.hit.b0), __float_as_uint(r.hit.b1));
    R.hit_b2[id] = r.hit.b2;
    if (R.scene.n_instances) R.hit_inst[id] = r.hit.inst;
    int bin = Q_MISS;
    if (r.found) {
        int m = R.scene.prims[r.hit.slot].material;
        if (m < 0) bin = Q_NOMAT;
        else { const pbrt_b200_material& mr = R.scene.materials[m]; bin = mr.textured ? Q_TEX : (int)mr.type; }
    }
    R.hit_bin[id] = (uint8_t)bin;
    return bin;
}
#if PB_EXACT_TU
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
#endif  // PB_EXACT_TU


// ---------------------------------------------------------------------------
// lights
// ---------------------------------------------------------------------------
PB_D uint32_t find_interval_cdf(const float* cdf, int size, float u) {  // pbrt.rs:184-204 with pred = cdf[i] <= u
    int first = 0, len_ = size;
    while (len_ > 0) {
        int half = len_ >> 1, middle = first + half;
        if (__ldg(cdf + middle) <= u) { first = middle + 1; len_ -= half + 1; } else len_ = half;
    }
    int r = first - 1;
    return (uint32_t)(r < 0 ? 0 : (r > size - 2 ? size - 2 : r));
}
PB_D float tiny_sample_continuous(const Tiny1D& d, float u, float* pdf, int* off) {  // sampling.rs:36-63
    int first = 0, len_ = 3;
    while (len_ > 0) {
        int half = len_ >> 1, middle = first + half;
        if (d.cdf[middle] <= u) { first = middle + 1; len_ -= half + 1; } else len_ = half;
    }
    int o = first - 1; o = o < 0 ? 0 : (o > 1 ? 1 : o);
    *off = o;
    float du = u - d.cdf[o];
    float diff = d.cdf[o + 1] - d.cdf[o];
    if (diff > 0.0f) du /= diff;
    *pdf = d.func_int > 0.0f ? d.func[o] / d.func_int : 0.0f;
    return ((float)o + du) / 2.0f;
}

struct LightSample { rgb Li; f3 wi; float pdf; f3 p1, p1_err, p1_n; };

// Triangle::sample + Shape::sample_interaction (shapes/triangle.rs:556-584, core/shape.rs:40-58)
PB_D void triangle_light_sample(const DevScene& s, const pbrt_b200_light& l, f3 ref_p, float2 u, LightSample& r) {
    float su0 = sqrtf(u.x);
    float b0 = 1.0f - su0, b1 = u.y * su0;  // uniform_sample_triangle, sampling.rs:244-248
    // the emitting triangle's vertices and normals, pre-gathered per light (DevScene::light_tris)
    const float4* lt = s.light_tris + 6ull * (size_t)(&l - s.lights);
    const float4 q0 = __ldg(lt), q1 = __ldg(lt + 1), q2 = __ldg(lt + 2);
    f3 p0(q0.x, q0.y, q0.z), p1(q1.x, q1.y, q1.z), p2(q2.x, q2.y, q2.z);
    float b2 = 1.0f - b0 - b1;
    f3 p = p0 * b0 + p1 * b1 + p2 * b2;
    f3 n = normalize(cross(p1 - p0, p2 - p0));
    if ((l.shape_flags & PBRT_B200_PRIM_HAS_N) && s.vertex_n) {
        const float4 n0 = __ldg(lt + 3), n1 = __ldg(lt + 4), n2 = __ldg(lt + 5);
        f3 ns = f3(n0.x, n0.y, n0.z) * b0 + f3(n1.x, n1.y, n1.z) * b1 + f3(n2.x, n2.y, n2.z) * b2;
        n = face_forward(n, ns);
    } else if (((l.shape_flags & PBRT_B200_PRIM_REVERSE_ORIENTATION) != 0) != ((l.shape_flags & PBRT_B200_PRIM_SWAPS_HANDEDNESS) != 0)) {
        n = n * -1.0f;
    }
    f3 pabs = vabs(p0 * b0) + vabs(p1 * b1) + vabs(p2 * b2);
    r.p1 = p; r.p1_n = n; r.p1_err = pabs * gamma_n(6);
    float pdf = 1.0f / l.area;
    f3 wi = p - ref_p;
    if (len2(wi) == 0.0f) pdf = 0.0f;
    else {
        wi = normalize(wi);
        f3 dd = ref_p - p;
        pdf *= len2(dd) / absdot(n, -wi);
        if (isinf(pdf)) pdf = 0.0f;
    }
    r.pdf = pdf;
}

// ---- Sphere as an area-light shape: Sphere::sample / sample_interaction / pdf_wi (shapes/sphere.rs:295-395, full spheres).
// Out of line and fed through the HBM copy of the scene (DevScene::self_dev): scenes without sphere lights pay one
// predicated call, and the shade kernels' register allocation does not move.
struct SphereLightSample { f3 p, p_err, n; float pdf; };
static __device__ __noinline__ void sphere_light_sample(const DevScene* sp, uint32_t li, f3 ref_p, f3 ref_perr, f3 ref_n, float ux, float uy, SphereLightSample* out) {
    const DevScene& s = *sp;
    const pbrt_b200_light& l = s.lights[li];
    const pbrt_b200_sphere& sph = s.spheres[l.shape_index];
    f3 pcenter = xf_point(sph.object_to_world, f3(0.f, 0.f, 0.f));
    f3 porigin = offset_ray_origin(ref_p, ref_perr, ref_n, pcenter - ref_p);
    f3 dco = porigin - pcenter;
    if (len2(dco) <= sph.radius * sph.radius) {  // inside: Sphere::sample (uniform over the surface), converted to solid angle
        float z = 1.0f - 2.0f * ux;
        float rr = sqrtf(fmaxf(1.0f - z * z, 0.0f));
        float phi = 2.0f * PB_PI * uy;
        f3 pobj = f3(rr * cosf(phi), rr * sinf(phi), z) * sph.radius;
        f3 n = normalize(xf_normal(sph.world_to_object, pobj));
        if (l.shape_flags & PBRT_B200_PRIM_REVERSE_ORIENTATION) n = n * -1.0f;
        pobj = pobj * (sph.radius / len(pobj));
        f3 pe = vabs(pobj) * gamma_n(5);
        out->p = xf_point_abs_err(sph.object_to_world, pobj, pe, &out->p_err);
        out->n = n;
        float pdf = 1.0f / l.area;
        f3 wi = out->p - ref_p;
        if (len2(wi) == 0.0f) pdf = 0.0f;
        else {
            wi = normalize(wi);
            f3 dd = ref_p - out->p;
            pdf *= len2(dd) / absdot(n, -wi);
        }
        if (isinf(pdf)) pdf = 0.0f;
        out->pdf = pdf;
        return;
    }
    // uniform inside the subtended cone (sphere.rs:335-378)
    f3 dcv = ref_p - pcenter;
    float dc = len(dcv);
    float invdc = 1.0f / dc;
    f3 wc = (pcenter - ref_p) * invdc, wcx, wcy;
    coordinate_system(wc, &wcx, &wcy);
    float stm = sph.radius * invdc;
    float stm2 = stm * stm;
    float istm = 1.0f / stm;
    float ctm = sqrtf(fmaxf(1.0f - stm2, 0.0f));
    float ct = (ctm - 1.0f) * ux + 1.0f;
    float st2 = 1.0f - ct * ct;
    if (stm2 < 0.00068523f) { st2 = stm2 * ux; ct = sqrtf(1.0f - st2); }
    float ca = st2 * istm + ct * sqrtf(fmaxf(1.0f - st2 * istm * istm, 0.0f));
    float sa = sqrtf(fmaxf(1.0f - ca * ca, 0.0f));
    float phi = uy * 2.0f * PB_PI;
    f3 nworld = (wcx * -1.0f) * sa * cosf(phi) + (wcy * -1.0f) * sa * sinf(phi) + (wc * -1.0f) * ca;  // spherical_direction_basis, geometry.rs:36-38
    f3 pworld = pcenter + nworld * sph.radius;
    out->p = pworld;
    out->p_err = vabs(pworld) * gamma_n(5);
    out->n = f3(0.f, 0.f, 0.f);  // sphere.rs:371-374 never sets it.n: only two-sided sphere lights emit through light sampling
    out->pdf = 1.0f / (2.0f * PB_PI * (1.0f - ctm));
}
static __device__ __noinline__ float sphere_light_pdf_wi(const DevScene* sp, uint32_t li, f3 ref_p, f3 ref_perr, f3 ref_n, f3 wi) {
    const DevScene& s = *sp;
    const pbrt_b200_light& l = s.lights[li];
    const pbrt_b200_sphere& sph = s.spheres[l.shape_index];
    f3 pcenter = xf_point(sph.object_to_world, f3(0.f, 0.f, 0.f));
    f3 porigin = offset_ray_origin(ref_p, ref_perr, ref_n, pcenter - ref_p);
    f3 dco = porigin - pcenter;
    if (len2(dco) <= sph.radius * sph.radius) {  // shape_pdfwi, core/shape.rs:117-136: re-intersect the shape, signed cosine
        f3 o = offset_ray_origin(ref_p, ref_perr, ref_n, wi);
        float t;
        if (!sphere_test(&sph, o, wi, PB_INF, &t)) return 0.0f;
        Surf ls = sphere_surface(&sph, o, wi, t);
        f3 dd = ref_p - ls.p;
        float pdf = len2(dd) / (dot(ls.n, -wi) * l.area);
        if (isinf(pdf)) pdf = 0.0f;
        return pdf;
    }
    f3 dcv = ref_p - pcenter;
    float stm2 = sph.radius * sph.radius / len2(dcv);
    float ctm = sqrtf(fmaxf(1.0f - stm2, 0.0f));
    return 1.0f / (2.0f * PB_PI * (1.0f - ctm));  // uniform_cone_pdf
}

// Light::sample_li for every light kind on the hot path.  ref_perr / ref_n: the reference point's error bounds and normal
// (only a sphere light's inside test looks at them, through offset_ray_origin).  SPH: sphere area lights are compiled in
// (the kernels of the full-featured family, selected when the scene has object instances or sphere lights; the lean family
// keeps the code -- and the register allocation -- it had without them).
template <bool SPH = false>
PB_D void light_sample_li(const RenderDev& R, uint32_t li, f3 ref_p, float2 u, LightSample& r, f3 ref_perr = f3(0.f, 0.f, 0.f), f3 ref_n = f3(0.f, 0.f, 0.f)) {
    const pbrt_b200_light& l = R.scene.lights[li];
    rgb L = rgb3(l.L);
    r.p1_err = f3(0.f, 0.f, 0.f); r.p1_n = f3(0.f, 0.f, 0.f);
    switch (l.type) {
        case PBRT_B200_LIGHT_POINT: {  // lights/point.rs:53-69
            f3 pl(l.pos[0], l.pos[1], l.pos[2]);
            r.wi = normalize(pl - ref_p); r.pdf = 1.0f; r.p1 = pl;
            r.Li = L / len2(pl - ref_p);
            break;
        }
        case PBRT_B200_LIGHT_SPOT: {  // lights/spot.rs:46-59,70-85
            f3 pl(l.pos[0], l.pos[1], l.pos[2]);
            r.wi = normalize(pl - ref_p); r.pdf = 1.0f; r.p1 = pl;
            f3 wl = normalize(xf_vector(l.world_to_light, -r.wi));
            float ct = wl.z, fall;
            if (ct < l.cos_total_width) fall = 0.0f;
            else if (ct >= l.cos_falloff_start) fall = 1.0f;
            else { float dl = (ct - l.cos_total_width) / (l.cos_falloff_start - l.cos_total_width); fall = (dl * dl) * (dl * dl); }
            r.Li = L * fall / len2(pl - ref_p);
            break;
        }
        case PBRT_B200_LIGHT_DISTANT: {  // lights/distant.rs:66-83
            f3 w(l.dir[0], l.dir[1], l.dir[2]);
            r.wi = w; r.pdf = 1.0f;
            r.p1 = ref_p + w * (2.0f * R.scene.world_radius);
            r.Li = L;
            break;
        }
        case PBRT_B200_LIGHT_DIFFUSE: {  // lights/diffuse.rs:91-106
            if (SPH && l.shape_kind == PBRT_B200_SHAPE_SPHERE) {
                SphereLightSample so;
                sphere_light_sample(R.scene.self_dev, li, ref_p, ref_perr, ref_n, u.x, u.y, &so);
                r.p1 = so.p; r.p1_err = so.p_err; r.p1_n = so.n; r.pdf = so.pdf;
            } else triangle_light_sample(R.scene, l, ref_p, u, r);
            f3 dlt = r.p1 - ref_p;
            if (r.pdf == 0.0f || len2(dlt) == 0.0f) { r.pdf = 0.0f; r.Li = rgb(0.0f); r.wi = f3(0.f, 0.f, 0.f); return; }
            r.wi = normalize(dlt);
            r.Li = (l.two_sided || dot(r.p1_n, -r.wi) > 0.0f) ? L : rgb(0.0f);  // AreaLight::l, diffuse.rs:68-75
            break;
        }
        default: {  // PBRT_B200_LIGHT_INFINITE, lights/infinite.rs:141-170 with a constant map
            const InfDistrib& D = R.inf_distrib[li];
            float pm, pc;
            int v, dummy;
            float d1 = tiny_sample_continuous(D.marg, u.y, &pm, &v);
            float d0 = tiny_sample_continuous(D.cond[v], u.x, &pc, &dummy);
            float map_pdf = pc * pm;
            if (map_pdf == 0.0f) { r.Li = rgb(0.0f); r.pdf = 0.0f; r.wi = f3(0.f, 0.f, 0.f); return; }
            float theta = d1 * PB_PI, phi = d0 * 2.0f * PB_PI;
            float ct = cosf(theta), st = sinf(theta), sp = sinf(phi), cp = cosf(phi);
            r.wi = f3(st * cp, st * sp, ct);
            r.pdf = map_pdf / (2.0f * PB_PI * PB_PI * st);
            if (st == 0.0f) r.pdf = 0.0f;
            r.p1 = ref_p + r.wi * (2.0f * R.scene.world_radius);
            r.Li = L;
            break;
        }
    }
}

// Shape::pdf_wi for a triangle light (core/shape.rs:63-82): re-intersects that one shape
// (Triangle::intersect with s = None) and converts to solid angle with the SIGNED cosine.
PB_D float triangle_light_pdf_wi(const DevScene& s, const pbrt_b200_light& l, const Surf& ref, f3 wi) {
    f3 o = offset_ray_origin(ref.p, ref.p_error, ref.n, wi);
    const float4* lt = s.light_tris + 6ull * (size_t)(&l - s.lights);
    const float4 q0 = __ldg(lt), q1 = __ldg(lt + 1), q2 = __ldg(lt + 2);
    f3 p0(q0.x, q0.y, q0.z), p1(q1.x, q1.y, q1.z), p2(q2.x, q2.y, q2.z);
    f3 ad = vabs(wi);
    int kz = (ad.x > ad.y) ? ((ad.x > ad.z) ? 0 : 2) : ((ad.y > ad.z) ? 1 : 2);
    int kx = (kz + 1 == 3) ? 0 : kz + 1, ky = (kx + 1 == 3) ? 0 : kx + 1;
    float dz = comp(wi, kz);
    float Sx = -comp(wi, kx) / dz, Sy = -comp(wi, ky) / dz, Sz = 1.0f / dz;
    float t, b0, b1, b2;
    if (!triangle_test<true>(o, wi, PB_INF, p0, p1, p2, kx, ky, kz, Sx, Sy, Sz, &t, &b0, &b1, &b2)) return 0.0f;
    float2 uv0, uv1, uv2;
    fetch_uv(s, l.shape_flags, l.shape_index, &uv0, &uv1, &uv2);
    if (triangle_bogus(p0, p1, p2, uv0, uv1, uv2)) return 0.0f;
    Surf ls = triangle_surface(s, p0, p1, p2, l.shape_flags, l.shape_index, wi, b0, b1, b2, false, PB_NO_SLOT, lt + 3);
    f3 dd = ref.p - ls.p;
    float pdf = len2(dd) / (dot(ls.n, -wi) * l.area);
    if (isinf(pdf)) pdf = 0.0f;
    return pdf;
}
template <bool SPH = false>
PB_D float light_pdf_li(const RenderDev& R, uint32_t li, const Surf& ref, f3 wi) {
    const pbrt_b200_light& l = R.scene.lights[li];
    if (l.type == PBRT_B200_LIGHT_DIFFUSE)
        return (SPH && l.shape_kind == PBRT_B200_SHAPE_SPHERE) ? sphere_light_pdf_wi(R.scene.self_dev, li, ref.p, ref.p_error, ref.n, wi) : triangle_light_pdf_wi(R.scene, l, ref, wi);
    if (l.type == PBRT_B200_LIGHT_INFINITE) {  // lights/infinite.rs:131-139, Distribution2D::pdf sampling.rs:131-143
        float theta = acosf(clampf(wi.z, -1.0f, 1.0f));
        float phi = atan2f(wi.y, wi.x);
        if (phi < 0.0f) phi += 2.0f * PB_PI;
        float st = sinf(theta);
        if (st == 0.0f) return 0.0f;
        const InfDistrib& D = R.inf_distrib[li];
        float pu = phi * 0.15915494309189533577f * 2.0f, pv = theta * PB_INV_PI * 2.0f;
        int iu = (pu != pu || pu <= 0.0f) ? 0 : (int)fminf(pu, 1.0e9f), iv = (pv != pv || pv <= 0.0f) ? 0 : (int)fminf(pv, 1.0e9f);
        iu = min(max(iu, 0), 1); iv = min(max(iv, 0), 1);
        return (D.cond[iv].func[iu] / D.marg.func_int) / (2.0f * PB_PI * PB_PI * st);
    }
    return 0.0f;
}
PB_D bool is_delta_light(const pbrt_b200_light& l) { return l.type == PBRT_B200_LIGHT_POINT || l.type == PBRT_B200_LIGHT_DISTANT || l.type == PBRT_B200_LIGHT_SPOT; }

// ---------------------------------------------------------------------------
// SpatialLightDistribution
// ---------------------------------------------------------------------------
// lookup(): point -> integer voxel, lightdistrib.rs:236-246 (Bounds3::offset bounds.rs:372-390, `as isize` saturates)
PB_D int spatial_voxel(const RenderDev& R, f3 p) {
    const float* wb = R.scene.root_box;
    float o[3] = {p.x - wb[0], p.y - wb[1], p.z - wb[2]};
#pragma unroll
    for (int k = 0; k < 3; ++k)
        if (wb[3 + k] > wb[k]) o[k] /= wb[3 + k] - wb[k];
    int pi[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float v = o[k] * (float)R.sp.nvox[k];
        long long q = (v != v) ? 0ll : __float2ll_rz(v);
        long long hi = (long long)R.sp.nvox[k] - 1;
        pi[k] = (int)(q < 0 ? 0 : (q > hi ? hi : q));
    }
    return (pi[2] * R.sp.nvox[1] + pi[1]) * R.sp.nvox[0] + pi[0];
}

#if PB_EXACT_TU
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
#endif  // PB_EXACT_TU


// ---------------------------------------------------------------------------
// sampler pre-pass and Sobol' table builders
// ---------------------------------------------------------------------------
#if PB_EXACT_TU
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
#endif  // PB_EXACT_TU


// ---------------------------------------------------------------------------
// K5/K6: shade
// ---------------------------------------------------------------------------
PB_D void store_ray(float4* rays, uint32_t id, f3 o, f3 d, float t_max, float time) {
    rays[2 * id] = make_float4(o.x, o.y, o.z, t_max);
    rays[2 * id + 1] = make_float4(d.x, d.y, d.z, time);
}

template <int BIN> struct BinKinds { static constexpr int KM = KM_ALL, MAT = -1, NL = 2; };
template <> struct BinKinds<Q_MATTE> { static constexpr int KM = KM_MATTE, MAT = PBRT_B200_MAT_MATTE, NL = 2; };
template <> struct BinKinds<Q_PLASTIC> { static constexpr int KM = KM_PLASTIC, MAT = PBRT_B200_MAT_PLASTIC, NL = 2; };
template <> struct BinKinds<Q_MIRROR> { static constexpr int KM = KM_MIRROR, MAT = PBRT_B200_MAT_MIRROR, NL = 2; };
template <> struct BinKinds<Q_GLASS> { static constexpr int KM = KM_GLASS, MAT = PBRT_B200_MAT_GLASS, NL = 2; };
template <> struct BinKinds<Q_METAL> { static constexpr int KM = KM_METAL, MAT = PBRT_B200_MAT_METAL, NL = 2; };
template <> struct BinKinds<Q_TEX> { static constexpr int KM = KM_TEX, MAT = -1, NL = 5; };

// One path of a material queue: PathIntegrator::li from the hit to the next ray (path.rs:104-214).  Shared by the wavefront
// kernel k_shade and the tile-serial megakernel k_zt_mega.
struct ShadeOut { bool push_next, push_shadow, push_mis, push_dead, zero_rad; };
// VOL: VolPathIntegrator::li's surface branch (volpath.rs:134-189) -- the same vertex, except that the light is sampled whatever the
// BSDF's lobes are (no num_components test), rays carry a medium (`vs`), and a material-less surface LOWERS the bounce count
// (`bounces -= 1; continue` skips the loop's increment; at 0 the usize wraps and the path ends at its next depth test).
template <int BIN, bool INST, bool ZT, bool VOL = false>
PB_D ShadeOut shade_path(const RenderDev& R, uint32_t id, VolState* vs = nullptr) {
    constexpr int KM = BinKinds<BIN>::KM;
    (void)KM;
    bool push_next = false, push_shadow = false, push_mis = false, push_dead = false, zero_rad = false;
    {
    float4 ra = R.ray[2 * id], rb = R.ray[2 * id + 1];
    f3 ro(ra.x, ra.y, ra.z), rd(rb.x, rb.y, rb.z);
    float time = rb.w;
    float4 Le = R.L_eta[id], bs = R.beta_st[id];
    rgb L(Le.x, Le.y, Le.z), beta(bs.x, bs.y, bs.z);
    float etascale = Le.w;
    uint32_t st = __float_as_uint(bs.w);
    uint32_t bounces = st & 0xffffu;
    bool specular_bounce = (st >> 16) & 1u;
    if (BIN == Q_MISS) {
        // path.rs:106-120: escaped ray
        if (bounces == 0 || specular_bounce)
            for (uint32_t k = 0; k < R.n_infinite; ++k) L = L + rgb3(R.scene.lights[R.infinite_lights[k]].L) * beta;
        R.L_eta[id] = make_float4(L.r, L.g, L.b, etascale);
        push_dead = true;
    } else {
        uint4 h = R.hit[id];
        typename SamplerSel<ZT, VOL>::type smp;
        smp.prefetch(R, id);
        uint32_t fl;
        const uint32_t hinst = (INST && R.scene.n_instances) ? R.hit_inst[id] : PBRT_B200_NO_HIT;
        Surf si;
        SurfX sx;
        if (BIN == Q_TEX) surface_full(R.scene.self_dev, hinst, h.x, ro, rd, __uint_as_float(h.y), __uint_as_float(h.z), __uint_as_float(h.w), R.hit_b2[id], &si, &sx, &fl);
        else si = surface_at_hit<INST>(R.scene, hinst, h.x, ro, rd, __uint_as_float(h.y), __uint_as_float(h.z), __uint_as_float(h.w), R.hit_b2[id], &fl);
        const pbrt_b200_prim pr = R.scene.prims[h.x];
        // SurfaceInteraction::le, interaction.rs:344-349 + AreaLight::l, diffuse.rs:68-75
        if ((bounces == 0 || specular_bounce) && pr.area_light >= 0) {
            const pbrt_b200_light& al = R.scene.lights[pr.area_light];
            if (al.two_sided || dot(si.n, -rd) > 0.0f) L = L + rgb3(al.L) * beta;
        }
        VolInterface vmi{-1, -1};
        if (VOL) vmi = vol_hit_interface(R.scene, h.x, vs->medium);
        if (bounces >= (uint32_t)R.max_depth) {
            R.L_eta[id] = make_float4(L.r, L.g, L.b, etascale);
            push_dead = true;
        } else {
            BsdfN<BinKinds<BIN>::NL> bsdf;
            bsdf.valid = false;
            if (BIN == Q_TEX) {
                const RayDiff rdf = load_diff(R.rdiff, id, R.rdiff != nullptr && (st & PB_ST_HAS_DIFF) != 0u);
                material_bsdf_tex<true>(R.scene.self_dev, pr.material, &si, &sx, &rdf, &bsdf);
            } else if (BIN != Q_NOMAT && BIN != Q_MISS) material_bsdf<BinKinds<BIN>::MAT>(R.scene.materials[pr.material], si, bsdf);
            if (!bsdf.valid) {
                // path.rs:124-129: skip the surface, bounces NOT incremented
                f3 o = offset_ray_origin(si.p, si.p_error, si.n, rd);
                store_ray(R.ray, id, o, rd, PB_INF, time);
                R.L_eta[id] = make_float4(L.r, L.g, L.b, etascale);
                if (!VOL && R.rdiff && (st & PB_ST_HAS_DIFF))  // the spawned ray has no differentials (interaction.rs:32-37)
                    R.beta_st[id] = make_float4(beta.r, beta.g, beta.b, __uint_as_float(st & ~PB_ST_HAS_DIFF));
                if (VOL) {  // volpath.rs:131-135
                    vs->medium = vol_medium_for(vmi, si.n, rd);
                    bounces = (bounces - 1u) & 0xffffu;
                    R.beta_st[id] = make_float4(beta.r, beta.g, beta.b, __uint_as_float(bounces | (specular_bounce ? 0x10000u : 0u)));
                }
                push_next = true;
            } else {
                smp.begin(R, id);
                const int NONSPEC = BX_ALL & ~BX_SPECULAR;
                // ---- uniform_sample_onelight + estimate_direct, integrator.rs:81-237
                if ((VOL || bsdf_count(bsdf, NONSPEC) > 0) && R.n_lights > 0) {
                    float u1 = smp.get_1d();
                    // light_distrib.lookup(isect.p), path.rs:132
                    const float* ld_cdf = R.ld_cdf; const float* ld_func = R.ld_func; float ld_func_int = R.ld_func_int;
                    if (R.sp.enabled) {
                        int sl = R.sp.slot[(R.sp.lazy && !ZT && !VOL) ? R.sp_voxel[id] : spatial_voxel(R, si.p)];  // (the megakernels have no mark pass)
                        if (sl >= 0) { ld_cdf = R.sp.cdf + (size_t)sl * (R.n_lights + 1); ld_func = R.sp.func + (size_t)sl * R.n_lights; ld_func_int = R.sp.func_int[sl]; }
                        else atomicExch(R.sp.counters + 2, 1u);  // cannot happen unless the slot table overflowed: the host fails the call
                    }
                    uint32_t ln = find_interval_cdf(ld_cdf, (int)R.n_lights + 1, u1);  // Distribution1D::sample_discrete
                    float selpdf = ld_func_int > 0.0f ? ld_func[ln] / (ld_func_int * (float)R.n_lights) : 0.0f;
                    bool zero = true;
                    if (selpdf != 0.0f) {
                        float2 ulight = smp.get_2d();
                        float2 uscatt = smp.get_2d();
                        const pbrt_b200_light& light = R.scene.lights[ln];
                        bool delta = is_delta_light(light);
                        LightSample ls;
                        light_sample_li<INST>(R, ln, si.p, ulight, ls, si.p_error, si.n);
                        float scattpdf = 0.0f;
                        if (ls.pdf > 0.0f && !is_black(ls.Li)) {
                            rgb f = bsdf_f<KM>(bsdf, si.wo, ls.wi, NONSPEC) * absdot(ls.wi, si.sh_n);
                            scattpdf = bsdf_pdf<KM>(bsdf, si.wo, ls.wi, NONSPEC);
                            if (!is_black(f)) {
                                // VisibilityTester::unoccluded -> spawn_rayto_interaction, interaction.rs:46-52
                                f3 o = offset_ray_origin(si.p, si.p_error, si.n, ls.p1 - si.p);
                                f3 tg = offset_ray_origin(ls.p1, ls.p1_err, ls.p1_n, o - ls.p1);
                                f3 d = tg - o;
                                rgb Ld = delta ? f * ls.Li / ls.pdf : f * ls.Li * power_heuristic(ls.pdf, scattpdf) / ls.pdf;
                                rgb add = beta * (Ld / selpdf);
                                store_ray(R.sh_ray, id, o, d, 1.0f - PB_SHADOW_EPSILON, time);
                                R.sh_contrib[id] = make_float4(add.r, add.g, add.b, 0.f);
                                if (VOL) { vs->sh_medium = vol_medium_for(vmi, si.n, d); vs->p1 = ls.p1; vs->p1_err = ls.p1_err; vs->p1_n = ls.p1_n; }
                                push_shadow = true;
                                zero = false;
                            }
                        }
                        if (!delta) {
                            f3 wi(0.f, 0.f, 0.f);
                            int stype = 0;
                            rgb f = bsdf_sample<KM>(bsdf, si.wo, &wi, uscatt, &scattpdf, NONSPEC, &stype);
                            f = f * absdot(wi, si.sh_n);
                            if (!is_black(f) && scattpdf > 0.0f) {
                                float weight = 1.0f;
                                bool go = true;
                                if (!(stype & BX_SPECULAR)) {
                                    float lpdf = light_pdf_li<INST>(R, ln, si, wi);
                                    if (lpdf == 0.0f) go = false;
                                    else weight = power_heuristic(scattpdf, lpdf);
                                }
                                if (go) {
                                    f3 o = offset_ray_origin(si.p, si.p_error, si.n, wi);
                                    rgb fac = beta * (f * weight / scattpdf / selpdf);
                                    store_ray(R.mis_ray, id, o, wi, PB_INF, time);
                                    R.mis_contrib[id] = make_float4(fac.r, fac.g, fac.b, __uint_as_float(ln));
                                    if (VOL) vs->mis_medium = vol_medium_for(vmi, si.n, wi);
                                    push_mis = true;
                                    zero = false;
                                }
                            }
                        }
                    }
                    zero_rad = zero;
                }
                // ---- sample the BSDF for the next direction, path.rs:147-174
                f3 wo = -rd, wi(0.f, 0.f, 0.f);
                float pdf = 0.0f;
                int flags = 0;
                float2 ub = smp.get_2d();
                rgb f = bsdf_sample<KM>(bsdf, wo, &wi, ub, &pdf, BX_ALL, &flags);
                bool alive = !(is_black(f) || pdf == 0.0f);
                if (alive) {
                    beta = beta * (f * absdot(wi, si.sh_n) / pdf);
                    specular_bounce = (flags & BX_SPECULAR) != 0;
                    if ((flags & BX_SPECULAR) && (flags & BX_TRANSMISSION)) {
                        float eta = bsdf.eta;
                        etascale *= (dot(wo, si.n) > 0.0f) ? eta * eta : 1.0f / (eta * eta);
                    }
                    f3 o = offset_ray_origin(si.p, si.p_error, si.n, wi);
                    // Russian roulette, path.rs:206-214
                    rgb rrbeta = beta * etascale;
                    float mc = max_comp(rrbeta);
                    if (mc < R.rr_threshold && bounces > 3) {
                        float qv = fmaxf(1.0f - mc, 0.05f);
                        if (smp.get_1d() < qv) alive = false;
                        else beta = beta / (1.0f - qv);
                    }
                    if (alive) {
                        store_ray(R.ray, id, o, wi, PB_INF, time);
                        if (VOL) vs->medium = vol_medium_for(vmi, si.n, wi);
                        bounces += 1;
                        R.beta_st[id] = make_float4(beta.r, beta.g, beta.b, __uint_as_float(bounces | (specular_bounce ? 0x10000u : 0u)));
                        push_next = true;
                    }
                }
                if (!alive) push_dead = true;
                R.L_eta[id] = make_float4(L.r, L.g, L.b, etascale);
                smp.end(R, id);
            }
        }
    }
    }
    return ShadeOut{push_next, push_shadow, push_mis, push_dead, zero_rad};
}

#if PB_SHADE_TU
template <int BIN, bool INST, bool ZT>
__global__ void __launch_bounds__(BIN == Q_TEX ? PB_TEX_BLOCK : 128) k_shade(RenderDev R, int parity) {
    const uint32_t n = R.cnt->n_mat[BIN];
    const uint32_t* q = R.q_mat[BIN];
    uint32_t* q_next = R.q_path[parity ^ 1];
    // Q_TEX reads its queue ordered by material (k_tex_count / k_tex_scan / k_tex_scatter below wrote it to the path queue that k_classify has consumed)
    if (BIN == Q_TEX) q = R.q_path[parity];
    // Q_TEX: 22 k instructions of texture interpreter, noise and EWA code -- ncu had 28 of 34 stall cycles per issued instruction on `no_instruction`
    // (instruction-cache misses) at 11 % issue-slot use.  Its CTA is the whole SM (PB_TEX_BLOCK threads at 128 registers) and its warps start every
    // path TOGETHER (barrier at the top of a trip; the queue is sorted by material, so they run the same programs): they fetch the same lines at
    // about the same time.  The trip count is CTA-uniform for the barrier.
    const bool lockstep = BIN == Q_TEX;
    const uint32_t nround = lockstep ? ((n + blockDim.x - 1u) / blockDim.x) * blockDim.x : ((n + 31u) & ~31u);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nround; i += gridDim.x * blockDim.x) {
        if (lockstep) __syncthreads();
        ShadeOut o = {false, false, false, false, false};
        uint32_t id = 0;
        const bool valid = i < n;
        if (valid) id = q[i];
        if (valid) o = shade_path<BIN, INST, ZT>(R, id);
        {
            unsigned zm = __ballot_sync(0xffffffffu, o.zero_rad);
            if (zm && (threadIdx.x & 31) == 0) atomicAdd(&R.cnt->zero_radiance, (unsigned long long)__popc(zm));
        }
        // the four appends of an iteration: lane 0 issues all the counter atomics back to back, THEN the bases are broadcast --
        // one atomic round trip per iteration instead of four dependent ones (17 % of the matte kernel's stall samples sat on
        // the first broadcast, profiles/r02_ncu_shade.md).  All 32 lanes are here: the loop runs over n rounded up to a warp.
        {
            const unsigned m0 = __ballot_sync(0xffffffffu, o.push_next), m1 = __ballot_sync(0xffffffffu, o.push_shadow);
            const unsigned m2 = __ballot_sync(0xffffffffu, o.push_mis), m3 = __ballot_sync(0xffffffffu, o.push_dead);
            const unsigned lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
            uint32_t b0 = 0, b1 = 0, b2 = 0, b3 = 0;
            if (lane == 0) {
                if (m0) b0 = atomicAdd(&R.cnt->n_next, (uint32_t)__popc(m0));
                if (m1) b1 = atomicAdd(&R.cnt->n_shadow, (uint32_t)__popc(m1));
                if (m2) b2 = atomicAdd(&R.cnt->n_mis, (uint32_t)__popc(m2));
                if (m3) b3 = atomicAdd(&R.cnt->n_dead, (uint32_t)__popc(m3));
            }
            b0 = __shfl_sync(0xffffffffu, b0, 0); b1 = __shfl_sync(0xffffffffu, b1, 0);
            b2 = __shfl_sync(0xffffffffu, b2, 0); b3 = __shfl_sync(0xffffffffu, b3, 0);
            if (o.push_next) q_next[b0 + __popc(m0 & below)] = id;
            if (o.push_shadow) R.q_shadow[b1 + __popc(m1 & below)] = id;
            if (o.push_mis) R.q_mis[b2 + __popc(m2 & below)] = id;
            if (o.push_dead) R.q_dead[parity][b3 + __popc(m3 & below)] = id;
        }
    }
}

// The textured bin holds every textured material of the scene and each one runs its own texture programs: a warp whose lanes carry different
// materials executes them one after the other (ncu, T1 scene: 8 of 32 lanes active per instruction after the first bounce; 13 with the CTA-local
// sort this pass replaces, whose barriers held 30 % of the stall samples -- profiles/r02_textures.md).  A counting sort of the WHOLE queue by
// material makes every warp uniform but the ones that straddle two materials: count, exclusive scan (which also re-zeroes the counts), scatter.
// Groups of equal material inside a warp (match.any) issue one atomic each.
PB_D uint32_t tex_sort_key(const RenderDev& R, uint32_t id) { return (uint32_t)R.scene.prims[R.hit[id].x].material; }
__global__ void __launch_bounds__(256) k_tex_count(RenderDev R) {
    const uint32_t n = R.cnt->n_mat[Q_TEX], nround = (n + 31u) & ~31u;
    const uint32_t* q = R.q_mat[Q_TEX];
    const unsigned lane = threadIdx.x & 31u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nround; i += gridDim.x * blockDim.x) {
        const uint32_t key = i < n ? tex_sort_key(R, q[i]) : 0xffffffffu;
        const unsigned peers = __match_any_sync(0xffffffffu, key);
        if (i < n && lane == (unsigned)__ffs(peers) - 1u) atomicAdd(&R.tex_sort[key], (uint32_t)__popc(peers));
    }
}
__global__ void __launch_bounds__(32) k_tex_scan(RenderDev R) {
    const uint32_t nm = R.scene.n_materials;
    uint32_t* count = R.tex_sort;
    uint32_t* cursor = R.tex_sort + nm;
    const unsigned lane = threadIdx.x;
    uint32_t carry = 0;
    for (uint32_t base = 0; base < nm; base += 32u) {
        const uint32_t m = base + lane;
        const uint32_t c = m < nm ? count[m] : 0u;
        uint32_t inc = c;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= (unsigned)o) inc += t; }
        if (m < nm) { cursor[m] = carry + inc - c; count[m] = 0u; }
        carry += __shfl_sync(0xffffffffu, inc, 31);
    }
}
__global__ void __launch_bounds__(256) k_tex_scatter(RenderDev R, int parity) {
    const uint32_t n = R.cnt->n_mat[Q_TEX], nround = (n + 31u) & ~31u, nm = R.scene.n_materials;
    const uint32_t* q = R.q_mat[Q_TEX];
    uint32_t* out = R.q_path[parity];  // consumed by k_classify: free until the next iteration's k_finish_regen
    const unsigned lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nround; i += gridDim.x * blockDim.x) {
        const uint32_t id = i < n ? q[i] : 0u;
        const uint32_t key = i < n ? tex_sort_key(R, id) : 0xffffffffu;
        const unsigned peers = __match_any_sync(0xffffffffu, key);
        const unsigned leader = (unsigned)__ffs(peers) - 1u;
        uint32_t base = 0;
        if (i < n && lane == leader) base = atomicAdd(&R.tex_sort[nm + key], (uint32_t)__popc(peers));
        base = __shfl_sync(0xffffffffu, base, (int)leader);
        if (i < n) out[base + (uint32_t)__popc(peers & below)] = id;
    }
}
#endif  // PB_SHADE_TU

#if PB_EXACT_TU || PB_MEGA_TU
// ---------------------------------------------------------------------------
// K3: shadow rays (VisibilityTester::unoccluded, core/light.rs:120-123)
// ---------------------------------------------------------------------------
PB_D void shadow_unoccluded(const RenderDev& R, uint32_t id) {  // the light sample's contribution reaches the path
    float4 c = R.sh_contrib[id];
    float4 L = R.L_eta[id];
    L.x += c.x; L.y += c.y; L.z += c.z;
    R.L_eta[id] = L;
}
#if PB_EXACT_TU
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
#endif  // PB_EXACT_TU

// ---------------------------------------------------------------------------
// K7: MIS rays (estimate_direct's BSDF-sampled branch, integrator.rs:205-234)
// ---------------------------------------------------------------------------
// estimate_direct's BSDF-sampled ray came back (integrator.rs:205-234): emission of the sampled light if the ray found it
template <bool INST>
PB_D void mis_resolve(const RenderDev& R, uint32_t id, const TravRay& r) {
    float4 c = R.mis_contrib[id];
    uint32_t ln = __float_as_uint(c.w);
    rgb li(0.0f);
    if (r.found) {
        const pbrt_b200_prim pr = R.scene.prims[r.hit.slot];
        if (pr.area_light == (int)ln) {  // Arc::ptr_eq(light, hit primitive's area light)
            uint32_t fl;
            Surf ls = surface_at_hit<INST>(R.scene, r.hit.inst, r.hit.slot, r.o, r.d, r.hit.t, r.hit.b0, r.hit.b1, r.hit.b2, &fl);
            const pbrt_b200_light& al = R.scene.lights[ln];
            if (al.two_sided || dot(ls.n, -r.d) > 0.0f) li = rgb3(al.L);
        }
    } else {
        const pbrt_b200_light& l = R.scene.lights[ln];
        if (l.type == PBRT_B200_LIGHT_INFINITE) li = rgb3(l.L);  // light.le(ray)
    }
    if (!is_black(li)) {
        float4 L = R.L_eta[id];
        L.x += c.x * li.r; L.y += c.y * li.g; L.z += c.z * li.b;
        R.L_eta[id] = L;
    }
}
#if PB_EXACT_TU
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
#endif  // PB_EXACT_TU

#endif  // PB_EXACT_TU || PB_MEGA_TU
}  // namespace pb
#include "recursive.cuh"
namespace pb {

// Launchers of the kernels that live in the other translation unit (shade.o, see the top of this file)
void launch_shade_kernels(const RenderDev& R, int parity, bool full, int grid_small, int grid_shade, cudaStream_t stream);
void launch_rec_shade(const RenderDev& R, int parity, bool zt, bool full, cudaStream_t stream);
// ... and in mega.o
void launch_zt_mega(const RenderDev& R, const RenderDev* rdev, uint32_t lanes, uint32_t nblk, cudaStream_t stream);
void launch_vol_mega(const RenderDev& R, const RenderDev* rdev, unsigned long long total_items, int camera_medium, bool full, int grid, cudaStream_t stream);
int vol_mega_blocks_per_sm(bool full);
#if PB_SHADE_TU
// one launch per material queue (sort/compact-by-material); INST selects the kernel family (trace.cuh, sphere lights)
template <bool INST>
static void launch_shade_family(const RenderDev& R, int parity, int grid_small, int grid_shade, cudaStream_t stream) {
    k_shade<Q_MISS, INST, false><<<grid_small, 128, 0, stream>>>(R, parity);
    k_shade<Q_MATTE, INST, false><<<grid_shade, 128, 0, stream>>>(R, parity);
    k_shade<Q_PLASTIC, INST, false><<<grid_shade, 128, 0, stream>>>(R, parity);
    k_shade<Q_MIRROR, INST, false><<<grid_shade, 128, 0, stream>>>(R, parity);
    k_shade<Q_GLASS, INST, false><<<grid_shade, 128, 0, stream>>>(R, parity);
    k_shade<Q_METAL, INST, false><<<grid_shade, 128, 0, stream>>>(R, parity);
    k_shade<Q_NOMAT, INST, false><<<grid_small, 128, 0, stream>>>(R, parity);
    if (INST && R.scene.material_ext) {  // textured scenes run the full-featured family
        k_tex_count<<<grid_small, 256, 0, stream>>>(R);
        k_tex_scan<<<1, 32, 0, stream>>>(R);
        k_tex_scatter<<<grid_small, 256, 0, stream>>>(R, parity);
        static int tex_grid = 0;  // one CTA per SM
        if (!tex_grid) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&tex_grid, cudaDevAttrMultiProcessorCount, dev); tex_grid = std::max(tex_grid, 1); }
        k_shade<Q_TEX, true, false><<<tex_grid, PB_TEX_BLOCK, 0, stream>>>(R, parity);
    }
}
void launch_shade_kernels(const RenderDev& R, int parity, bool full, int grid_small, int grid_shade, cudaStream_t stream) {
    if (full) launch_shade_family<true>(R, parity, grid_small, grid_shade, stream);
    else launch_shade_family<false>(R, parity, grid_small, grid_shade, stream);
}
void launch_rec_shade(const RenderDev& R, int parity, bool zt, bool full, cudaStream_t stream) {
    static int g = 0;  // one CTA per SM
    if (!g) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&g, cudaDevAttrMultiProcessorCount, dev); g = std::max(g, 1); }
    if (R.scene.material_ext) {
        if (zt) k_rec_shade<true, true, true><<<g, PB_REC_BLOCK, 0, stream>>>(R, parity);
        else k_rec_shade<true, false, true><<<g, PB_REC_BLOCK, 0, stream>>>(R, parity);
    } else {
        if (zt) k_rec_shade<true, true, false><<<g, PB_REC_BLOCK, 0, stream>>>(R, parity);
        else if (full) k_rec_shade<true, false, false><<<g, PB_REC_BLOCK, 0, stream>>>(R, parity);
        else k_rec_shade<false, false, false><<<g, PB_REC_BLOCK, 0, stream>>>(R, parity);
    }
}
}  // namespace pb (shade.o ends here)
#endif  // PB_SHADE_TU
#if PB_EXACT_TU || PB_MEGA_TU
#if PB_EXACT_TU

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

#endif  // PB_EXACT_TU
// ---- (0,2)-sequence: tile-serial sample generation (the pixel / sample loops of integrator.rs:320-380 per tile)
// Advances tile `j` (slot == tile ordinal) to its next camera sample and writes the path into the slot.  `first`: the tile
// has not started (start_pixel of its first pixel is due).  Returns false when the tile is finished.
PB_D bool zt_next_path(const RenderDev& R, uint32_t j, bool first) {
    ZtTile* tp = R.zt.tiles + j;
    float* s1d = R.zt.s1d + (size_t)j * R.zt.ndims * R.zt.spp;
    float2* s2d = R.zt.s2d + (size_t)j * R.zt.n2d * R.zt.spp;
    const uint32_t s_begin = R.sample_begin, s_end = R.sample_begin + R.n_samples_sel;
    bool have = false;
    if (!first) {  // start_next_sample(), sampler.rs:206-216
        tp->cur1d = 0; tp->cur2d = 0;
        tp->sample_idx += 1;
        have = tp->sample_idx < R.zt.spp && tp->sample_idx < s_end;
        if (!have) tp->pixel_idx += 1;
    }
    while (!have) {
        if (tp->pixel_idx >= tp->npix) return false;
        zt_start_pixel(tp, s1d, s2d, R.zt.spp, R.zt.ndims, R.zt.n2d);  // every pixel of the tile, inside the pixel bounds or not (integrator.rs:322-330)
        int x = tp->x0 + (int)(tp->pixel_idx % tp->w), y = tp->y0 + (int)(tp->pixel_idx / tp->w);
        bool inside = x >= R.pixel_bounds[0] && x < R.pixel_bounds[2] && y >= R.pixel_bounds[1] && y < R.pixel_bounds[3];
        if (inside && s_begin < R.zt.spp && s_begin < s_end) { tp->sample_idx = s_begin; have = true; }  // set_sample_number
        else tp->pixel_idx += 1;
    }
    const int x = tp->x0 + (int)(tp->pixel_idx % tp->w), y = tp->y0 + (int)(tp->pixel_idx / tp->w);
    ZtCursor c = zt_cursor(R, j);
    // get_camera_sample, sampler.rs:170-180
    float2 u = get_2d(c);
    float2 pfilm = make_float2((float)x + u.x, (float)y + u.y);
    float tu = get_1d(c);
    float2 plens = get_2d(c);
    f3 o, d;
    float time;
    generate_ray(R.camera, pfilm, tu, plens, &o, &d, &time);
    R.ray[2 * j] = make_float4(o.x, o.y, o.z, PB_INF);
    R.ray[2 * j + 1] = make_float4(d.x, d.y, d.z, time);
    R.L_eta[j] = make_float4(0.f, 0.f, 0.f, 1.0f);
    R.beta_st[j] = make_float4(1.f, 1.f, 1.f, __uint_as_float(R.rdiff ? PB_ST_HAS_DIFF : 0u));
    if (R.rdiff) camera_differentials(R.camera, pfilm, plens, o, d, R.zt.spp, R.rdiff, j);
    R.pfilm[j] = pfilm;
    R.pixel[j] = (uint32_t)(x - R.sampler.sb[0]) | ((uint32_t)(y - R.sampler.sb[1]) << 16);
    if (R.rec.kind) { R.rec.sp[j] = 0; R.rec.arr[j] = 0; }
    return true;
}
#if PB_EXACT_TU
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

#endif  // PB_EXACT_TU
#if PB_MEGA_TU
// The (0,2)-sequence sampler under the PathIntegrator, one kernel: a tile's paths are inherently serial (every draw of
// every path advances the tile's PCG32), so the wavefront form spends its time launching 13 kernels per path segment for a
// few hundred threads.  Here ONE thread per tile (one warp per CTA, lane 0 working) walks its tile's pixels, samples and
// bounces start to finish -- camera sample, closest hit, shade, shadow ray, MIS ray, film -- with the same device
// functions, in the same order per tile, hence the same random stream and the same image as the wavefront form.
PB_D void film_add_sample_lane(const RenderDev& R, float2 pfilm, rgb L);  // defined with k_vol_mega below
template <int BIN, bool INST>
static __device__ __noinline__ ShadeOut zt_shade(const RenderDev* Rp, uint32_t id) { return shade_path<BIN, INST, true>(*Rp, id); }
template <bool INST>
__global__ void __launch_bounds__(32 * PB_ZT_WARPS) k_zt_mega(RenderDev R, const RenderDev* Rdev, uint32_t lanes) {
    // `lanes` tiles per warp: 1 when there are few tiles (pure latency), more when one-lane warps would fill the issue slots.  The warps of a CTA pass
    // the phases of a trip together (barriers between them), as k_vol_mega's do and for the same reason: the instruction cache.
    const uint32_t warp = threadIdx.x >> 5, ln = threadIdx.x & 31u;
    const uint32_t j = (blockIdx.x * (blockDim.x >> 5) + warp) * lanes + ln;
    unsigned long long n_camera = 0, n_closest = 0, n_shadow = 0, n_zero = 0, n_iter = 0;
    bool ok = false;
    if (ln < lanes && j < R.n_tiles_sel) {
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
    uint2 stack_mem[PB_STACK_SIZE(INST)];
    LocalStack stack{stack_mem};
    // ONE flat loop, a path vertex per trip: a lane whose path has ended goes on to its tile's next sample in the same trip count as its
    // neighbours' next vertex, instead of waiting at the end of a nested path loop for the warp's longest path.
    if (ok) n_camera += 1;
    for (;;) {
        if (!__syncthreads_or(ok)) break;
        int bin = Q_MISS;
        TravRay r;
        if (ok) {
            n_iter += 1;
            float4 a = R.ray[2 * j], b = R.ray[2 * j + 1];
            trav_init(R.scene, r, f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), a.w);
            trav_run<false, INST>(R.scene, r, stack, 0);
            n_closest += 1;
            bin = store_closest_hit(R, j, r);
        }
        __syncthreads();
        ShadeOut o = {false, false, false, false, false};
        if (ok) {
            switch (bin) {
                case Q_MATTE: o = zt_shade<Q_MATTE, INST>(Rdev, j); break;
                case Q_PLASTIC: o = zt_shade<Q_PLASTIC, INST>(Rdev, j); break;
                case Q_MIRROR: o = zt_shade<Q_MIRROR, INST>(Rdev, j); break;
                case Q_GLASS: o = zt_shade<Q_GLASS, INST>(Rdev, j); break;
                case Q_METAL: o = zt_shade<Q_METAL, INST>(Rdev, j); break;
                case Q_NOMAT: o = zt_shade<Q_NOMAT, INST>(Rdev, j); break;
                case Q_TEX: o = zt_shade<Q_TEX, INST>(Rdev, j); break;
                default: o = zt_shade<Q_MISS, INST>(Rdev, j); break;
            }
            if (o.zero_rad) n_zero += 1;
        }
        __syncthreads();
        if (ok && o.push_shadow) {
            float4 a = R.sh_ray[2 * j], b = R.sh_ray[2 * j + 1];
            trav_init(R.scene, r, f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), a.w);
            trav_run<true, INST>(R.scene, r, stack, 0);
            n_shadow += 1;
            if (!r.found) shadow_unoccluded(R, j);
        }
        __syncthreads();
        if (ok && o.push_mis) {
            float4 a = R.mis_ray[2 * j], b = R.mis_ray[2 * j + 1];
            trav_init(R.scene, r, f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), a.w);
            trav_run<false, INST>(R.scene, r, stack, 0);
            n_closest += 1;
            mis_resolve<INST>(R, j, r);
        }
        if (ok && !o.push_next) {
            // finished path -> film (integrator.rs:350-368 sanity rule), then the tile's next sample
            float4 Le = R.L_eta[j];
            rgb L(Le.x, Le.y, Le.z);
            float y = lum(L);
            if (L.r != L.r || L.g != L.g || L.b != L.b) L = rgb(0.0f);
            else if (y < -1.0e-5f) L = rgb(0.0f);
            else if (isinf(y)) L = rgb(0.0f);
            film_add_sample_lane(R, R.pfilm[j], L);
            ok = zt_next_path(R, j, false);
            if (ok) n_camera += 1;
        }
    }
    atomicAdd(&R.cnt->camera_rays, n_camera); atomicAdd(&R.cnt->closest_rays, n_closest); atomicAdd(&R.cnt->shadow_rays, n_shadow);
    atomicAdd(&R.cnt->zero_radiance, n_zero); atomicMax(&R.cnt->iterations, n_iter);
}


// ---------------------------------------------------------------------------
// VolPathIntegrator (src/integrators/volpath.rs:82-221) with homogeneous media: one kernel, a thread per path
// ---------------------------------------------------------------------------
// A volumetric path is a chain of data-dependent loops -- medium sampling in front of every vertex, the two transmittance loops of
// estimate_direct (VisibilityTester::tr, Scene::intersect_tr) that walk through any number of material-less boundaries, a sample
// stream whose length depends on which of them ran -- so it is written as the reference writes it: one thread owns a path from its
// camera sample to the film, claims the next camera sample when it is done (warp-aggregated fetch-add on the call's item cursor),
// and calls the same traversal (exact TU) and shading functions as the surface path integrator.  Path state lives in the slot
// arrays of RenderDev (slot = global thread index), the volume-only state in the thread (VolState).

// FilmTile::add_sample without the warp aggregation of film_add_sample (the lanes of this kernel are not converged)
PB_D void film_add_sample_lane(const RenderDev& R, float2 pfilm, rgb L) {
    const float rx = R.filter_radius[0], ry = R.filter_radius[1];
    const float ly = lum(L);
    if (ly > R.max_sample_luminance) L = L * rgb(R.max_sample_luminance / ly);
    const float dx = pfilm.x - 0.5f, dy = pfilm.y - 0.5f;
    const int p0x = max((int)ceilf(dx - rx), R.crop[0]), p0y = max((int)ceilf(dy - ry), R.crop[1]);
    const int p1x = min((int)floorf(dx + rx) + 1, R.crop[2]), p1y = min((int)floorf(dy + ry) + 1, R.crop[3]);
    const int width = R.crop[2] - R.crop[0];
    for (int y = p0y; y < p1y; ++y)
        for (int x = p0x; x < p1x; ++x) {
            float fx = fabsf(((float)x - dx) * R.inv_filter_radius[0] * 16.0f);
            float fy = fabsf(((float)y - dy) * R.inv_filter_radius[1] * 16.0f);
            int ix = min((int)floorf(fx), 15), iy = min((int)floorf(fy), 15);
            float fw = __ldg(R.filter_table + iy * 16 + ix);
            rgb c = L * rgb(1.0f) * rgb(fw);
            atomicAdd(R.film + (size_t)(y - R.crop[1]) * width + (x - R.crop[0]), make_float4(c.r, c.g, c.b, fw));
        }
}

// HomogeneousMedium::sample (homogeneous.rs:35-72) in front of the vertex the path ray of slot `id` has just found, then volpath.rs:114.
// Returns 0: no medium interaction (go on with the surface / the miss), 1: interaction sampled at vs->mi_p, 2: beta is black.
PB_D int vol_sample_medium(const RenderDev& R, uint32_t id, VolState* vs, bool found, float t_hit) {
    float4 bs = R.beta_st[id];
    rgb beta(bs.x, bs.y, bs.z);
    bool sampled = false;
    if (vs->medium >= 0) {
        const float4 ra = R.ray[2 * id], rb = R.ray[2 * id + 1];
        const f3 o(ra.x, ra.y, ra.z), d(rb.x, rb.y, rb.z);
        const float t_max = found ? t_hit : ra.w;  // Scene::intersect leaves the hit distance in ray.t_max
        DirectSampler smp;
        smp.prefetch(R, id);
        const pbrt_b200_medium m = R.scene.media[vs->medium];
        const rgb st = medium_sigma_t(m), ss = rgb3(m.sigma_s);
        const int channel = min((int)(smp.get_1d() * 3.0f), 2);
        const float stc = channel == 0 ? st.r : (channel == 1 ? st.g : st.b);
        const float dist = -logf(1.0f - smp.get_1d()) / stc;
        const float dl = len(d);
        const float t = fminf(dist / dl, t_max);
        sampled = t < t_max;
        if (sampled) vs->mi_p = o + d * t;
        const float tt = fminf(t, PB_FLT_MAX);
        const rgb Tr(expf((-st.r * tt) * dl), expf((-st.g * tt) * dl), expf((-st.b * tt) * dl));
        const rgb density = sampled ? st * Tr : Tr;
        float pdf = 0.0f;
        pdf += density.r; pdf += density.g; pdf += density.b;
        pdf *= 1.0f / 3.0f;
        if (pdf == 0.0f) pdf = 1.0f;
        beta = beta * (sampled ? Tr * ss / pdf : Tr / pdf);
        R.beta_st[id] = make_float4(beta.r, beta.g, beta.b, bs.w);
        smp.end(R, id);
    }
    if (is_black(beta)) return 2;
    return sampled ? 1 : 0;
}

// The medium branch of VolPathIntegrator::li (volpath.rs:117-133): uniform_sample_onelight / estimate_direct with the phase function
// in the BSDF's place (integrator.rs:140-146,183-188), then HenyeyGreenstein::sample_p for the next direction.
template <bool INST>
static __device__ __noinline__ ShadeOut vol_shade_medium(const RenderDev* Rp, uint32_t id, VolState* vs) {
    const RenderDev& R = *Rp;
    ShadeOut out{false, false, false, false, false};
    const float4 rb = R.ray[2 * id + 1];
    const f3 rd(rb.x, rb.y, rb.z);
    const float time = rb.w;
    float4 Le = R.L_eta[id], bs = R.beta_st[id];
    rgb beta(bs.x, bs.y, bs.z);
    uint32_t st = __float_as_uint(bs.w);
    uint32_t bounces = st & 0xffffu;
    if (bounces >= (uint32_t)R.max_depth) { out.push_dead = true; return out; }
    DirectSampler smp;
    smp.prefetch(R, id);
    const f3 p = vs->mi_p, wo = -rd, zero(0.f, 0.f, 0.f);
    const float g = R.scene.media[vs->medium].g;
    if (R.n_lights > 0) {
        float u1 = smp.get_1d();
        const float* ld_cdf = R.ld_cdf; const float* ld_func = R.ld_func; float ld_func_int = R.ld_func_int;
        if (R.sp.enabled) {
            int sl = R.sp.slot[spatial_voxel(R, p)];
            if (sl >= 0) { ld_cdf = R.sp.cdf + (size_t)sl * (R.n_lights + 1); ld_func = R.sp.func + (size_t)sl * R.n_lights; ld_func_int = R.sp.func_int[sl]; }
            else atomicExch(R.sp.counters + 2, 1u);
        }
        uint32_t ln = find_interval_cdf(ld_cdf, (int)R.n_lights + 1, u1);
        float selpdf = ld_func_int > 0.0f ? ld_func[ln] / (ld_func_int * (float)R.n_lights) : 0.0f;
        bool zero_rad = true;
        if (selpdf != 0.0f) {
            float2 ulight = smp.get_2d();
            float2 uscatt = smp.get_2d();
            const pbrt_b200_light& light = R.scene.lights[ln];
            bool delta = is_delta_light(light);
            LightSample ls;
            light_sample_li<INST>(R, ln, p, ulight, ls, zero, zero);
            if (ls.pdf > 0.0f && !is_black(ls.Li)) {
                float ph = phase_hg(dot(wo, ls.wi), g);
                if (ph != 0.0f) {
                    f3 o = offset_ray_origin(p, zero, zero, ls.p1 - p);
                    f3 tg = offset_ray_origin(ls.p1, ls.p1_err, ls.p1_n, o - ls.p1);
                    f3 d = tg - o;
                    rgb f(ph);
                    rgb Ld = delta ? f * ls.Li / ls.pdf : f * ls.Li * power_heuristic(ls.pdf, ph) / ls.pdf;
                    rgb add = beta * (Ld / selpdf);
                    store_ray(R.sh_ray, id, o, d, 1.0f - PB_SHADOW_EPSILON, time);
                    R.sh_contrib[id] = make_float4(add.r, add.g, add.b, 0.f);
                    vs->sh_medium = vs->medium; vs->p1 = ls.p1; vs->p1_err = ls.p1_err; vs->p1_n = ls.p1_n;
                    out.push_shadow = true;
                    zero_rad = false;
                }
            }
            if (!delta) {
                f3 wi(0.f, 0.f, 0.f);
                float ph = hg_sample_p(g, wo, &wi, uscatt);
                if (ph != 0.0f && ph > 0.0f) {
                    Surf ref;
                    ref.p = p; ref.p_error = zero; ref.n = zero; ref.wo = wo; ref.sh_n = zero; ref.sh_dpdu = zero;
                    float lpdf = light_pdf_li<INST>(R, ln, ref, wi);
                    if (lpdf != 0.0f) {
                        float weight = power_heuristic(ph, lpdf);
                        rgb fac = beta * (rgb(ph) * weight / ph / selpdf);
                        store_ray(R.mis_ray, id, offset_ray_origin(p, zero, zero, wi), wi, PB_INF, time);
                        R.mis_contrib[id] = make_float4(fac.r, fac.g, fac.b, __uint_as_float(ln));
                        vs->mis_medium = vs->medium;
                        out.push_mis = true;
                        zero_rad = false;
                    }
                }
            }
        }
        out.zero_rad = zero_rad;
    }
    // volpath.rs:127-132: new direction from the phase function; the ray stays in the medium
    f3 wi(0.f, 0.f, 0.f);
    hg_sample_p(g, wo, &wi, smp.get_2d());
    store_ray(R.ray, id, offset_ray_origin(p, zero, zero, wi), wi, PB_INF, time);
    bool alive = true;
    {   // Russian roulette, volpath.rs:206-214 (specular_bounce = false)
        rgb rrbeta = beta * Le.w;
        float mc = max_comp(rrbeta);
        if (mc < R.rr_threshold && bounces > 3) {
            float qv = fmaxf(1.0f - mc, 0.05f);
            if (smp.get_1d() < qv) alive = false;
            else beta = beta / (1.0f - qv);
        }
    }
    smp.end(R, id);
    if (alive) {
        bounces += 1;
        R.beta_st[id] = make_float4(beta.r, beta.g, beta.b, __uint_as_float(bounces));
        out.push_next = true;
    } else out.push_dead = true;
    return out;
}

template <int BIN, bool INST>
static __device__ __noinline__ ShadeOut vol_shade(const RenderDev* Rp, uint32_t id, VolState* vs) { return shade_path<BIN, INST, false, true>(*Rp, id, vs); }

#define PB_VOL_SEGMENT_CAP 4096u   /* transmittance loops: boundaries crossed by one shadow / MIS ray before it is given up (hang guard) */
#define PB_VOL_VERTEX_CAP 65536u   /* path loop: boundary crossings lower the bounce count, so max_depth alone does not bound it */
template <bool INST>
__global__ void __launch_bounds__(PB_VOL_BLOCK) k_vol_mega(RenderDev R, const RenderDev* Rdev, unsigned long long total_items, int camera_medium) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;  // slot
    const unsigned lane = threadIdx.x & 31u;
    unsigned long long n_camera = 0, n_closest = 0, n_zero = 0, n_iter = 0;
    uint2 stack_mem[PB_STACK_SIZE(INST)];
    LocalStack stack{stack_mem};
    VolState vs;
    // ONE flat loop, a path vertex per trip: a lane whose path has ended claims its next camera sample at the top of the following trip, so the
    // warp stays full and every lane is in the same phase of a vertex (trace, medium / surface shade, shadow walk, MIS walk).  The nested form
    // (a path loop inside a sample loop) reconverged only when the warp's LONGEST path had ended: lanes idled for the rest of it.
    bool have = false, exhausted = false, alive = false;
    uint32_t vertices = 0;
    for (;;) {
        {   // lanes without a path share one fetch-add
            const bool need = !have && !exhausted;
            const unsigned m = __ballot_sync(0xffffffffu, need);
            if (need) {
                const int leader = __ffs(m) - 1;
                unsigned long long base = 0;
                if ((int)lane == leader) base = atomicAdd(&R.cnt->item_cursor, (unsigned long long)__popc(m));
                base = __shfl_sync(m, base, leader);
                const unsigned long long item = base + (unsigned long long)__popc(m & ((1u << lane) - 1u));
                if (item >= total_items) exhausted = true;
                else if (gen_camera_path(R, item, j)) {
                    n_camera += 1;
                    vs.medium = camera_medium;
                    have = true; alive = true; vertices = 0;
                }
            }
        }
        // ncu on the 64-thread form: issue slots 7 % busy, 52 of 57 stall cycles per instruction are `no_instruction` -- sixteen warps per SM each
        // somewhere else in 100s of KB of code miss the instruction cache all the time.  One 512-thread CTA per SM whose warps pass the phases of a
        // trip TOGETHER (barriers between trace / shade / shadow walk / MIS walk) keeps the SM inside one region of the code at a time.
        if (!__syncthreads_or(have || !exhausted)) break;
        if (have) {
            if (vertices++ >= PB_VOL_VERTEX_CAP) alive = false;
        }
        int bin = Q_MISS, ms = 2;
        TravRay r;
        if (have && alive) {
            n_iter += 1;
            {
                float4 a = R.ray[2 * j], b = R.ray[2 * j + 1];
                trav_init(R.scene, r, f3(a.x, a.y, a.z), f3(b.x, b.y, b.z), a.w);
                trav_run<false, INST>(R.scene, r, stack, 0);
                n_closest += 1;
            }
            bin = store_closest_hit(R, j, r);
            ms = vol_sample_medium(R, j, &vs, r.found, r.hit.t);
        }
        __syncthreads();
        ShadeOut o = {false, false, false, false, false};  // ms == 2: the path ends here (volpath.rs:114)
        if (have && alive) {
            if (ms == 2) {}
            else if (ms == 1) o = vol_shade_medium<INST>(Rdev, j, &vs);
            else switch (bin) {
                case Q_MATTE: o = vol_shade<Q_MATTE, INST>(Rdev, j, &vs); break;
                case Q_PLASTIC: o = vol_shade<Q_PLASTIC, INST>(Rdev, j, &vs); break;
                case Q_MIRROR: o = vol_shade<Q_MIRROR, INST>(Rdev, j, &vs); break;
                case Q_GLASS: o = vol_shade<Q_GLASS, INST>(Rdev, j, &vs); break;
                case Q_METAL: o = vol_shade<Q_METAL, INST>(Rdev, j, &vs); break;
                case Q_NOMAT: o = vol_shade<Q_NOMAT, INST>(Rdev, j, &vs); break;
                case Q_TEX: if (INST) { o = vol_shade<Q_TEX, true>(Rdev, j, &vs); break; }  // textured scenes run the full-featured family (launch_vol_mega)
                default: o = vol_shade<Q_MISS, INST>(Rdev, j, &vs); break;
            }
            if (o.zero_rad) n_zero += 1;
        }
        __syncthreads();
        if (have && alive) {
            if (o.push_shadow) {  // VisibilityTester::tr, light.rs:125-150
                float4 a = R.sh_ray[2 * j], b = R.sh_ray[2 * j + 1];
                f3 ro(a.x, a.y, a.z), rdir(b.x, b.y, b.z);
                float t_max = a.w;
                int med = vs.sh_medium;
                rgb Tr(1.0f);
                bool blocked = false;
                for (uint32_t seg = 0;; ++seg) {
                    if (seg >= PB_VOL_SEGMENT_CAP) { blocked = true; break; }
                    trav_init(R.scene, r, ro, rdir, t_max);
                    trav_run<false, INST>(R.scene, r, stack, 0);
                    n_closest += 1;
                    if (r.found && R.scene.prims[r.hit.slot].material >= 0) { blocked = true; break; }
                    if (med >= 0) Tr = Tr * medium_tr(R.scene.media[med], rdir, r.found ? r.hit.t : t_max);
                    if (!r.found) break;
                    uint32_t fl;
                    Surf si = surface_at_hit<INST>(R.scene, r.hit.inst, r.hit.slot, ro, rdir, r.hit.t, r.hit.b0, r.hit.b1, r.hit.b2, &fl);
                    const VolInterface mi = vol_hit_interface(R.scene, r.hit.slot, med);
                    const f3 o2 = offset_ray_origin(si.p, si.p_error, si.n, vs.p1 - si.p);  // spawn_rayto_interaction, interaction.rs:46-52
                    const f3 tg = offset_ray_origin(vs.p1, vs.p1_err, vs.p1_n, o2 - vs.p1);
                    rdir = tg - o2; ro = o2; t_max = 1.0f - PB_SHADOW_EPSILON;
                    med = vol_medium_for(mi, si.n, rdir);
                }
                if (!blocked) {
                    float4 c = R.sh_contrib[j], L = R.L_eta[j];
                    L.x += c.x * Tr.r; L.y += c.y * Tr.g; L.z += c.z * Tr.b;
                    R.L_eta[j] = L;
                }
            }
        }
        __syncthreads();
        if (have && alive) {
            if (o.push_mis) {  // Scene::intersect_tr, scene.rs:68-87, then integrator.rs:218-232
                float4 a = R.mis_ray[2 * j], b = R.mis_ray[2 * j + 1];
                f3 ro(a.x, a.y, a.z);
                const f3 rdir(b.x, b.y, b.z);
                int med = vs.mis_medium;
                const float4 c = R.mis_contrib[j];
                const uint32_t ln = __float_as_uint(c.w);
                rgb Tr(1.0f), li(0.0f);
                for (uint32_t seg = 0; seg < PB_VOL_SEGMENT_CAP; ++seg) {
                    trav_init(R.scene, r, ro, rdir, PB_INF);
                    trav_run<false, INST>(R.scene, r, stack, 0);
                    n_closest += 1;
                    if (med >= 0) Tr = Tr * medium_tr(R.scene.media[med], rdir, r.found ? r.hit.t : PB_INF);
                    if (!r.found) {
                        const pbrt_b200_light& l = R.scene.lights[ln];
                        if (l.type == PBRT_B200_LIGHT_INFINITE) li = rgb3(l.L);
                        break;
                    }
                    const pbrt_b200_prim pr = R.scene.prims[r.hit.slot];
                    uint32_t fl;
                    Surf si = surface_at_hit<INST>(R.scene, r.hit.inst, r.hit.slot, ro, rdir, r.hit.t, r.hit.b0, r.hit.b1, r.hit.b2, &fl);
                    if (pr.material >= 0) {
                        if (pr.area_light == (int)ln) {
                            const pbrt_b200_light& al = R.scene.lights[ln];
                            if (al.two_sided || dot(si.n, -rdir) > 0.0f) li = rgb3(al.L);
                        }
                        break;
                    }
                    const VolInterface mi = vol_hit_interface(R.scene, r.hit.slot, med);
                    ro = offset_ray_origin(si.p, si.p_error, si.n, rdir);
                    med = vol_medium_for(mi, si.n, rdir);
                }
                if (!is_black(li)) {
                    float4 L = R.L_eta[j];
                    L.x += c.x * li.r * Tr.r; L.y += c.y * li.g * Tr.g; L.z += c.z * li.b * Tr.b;
                    R.L_eta[j] = L;
                }
            }
            alive = o.push_next;
        }
        if (have && !alive) {
            float4 Le = R.L_eta[j];
            rgb L(Le.x, Le.y, Le.z);
            float y = lum(L);  // integrator.rs:350-368
            if (L.r != L.r || L.g != L.g || L.b != L.b) L = rgb(0.0f);
            else if (y < -1.0e-5f) L = rgb(0.0f);
            else if (isinf(y)) L = rgb(0.0f);
            film_add_sample_lane(R, R.pfilm[j], L);
            have = false;
        }
    }
    atomicAdd(&R.cnt->camera_rays, n_camera); atomicAdd(&R.cnt->closest_rays, n_closest);
    atomicAdd(&R.cnt->zero_radiance, n_zero); atomicMax(&R.cnt->iterations, n_iter);
}

void launch_zt_mega(const RenderDev& R, const RenderDev* rdev, uint32_t lanes, uint32_t nblk, cudaStream_t stream) {
    k_zt_mega<true><<<nblk, 32 * PB_ZT_WARPS, 0, stream>>>(R, rdev, lanes);
}
void launch_vol_mega(const RenderDev& R, const RenderDev* rdev, unsigned long long total_items, int camera_medium, bool full, int grid, cudaStream_t stream) {
    if (full) k_vol_mega<true><<<grid, PB_VOL_BLOCK, 0, stream>>>(R, rdev, total_items, camera_medium);
    else k_vol_mega<false><<<grid, PB_VOL_BLOCK, 0, stream>>>(R, rdev, total_items, camera_medium);
}
int vol_mega_blocks_per_sm(bool full) {
    int per_sm = 1;
    if (full) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_vol_mega<true>, PB_VOL_BLOCK, 0);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_vol_mega<false>, PB_VOL_BLOCK, 0);
    return per_sm;
}
}  // namespace pb (mega.o ends here)
#endif  // PB_MEGA_TU
#endif  // PB_EXACT_TU || PB_MEGA_TU
#if PB_EXACT_TU
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

extern "C" int pbrt_b200_render(pbrt_b200_scene* sc, const pbrt_b200_render_desc* rd, float* rgbw_out, pbrt_b200_render_stats* stats) {
    if (!sc || !rd || !rgbw_out) return fail(PBRT_B200_ERR_INVALID, "render: null argument");
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
    if (ikind > PBRT_B200_INTEGRATOR_VOLPATH) return fail(PBRT_B200_ERR_INVALID, "render: unknown integrator kind");
    const bool vol = ikind == PBRT_B200_INTEGRATOR_VOLPATH;
    const bool path_like = ikind == PBRT_B200_INTEGRATOR_PATH || vol;  // no recursion state
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
    // volpath: one slot per thread of the megakernel's single resident wave
    int vol_grid = 0;
    if (vol) {
        int smc = 148, per_sm = 1;
        cudaDeviceGetAttribute(&smc, cudaDevAttrMultiProcessorCount, sc->device);
        per_sm = vol_mega_blocks_per_sm(sc->dev.n_instances || sc->dev.n_sphere_lights || sc->dev.material_ext);
        const unsigned long long want = (total_items + (unsigned long long)PB_VOL_BLOCK - 1ull) / (unsigned long long)PB_VOL_BLOCK;
        vol_grid = (int)std::max<unsigned long long>(1ull, std::min<unsigned long long>((unsigned long long)smc * (unsigned long long)std::max(per_sm, 1), want));
        capacity = ((uint32_t)vol_grid * (uint32_t)PB_VOL_BLOCK + 255u) & ~255u;
    }
    if (capacity == 0) capacity = 256;
    if ((rc = ensure_buffers(st, &capacity))) return rc;
    if (vol && capacity < (uint32_t)vol_grid * (uint32_t)PB_VOL_BLOCK) vol_grid = (int)(capacity / (uint32_t)PB_VOL_BLOCK);
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
    bool sample_prepass = !zt && !R.rec.kind && !vol;  // k_sample_block serves every path the tables do not
    R.u8 = nullptr;
    if (!zt && !R.rec.kind && !vol && S.kind == PBRT_B200_SAMPLER_SOBOL && S.log2_resolution > 0 && !getenv("PBRT_B200_NO_SOBOL_TABLES")) {
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
    if (vol && R.sp.enabled && R.sp.lazy)
        return fail(PBRT_B200_ERR_UNSUPPORTED, "render: volpath with lightsamplestrategy \"spatial\" needs the eagerly built voxel table (voxels x lights <= 2^25)");
    PB_CUDA_TRY(cudaEventRecord(ev0, stream));
    if (vol) {
        if (total_items > 0) {
            // R in device memory for the out-of-line shade calls (as k_zt_mega)
            size_t rdev_bytes = 0;
            RenderDev* rdev = reinterpret_cast<RenderDev*>(pool_alloc(sizeof(RenderDev), &rdev_bytes));
            if (!rdev) return fail(PBRT_B200_ERR_CUDA, "render: out of device memory");
            ZtRelease rdev_release{rdev, rdev_bytes};
            PB_CUDA_TRY(cudaMemcpyAsync(rdev, &R, sizeof(RenderDev), cudaMemcpyHostToDevice, stream));
            launch_vol_mega(R, rdev, total_items, rd->integrator.camera_medium, sc->dev.n_instances || sc->dev.n_sphere_lights || sc->dev.material_ext, vol_grid, stream);
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
#endif  // PB_EXACT_TU
