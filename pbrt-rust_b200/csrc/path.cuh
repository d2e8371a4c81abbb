// Device side of the wavefront path tracer that more than one translation unit needs (render.cu, shade.cu, mega.cu): path state
// (RenderDev and its queues), samplers, media, film, ray generation, light sampling, and shade_path -- one path vertex of
// PathIntegrator::li / VolPathIntegrator::li -- that the wavefront kernels and the one-kernel forms share.  Kernels live in the units.
#pragma once
#include <cuda_runtime.h>
#include <cmath>
#include "scene.cuh"
#include "shading.cuh"
#include "trace.cuh"
#include "texture.cuh"
#include "util.cuh"

#define PB_ZT_WARPS 4u    /* warps per CTA of k_zt_mega (the host aims at ~4 warps per SM: one CTA), phases of a trip passed together */
#define PB_VOL_BLOCK 512  /* threads per CTA of k_vol_mega: the CTA's warps pass the phases of a trip together (barriers between them): see the kernel */

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

// FilmTile::add_sample without the warp aggregation of film_add_sample (the lanes of the one-kernel forms are not converged)
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

// hit record + material bin of a path's closest-hit ray (k_trace_closest, and the path rays of the one-kernel forms)
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
// PART (volpath with grid media, where estimate_direct's transmittance loops draw from the sampler and so must run between the two
// halves of the vertex): 0 = the whole vertex; 1 = up to and including the light sample -- a vertex that goes on returns neither
// push_next nor push_dead, its continuation is pending; 2 = the continuation (next direction, roulette), which recomputes the
// interaction and the BSDF from the hit record still in the slot.
template <int BIN, bool INST, bool ZT, bool VOL = false, int PART = 0>
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
        if constexpr (PART != 2) if ((bounces == 0 || specular_bounce) && pr.area_light >= 0) {
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
                if constexpr (PART != 2) if ((VOL || bsdf_count(bsdf, NONSPEC) > 0) && R.n_lights > 0) {
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
                if constexpr (PART == 1) {  // the continuation is pending (phase 5 of k_vol_mega<.., true>)
                    R.L_eta[id] = make_float4(L.r, L.g, L.b, etascale);
                    smp.end(R, id);
                    return ShadeOut{false, push_shadow, push_mis, false, zero_rad};
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

// ---------------------------------------------------------------------------
// what a traced shadow / MIS ray adds to its path (k_trace_shadow / k_trace_mis, and the one-kernel forms)
// ---------------------------------------------------------------------------
// VisibilityTester::unoccluded (core/light.rs:120-123)
PB_D void shadow_unoccluded(const RenderDev& R, uint32_t id) {  // the light sample's contribution reaches the path
    float4 c = R.sh_contrib[id];
    float4 L = R.L_eta[id];
    L.x += c.x; L.y += c.y; L.z += c.z;
    R.L_eta[id] = L;
}
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

// Launchers of the kernels in shade.cu ...
void launch_shade_kernels(const RenderDev& R, int parity, bool full, int grid_small, int grid_shade, cudaStream_t stream);
void launch_rec_shade(const RenderDev& R, int parity, bool zt, bool full, cudaStream_t stream);
// ... and in mega.cu
void launch_zt_mega(const RenderDev& R, const RenderDev* rdev, uint32_t lanes, uint32_t nblk, cudaStream_t stream);
void launch_vol_mega(const RenderDev& R, const RenderDev* rdev, unsigned long long total_items, int camera_medium, bool full, const DevGrid* grids, int grid,
                     cudaStream_t stream);
int vol_mega_blocks_per_sm(bool full, bool grids);

// ... and in bdpt.cu: PerspectiveCamera's importance functions need the inverse matrices, which the host computes once per call
struct BdptCam {
    float c2w[16], w2c[16], c2r[16];
    f3 fwd;             // CameraToWorld(0, 0, 1) as a vector: cos(theta) of a ray leaving the lens
    f3 n_lens;          // ... as a normal: the lens interaction's n
    float A;            // image-plane area at z = 1 (pbrt-v3 perspective.cpp:55-62)
    float lens_radius, focal_distance;
    int sb[4];          // Film::get_sample_bounds
    const float* spot_l2w;  // [n_lights][16] LightToWorld of spot lights (inverse of world_to_light), device memory
};
size_t bdpt_vertex_bytes();
int bdpt_blocks_per_sm(bool inst);
void launch_bdpt(const RenderDev& R, const BdptCam& C, void* verts, float* splat, unsigned long long total_items, bool inst, int grid, cudaStream_t stream);

}  // namespace pb
