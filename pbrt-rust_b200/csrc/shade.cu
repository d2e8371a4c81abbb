// The shade kernels of the wavefront path tracer (k_shade<material>, k_rec_shade) and their launchers, compiled with --use_fast_math
// (csrc/Makefile).  Shading is tolerance-parity by nature (libm differs from CUDA's transcendentals, SURVEY App. A.7): here the ~200 IEEE
// divisions and square roots per path (8-10 SASS instructions each, with a slow-path call) become MUFU.RCP / MUFU.RSQ sequences and
// a*b+c contracts to FFMA.  Nothing here is pinned bit for bit: BSDF / light / material arithmetic is checked against the oracle by
// image relMSE <= 1e-3 (tests/test_gpu_render.py), while every ray the shade kernels emit is still traced by the exactly rounded
// kernels of render.cu.
// PB_TU_SHADE comes before the first include: vecmath.cuh then takes the plain f32 cross product instead of the f64-exact one.
#define PB_TU_SHADE 1
#include <algorithm>

#include "path.cuh"
#include "recursive.cuh"

namespace pb {

// Min resident CTAs per SM in __launch_bounds__, A/B-measured with tools/step_diag.py on S3: shade 5/6/8 CTAs (96/80/64 registers) and
// trace 6/8/10 CTAs are all within +-1% or slower than the compiler's default choice, so the shade kernels and the plain trace kernels
// set none.
#define PB_REC_BLOCK 384  /* threads per CTA of k_rec_shade (168 registers: one CTA per SM whose warps start every path together, see the kernel) */
#define PB_TEX_BLOCK 512  /* threads per CTA of k_shade<Q_TEX>: one CTA per SM whose warps start every path together (see k_shade) */

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

// WhittedIntegrator / DirectLightingIntegrator (recursive.cuh): one step of the depth-first recursion for every live camera sample --
// shade the hit of its current ray.
// TEX: the scene has textured materials (texture.cuh) -- every surface then gets its full interaction and its ray differentials
// (compute_scattering_functions always runs compute_differentials, interaction.rs:258-267), and specular_reflect / specular_transmit
// hand differentials on to the rays they spawn (integrator.rs:427-452, 476-513).
template <bool INST, bool ZT, bool TEX>
__global__ void __launch_bounds__(PB_REC_BLOCK) k_rec_shade(RenderDev R, int parity) {
    constexpr int KM = TEX ? KM_TEX : KM_ALL;
    const uint32_t n = R.cnt->n_path;
    const uint32_t* q = R.q_path[parity];
    uint32_t* q_next = R.q_path[parity ^ 1];
    // 35 k instructions (TEX: 56 k, the texture interpreter on top of every BSDF and the recursion frames) -- as k_shade<Q_TEX>, the CTA is
    // the whole SM and its warps start every path behind a barrier, so that they stay close to each other in the code (instruction cache)
    const uint32_t nround = ((n + blockDim.x - 1u) / blockDim.x) * blockDim.x;
    const uint32_t D = R.rec.stack_depth;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nround; i += gridDim.x * blockDim.x) {
        __syncthreads();
        bool push_next = false, push_dead = false;
        uint32_t id = 0;
        if (i < n) {
            id = q[i];
            float4 ra = R.ray[2 * id], rb = R.ray[2 * id + 1];
            f3 ro(ra.x, ra.y, ra.z), rd(rb.x, rb.y, rb.z);
            const float time = rb.w;
            float4 bs = R.beta_st[id];
            rgb beta(bs.x, bs.y, bs.z), Ladd(0.0f);
            uint32_t depth = __float_as_uint(bs.w) & 0xffffu;
            bool has_diff = TEX && (__float_as_uint(bs.w) & PB_ST_HAS_DIFF) != 0u;
            RecSampler<ZT> smp;
            smp.begin(R, id);
            uint32_t sp = R.rec.sp[id];
            const int bin = (int)R.hit_bin[id];
            bool pop = false;
            if (bin == Q_MISS) {
                // every light's le(ray): non-zero for infinite lights only (whitted.rs:60-65, directlighting.rs:83-86)
                for (uint32_t k = 0; k < R.n_infinite; ++k) Ladd = Ladd + rgb3(R.scene.lights[R.infinite_lights[k]].L) * beta;
                pop = true;
            } else {
                uint4 h = R.hit[id];
                uint32_t fl;
                const uint32_t hinst = (INST && R.scene.n_instances) ? R.hit_inst[id] : PBRT_B200_NO_HIT;
                Surf si;
                SurfX sx;
                RayDiff rdf;
                rdf.has = false;
                if (TEX) {
                    surface_full(R.scene.self_dev, hinst, h.x, ro, rd, __uint_as_float(h.y), __uint_as_float(h.z), __uint_as_float(h.w), R.hit_b2[id], &si, &sx, &fl);
                    rdf = load_diff(R.rdiff, id, has_diff);
                } else si = surface_at_hit<INST>(R.scene, hinst, h.x, ro, rd, __uint_as_float(h.y), __uint_as_float(h.z), __uint_as_float(h.w), R.hit_b2[id], &fl);
                const pbrt_b200_prim pr = R.scene.prims[h.x];
                BsdfN<TEX ? 5 : 2> bsdf;
                bsdf.valid = false;
                if (pr.material >= 0) {
                    if (TEX && R.scene.materials[pr.material].textured) material_bsdf_tex<false>(R.scene.self_dev, pr.material, &si, &sx, &rdf, &bsdf);
                    else {
                        if (TEX) compute_differentials(si, sx, rdf);
                        material_bsdf<-1, false>(R.scene.materials[pr.material], si, bsdf);
                    }
                }
                if (!bsdf.valid) {  // same depth, nothing drawn from the sampler (whitted.rs:76-80, directlighting.rs:91-94)
                    f3 o = offset_ray_origin(si.p, si.p_error, si.n, rd);
                    store_ray(R.ray, id, o, rd, PB_INF, time);
                    has_diff = false;  // spawn_ray: no differentials
                    push_next = true;
                } else {
                    if (pr.area_light >= 0) {  // isect.le(wo)
                        const pbrt_b200_light& al = R.scene.lights[pr.area_light];
                        if (al.two_sided || dot(si.n, si.wo) > 0.0f) Ladd = Ladd + rgb3(al.L) * beta;
                    }
                    const uint32_t nl = R.n_lights;
                    if (R.rec.kind == PBRT_B200_INTEGRATOR_WHITTED) {  // whitted.rs:85-97
                        for (uint32_t li = 0; li < nl; ++li) {
                            float2 u = smp.get_2d(R);
                            LightSample ls;
                            light_sample_li<INST>(R, li, si.p, u, ls, si.p_error, si.n);
                            if (is_black(ls.Li) || ls.pdf == 0.0f) continue;
                            rgb f = bsdf_f<KM>(bsdf, si.wo, ls.wi, BX_ALL);
                            if (is_black(f)) continue;
                            f3 o = offset_ray_origin(si.p, si.p_error, si.n, ls.p1 - si.p);
                            f3 tg = offset_ray_origin(ls.p1, ls.p1_err, ls.p1_n, o - ls.p1);
                            rgb add = beta * (f * ls.Li * absdot(ls.wi, si.n) / ls.pdf);
                            uint32_t e = atomicAdd(&R.cnt->n_shadow, 1u);
                            store_ray(R.rec.e_sh_ray, e, o, tg - o, 1.0f - PB_SHADOW_EPSILON, time);
                            R.rec.e_sh_contrib[e] = make_float4(add.r, add.g, add.b, __uint_as_float(id));
                        }
                    } else if (nl > 0) {
                        if (R.rec.kind == PBRT_B200_INTEGRATOR_DIRECT_ALL) {  // uniform_sample_all_lights, integrator.rs:40-79
                            for (uint32_t li = 0; li < nl; ++li) {
                                float2 ulight, uscatt;
                                const uint32_t ns = R.rec.multi ? max(R.scene.lights[li].n_samples, 1u) : 1u;
                                if (!ZT && ns > 1u) {  // Ld = sum_k estimate_direct(array element k) / nsamples, integrator.rs:63-74
                                    if (smp.arr + 2u <= R.rec.n_arrays) {
                                        const uint32_t a0 = smp.arr, sn = R.rec.sample_num[id];
                                        smp.arr += 2u;
                                        for (uint32_t k = 0; k < ns; ++k) {
                                            ulight = smp.array_element(R, a0, sn, ns, k);
                                            uscatt = smp.array_element(R, a0 + 1u, sn, ns, k);
                                            rec_estimate_direct<INST, KM>(R, id, si, bsdf, li, ulight, uscatt, beta, 1.0f / (float)ns, time);
                                        }
                                        continue;
                                    }
                                    smp.arr = R.rec.n_arrays;  // requests exhausted: get_2d_array returns None from here on
                                    ulight = smp.get_2d(R); uscatt = smp.get_2d(R);
                                    rec_estimate_direct<INST, KM>(R, id, si, bsdf, li, ulight, uscatt, beta, 1.0f, time);
                                    continue;
                                }
                                bool hl = smp.get_2d_array(R, &ulight);
                                bool hs = smp.get_2d_array(R, &uscatt);
                                if (!hl || !hs) { ulight = smp.get_2d(R); uscatt = smp.get_2d(R); }
                                rec_estimate_direct<INST, KM>(R, id, si, bsdf, li, ulight, uscatt, beta, 1.0f, time);
                            }
                        } else {  // uniform_sample_onelight without a distribution, integrator.rs:81-106
                            float u1 = smp.get_1d(R);
                            float fl1 = u1 * (float)nl;
                            uint32_t ln = (fl1 != fl1 || fl1 <= 0.0f) ? 0u : (fl1 >= 4294967040.0f ? 0xffffffffu : (uint32_t)fl1);  // `as usize`
                            ln = min(ln, nl - 1u);
                            float lightpdf = 1.0f / (float)nl;
                            float2 ulight = smp.get_2d(R);
                            float2 uscatt = smp.get_2d(R);
                            rec_estimate_direct<INST, KM>(R, id, si, bsdf, ln, ulight, uscatt, beta, 1.0f / lightpdf, time);
                        }
                    }
                    pop = true;
                    if ((int)depth + 1 < R.max_depth) {
                        // specular_reflect (integrator.rs:413-455): the 2D sample is drawn whatever the BSDF holds
                        float2 ur = smp.get_2d(R);
                        f3 wir(0.f, 0.f, 0.f), wit(0.f, 0.f, 0.f);
                        float pdfr = 0.0f, pdft = 0.0f;
                        int st = 0;
                        rgb fr = bsdf_sample<KM>(bsdf, si.wo, &wir, ur, &pdfr, BX_REFLECTION | BX_SPECULAR, &st);
                        const bool okr = pdfr > 0.0f && !is_black(fr) && absdot(wir, si.sh_n) != 0.0f;
                        // specular_transmit (integrator.rs:457-520): a specular lobe ignores its sample, so the direction and
                        // weight are known now; the two dimensions are drawn when the reference draws them (after the
                        // reflection sub-tree)
                        rgb ft = bsdf_sample<KM>(bsdf, si.wo, &wit, make_float2(0.0f, 0.0f), &pdft, BX_TRANSMISSION | BX_SPECULAR, &st);
                        bool okt = pdft > 0.0f && !is_black(ft) && absdot(wit, si.sh_n) != 0.0f;
                        rgb beta_t = okt ? beta * (ft * (absdot(wit, si.sh_n) / pdft)) : rgb(0.0f);
                        f3 ot = okt ? offset_ray_origin(si.p, si.p_error, si.n, wit) : f3(0.f, 0.f, 0.f);
                        // uber with partial opacity holds TWO specular transmission lobes (uber.rs:52-56,102-106): the sample's first
                        // dimension picks one (BSDF::sample_f), so both candidates are prepared and the choice is made when the sample is drawn
                        const bool two = TEX && bsdf_count(bsdf, BX_TRANSMISSION | BX_SPECULAR) == 2;
                        f3 wit2(0.f, 0.f, 0.f), ot2(0.f, 0.f, 0.f);
                        rgb beta_t2(0.0f);
                        bool okt2 = false;
                        if (two) {
                            float pdf2 = 0.0f;
                            rgb ft2 = bsdf_sample<KM>(bsdf, si.wo, &wit2, make_float2(0.75f, 0.0f), &pdf2, BX_TRANSMISSION | BX_SPECULAR, &st);
                            okt2 = pdf2 > 0.0f && !is_black(ft2) && absdot(wit2, si.sh_n) != 0.0f;
                            if (okt2) { beta_t2 = beta * (ft2 * (absdot(wit2, si.sh_n) / pdf2)); ot2 = offset_ray_origin(si.p, si.p_error, si.n, wit2); }
                        }
                        const size_t FS = (size_t)R.capacity * D;  // second-candidate frames live one stack array further
                        // a spawned ray has differentials iff its parent has (`if let Some(ref diff) = r.diff`)
                        if (okr) {
                            if (sp < D) {
                                const size_t fi = (size_t)id * D + sp;
                                R.rec.st_ray[2 * fi] = make_float4(ot.x, ot.y, ot.z, okt ? 1.0f : 0.0f);
                                R.rec.st_ray[2 * fi + 1] = make_float4(wit.x, wit.y, wit.z, time);
                                R.rec.st_beta[fi] = make_float4(beta_t.r, beta_t.g, beta_t.b,
                                                                __uint_as_float((depth + 1u) | (has_diff ? PB_ST_HAS_DIFF : 0u) | (two ? PB_ST_TWO_LOBES : 0u)));
                                if (TEX && has_diff && okt) store_diff(R.rec.st_diff, fi, specular_differentials(si, sx, rdf, si.wo, wit, bsdf.eta, true));
                                if (two) {
                                    R.rec.st_ray[2 * (fi + FS)] = make_float4(ot2.x, ot2.y, ot2.z, okt2 ? 1.0f : 0.0f);
                                    R.rec.st_ray[2 * (fi + FS) + 1] = make_float4(wit2.x, wit2.y, wit2.z, time);
                                    R.rec.st_beta[fi + FS] = make_float4(beta_t2.r, beta_t2.g, beta_t2.b, 0.0f);
                                    if (has_diff && okt2) store_diff(R.rec.st_diff, fi + FS, specular_differentials(si, sx, rdf, si.wo, wit2, bsdf.eta, true));
                                }
                                sp += 1;
                            }
                            beta = beta * (fr * absdot(wir, si.sh_n) / pdfr);
                            f3 o = offset_ray_origin(si.p, si.p_error, si.n, wir);
                            store_ray(R.ray, id, o, wir, PB_INF, time);
                            if (TEX && has_diff) store_diff(R.rdiff, id, specular_differentials(si, sx, rdf, si.wo, wir, bsdf.eta, false));
                            depth += 1;
                            push_next = true; pop = false;
                        } else {
                            if (two) {  // specular_transmit's get_2d: its first dimension picks the lobe
                                const float2 u2 = smp.get_2d(R);
                                if (floorf(u2.x * 2.0f) >= 1.0f) { okt = okt2; beta_t = beta_t2; ot = ot2; wit = wit2; }
                            } else smp.skip_2d(R);
                            if (okt) {
                                beta = beta_t;
                                store_ray(R.ray, id, ot, wit, PB_INF, time);
                                if (TEX && has_diff) store_diff(R.rdiff, id, specular_differentials(si, sx, rdf, si.wo, wit, bsdf.eta, true));
                                depth += 1;
                                push_next = true; pop = false;
                            }
                        }
                    }
                }
            }
            if (pop) {
                // this `li` has returned: resume the innermost pending specular_transmit
                while (sp > 0 && !push_next) {
                    sp -= 1;
                    const size_t fi = (size_t)id * D + sp;
                    float4 a = R.rec.st_ray[2 * fi], b = R.rec.st_ray[2 * fi + 1], w = R.rec.st_beta[fi];
                    const uint32_t wbits = __float_as_uint(w.w);
                    size_t fsel = fi;
                    if (TEX && (wbits & PB_ST_TWO_LOBES)) {
                        const float2 u2 = smp.get_2d(R);
                        if (floorf(u2.x * 2.0f) >= 1.0f) {
                            fsel = fi + (size_t)R.capacity * D;
                            a = R.rec.st_ray[2 * fsel]; b = R.rec.st_ray[2 * fsel + 1];
                            const float4 w2 = R.rec.st_beta[fsel];
                            w.x = w2.x; w.y = w2.y; w.z = w2.z;
                        }
                    } else smp.skip_2d(R);
                    if (a.w != 0.0f) {
                        R.ray[2 * id] = make_float4(a.x, a.y, a.z, PB_INF);
                        R.ray[2 * id + 1] = b;
                        beta = rgb(w.x, w.y, w.z);
                        depth = __float_as_uint(w.w) & 0xffffu;
                        has_diff = TEX && (__float_as_uint(w.w) & PB_ST_HAS_DIFF) != 0u;
                        if (has_diff) { R.rdiff[3 * (size_t)id] = R.rec.st_diff[3 * fsel]; R.rdiff[3 * (size_t)id + 1] = R.rec.st_diff[3 * fsel + 1]; R.rdiff[3 * (size_t)id + 2] = R.rec.st_diff[3 * fsel + 2]; }
                        push_next = true;
                    }
                }
                if (!push_next) push_dead = true;
            }
            if (!is_black(Ladd)) rec_atomic_add(R.L_eta, id, Ladd);
            R.beta_st[id] = make_float4(beta.r, beta.g, beta.b, __uint_as_float(depth | (has_diff ? PB_ST_HAS_DIFF : 0u)));
            smp.end(R, id);
            R.rec.sp[id] = sp;
        }
        queue_push(q_next, &R.cnt->n_next, id, push_next);
        queue_push(R.q_dead[parity], &R.cnt->n_dead, id, push_dead);
    }
}

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
}  // namespace pb
