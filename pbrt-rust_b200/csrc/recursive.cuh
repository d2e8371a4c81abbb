// WhittedIntegrator::li (src/integrators/whitted.rs:52-105) and DirectLightingIntegrator::li
// (src/integrators/directlighting.rs:78-119) as wavefront kernels on the PathIntegrator's queues.
// Included by render.cu after the path kernels; everything it calls (surface_at_hit, material_bsdf, light_sample_li,
// trace_queue, film, k_finish_regen) is the path integrator's.
//
// Both integrators recurse: `li` calls `specular_reflect` and then `specular_transmit` (integrator.rs:409-520), each of
// which draws a 2D sample and may call `li` again one level deeper.  A Sobol' / Halton sampler hands out dimensions in
// call order, so the numbers a radiance evaluation sees depend on everything evaluated before it for the same camera
// sample.  The recursion is therefore run depth-first per camera sample, one ray at a time: a path slot owns a small
// stack of pending `specular_transmit` calls (ray and weight are fixed when the parent surface is shaded -- a specular
// lobe ignores its 2D sample -- but the sample's two dimensions are only consumed when the frame is popped, which is
// when the reference draws them).  Radiance is linear in the recursion, so each frame carries the product of the
// f * |cos| / pdf factors above it and adds straight into the camera sample's L.
//
// Direct lighting produces up to `entries_per_slot` shadow rays (and MIS rays) per shaded surface; they go to global
// entry arrays {ray, weight, slot} appended with one atomic each, are traced by the any-hit / closest-hit queue
// kernels, and add into L with float atomics (several entries of one slot can finish at the same time).
#pragma once

namespace pb {

PB_D void rec_atomic_add(float4* L, uint32_t slot, rgb v) {
    float* p = reinterpret_cast<float*>(L + slot);
    if (v.r != 0.0f) atomicAdd(p, v.r);
    if (v.g != 0.0f) atomicAdd(p + 1, v.g);
    if (v.b != 0.0f) atomicAdd(p + 2, v.b);
}

// GlobalSampler::get_1d / get_2d with the sample-array dimensions skipped (sampler.rs:322-353)
PB_D float rec_get_1d(const RenderDev& R, SampleCursor& c) {
    const uint32_t end = 5u + 2u * R.rec.n_arrays;
    if (c.dim >= 5u && c.dim < end) c.dim = end;
    float r = c.dim < 1024u || R.sampler.kind != PBRT_B200_SAMPLER_SOBOL ? sample_dimension(R.sampler, c, c.dim) : 0.5f;
    c.dim += 1;
    return r;
}
PB_D void rec_skip_2d(const RenderDev& R, SampleCursor& c) {
    const uint32_t end = 5u + 2u * R.rec.n_arrays;
    if (c.dim + 1u >= 5u && c.dim < end) c.dim = end;
}
PB_D float2 rec_get_2d(const RenderDev& R, SampleCursor& c) {
    rec_skip_2d(R, c);
    const bool ok = c.dim + 1u < 1024u || R.sampler.kind != PBRT_B200_SAMPLER_SOBOL;
    float y = ok ? sample_dimension(R.sampler, c, c.dim + 1) : 0.5f;
    float x = ok ? sample_dimension(R.sampler, c, c.dim) : 0.5f;
    c.dim += 2;
    return make_float2(x, y);
}
// Sampler::get_2d_array(1) (sampler.rs:149-166): array `arr` of a global sampler lives in dimensions 5+2*arr, 5+2*arr+1
// and its element for pixel sample s is that sample's own index (one element per sample).
PB_D bool rec_get_2d_array(const RenderDev& R, const SampleCursor& c, uint32_t& arr, float2* out) {
    if (arr == R.rec.n_arrays) return false;
    const uint32_t dim = 5u + 2u * arr;
    float y = sample_dimension(R.sampler, c, dim + 1);
    float x = sample_dimension(R.sampler, c, dim);
    *out = make_float2(x, y);
    arr += 1;
    return true;
}
// element k of an n-element array (a light asking for n samples): the array holds n * spp points, point j is evaluated at
// get_index_for_sample(j) (global_start_pixel!, sampler.rs:268-303), and pixel sample s reads j = s * n + k
PB_D float2 rec_array_element(const RenderDev& R, const SampleCursor& c, uint32_t arr_index, uint32_t sample_num, uint32_t n, uint32_t k) {
    SampleCursor e = c;
    const unsigned long long j = (unsigned long long)sample_num * n + k;
    e.index = R.sampler.kind == PBRT_B200_SAMPLER_SOBOL
                  ? sobol_interval_to_index(R.sampler, (uint32_t)R.sampler.log2_resolution, j, c.px - R.sampler.sb[0], c.py - R.sampler.sb[1])
                  : halton_index(R.sampler, j, c.px, c.py);
    const uint32_t dim = 5u + 2u * arr_index;
    float y = sample_dimension(R.sampler, e, dim + 1);
    float x = sample_dimension(R.sampler, e, dim);
    return make_float2(x, y);
}

// The sampler as the recursion sees it: get_1d / get_2d / get_2d_array(1).  ZT = false: the global samplers above
// (state = cursor + array offset in registers, written back by end()); ZT = true: the tile's (0,2)-sequence state in HBM
// (PixelSampler: arrays are extra rows of the tile's 2D table, filled by start_pixel).
template <bool ZT> struct RecSampler;
template <> struct RecSampler<false> {
    SampleCursor c; uint32_t arr;
    PB_D void begin(const RenderDev& R, uint32_t id) {
        c.index = R.s_index[id]; c.dim = R.s_dim[id];
        const uint32_t pxy = R.pixel[id];
        c.px = (int)(pxy & 0xffffu) + R.sampler.sb[0]; c.py = (int)(pxy >> 16) + R.sampler.sb[1];
        arr = R.rec.arr[id];
    }
    PB_D float get_1d(const RenderDev& R) { return rec_get_1d(R, c); }
    PB_D float2 get_2d(const RenderDev& R) { return rec_get_2d(R, c); }
    PB_D void skip_2d(const RenderDev& R) { rec_skip_2d(R, c); c.dim += 2; }  // a get_2d whose value nobody looks at
    PB_D bool get_2d_array(const RenderDev& R, float2* out) { return rec_get_2d_array(R, c, arr, out); }
    PB_D float2 array_element(const RenderDev& R, uint32_t a, uint32_t sn, uint32_t n, uint32_t k) { return rec_array_element(R, c, a, sn, n, k); }
    PB_D void end(const RenderDev& R, uint32_t id) { R.s_dim[id] = c.dim; R.rec.arr[id] = arr; }
};
template <> struct RecSampler<true> {
    ZtCursor z; uint32_t arr;
    PB_D void begin(const RenderDev& R, uint32_t id) { z = zt_cursor(R, id); arr = R.rec.arr[id]; }  // slot == tile ordinal
    PB_D float get_1d(const RenderDev&) { return pb::get_1d(z); }
    PB_D float2 get_2d(const RenderDev&) { return pb::get_2d(z); }
    PB_D void skip_2d(const RenderDev&) { (void)pb::get_2d(z); }  // the draw happens (table row or two RNG numbers)
    PB_D float2 array_element(const RenderDev&, uint32_t, uint32_t, uint32_t, uint32_t) { return make_float2(0.5f, 0.5f); }  // multi-sample arrays: global samplers only
    PB_D bool get_2d_array(const RenderDev& R, float2* out) {
        if (arr == R.rec.n_arrays) return false;
        *out = z.s2d[(size_t)(z.ndims + arr) * z.spp + z.t->sample_idx];
        arr += 1;
        return true;
    }
    PB_D void end(const RenderDev& R, uint32_t id) { R.rec.arr[id] = arr; }
};

// estimate_direct (integrator.rs:109-237, handle_media = false, specular = false): the light-sampled half becomes a
// shadow entry, the BSDF-sampled half a MIS entry; `scale` = 1 / (light selection pdf).
template <bool INST, int KM = KM_ALL, class B>
PB_D void rec_estimate_direct(const RenderDev& R, uint32_t id, const Surf& si, const B& bsdf, uint32_t ln, float2 ulight, float2 uscatt, rgb beta,
                              float inv_selpdf, float time) {
    const int NONSPEC = BX_ALL & ~BX_SPECULAR;
    const pbrt_b200_light& light = R.scene.lights[ln];
    const bool delta = is_delta_light(light);
    LightSample ls;
    light_sample_li<INST>(R, ln, si.p, ulight, ls, si.p_error, si.n);
    float scattpdf = 0.0f;
    if (ls.pdf > 0.0f && !is_black(ls.Li)) {
        rgb f = bsdf_f<KM>(bsdf, si.wo, ls.wi, NONSPEC) * absdot(ls.wi, si.sh_n);
        scattpdf = bsdf_pdf<KM>(bsdf, si.wo, ls.wi, NONSPEC);
        if (!is_black(f)) {
            f3 o = offset_ray_origin(si.p, si.p_error, si.n, ls.p1 - si.p);
            f3 tg = offset_ray_origin(ls.p1, ls.p1_err, ls.p1_n, o - ls.p1);
            rgb Ld = delta ? f * ls.Li / ls.pdf : f * ls.Li * power_heuristic(ls.pdf, scattpdf) / ls.pdf;
            rgb add = beta * (Ld * inv_selpdf);
            uint32_t e = atomicAdd(&R.cnt->n_shadow, 1u);
            store_ray(R.rec.e_sh_ray, e, o, tg - o, 1.0f - PB_SHADOW_EPSILON, time);
            R.rec.e_sh_contrib[e] = make_float4(add.r, add.g, add.b, __uint_as_float(id));
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
                rgb fac = beta * (f * weight / scattpdf * inv_selpdf);
                uint32_t e = atomicAdd(&R.cnt->n_mis, 1u);
                store_ray(R.rec.e_mis_ray, e, o, wi, PB_INF, time);
                R.rec.e_mis_contrib[e] = make_float4(fac.r, fac.g, fac.b, __uint_as_float(ln));
                R.rec.e_mis_slot[e] = id;
            }
        }
    }
}

// One step of the depth-first recursion for every live camera sample: shade the hit of its current ray.
#if PB_SHADE_TU
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

#endif  // PB_SHADE_TU

#if PB_EXACT_TU
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

#endif  // PB_EXACT_TU

}  // namespace pb
