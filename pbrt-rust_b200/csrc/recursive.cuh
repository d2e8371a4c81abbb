// WhittedIntegrator::li (src/integrators/whitted.rs:52-105) and DirectLightingIntegrator::li
// (src/integrators/directlighting.rs:78-119) as wavefront kernels on the PathIntegrator's queues.
// The kernels are k_rec_shade (shade.cu) and k_rec_shadow / k_rec_mis (render.cu); this header holds the device code they share.
// Everything else they use (surface_at_hit, material_bsdf, light_sample_li, trace_queue, film, k_finish_regen) is the path integrator's.
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
#include "path.cuh"

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


}  // namespace pb
