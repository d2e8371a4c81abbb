// BDPTIntegrator (src/integrators/bdpt.rs, a port of pbrt-v3's integrators/bdpt.cpp) on the device: k_bdpt, one thread per camera sample.
// A sample builds its camera subpath, then its light subpath (RandomWalk without Russian roulette), then evaluates every (s, t)
// connection with its visibility walk and the balance-heuristic MISWeight; L goes to the film, the t = 1 strategies to the splat film.
// Compiled with the exact-arithmetic flags of render.cu / mega.cu.  The CPU oracle is oracle/oracle_bdpt.hpp; DESIGN.md §4f.
//
// Subpath vertices live in per-slot scratch in device memory (BVert).  A surface vertex keeps its hit record, and the BSDF is rebuilt
// from it wherever a connection needs it (surface_at_hit / surface_full + material_bsdf / material_bsdf_tex are pure functions of the
// record and, for the camera subpath's first hit, of the camera ray's differentials, which stay in the slot's R.rdiff entry).
// FULL: the full-featured family (instances, sphere area lights, textured materials), chosen per scene as for the other kernels.
#include <type_traits>
#include "path.cuh"

namespace pb {

enum { BV_CAMERA = 0, BV_LIGHT = 1, BV_SURFACE = 2 };

struct BVert {
    f3 p, p_err, n, ns;     // n = 0: not on a surface
    rgb beta;
    float pdf_fwd, pdf_rev, time;
    uint32_t type, delta;
    uint32_t diff;          // BV_SURFACE: 1 = found by the camera ray, whose differentials (R.rdiff) filter its textures
    int light;              // BV_LIGHT: the light, -1 = the escaped camera ray's endpoint
    uint32_t slot, inst;    // BV_SURFACE: the hit record ...
    float t, b0, b1, b2;
    f3 ro, rd;              // ... and the ray that found it
};

PB_D bool bv_on_surface(const BVert& v) { return !(v.n.x == 0.0f && v.n.y == 0.0f && v.n.z == 0.0f); }

struct BdptCtx {
    const RenderDev& R;
    const BdptCam& C;
    const float* ld_func;
    const float* ld_cdf;
    float ld_func_int;
    unsigned long long* n_closest;
    LocalStack stack;
    uint32_t slot;
};
template <bool FULL> using BsdfT = typename std::conditional<FULL, BsdfX, Bsdf>::type;

// a surface vertex's interaction and BSDF, rebuilt from its hit record
template <bool INST>
PB_D void bv_bsdf(const BdptCtx& c, const BVert& v, Surf* si, BsdfT<INST>* b) {
    uint32_t fl;
    b->valid = false; b->n = 0;
    const int m = c.R.scene.prims[v.slot].material;
    if (INST && m >= 0 && c.R.scene.materials[m].textured) {  // as shade_path's Q_TEX bin
        SurfX sx;
        surface_full(c.R.scene.self_dev, v.inst, v.slot, v.ro, v.rd, v.t, v.b0, v.b1, v.b2, si, &sx, &fl);
        const RayDiff rdf = load_diff(c.R.rdiff, c.slot, c.R.rdiff != nullptr && v.diff != 0u);
        material_bsdf_tex<true>(c.R.scene.self_dev, m, si, &sx, &rdf, b);
        return;
    }
    *si = surface_at_hit<INST>(c.R.scene, v.inst, v.slot, v.ro, v.rd, v.t, v.b0, v.b1, v.b2, &fl);
    if (m >= 0) material_bsdf<-1, true>(c.R.scene.materials[m], *si, *b);
}

PB_D bool bv_infinite_light(const BdptCtx& c, const BVert& v) {
    if (v.type != BV_LIGHT) return false;
    if (v.light < 0) return true;
    const uint32_t t = c.R.scene.lights[v.light].type;
    return t == PBRT_B200_LIGHT_INFINITE || t == PBRT_B200_LIGHT_DISTANT;
}
PB_D int bv_area_light(const BdptCtx& c, const BVert& v) { return v.type == BV_SURFACE ? c.R.scene.prims[v.slot].area_light : -1; }
PB_D bool bv_is_light(const BdptCtx& c, const BVert& v) { return v.type == BV_LIGHT || bv_area_light(c, v) >= 0; }
PB_D bool bv_delta_light(const BdptCtx& c, const BVert& v) { return v.type == BV_LIGHT && v.light >= 0 && is_delta_light(c.R.scene.lights[v.light]); }
template <bool INST>
PB_D bool bv_connectible(const BdptCtx& c, const BVert& v) {
    if (v.type == BV_CAMERA) return true;
    if (v.type == BV_LIGHT) return v.light < 0 || c.R.scene.lights[v.light].type != PBRT_B200_LIGHT_DISTANT;
    Surf si; BsdfT<INST> b;
    bv_bsdf<INST>(c, v, &si, &b);
    return bsdf_count(b, BX_DIFFUSE | BX_GLOSSY | BX_REFLECTION | BX_TRANSMISSION) > 0;
}

// TransportMode::Importance: the shared lobes apply the Radiance (etai/etat)^2 scale to specular and microfacet transmission
template <class B>
PB_D float importance_scale(const B& b, f3 wo, bool trans) {
    if (!trans || b.eta == 1.0f) return 1.0f;
    const float e = to_local(b, wo).z > 0.0f ? b.eta : 1.0f / b.eta;
    return e * e;
}
PB_D float correct_shading_normal(const Surf& si, f3 wo, f3 wi, bool importance) {  // pbrt-v3 bdpt.cpp:48-59
    if (!importance) return 1.0f;
    const float num = absdot(wo, si.sh_n) * absdot(wi, si.n), den = absdot(wo, si.n) * absdot(wi, si.sh_n);
    if (den == 0.0f) return 0.0f;
    return num / den;
}
template <bool INST>
PB_D rgb bv_f(const BdptCtx& c, const BVert& v, const BVert& next, bool importance) {
    f3 wi = next.p - v.p;
    if (len2(wi) == 0.0f) return rgb(0.0f);
    wi = normalize(wi);
    if (v.type != BV_SURFACE) return rgb(0.0f);
    Surf si; BsdfT<INST> b;
    bv_bsdf<INST>(c, v, &si, &b);
    const f3 wo = si.wo;
    rgb f = bsdf_f<INST ? KM_TEX : KM_ALL>(b, wo, wi, BX_ALL);
    if (importance) f = f * rgb(importance_scale(b, wo, !(dot(wi, b.ng) * dot(wo, b.ng) > 0.0f)));
    return f * rgb(correct_shading_normal(si, wo, wi, importance));
}
PB_D float bv_convert_density(const BdptCtx& c, const BVert& v, float pdf, const BVert& next) {
    if (bv_infinite_light(c, next)) return pdf;
    const f3 w = next.p - v.p;
    if (len2(w) == 0.0f) return 0.0f;
    const float inv_d2 = 1.0f / len2(w);
    if (bv_on_surface(next)) pdf *= absdot(next.n, w * sqrtf(inv_d2));
    return pdf * inv_d2;
}

// ---- Light::sample_le / pdf_le (pbrt-v3 lights/*.cpp)
// Sphere::sample (shapes/sphere.rs:295-311): a uniform point on a full sphere, pdf 1 / area.  Out of line, as sphere_light_sample.
static __device__ __noinline__ void sphere_sample_area(const DevScene* sp, uint32_t li, float ux, float uy, SphereLightSample* out) {
    const DevScene& s = *sp;
    const pbrt_b200_light& l = s.lights[li];
    const pbrt_b200_sphere& sph = s.spheres[l.shape_index];
    const float z = 1.0f - 2.0f * ux, rr = sqrtf(fmaxf(1.0f - z * z, 0.0f)), phi = 2.0f * PB_PI * uy;
    f3 pobj = f3(rr * cosf(phi), rr * sinf(phi), z) * sph.radius;
    f3 n = normalize(xf_normal(sph.world_to_object, pobj));
    if (l.shape_flags & PBRT_B200_PRIM_REVERSE_ORIENTATION) n = n * -1.0f;
    pobj = pobj * (sph.radius / len(pobj));
    const f3 pe = vabs(pobj) * gamma_n(5);
    out->p = xf_point_abs_err(sph.object_to_world, pobj, pe, &out->p_err);
    out->n = n;
    out->pdf = 1.0f / l.area;
}
PB_D f3 uniform_sphere(float2 u) {
    const float z = 1.0f - 2.0f * u.x, r = sqrtf(fmaxf(1.0f - z * z, 0.0f)), phi = 2.0f * PB_PI * u.y;
    return f3(r * cosf(phi), r * sinf(phi), z);
}
struct LeSample { rgb Le; f3 o, d, n; float pdf_pos, pdf_dir; };
template <bool INST>
PB_D void light_sample_le(const BdptCtx& c, int li, float2 u1, float2 u2, LeSample& r) {
    const RenderDev& R = c.R;
    const pbrt_b200_light& l = R.scene.lights[li];
    const rgb L = rgb3(l.L);
    r.pdf_pos = 0.0f; r.pdf_dir = 0.0f; r.Le = rgb(0.0f);
    switch (l.type) {
        case PBRT_B200_LIGHT_POINT:
            r.o = f3(l.pos[0], l.pos[1], l.pos[2]); r.d = uniform_sphere(u1); r.n = r.d;
            r.pdf_pos = 1.0f; r.pdf_dir = 1.0f / (4.0f * PB_PI); r.Le = L;
            break;
        case PBRT_B200_LIGHT_SPOT: {
            const float ct = (1.0f - u1.x) + u1.x * l.cos_total_width, st = sqrtf(1.0f - ct * ct), phi = u1.y * 2.0f * PB_PI;
            r.o = f3(l.pos[0], l.pos[1], l.pos[2]);
            r.d = xf_vector(c.C.spot_l2w + 16 * li, f3(cosf(phi) * st, sinf(phi) * st, ct)); r.n = r.d;
            r.pdf_pos = 1.0f; r.pdf_dir = 1.0f / (2.0f * PB_PI * (1.0f - l.cos_total_width));
            const f3 wl = normalize(xf_vector(l.world_to_light, r.d));
            float fall;
            if (wl.z < l.cos_total_width) fall = 0.0f;
            else if (wl.z >= l.cos_falloff_start) fall = 1.0f;
            else { const float dl = (wl.z - l.cos_total_width) / (l.cos_falloff_start - l.cos_total_width); fall = (dl * dl) * (dl * dl); }
            r.Le = L * rgb(fall);
            break;
        }
        case PBRT_B200_LIGHT_DISTANT: {
            f3 w(l.dir[0], l.dir[1], l.dir[2]), v1, v2;
            coordinate_system(w, &v1, &v2);
            const float2 cd = concentric_disk(u1);
            const f3 pdisk = f3(R.scene.world_center[0], R.scene.world_center[1], R.scene.world_center[2]) + (v1 * cd.x + v2 * cd.y) * R.scene.world_radius;
            r.o = pdisk + w * R.scene.world_radius; r.d = -w; r.n = r.d;
            r.pdf_pos = 1.0f / (PB_PI * R.scene.world_radius * R.scene.world_radius); r.pdf_dir = 1.0f; r.Le = L;
            break;
        }
        case PBRT_B200_LIGHT_DIFFUSE: {
            LightSample ls;
            if (INST && l.shape_kind == PBRT_B200_SHAPE_SPHERE) {
                SphereLightSample so;
                sphere_sample_area(R.scene.self_dev, (uint32_t)li, u1.x, u1.y, &so);
                ls.p1 = so.p; ls.p1_err = so.p_err; ls.p1_n = so.n;
            } else triangle_light_sample(R.scene, l, f3(0.f, 0.f, 0.f), u1, ls);
            r.pdf_pos = 1.0f / l.area;
            f3 w;
            if (l.two_sided) {
                float2 u = u2;
                if (u.x < 0.5f) { u.x = fminf(u.x * 2.0f, PB_ONE_MINUS_EPSILON); w = cosine_hemisphere(u); }
                else { u.x = fminf((u.x - 0.5f) * 2.0f, PB_ONE_MINUS_EPSILON); w = cosine_hemisphere(u); w.z *= -1.0f; }
                r.pdf_dir = 0.5f * fabsf(w.z) * PB_INV_PI;
            } else {
                w = cosine_hemisphere(u2);
                r.pdf_dir = w.z * PB_INV_PI;
            }
            f3 v1, v2;
            const f3 n = ls.p1_n;
            coordinate_system(n, &v1, &v2);
            w = v1 * w.x + v2 * w.y + n * w.z;
            r.o = offset_ray_origin(ls.p1, ls.p1_err, n, w); r.d = w; r.n = n;
            r.Le = (l.two_sided || dot(n, w) > 0.0f) ? L : rgb(0.0f);
            break;
        }
        default: {  // constant infinite light
            const InfDistrib& D = R.inf_distrib[li];
            float pm, pc;
            int v, dummy;
            const float d1 = tiny_sample_continuous(D.marg, u1.y, &pm, &v);
            const float d0 = tiny_sample_continuous(D.cond[v], u1.x, &pc, &dummy);
            const float map_pdf = pc * pm;
            if (map_pdf == 0.0f) return;
            const float theta = d1 * PB_PI, phi = d0 * 2.0f * PB_PI;
            const float ct = cosf(theta), st = sinf(theta), sp = sinf(phi), cp = cosf(phi);
            const f3 d = -f3(st * cp, st * sp, ct);
            f3 v1, v2;
            coordinate_system(-d, &v1, &v2);
            const float2 cd = concentric_disk(u2);
            const f3 pdisk = f3(R.scene.world_center[0], R.scene.world_center[1], R.scene.world_center[2]) + (v1 * cd.x + v2 * cd.y) * R.scene.world_radius;
            r.o = pdisk + (-d) * R.scene.world_radius; r.d = d; r.n = d;
            r.pdf_dir = st == 0.0f ? 0.0f : map_pdf / (2.0f * PB_PI * PB_PI * st);
            r.pdf_pos = 1.0f / (PB_PI * R.scene.world_radius * R.scene.world_radius);
            r.Le = L;
            break;
        }
    }
}
PB_D void light_pdf_le(const BdptCtx& c, int li, f3 d, f3 n, float* pdf_pos, float* pdf_dir) {
    const RenderDev& R = c.R;
    const pbrt_b200_light& l = R.scene.lights[li];
    switch (l.type) {
        case PBRT_B200_LIGHT_POINT: *pdf_pos = 0.0f; *pdf_dir = 1.0f / (4.0f * PB_PI); break;
        case PBRT_B200_LIGHT_SPOT: {
            *pdf_pos = 0.0f;
            const f3 wl = xf_vector(l.world_to_light, d);
            *pdf_dir = wl.z >= l.cos_total_width ? 1.0f / (2.0f * PB_PI * (1.0f - l.cos_total_width)) : 0.0f;
            break;
        }
        case PBRT_B200_LIGHT_DISTANT: *pdf_pos = 1.0f / (PB_PI * R.scene.world_radius * R.scene.world_radius); *pdf_dir = 0.0f; break;
        case PBRT_B200_LIGHT_DIFFUSE:
            *pdf_pos = 1.0f / l.area;
            *pdf_dir = l.two_sided ? 0.5f * absdot(n, d) * PB_INV_PI : dot(n, d) * PB_INV_PI;
            break;
        default: {
            Surf ref;
            ref.p = f3(0.f, 0.f, 0.f); ref.p_error = ref.p; ref.n = ref.p;
            *pdf_dir = light_pdf_li(R, (uint32_t)li, ref, -d);
            *pdf_pos = 1.0f / (PB_PI * R.scene.world_radius * R.scene.world_radius);
            break;
        }
    }
}
PB_D float infinite_light_density(const BdptCtx& c, f3 w) {
    float pdf = 0.0f;
    Surf ref;
    ref.p = f3(0.f, 0.f, 0.f); ref.p_error = ref.p; ref.n = ref.p;
    for (uint32_t k = 0; k < c.R.n_infinite; ++k) {
        const uint32_t li = c.R.infinite_lights[k];
        pdf += light_pdf_li(c.R, li, ref, -w) * c.ld_func[li];
    }
    return pdf / (c.ld_func_int * (float)c.R.n_lights);
}
PB_D float bv_pdf_light(const BdptCtx& c, const BVert& v, const BVert& next) {
    f3 w = next.p - v.p;
    const float inv_d2 = 1.0f / len2(w);
    w = w * sqrtf(inv_d2);
    float pdf;
    if (bv_infinite_light(c, v)) pdf = 1.0f / (PB_PI * c.R.scene.world_radius * c.R.scene.world_radius);
    else {
        float pp, pd;
        light_pdf_le(c, v.type == BV_LIGHT ? v.light : bv_area_light(c, v), w, v.n, &pp, &pd);
        pdf = pd * inv_d2;
    }
    if (bv_on_surface(next)) pdf *= absdot(next.n, w);
    return pdf;
}
PB_D float bv_pdf_light_origin(const BdptCtx& c, const BVert& v, const BVert& next) {
    f3 w = next.p - v.p;
    if (len2(w) == 0.0f) return 0.0f;
    w = normalize(w);
    if (bv_infinite_light(c, v)) return infinite_light_density(c, w);
    const int li = v.type == BV_LIGHT ? v.light : bv_area_light(c, v);
    float pp, pd;
    light_pdf_le(c, li, w, v.n, &pp, &pd);
    return pp * (c.ld_func[li] / (c.ld_func_int * (float)c.R.n_lights));
}

// PerspectiveCamera::we / pdf_we (pbrt-v3 cameras/perspective.cpp:150-215)
PB_D bool cam_raster(const BdptCam& C, f3 o, f3 d, float2* pr, float* ct) {
    *ct = dot(d, C.fwd);
    if (*ct <= 0.0f) return false;
    const f3 pfocus = o + d * ((C.lens_radius > 0.0f ? C.focal_distance : 1.0f) / *ct);
    const f3 p = xf_point(C.c2r, xf_point(C.w2c, pfocus));
    *pr = make_float2(p.x, p.y);
    return !(p.x < (float)C.sb[0] || p.x >= (float)C.sb[2] || p.y < (float)C.sb[1] || p.y >= (float)C.sb[3]);
}
PB_D float cam_lens_area(const BdptCam& C) { return C.lens_radius != 0.0f ? PB_PI * C.lens_radius * C.lens_radius : 1.0f; }
PB_D void cam_pdf_we(const BdptCam& C, f3 o, f3 d, float* pdf_pos, float* pdf_dir) {
    float ct; float2 pr;
    if (!cam_raster(C, o, d, &pr, &ct)) { *pdf_pos = 0.0f; *pdf_dir = 0.0f; return; }
    *pdf_pos = 1.0f / cam_lens_area(C);
    *pdf_dir = 1.0f / (C.A * ct * ct * ct);
}

template <bool INST>
PB_D float bv_pdf(const BdptCtx& c, const BVert& v, const BVert* prev, const BVert& next) {
    if (v.type == BV_LIGHT) return bv_pdf_light(c, v, next);
    f3 wn = next.p - v.p;
    if (len2(wn) == 0.0f) return 0.0f;
    wn = normalize(wn);
    float pdf = 0.0f;
    if (v.type == BV_CAMERA) { float pp; cam_pdf_we(c.C, v.p, wn, &pp, &pdf); }
    else {
        Surf si; BsdfT<INST> b;
        bv_bsdf<INST>(c, v, &si, &b);
        pdf = bsdf_pdf<INST ? KM_TEX : KM_ALL>(b, normalize(prev->p - v.p), wn, BX_ALL);
    }
    return bv_convert_density(c, v, pdf, next);
}
PB_D rgb bv_le(const BdptCtx& c, const BVert& v, const BVert& to) {
    if (!bv_is_light(c, v)) return rgb(0.0f);
    f3 w = to.p - v.p;
    if (len2(w) == 0.0f) return rgb(0.0f);
    w = normalize(w);
    if (bv_infinite_light(c, v)) {
        rgb Le(0.0f);
        for (uint32_t k = 0; k < c.R.n_infinite; ++k) Le = Le + rgb3(c.R.scene.lights[c.R.infinite_lights[k]].L);
        return Le;
    }
    const pbrt_b200_light& l = c.R.scene.lights[bv_area_light(c, v)];
    return (l.two_sided || dot(v.n, w) > 0.0f) ? rgb3(l.L) : rgb(0.0f);
}

// VisibilityTester::tr without media (light.rs:125-150): closest hits through material-less surfaces
template <bool INST>
PB_D bool unoccluded(BdptCtx& c, f3 ap, f3 aerr, f3 an, f3 bp, f3 berr, f3 bn) {
    f3 o = offset_ray_origin(ap, aerr, an, bp - ap);
    f3 tg = offset_ray_origin(bp, berr, bn, o - bp);
    f3 d = tg - o;
    for (uint32_t seg = 0; seg < 4096u; ++seg) {
        TravRay r;
        trav_init(c.R.scene, r, o, d, 1.0f - PB_SHADOW_EPSILON);
        trav_run<false, INST>(c.R.scene, r, c.stack, 0);
        *c.n_closest += 1;
        if (!r.found) return true;
        if (c.R.scene.prims[r.hit.slot].material >= 0) return false;
        uint32_t fl;
        const Surf si = surface_at_hit<INST>(c.R.scene, r.hit.inst, r.hit.slot, o, d, r.hit.t, r.hit.b0, r.hit.b1, r.hit.b2, &fl);
        o = offset_ray_origin(si.p, si.p_error, si.n, bp - si.p);
        tg = offset_ray_origin(bp, berr, bn, o - bp);
        d = tg - o;
    }
    return false;
}

// RandomWalk (pbrt-v3 bdpt.cpp:191-269) without media
template <bool INST>
PB_D int random_walk(BdptCtx& c, DirectSampler& smp, f3 ro, f3 rd, float time, rgb beta, float pdf, int max_depth, bool importance, BVert* path) {
    if (max_depth == 0) return 0;
    int bounces = 0;
    float pdf_fwd = pdf, pdf_rev = 0.0f;
    uint32_t diff = importance ? 0u : 1u;  // the camera ray carries differentials; spawned rays do not (interaction.rs:32-37)
    for (uint32_t guard = 0; guard < 65536u; ++guard) {
        TravRay r;
        trav_init(c.R.scene, r, ro, rd, PB_INF);
        trav_run<false, INST>(c.R.scene, r, c.stack, 0);
        *c.n_closest += 1;
        if (is_black(beta)) break;
        BVert& v = path[bounces];
        BVert& prev = path[bounces - 1];
        if (!r.found) {
            if (!importance) {
                v.type = BV_LIGHT; v.delta = 0; v.diff = 0; v.light = -1; v.beta = beta; v.pdf_fwd = pdf_fwd; v.pdf_rev = 0.0f;
                v.p = ro + rd; v.n = -rd; v.ns = v.n; v.p_err = f3(0.f, 0.f, 0.f); v.time = time;
                ++bounces;
            }
            break;
        }
        v.type = BV_SURFACE; v.delta = 0; v.diff = diff; v.light = -1; v.beta = beta; v.pdf_rev = 0.0f; v.time = time;
        v.slot = r.hit.slot; v.inst = r.hit.inst; v.t = r.hit.t; v.b0 = r.hit.b0; v.b1 = r.hit.b1; v.b2 = r.hit.b2; v.ro = ro; v.rd = rd;
        Surf si; BsdfT<INST> b;
        bv_bsdf<INST>(c, v, &si, &b);
        diff = 0u;
        if (!b.valid) { ro = offset_ray_origin(si.p, si.p_error, si.n, rd); continue; }
        v.p = si.p; v.p_err = si.p_error; v.n = si.n; v.ns = si.sh_n;
        v.pdf_fwd = bv_convert_density(c, prev, pdf_fwd, v);
        if (++bounces >= max_depth) break;
        const f3 wo = si.wo;
        f3 wi(0.f, 0.f, 0.f);
        int type = 0;
        pdf_fwd = 0.0f;
        rgb f = bsdf_sample<INST ? KM_TEX : KM_ALL>(b, wo, &wi, smp.get_2d(), &pdf_fwd, BX_ALL, &type);
        if (is_black(f) || pdf_fwd == 0.0f) break;
        if (importance) f = f * rgb(importance_scale(b, wo, (type & BX_SPECULAR) ? (type & BX_TRANSMISSION) != 0 : !(dot(wi, b.ng) * dot(wo, b.ng) > 0.0f)));
        beta = beta * (f * absdot(wi, si.sh_n) / pdf_fwd);
        pdf_rev = bsdf_pdf<INST ? KM_TEX : KM_ALL>(b, wi, wo, BX_ALL);
        if (type & BX_SPECULAR) { v.delta = 1; pdf_rev = pdf_fwd = 0.0f; }
        beta = beta * rgb(correct_shading_normal(si, wo, wi, importance));
        ro = offset_ray_origin(si.p, si.p_error, si.n, wi); rd = wi;
        prev.pdf_rev = bv_convert_density(c, v, pdf_rev, prev);
    }
    return bounces;
}

template <bool INST>
PB_D float mis_weight(const BdptCtx& c, BVert* lv, BVert* cv, const BVert& sampled, int s, int t) {
    if (s + t == 2) return 1.0f;
    BVert* qs = s > 0 ? &lv[s - 1] : nullptr;
    BVert* pt = t > 0 ? &cv[t - 1] : nullptr;
    BVert* qsm = s > 1 ? &lv[s - 2] : nullptr;
    BVert* ptm = t > 1 ? &cv[t - 2] : nullptr;
    // the scoped assignments of bdpt.cpp:433-460, undone on return
    BVert save_q, save_p;
    if (qs) save_q = *qs;
    if (pt) save_p = *pt;
    const float save_ptm = ptm ? ptm->pdf_rev : 0.0f, save_qsm = qsm ? qsm->pdf_rev : 0.0f;
    if (s == 1) *qs = sampled;
    else if (t == 1) *pt = sampled;
    if (pt) pt->delta = 0;
    if (qs) qs->delta = 0;
    if (pt) pt->pdf_rev = s > 0 ? bv_pdf<INST>(c, *qs, qsm, *pt) : bv_pdf_light_origin(c, *pt, *ptm);
    if (ptm) ptm->pdf_rev = s > 0 ? bv_pdf<INST>(c, *pt, qs, *ptm) : bv_pdf_light(c, *pt, *ptm);
    if (qs) qs->pdf_rev = bv_pdf<INST>(c, *pt, ptm, *qs);
    if (qsm) qsm->pdf_rev = bv_pdf<INST>(c, *qs, pt, *qsm);
    float sum = 0.0f, ri = 1.0f;
    for (int i = t - 1; i > 0; --i) {
        ri *= (cv[i].pdf_rev != 0.0f ? cv[i].pdf_rev : 1.0f) / (cv[i].pdf_fwd != 0.0f ? cv[i].pdf_fwd : 1.0f);
        if (!cv[i].delta && !cv[i - 1].delta) sum += ri;
    }
    ri = 1.0f;
    for (int i = s - 1; i >= 0; --i) {
        ri *= (lv[i].pdf_rev != 0.0f ? lv[i].pdf_rev : 1.0f) / (lv[i].pdf_fwd != 0.0f ? lv[i].pdf_fwd : 1.0f);
        const bool dl = i > 0 ? lv[i - 1].delta != 0 : bv_delta_light(c, lv[0]);
        if (!lv[i].delta && !dl) sum += ri;
    }
    if (qs) *qs = save_q;
    if (pt) *pt = save_p;
    if (ptm) ptm->pdf_rev = save_ptm;
    if (qsm) qsm->pdf_rev = save_qsm;
    return 1.0f / (1.0f + sum);
}

// ConnectBDPT (pbrt-v3 bdpt.cpp:462-560)
template <bool INST>
PB_D rgb connect(BdptCtx& c, DirectSampler& smp, BVert* lv, BVert* cv, int s, int t, float2* praster) {
    rgb L(0.0f);
    if (t > 1 && s != 0 && cv[t - 1].type == BV_LIGHT) return L;
    BVert sampled;
    sampled.type = BV_CAMERA; sampled.delta = 0; sampled.diff = 0; sampled.light = -1; sampled.pdf_fwd = 0.0f; sampled.pdf_rev = 0.0f;
    if (s == 0) {
        const BVert& pt = cv[t - 1];
        if (bv_is_light(c, pt)) L = bv_le(c, pt, cv[t - 2]) * pt.beta;
    } else if (t == 1) {
        const BVert& qs = lv[s - 1];
        if (bv_connectible<INST>(c, qs)) {
            const BdptCam& C = c.C;
            float2 pl = concentric_disk(smp.get_2d());
            pl.x *= C.lens_radius; pl.y *= C.lens_radius;
            const f3 plw = xf_point(C.c2w, f3(pl.x, pl.y, 0.0f));
            f3 wi = plw - qs.p;
            const float dist = len(wi);
            wi = f3(wi.x / dist, wi.y / dist, wi.z / dist);
            const float pdf = (dist * dist) / (absdot(C.n_lens, wi) * cam_lens_area(C));
            float We = 0.0f, ct;
            if (cam_raster(C, offset_ray_origin(plw, f3(0.f, 0.f, 0.f), C.n_lens, -wi), -wi, praster, &ct)) We = 1.0f / (C.A * cam_lens_area(C) * (ct * ct) * (ct * ct));
            if (pdf > 0.0f && We != 0.0f) {
                sampled.type = BV_CAMERA; sampled.beta = rgb(We / pdf); sampled.p = plw; sampled.p_err = f3(0.f, 0.f, 0.f);
                sampled.n = C.n_lens; sampled.ns = sampled.n; sampled.time = qs.time;
                L = qs.beta * bv_f<INST>(c, qs, sampled, true) * sampled.beta;
                if (bv_on_surface(qs)) L = L * rgb(absdot(wi, qs.ns));
                if (!is_black(L) && !unoccluded<INST>(c, qs.p, qs.p_err, qs.n, sampled.p, sampled.p_err, sampled.n)) L = rgb(0.0f);
            }
        }
    } else if (s == 1) {
        const BVert& pt = cv[t - 1];
        if (bv_connectible<INST>(c, pt)) {
            const float u = smp.get_1d();
            const uint32_t ln = find_interval_cdf(c.ld_cdf, (int)c.R.n_lights + 1, u);
            const float light_pdf = c.ld_func[ln] / (c.ld_func_int * (float)c.R.n_lights);
            LightSample ls;
            light_sample_li<INST>(c.R, ln, pt.p, smp.get_2d(), ls, pt.p_err, pt.n);
            if (ls.pdf > 0.0f && !is_black(ls.Li)) {
                sampled.type = BV_LIGHT; sampled.light = (int)ln; sampled.beta = ls.Li / rgb(ls.pdf * light_pdf);
                sampled.p = ls.p1; sampled.p_err = ls.p1_err; sampled.n = ls.p1_n; sampled.ns = sampled.n; sampled.time = pt.time;
                sampled.pdf_fwd = bv_pdf_light_origin(c, sampled, pt);
                L = pt.beta * bv_f<INST>(c, pt, sampled, false) * sampled.beta;
                if (bv_on_surface(pt)) L = L * rgb(absdot(ls.wi, pt.ns));
                if (!is_black(L) && !unoccluded<INST>(c, pt.p, pt.p_err, pt.n, ls.p1, ls.p1_err, ls.p1_n)) L = rgb(0.0f);
            }
        }
    } else {
        const BVert& qs = lv[s - 1];
        const BVert& pt = cv[t - 1];
        if (bv_connectible<INST>(c, qs) && bv_connectible<INST>(c, pt)) {
            L = qs.beta * bv_f<INST>(c, qs, pt, true) * bv_f<INST>(c, pt, qs, false) * pt.beta;
            if (!is_black(L)) {  // G (bdpt.cpp:170-180)
                f3 d = qs.p - pt.p;
                float g = 1.0f / len2(d);
                d = d * sqrtf(g);
                if (bv_on_surface(qs)) g *= absdot(qs.ns, d);
                if (bv_on_surface(pt)) g *= absdot(pt.ns, d);
                if (!unoccluded<INST>(c, qs.p, qs.p_err, qs.n, pt.p, pt.p_err, pt.n)) g = 0.0f;
                L = L * rgb(g);
            }
        }
    }
    if (is_black(L)) return L;
    return L * rgb(mis_weight<INST>(c, lv, cv, sampled, s, t));
}

// Film::add_splat (pbrt-v3 film.cpp:126-146) into the splat film, RGB per cropped pixel
PB_D void film_add_splat(const RenderDev& R, float* splat, float2 p, rgb v) {
    const float y = lum(v);
    if (v.r != v.r || v.g != v.g || v.b != v.b || y < 0.0f || isinf(y)) return;
    const float fx = floorf(p.x), fy = floorf(p.y);
    if (!(fx >= (float)R.crop[0] && fx < (float)R.crop[2] && fy >= (float)R.crop[1] && fy < (float)R.crop[3])) return;
    if (y > R.max_sample_luminance) v = v * rgb(R.max_sample_luminance / y);
    const size_t o = 3 * ((size_t)((int)fy - R.crop[1]) * (size_t)(R.crop[2] - R.crop[0]) + (size_t)((int)fx - R.crop[0]));
    atomicAdd(splat + o, v.r); atomicAdd(splat + o + 1, v.g); atomicAdd(splat + o + 2, v.b);
}

// One 512-thread CTA per SM (the §4e structure): a trip is one camera sample per thread, and the CTA's warps pass its phases -- camera
// subpath, light subpath, connections -- together, with barriers between them, so that the SM stays inside one region of the code.
template <bool INST>
__global__ void __launch_bounds__(PB_VOL_BLOCK) k_bdpt(RenderDev R, BdptCam C, BVert* verts, float* splat, unsigned long long total_items) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    const int max_depth = R.max_depth;
    BVert* cv = verts + (size_t)j * (size_t)(2 * max_depth + 3);
    BVert* lv = cv + (max_depth + 2);
    unsigned long long n_camera = 0, n_closest = 0;
    uint2 stack_mem[PB_STACK_SIZE(INST)];
    BdptCtx c{R, C, R.ld_func, R.ld_cdf, R.ld_func_int, &n_closest, LocalStack{stack_mem}, j};
    bool exhausted = false;
    for (;;) {
        bool have = false;
        {
            const bool need = !exhausted;
            const unsigned m = __ballot_sync(0xffffffffu, need);
            if (need) {
                const int leader = __ffs(m) - 1;
                unsigned long long base = 0;
                if ((int)lane == leader) base = atomicAdd(&R.cnt->item_cursor, (unsigned long long)__popc(m));
                base = __shfl_sync(m, base, leader);
                const unsigned long long item = base + (unsigned long long)__popc(m & ((1u << lane) - 1u));
                if (item >= total_items) exhausted = true;
                else have = gen_camera_path(R, item, j);
            }
        }
        if (!__syncthreads_or(have || !exhausted)) break;
        DirectSampler smp;
        float2 pfilm = make_float2(0.f, 0.f);
        int nc = 0, nl = 0;
        if (have) {  // camera subpath (GenerateCameraSubpath, bdpt.cpp:271-292)
            n_camera += 1;
            smp.prefetch(R, j);
            pfilm = R.pfilm[j];
            const float4 a = R.ray[2 * j], b = R.ray[2 * j + 1];
            const f3 ro(a.x, a.y, a.z), rd(b.x, b.y, b.z);
            BVert& v0 = cv[0];
            v0.type = BV_CAMERA; v0.delta = 0; v0.diff = 0; v0.light = -1; v0.beta = rgb(1.0f); v0.pdf_fwd = 0.0f; v0.pdf_rev = 0.0f;
            v0.p = ro; v0.p_err = f3(0.f, 0.f, 0.f); v0.n = v0.p_err; v0.ns = v0.p_err; v0.time = b.w;
            float pdf_pos, pdf_dir;
            cam_pdf_we(C, ro, rd, &pdf_pos, &pdf_dir);
            nc = random_walk<INST>(c, smp, ro, rd, b.w, rgb(1.0f), pdf_dir, max_depth + 1, false, cv + 1) + 1;
            c.ld_cdf = R.ld_cdf; c.ld_func = R.ld_func; c.ld_func_int = R.ld_func_int;
            if (R.sp.enabled) {  // SpatialLightDistribution looked up at the camera vertex
                const int sl = R.sp.slot[spatial_voxel(R, ro)];
                if (sl >= 0) { c.ld_cdf = R.sp.cdf + (size_t)sl * (R.n_lights + 1); c.ld_func = R.sp.func + (size_t)sl * R.n_lights; c.ld_func_int = R.sp.func_int[sl]; }
                else atomicExch(R.sp.counters + 2, 1u);  // cannot happen with the eager table; the host fails the call
            }
        }
        __syncthreads();
        if (have && R.n_lights > 0) {  // light subpath (GenerateLightSubpath, bdpt.cpp:294-316)
            const float u = smp.get_1d();
            const uint32_t ln = find_interval_cdf(c.ld_cdf, (int)R.n_lights + 1, u);
            const float light_pdf = c.ld_func[ln] / (c.ld_func_int * (float)R.n_lights);
            const float2 u1 = smp.get_2d(), u2 = smp.get_2d();
            LeSample ls;
            light_sample_le<INST>(c, (int)ln, u1, u2, ls);
            if (!(ls.pdf_pos == 0.0f || ls.pdf_dir == 0.0f || is_black(ls.Le))) {
                BVert& v0 = lv[0];
                v0.type = BV_LIGHT; v0.delta = 0; v0.diff = 0; v0.light = (int)ln; v0.beta = ls.Le; v0.pdf_fwd = ls.pdf_pos * light_pdf; v0.pdf_rev = 0.0f;
                v0.p = ls.o; v0.p_err = f3(0.f, 0.f, 0.f); v0.n = ls.n; v0.ns = ls.n; v0.time = cv[0].time;
                const rgb beta = ls.Le * rgb(absdot(ls.n, ls.d) / (light_pdf * ls.pdf_pos * ls.pdf_dir));
                const int nv = random_walk<INST>(c, smp, ls.o, ls.d, cv[0].time, beta, ls.pdf_dir, max_depth, true, lv + 1);
                if (bv_infinite_light(c, v0)) {
                    if (nv > 0) {
                        lv[1].pdf_fwd = ls.pdf_pos;
                        if (bv_on_surface(lv[1])) lv[1].pdf_fwd *= absdot(ls.d, lv[1].n);
                    }
                    v0.pdf_fwd = infinite_light_density(c, ls.d);
                }
                nl = nv + 1;
            }
        }
        __syncthreads();
        if (have) {  // every strategy (bdpt.cpp:382-425)
            rgb L(0.0f);
            for (int t = 1; t <= nc; ++t)
                for (int s = 0; s <= nl; ++s) {
                    const int depth = t + s - 2;
                    if ((s == 1 && t == 1) || depth < 0 || depth > max_depth) continue;
                    float2 praster = pfilm;
                    const rgb Lp = connect<INST>(c, smp, lv, cv, s, t, &praster);
                    if (t != 1) L = L + Lp;
                    else film_add_splat(R, splat, praster, Lp);
                }
            const float y = lum(L);  // integrator.rs:350-368
            if (L.r != L.r || L.g != L.g || L.b != L.b) L = rgb(0.0f);
            else if (y < -1.0e-5f) L = rgb(0.0f);
            else if (isinf(y)) L = rgb(0.0f);
            film_add_sample_lane(R, pfilm, L);
        }
    }
    atomicAdd(&R.cnt->camera_rays, n_camera); atomicAdd(&R.cnt->closest_rays, n_closest);
}

size_t bdpt_vertex_bytes() { return sizeof(BVert); }
int bdpt_blocks_per_sm(bool inst) {
    int per_sm = 1;
    if (inst) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_bdpt<true>, PB_VOL_BLOCK, 0);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_bdpt<false>, PB_VOL_BLOCK, 0);
    return per_sm;
}
void launch_bdpt(const RenderDev& R, const BdptCam& C, void* verts, float* splat, unsigned long long total_items, bool inst, int grid, cudaStream_t stream) {
    if (inst) k_bdpt<true><<<grid, PB_VOL_BLOCK, 0, stream>>>(R, C, static_cast<BVert*>(verts), splat, total_items);
    else k_bdpt<false><<<grid, PB_VOL_BLOCK, 0, stream>>>(R, C, static_cast<BVert*>(verts), splat, total_items);
}

}  // namespace pb
