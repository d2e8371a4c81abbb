// TEST INFRASTRUCTURE -- NOT PRODUCT CODE (see oracle_math.hpp header).
// oracle_bdpt.hpp: BDPTIntegrator (src/integrators/bdpt.rs, a port of pbrt-v3's integrators/bdpt.cpp) on surfaces: camera and light
// subpaths (RandomWalk, no Russian roulette), every (s, t) connection with its visibility walk, the balance-heuristic MISWeight,
// light-tracing splats.  Where the Rust port's behaviour could not be checked, pbrt-v3 is followed (DESIGN.md §4f lists each case).
// Traversal, shading, lights and the sampler come from the existing oracle headers, which this file does not change.
#pragma once
#include "oracle_render.hpp"

namespace orc {
namespace bdpt {

enum VType { V_CAMERA, V_LIGHT, V_SURFACE };

// PerspectiveCamera's importance functions (pbrt-v3 cameras/perspective.cpp:150-243).  The image-plane area A comes from
// raster_to_camera and the full resolution; the inverse matrices are computed here (pbrt_b200_camera carries the forward ones).
struct CameraImp {
    M4 r2c, c2w, c2r, w2c;
    Float A = 0, lens_radius = 0, focal_distance = 0;
    int sb[4];
    V3 n_lens;  // CameraToWorld applied to the normal (0, 0, 1)
    void init(const pbrt_b200_camera& c, const pbrt_b200_film& f, const int* sample_bounds) {
        r2c = m4_from(c.raster_to_camera); c2w = m4_from(c.camera_to_world);
        c2r = m4_inverse(r2c); w2c = m4_inverse(c2w);
        V3 pmin = m4_point(r2c, V3(0, 0, 0)), pmax = m4_point(r2c, V3((Float)f.full_resolution[0], (Float)f.full_resolution[1], 0));
        pmin = pmin / pmin.z; pmax = pmax / pmax.z;
        A = std::fabs((pmax.x - pmin.x) * (pmax.y - pmin.y));
        lens_radius = c.lens_radius; focal_distance = c.focal_distance;
        for (int i = 0; i < 4; ++i) sb[i] = sample_bounds[i];
        n_lens = m4_normal(w2c, V3(0, 0, 1));
    }
    Float lens_area() const { return lens_radius != 0.0f ? PI * lens_radius * lens_radius : 1.0f; }
    // pRaster of a ray leaving the lens; false when the ray points backwards or leaves the sample bounds
    bool raster(V3 o, V3 d, P2* pr, Float* cos_theta) const {
        *cos_theta = dot(d, m4_vector(c2w, V3(0, 0, 1)));
        if (*cos_theta <= 0.0f) return false;
        V3 pfocus = o + d * ((lens_radius > 0.0f ? focal_distance : 1.0f) / *cos_theta);
        V3 p = m4_point(c2r, m4_point(w2c, pfocus));
        *pr = P2(p.x, p.y);
        return !(p.x < (Float)sb[0] || p.x >= (Float)sb[2] || p.y < (Float)sb[1] || p.y >= (Float)sb[3]);
    }
    Float we(V3 o, V3 d, P2* pr) const {
        Float ct;
        if (!raster(o, d, pr, &ct)) return 0.0f;
        Float c2 = ct * ct;
        return 1.0f / (A * lens_area() * c2 * c2);
    }
    void pdf_we(V3 o, V3 d, Float* pdf_pos, Float* pdf_dir) const {
        Float ct; P2 pr;
        if (!raster(o, d, &pr, &ct)) { *pdf_pos = 0.0f; *pdf_dir = 0.0f; return; }
        *pdf_pos = 1.0f / lens_area();
        *pdf_dir = 1.0f / (A * ct * ct * ct);
    }
};

struct Vertex {
    VType type = V_SURFACE;
    Spectrum beta;
    bool delta = false;
    Float pdf_fwd = 0, pdf_rev = 0;
    V3 p, p_error, n, ns;  // n = 0: not on a surface
    Float time = 0;
    int light = -1;        // V_LIGHT: the light (-1: the escaped camera ray's "infinite" endpoint)
    // V_SURFACE
    SurfaceInteraction si;
    BSDF bsdf;
    bool on_surface() const { return !(n.x == 0.0f && n.y == 0.0f && n.z == 0.0f); }
};

struct Ctx {
    const RenderScene& s;
    const IntegratorParams& ip;
    const Distribution1D& ld;  // light distribution looked up at the camera vertex
    const CameraImp& cam;
    RenderCounters& rc;
};

inline bool is_infinite_light(const Ctx& c, const Vertex& v) {
    if (v.type != V_LIGHT) return false;
    if (v.light < 0) return true;
    uint32_t t = c.s.d.lights[v.light].type;
    return t == PBRT_B200_LIGHT_INFINITE || t == PBRT_B200_LIGHT_DISTANT;
}
inline bool is_delta_light_v(const Ctx& c, const Vertex& v) { return v.type == V_LIGHT && v.light >= 0 && is_delta_light(c.s.d.lights[v.light]); }
inline int area_light_of(const Ctx& c, const Vertex& v) { return v.type == V_SURFACE ? c.s.d.prims[v.si.slot].area_light : -1; }
inline bool is_light(const Ctx& c, const Vertex& v) { return v.type == V_LIGHT || area_light_of(c, v) >= 0; }
inline bool is_connectible(const Ctx& c, const Vertex& v) {
    if (v.type == V_CAMERA) return true;
    if (v.type == V_LIGHT) return v.light < 0 || c.s.d.lights[v.light].type != PBRT_B200_LIGHT_DISTANT;  // DeltaDirection
    return v.bsdf.num_components(BSDF_DIFFUSE | BSDF_GLOSSY | BSDF_REFLECTION | BSDF_TRANSMISSION) > 0;
}

// TransportMode::Importance where the shared BSDF code applies the Radiance scale: light subpaths undo the (etai/etat)^2 factor
// of specular and microfacet transmission.  `trans`: the pair of directions is a transmission.
inline Float importance_scale(const BSDF& b, V3 wo, bool trans) {
    if (!trans || b.eta == 1.0f) return 1.0f;
    Float e = b.world_to_local(wo).z > 0.0f ? b.eta : 1.0f / b.eta;
    return e * e;
}
// pbrt-v3 CorrectShadingNormal (bdpt.cpp:48-59)
inline Float correct_shading_normal(const SurfaceInteraction& si, V3 wo, V3 wi, bool importance) {
    if (!importance) return 1.0f;
    Float num = abs_dot(wo, si.sh_n) * abs_dot(wi, si.n), den = abs_dot(wo, si.n) * abs_dot(wi, si.sh_n);
    if (den == 0.0f) return 0.0f;
    return num / den;
}

// Vertex::f
inline Spectrum vertex_f(const Vertex& v, const Vertex& next, bool importance) {
    V3 wi = next.p - v.p;
    if (length_squared(wi) == 0.0f) return Spectrum(0.0f);
    wi = normalize(wi);
    if (v.type != V_SURFACE) return Spectrum(0.0f);
    const V3 wo = v.si.wo;
    Spectrum f = v.bsdf.f(wo, wi, BSDF_ALL);
    if (importance) f = f * Spectrum(importance_scale(v.bsdf, wo, !(dot(wi, v.bsdf.ng) * dot(wo, v.bsdf.ng) > 0.0f)));
    return f * Spectrum(correct_shading_normal(v.si, wo, wi, importance));
}

inline Float convert_density(const Ctx& c, const Vertex& v, Float pdf, const Vertex& next) {
    if (is_infinite_light(c, next)) return pdf;
    V3 w = next.p - v.p;
    if (length_squared(w) == 0.0f) return 0.0f;
    Float inv_d2 = 1.0f / length_squared(w);
    if (next.on_surface()) pdf *= abs_dot(next.n, w * std::sqrt(inv_d2));
    return pdf * inv_d2;
}

// ---- Light::sample_le / pdf_le (pbrt-v3 lights/*.cpp)
inline V3 uniform_sample_cone(P2 u, Float cos_max) {
    Float ct = (1.0f - u.x) + u.x * cos_max;
    Float st = std::sqrt(1.0f - ct * ct);
    Float phi = u.y * 2.0f * PI;
    return V3(std::cos(phi) * st, std::sin(phi) * st, ct);
}
inline Float spot_falloff(const pbrt_b200_light& l, V3 w) {
    V3 wl = normalize(m4_vector(m4_from(l.world_to_light), w));
    Float ct = wl.z;
    if (ct < l.cos_total_width) return 0.0f;
    if (ct >= l.cos_falloff_start) return 1.0f;
    Float d = (ct - l.cos_total_width) / (l.cos_falloff_start - l.cos_total_width);
    return (d * d) * (d * d);
}
struct LeSample { Spectrum Le; V3 o, d, n; Float pdf_pos = 0, pdf_dir = 0; };
inline LeSample light_sample_le(const RenderScene& s, int li, P2 u1, P2 u2) {
    const pbrt_b200_light& l = s.d.lights[li];
    LeSample r;
    Spectrum L = spec3(l.L);
    switch (l.type) {
        case PBRT_B200_LIGHT_POINT:
            r.o = V3(l.pos[0], l.pos[1], l.pos[2]); r.d = uniform_sample_sphere_(u1); r.n = r.d;
            r.pdf_pos = 1.0f; r.pdf_dir = 1.0f / (4.0f * PI); r.Le = L;
            break;
        case PBRT_B200_LIGHT_SPOT: {
            M4 l2w = m4_inverse(m4_from(l.world_to_light));
            r.o = V3(l.pos[0], l.pos[1], l.pos[2]); r.d = m4_vector(l2w, uniform_sample_cone(u1, l.cos_total_width)); r.n = r.d;
            r.pdf_pos = 1.0f; r.pdf_dir = 1.0f / (2.0f * PI * (1.0f - l.cos_total_width));
            r.Le = L * Spectrum(spot_falloff(l, r.d));
            break;
        }
        case PBRT_B200_LIGHT_DISTANT: {
            V3 w(l.dir[0], l.dir[1], l.dir[2]), v1, v2;
            coordinate_system(w, &v1, &v2);
            P2 cd = concentric_sample_disk(u1);
            V3 pdisk = s.world_center + (v1 * cd.x + v2 * cd.y) * s.world_radius;
            r.o = pdisk + w * s.world_radius; r.d = -w; r.n = r.d;
            r.pdf_pos = 1.0f / (PI * s.world_radius * s.world_radius); r.pdf_dir = 1.0f; r.Le = L;
            break;
        }
        case PBRT_B200_LIGHT_DIFFUSE: {
            InteractionData ps;
            Float pdf_pos;
            if (l.shape_kind == PBRT_B200_SHAPE_SPHERE) ps = sphere_sample(s.d.spheres[l.shape_index], l, u1, &pdf_pos);
            else {  // Triangle::sample (the area density; sample_interaction's solid-angle conversion is not used here)
                InteractionData ref; ref.p = V3(0, 0, 0);
                ps = triangle_sample_interaction(s, l, ref, u1, &pdf_pos);
                pdf_pos = 1.0f / l.area;
            }
            r.pdf_pos = pdf_pos;
            V3 w;
            if (l.two_sided) {
                P2 u = u2;
                if (u.x < 0.5f) { u.x = std::fmin(u.x * 2.0f, ONE_MINUS_EPSILON); w = cosine_sample_hemisphere(u); }
                else { u.x = std::fmin((u.x - 0.5f) * 2.0f, ONE_MINUS_EPSILON); w = cosine_sample_hemisphere(u); w.z *= -1.0f; }
                r.pdf_dir = 0.5f * std::fabs(w.z) * INV_PI;
            } else {
                w = cosine_sample_hemisphere(u2);
                r.pdf_dir = w.z * INV_PI;
            }
            V3 v1, v2, n = ps.n;
            coordinate_system(n, &v1, &v2);
            w = v1 * w.x + v2 * w.y + n * w.z;
            r.o = offset_ray_origin(ps.p, ps.p_error, ps.n, w); r.d = w; r.n = ps.n;
            r.Le = (l.two_sided || dot(ps.n, w) > 0.0f) ? L : Spectrum(0.0f);
            break;
        }
        default: {  // constant infinite light
            Float map_pdf = 0.0f;
            P2 uv = s.inf_distrib[li].sample_continuous(u1, &map_pdf);
            if (map_pdf == 0.0f) return r;
            Float theta = uv.y * PI, phi = uv.x * 2.0f * PI;
            Float ct = std::cos(theta), st = std::sin(theta), sp = std::sin(phi), cp = std::cos(phi);
            V3 d = -V3(st * cp, st * sp, ct), v1, v2;
            coordinate_system(-d, &v1, &v2);
            P2 cd = concentric_sample_disk(u2);
            V3 pdisk = s.world_center + (v1 * cd.x + v2 * cd.y) * s.world_radius;
            r.o = pdisk + (-d) * s.world_radius; r.d = d; r.n = d;
            r.pdf_dir = st == 0.0f ? 0.0f : map_pdf / (2.0f * PI * PI * st);
            r.pdf_pos = 1.0f / (PI * s.world_radius * s.world_radius);
            r.Le = L;
            break;
        }
    }
    return r;
}
inline void light_pdf_le(const RenderScene& s, int li, V3 d, V3 n, Float* pdf_pos, Float* pdf_dir) {
    const pbrt_b200_light& l = s.d.lights[li];
    switch (l.type) {
        case PBRT_B200_LIGHT_POINT: *pdf_pos = 0.0f; *pdf_dir = 1.0f / (4.0f * PI); break;
        case PBRT_B200_LIGHT_SPOT: {
            *pdf_pos = 0.0f;
            V3 wl = m4_vector(m4_from(l.world_to_light), d);
            *pdf_dir = wl.z >= l.cos_total_width ? 1.0f / (2.0f * PI * (1.0f - l.cos_total_width)) : 0.0f;
            break;
        }
        case PBRT_B200_LIGHT_DISTANT: *pdf_pos = 1.0f / (PI * s.world_radius * s.world_radius); *pdf_dir = 0.0f; break;
        case PBRT_B200_LIGHT_DIFFUSE:
            *pdf_pos = 1.0f / l.area;
            *pdf_dir = l.two_sided ? 0.5f * abs_dot(n, d) * INV_PI : dot(n, d) * INV_PI;
            break;
        default: {
            V3 wi = -d;
            Float theta = spherical_theta(wi), phi = spherical_phi(wi), st = std::sin(theta);
            *pdf_dir = st == 0.0f ? 0.0f : s.inf_distrib[li].pdf(P2(phi * INV2_PI, theta * INV_PI)) / (2.0f * PI * PI * st);
            *pdf_pos = 1.0f / (PI * s.world_radius * s.world_radius);
            break;
        }
    }
}

inline Float infinite_light_density(const Ctx& c, V3 w) {
    Float pdf = 0.0f;
    InteractionData ref;
    ref.p = V3(0, 0, 0); ref.p_error = V3(0, 0, 0); ref.n = V3(0, 0, 0);
    for (int li : c.s.infinite_lights) pdf += light_pdf_li(c.s, li, ref, -w) * c.ld.func[li];  // Scene.infinite_lights: no distant lights
    return pdf / (c.ld.func_int * (Float)c.ld.count());
}

inline Float pdf_light(const Ctx& c, const Vertex& v, const Vertex& next) {
    V3 w = next.p - v.p;
    Float inv_d2 = 1.0f / length_squared(w);
    w = w * std::sqrt(inv_d2);
    Float pdf;
    if (is_infinite_light(c, v)) pdf = 1.0f / (PI * c.s.world_radius * c.s.world_radius);
    else {
        int li = v.type == V_LIGHT ? v.light : area_light_of(c, v);
        Float pp, pd;
        light_pdf_le(c.s, li, w, v.n, &pp, &pd);
        pdf = pd * inv_d2;
    }
    if (next.on_surface()) pdf *= abs_dot(next.n, w);
    return pdf;
}
inline Float pdf_light_origin(const Ctx& c, const Vertex& v, const Vertex& next) {
    V3 w = next.p - v.p;
    if (length_squared(w) == 0.0f) return 0.0f;
    w = normalize(w);
    if (is_infinite_light(c, v)) return infinite_light_density(c, w);
    int li = v.type == V_LIGHT ? v.light : area_light_of(c, v);
    Float pp, pd;
    light_pdf_le(c.s, li, w, v.n, &pp, &pd);
    return pp * c.ld.discrete_pdf((size_t)li);
}
// Vertex::Pdf
inline Float vertex_pdf(const Ctx& c, const Vertex& v, const Vertex* prev, const Vertex& next) {
    if (v.type == V_LIGHT) return pdf_light(c, v, next);
    V3 wn = next.p - v.p;
    if (length_squared(wn) == 0.0f) return 0.0f;
    wn = normalize(wn);
    Float pdf = 0.0f;
    if (v.type == V_CAMERA) { Float pp; c.cam.pdf_we(v.p, wn, &pp, &pdf); }
    else {
        V3 wp = normalize(prev->p - v.p);
        pdf = v.bsdf.pdf(wp, wn, BSDF_ALL);
    }
    return convert_density(c, v, pdf, next);
}
// Vertex::Le
inline Spectrum vertex_le(const Ctx& c, const Vertex& v, const Vertex& to) {
    if (!is_light(c, v)) return Spectrum(0.0f);
    V3 w = to.p - v.p;
    if (length_squared(w) == 0.0f) return Spectrum(0.0f);
    w = normalize(w);
    if (is_infinite_light(c, v)) {
        Spectrum Le(0.0f);
        for (int li : c.s.infinite_lights) Le += light_le(c.s, li);
        return Le;
    }
    const pbrt_b200_light& l = c.s.d.lights[area_light_of(c, v)];
    return (l.two_sided || dot(v.n, w) > 0.0f) ? spec3(l.L) : Spectrum(0.0f);
}

// VisibilityTester::tr without media: closest hits through material-less surfaces
inline bool unoccluded(const Ctx& c, const InteractionData& a, const InteractionData& b) {
    Ray r = spawn_ray_to(a, b);
    for (;;) {
        Hit h;
        Ray r0 = r;
        c.rc.intersection_tests++;
        if (!scene_intersect(c.s, r, &h, &c.rc.trav_closest)) return true;
        if (c.s.d.prims[h.slot].material >= 0) return false;
        SurfaceInteraction si = make_interaction(c.s, r0, h);
        InteractionData ia; ia.p = si.p; ia.p_error = si.p_error; ia.n = si.n; ia.time = si.time;
        r = spawn_ray_to(ia, b);
    }
}
inline InteractionData idata(const Vertex& v) { InteractionData d; d.p = v.p; d.p_error = v.p_error; d.n = v.n; d.time = v.time; return d; }

// RandomWalk (bdpt.cpp:191-269) without media; `ray` carries differentials for the camera subpath's first hit only
inline int random_walk(const Ctx& c, Ray ray, Sampler& smp, Spectrum beta, Float pdf, int max_depth, bool importance, Vertex* path) {
    if (max_depth == 0) return 0;
    int bounces = 0;
    Float pdf_fwd = pdf, pdf_rev = 0.0f;
    for (;;) {
        Hit h;
        Ray r0 = ray;
        c.rc.intersection_tests++;
        bool found = scene_intersect(c.s, ray, &h, &c.rc.trav_closest);
        if (beta.is_black()) break;
        Vertex& v = path[bounces];
        Vertex& prev = path[bounces - 1];
        if (!found) {
            if (!importance) {
                v = Vertex(); v.type = V_LIGHT; v.light = -1; v.beta = beta; v.pdf_fwd = pdf_fwd;
                v.p = r0.o + r0.d; v.n = -r0.d; v.ns = v.n; v.p_error = V3(0, 0, 0); v.time = r0.time;  // EndpointInteraction(ray): ray(1)
                ++bounces;
            }
            break;
        }
        SurfaceInteraction isect = make_interaction(c.s, r0, h);
        BSDF bsdf;
        scattering_functions(c.s, ray, h.slot, isect, &bsdf, true);
        if (!bsdf.valid) { ray = spawn_ray(isect.p, isect.p_error, isect.n, ray.d, isect.time); continue; }
        v = Vertex(); v.type = V_SURFACE; v.si = isect; v.bsdf = bsdf; v.beta = beta;
        v.p = isect.p; v.p_error = isect.p_error; v.n = isect.n; v.ns = isect.sh_n; v.time = isect.time;
        v.pdf_fwd = convert_density(c, prev, pdf_fwd, v);
        if (++bounces >= max_depth) break;
        V3 wi, wo = isect.wo;
        int type = 0;
        pdf_fwd = 0.0f;
        Spectrum f = bsdf.sample_f(wo, &wi, smp.get_2d(), &pdf_fwd, BSDF_ALL, &type);
        if (f.is_black() || pdf_fwd == 0.0f) break;
        if (importance)
            f = f * Spectrum(importance_scale(bsdf, wo, (type & BSDF_SPECULAR) ? (type & BSDF_TRANSMISSION) != 0 : !(dot(wi, bsdf.ng) * dot(wo, bsdf.ng) > 0.0f)));
        beta *= f * abs_dot(wi, isect.sh_n) / pdf_fwd;
        pdf_rev = bsdf.pdf(wi, wo, BSDF_ALL);
        if (type & BSDF_SPECULAR) { v.delta = true; pdf_rev = pdf_fwd = 0.0f; }
        beta *= Spectrum(correct_shading_normal(isect, wo, wi, importance));
        ray = spawn_ray(isect.p, isect.p_error, isect.n, wi, isect.time);
        prev.pdf_rev = convert_density(c, v, pdf_rev, prev);
    }
    return bounces;
}

inline int camera_subpath(const Ctx& c, Sampler& smp, int max_depth, const Ray& ray, Vertex* path) {
    if (max_depth == 0) return 0;
    path[0] = Vertex(); path[0].type = V_CAMERA; path[0].beta = Spectrum(1.0f); path[0].p = ray.o; path[0].p_error = V3(0, 0, 0);
    path[0].n = V3(0, 0, 0); path[0].ns = V3(0, 0, 0); path[0].time = ray.time;
    Float pdf_pos, pdf_dir;
    c.cam.pdf_we(ray.o, ray.d, &pdf_pos, &pdf_dir);
    return random_walk(c, ray, smp, Spectrum(1.0f), pdf_dir, max_depth - 1, false, path + 1) + 1;
}

inline int light_subpath(const Ctx& c, Sampler& smp, int max_depth, Float time, Vertex* path) {
    if (max_depth == 0) return 0;
    Float light_pdf = 0.0f;
    int ln = (int)c.ld.sample_discrete(smp.get_1d(), &light_pdf);
    P2 u1 = smp.get_2d(), u2 = smp.get_2d();
    LeSample ls = light_sample_le(c.s, ln, u1, u2);
    if (ls.pdf_pos == 0.0f || ls.pdf_dir == 0.0f || ls.Le.is_black()) return 0;
    path[0] = Vertex(); path[0].type = V_LIGHT; path[0].light = ln; path[0].beta = ls.Le; path[0].pdf_fwd = ls.pdf_pos * light_pdf;
    path[0].p = ls.o; path[0].p_error = V3(0, 0, 0); path[0].n = ls.n; path[0].ns = ls.n; path[0].time = time;
    Spectrum beta = ls.Le * Spectrum(abs_dot(ls.n, ls.d) / (light_pdf * ls.pdf_pos * ls.pdf_dir));
    Ray ray(ls.o, ls.d, INFINITY_F, time);
    int nv = random_walk(c, ray, smp, beta, ls.pdf_dir, max_depth - 1, true, path + 1);
    if (is_infinite_light(c, path[0])) {
        if (nv > 0) {
            path[1].pdf_fwd = ls.pdf_pos;
            if (path[1].on_surface()) path[1].pdf_fwd *= abs_dot(ls.d, path[1].n);
        }
        path[0].pdf_fwd = infinite_light_density(c, ls.d);
    }
    return nv + 1;
}

inline Float mis_weight(const Ctx& c, Vertex* lv, Vertex* cv, const Vertex& sampled, int s, int t) {
    if (s + t == 2) return 1.0f;
    auto remap0 = [](Float f) { return f != 0.0f ? f : 1.0f; };
    Vertex* qs = s > 0 ? &lv[s - 1] : nullptr;
    Vertex* pt = t > 0 ? &cv[t - 1] : nullptr;
    Vertex* qsm = s > 1 ? &lv[s - 2] : nullptr;
    Vertex* ptm = t > 1 ? &cv[t - 2] : nullptr;
    // the scoped assignments of bdpt.cpp:433-460, undone on return
    Vertex save_q, save_p;
    if (qs) save_q = *qs;
    if (pt) save_p = *pt;
    Float save_ptm = ptm ? ptm->pdf_rev : 0.0f, save_qsm = qsm ? qsm->pdf_rev : 0.0f;
    if (s == 1) *qs = sampled;
    else if (t == 1) *pt = sampled;
    if (pt) pt->delta = false;
    if (qs) qs->delta = false;
    if (pt) pt->pdf_rev = s > 0 ? vertex_pdf(c, *qs, qsm, *pt) : pdf_light_origin(c, *pt, *ptm);
    if (ptm) ptm->pdf_rev = s > 0 ? vertex_pdf(c, *pt, qs, *ptm) : pdf_light(c, *pt, *ptm);
    if (qs) qs->pdf_rev = vertex_pdf(c, *pt, ptm, *qs);
    if (qsm) qsm->pdf_rev = vertex_pdf(c, *qs, pt, *qsm);
    Float sum = 0.0f, ri = 1.0f;
    for (int i = t - 1; i > 0; --i) {
        ri *= remap0(cv[i].pdf_rev) / remap0(cv[i].pdf_fwd);
        if (!cv[i].delta && !cv[i - 1].delta) sum += ri;
    }
    ri = 1.0f;
    for (int i = s - 1; i >= 0; --i) {
        ri *= remap0(lv[i].pdf_rev) / remap0(lv[i].pdf_fwd);
        bool dl = i > 0 ? lv[i - 1].delta : is_delta_light_v(c, lv[0]);
        if (!lv[i].delta && !dl) sum += ri;
    }
    if (qs) *qs = save_q;
    if (pt) *pt = save_p;
    if (ptm) ptm->pdf_rev = save_ptm;
    if (qsm) qsm->pdf_rev = save_qsm;
    return 1.0f / (1.0f + sum);
}

// ConnectBDPT (bdpt.cpp:462-560)
inline Spectrum connect(const Ctx& c, Vertex* lv, Vertex* cv, int s, int t, Sampler& smp, P2* praster, Float* weight_out) {
    Spectrum L(0.0f);
    if (t > 1 && s != 0 && cv[t - 1].type == V_LIGHT) { *weight_out = 0.0f; return L; }
    Vertex sampled;
    if (s == 0) {
        const Vertex& pt = cv[t - 1];
        if (is_light(c, pt)) L = vertex_le(c, pt, cv[t - 2]) * pt.beta;
    } else if (t == 1) {
        const Vertex& qs = lv[s - 1];
        if (is_connectible(c, qs)) {
            P2 u = smp.get_2d();
            // PerspectiveCamera::sample_wi
            P2 pl = concentric_sample_disk(u);
            pl = P2(pl.x * c.cam.lens_radius, pl.y * c.cam.lens_radius);
            V3 plw = m4_point(c.cam.c2w, V3(pl.x, pl.y, 0.0f));
            V3 wi = plw - qs.p;
            Float dist = length(wi);
            wi = wi / dist;
            Float pdf = (dist * dist) / (abs_dot(c.cam.n_lens, wi) * c.cam.lens_area());
            Float We = c.cam.we(offset_ray_origin(plw, V3(0, 0, 0), c.cam.n_lens, -wi), -wi, praster);
            if (pdf > 0.0f && We != 0.0f) {
                sampled.type = V_CAMERA; sampled.beta = Spectrum(We / pdf); sampled.p = plw; sampled.p_error = V3(0, 0, 0);
                sampled.n = c.cam.n_lens; sampled.ns = sampled.n; sampled.time = qs.time;
                L = qs.beta * vertex_f(qs, sampled, true) * sampled.beta;
                if (qs.on_surface()) L *= Spectrum(abs_dot(wi, qs.ns));
                if (!L.is_black() && !unoccluded(c, idata(qs), idata(sampled))) L = Spectrum(0.0f);
            }
        }
    } else if (s == 1) {
        const Vertex& pt = cv[t - 1];
        if (is_connectible(c, pt)) {
            Float light_pdf = 0.0f;
            int ln = (int)c.ld.sample_discrete(smp.get_1d(), &light_pdf);
            LightSample ls = light_sample_li(c.s, ln, idata(pt), smp.get_2d());
            if (ls.pdf > 0.0f && !ls.Li.is_black()) {
                sampled.type = V_LIGHT; sampled.light = ln; sampled.beta = ls.Li / Spectrum(ls.pdf * light_pdf); sampled.pdf_fwd = 0.0f;
                sampled.p = ls.p1.p; sampled.p_error = ls.p1.p_error; sampled.n = ls.p1.n; sampled.ns = sampled.n; sampled.time = pt.time;
                sampled.pdf_fwd = pdf_light_origin(c, sampled, pt);
                L = pt.beta * vertex_f(pt, sampled, false) * sampled.beta;
                if (pt.on_surface()) L *= Spectrum(abs_dot(ls.wi, pt.ns));
                if (!L.is_black() && !unoccluded(c, idata(pt), ls.p1)) L = Spectrum(0.0f);
            }
        }
    } else {
        const Vertex& qs = lv[s - 1];
        const Vertex& pt = cv[t - 1];
        if (is_connectible(c, qs) && is_connectible(c, pt)) {
            L = qs.beta * vertex_f(qs, pt, true) * vertex_f(pt, qs, false) * pt.beta;
            if (!L.is_black()) {  // G (bdpt.cpp:170-180)
                V3 d = qs.p - pt.p;
                Float g = 1.0f / length_squared(d);
                d = d * std::sqrt(g);
                if (qs.on_surface()) g *= abs_dot(qs.ns, d);
                if (pt.on_surface()) g *= abs_dot(pt.ns, d);
                if (!unoccluded(c, idata(qs), idata(pt))) g = 0.0f;
                L *= Spectrum(g);
            }
        }
    }
    Float w = L.is_black() ? 0.0f : mis_weight(c, lv, cv, sampled, s, t);
    *weight_out = w;
    return L * Spectrum(w);
}

}  // namespace bdpt
}  // namespace orc
