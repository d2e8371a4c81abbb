// TEST INFRASTRUCTURE (see oracle_grid.py): CPU restatement of pbrt-rust's VolPathIntegrator for scenes with grid-density media.
//
//   GridDensityMedium::{d, density, sample, tr}  src/media/grid.rs (a port of pbrt-v3 media/grid.{h,cpp}), api.rs make_medium
//
// oracle_volpath.hpp restates VolPathIntegrator::li with HomogeneousMedium, whose tr draws nothing.  GridDensityMedium::tr draws from the
// sampler, so both transmittance loops (VisibilityTester::tr, light.rs:125-150; Scene::intersect_tr, scene.rs:68-87), estimate_direct
// and li take the sampler here; every other piece -- traversal, interactions, BSDFs, lights, the phase function, medium interfaces,
// HomogeneousMedium -- is the one of oracle_render.hpp / oracle_volpath.hpp.  The functions below are those of oracle_volpath.hpp with
// the grid table added, in a namespace of their own; homogeneous rows (grid = 0) take the same path as there.
//
// Reproduced on purpose, as in the reference:
//   * GridDensityMedium::sample returns the interaction at ray_world(t) although t is measured along the normalised ray (exact for
//     the unit-direction path rays of this integrator).
//   * sigma_t is the first channel of sigma_a + sigma_s.
// Choices of this project, shared with the device (csrc/mega.cu):
//   * A grid whose sigma_t * max_density is 0 (an all-zero grid) is vacuum: sample and tr return weight 1 without drawing.
//   * A tracking loop that runs ORC_VOL_TRACK_CAP steps gives up, and the path ends there: the walk that gave up adds nothing,
//     what was added before stays.
#pragma once
#include "oracle_render.hpp"

namespace orc {
namespace grid_media {

// The density grids of the media rows with grid = k > 0 (grids[k - 1]) and their maxima (GridDensityMedium::new: max_density)
struct GridTable {
    const pbrt_b200_density_grid* grids = nullptr;
    std::vector<Float> max;
    GridTable(const pbrt_b200_density_grid* g, uint64_t n) : grids(g) {
        for (uint64_t i = 0; i < n; ++i) {
            const uint64_t cnt = (uint64_t)g[i].nx * g[i].ny * g[i].nz;
            Float m = 0.0f;
            for (uint64_t k = 0; k < cnt; ++k) m = g[i].density[k] > m ? g[i].density[k] : m;
            max.push_back(m);
        }
    }
};

// ---- GridDensityMedium (grid.rs)
#define ORC_VOL_TRACK_CAP 65536u  // = PB_VOL_TRACK_CAP (csrc/mega.cu)

inline Float grid_d(const pbrt_b200_density_grid& g, int x, int y, int z) {  // GridDensityMedium::d
    if (x < 0 || y < 0 || z < 0 || x >= (int)g.nx || y >= (int)g.ny || z >= (int)g.nz) return 0.0f;
    return g.density[((size_t)z * g.ny + (size_t)y) * g.nx + (size_t)x];
}
inline Float grid_lerp(Float t, Float a, Float b) { return (1.0f - t) * a + t * b; }
inline Float grid_density(const pbrt_b200_density_grid& g, V3 p) {  // GridDensityMedium::density
    const Float sx = p.x * (Float)g.nx - 0.5f, sy = p.y * (Float)g.ny - 0.5f, sz = p.z * (Float)g.nz - 0.5f;
    const Float fx = std::floor(sx), fy = std::floor(sy), fz = std::floor(sz);
    const int x = (int)fx, y = (int)fy, z = (int)fz;
    const Float dx = sx - fx, dy = sy - fy, dz = sz - fz;
    const Float d00 = grid_lerp(dx, grid_d(g, x, y, z), grid_d(g, x + 1, y, z));
    const Float d10 = grid_lerp(dx, grid_d(g, x, y + 1, z), grid_d(g, x + 1, y + 1, z));
    const Float d01 = grid_lerp(dx, grid_d(g, x, y, z + 1), grid_d(g, x + 1, y, z + 1));
    const Float d11 = grid_lerp(dx, grid_d(g, x, y + 1, z + 1), grid_d(g, x + 1, y + 1, z + 1));
    const Float d0 = grid_lerp(dy, d00, d10), d1 = grid_lerp(dy, d01, d11);
    return grid_lerp(dz, d0, d1);
}
// world_to_medium(Ray(o, normalize(d), t_max * |d|)) clipped to Bounds3(0,0,0)-(1,1,1) (the t0/t1 form of Bounds3::intersect_p)
inline bool grid_clip(const pbrt_b200_density_grid& g, const Ray& rw, Ray* mr, Float* t0_out, Float* t1_out) {
    *mr = m4_ray(m4_from(g.world_to_medium), Ray(rw.o, normalize(rw.d), rw.t_max * length(rw.d), rw.time));
    Float t0 = 0.0f, t1 = mr->t_max;
    const Float ro[3] = {mr->o.x, mr->o.y, mr->o.z}, rd[3] = {mr->d.x, mr->d.y, mr->d.z};
    for (int i = 0; i < 3; ++i) {
        const Float inv = 1.0f / rd[i];
        Float tn = (0.0f - ro[i]) * inv, tf = (1.0f - ro[i]) * inv;
        if (tn > tf) std::swap(tn, tf);
        tf *= 1.0f + 2.0f * gamma(3);
        t0 = tn > t0 ? tn : t0;
        t1 = tf < t1 ? tf : t1;
        if (t0 > t1) return false;
    }
    *t0_out = t0; *t1_out = t1;
    return true;
}
inline bool grid_is_vacuum(Float max_density, Float sigma_t) { return !(max_density > 0.0f && sigma_t > 0.0f); }
inline Float grid_step(Float inv_max, Float sigma_t, Float t, Float u) { return t - std::log(1.0f - u) * inv_max / sigma_t; }
// GridDensityMedium::sample (delta tracking): true with *p = ray_world(t), *w = sigma_s / sigma_t; else *w = 1
inline bool grid_sample(const RenderScene& s, const GridTable& gt, const pbrt_b200_medium& m, const Ray& rw, Sampler& sampler, V3* p, Spectrum* w, bool& gave_up) {
    *w = Spectrum(1.0f);
    const pbrt_b200_density_grid& g = gt.grids[m.grid - 1];
    const Float mx = gt.max[m.grid - 1], inv = 1.0f / mx;
    Ray mr; Float t0, t1;
    const Float st = m.sigma_a[0] + m.sigma_s[0];
    if (grid_is_vacuum(mx, st) || !grid_clip(g, rw, &mr, &t0, &t1)) return false;
    Float t = t0;
    for (uint32_t k = 0;; ++k) {
        if (k >= ORC_VOL_TRACK_CAP) { gave_up = true; return false; }
        t = grid_step(inv, st, t, sampler.get_1d());
        if (t >= t1) break;
        if (grid_density(g, mr.o + mr.d * t) * inv > sampler.get_1d()) {
            *p = rw.o + rw.d * t;
            *w = Spectrum(m.sigma_s[0] / st, m.sigma_s[1] / st, m.sigma_s[2] / st);
            return true;
        }
    }
    return false;
}
// GridDensityMedium::tr (ratio tracking with Russian roulette): draws from the sampler
inline Float grid_tr(const RenderScene& s, const GridTable& gt, const pbrt_b200_medium& m, const Ray& rw, Sampler& sampler, bool& gave_up) {
    const pbrt_b200_density_grid& g = gt.grids[m.grid - 1];
    const Float mx = gt.max[m.grid - 1], inv = 1.0f / mx;
    Ray mr; Float t0, t1;
    const Float st = m.sigma_a[0] + m.sigma_s[0];
    if (grid_is_vacuum(mx, st) || !grid_clip(g, rw, &mr, &t0, &t1)) return 1.0f;
    Float tr = 1.0f, t = t0;
    for (uint32_t k = 0;; ++k) {
        if (k >= ORC_VOL_TRACK_CAP) { gave_up = true; return 0.0f; }
        t = grid_step(inv, st, t, sampler.get_1d());
        if (t >= t1) break;
        tr *= 1.0f - std::fmax(0.0f, grid_density(g, mr.o + mr.d * t) * inv);
        if (tr < 0.1f) {
            const Float q = std::fmax(0.05f, 1.0f - tr);
            if (sampler.get_1d() < q) return 0.0f;
            tr /= 1.0f - q;
        }
    }
    return tr;
}
// Medium::tr of either kind
inline Spectrum any_medium_tr(const RenderScene& s, const GridTable& gt, int medium, const Ray& ray, Sampler& sampler, bool& gave_up) {
    const pbrt_b200_medium& m = s.d.media[medium];
    if (m.grid == 0) return medium_tr(m, ray);
    return Spectrum(grid_tr(s, gt, m, ray, sampler, gave_up));
}

// VisibilityTester::tr, light.rs:125-150: p0 -> p1 through every material-less surface on the way
inline Spectrum visibility_tr(const RenderScene& s, const GridTable& gt, const InteractionData& p0, const VolInterface& mi0, const InteractionData& p1, RenderCounters& rc,
                              Sampler& sampler, bool& gave_up) {
    VolRay vr;
    vr.r = spawn_ray_to(p0, p1);
    vr.medium = medium_for(mi0, p0.n, vr.r.d);
    Spectrum Tr(1.0f);
    for (;;) {
        Hit h;
        Ray r0 = vr.r;
        rc.intersection_tests++;  // Scene::intersect, not intersect_p
        bool hit = scene_intersect(s, vr.r, &h, &rc.trav_closest);
        if (hit && s.d.prims[h.slot].material >= 0) return Spectrum(0.0f);
        if (vr.medium >= 0) Tr *= any_medium_tr(s, gt, vr.medium, vr.r, sampler, gave_up);
        if (gave_up) return Spectrum(0.0f);
        if (!hit) break;
        SurfaceInteraction isect = make_interaction(s, r0, h);
        InteractionData a; a.p = isect.p; a.p_error = isect.p_error; a.n = isect.n; a.time = isect.time;
        VolInterface mi = hit_interface(s, h.slot, vr.medium);
        vr.r = spawn_ray_to(a, p1);
        vr.medium = medium_for(mi, isect.n, vr.r.d);
    }
    return Tr;
}

// Scene::intersect_tr, scene.rs:68-87
inline bool intersect_tr(const RenderScene& s, const GridTable& gt, VolRay vr, Hit* h_out, Ray* r_hit, Spectrum* Tr, RenderCounters& rc, Sampler& sampler, bool& gave_up) {
    *Tr = Spectrum(1.0f);
    for (;;) {
        Hit h;
        Ray r0 = vr.r;
        rc.intersection_tests++;
        bool hit = scene_intersect(s, vr.r, &h, &rc.trav_closest);
        if (vr.medium >= 0) *Tr *= any_medium_tr(s, gt, vr.medium, vr.r, sampler, gave_up);
        if (gave_up) return false;
        if (!hit) return false;
        if (s.d.prims[h.slot].material >= 0) { *h_out = h; *r_hit = r0; return true; }
        SurfaceInteraction isect = make_interaction(s, r0, h);
        VolInterface mi = hit_interface(s, h.slot, vr.medium);
        vr.r = spawn_ray(isect.p, isect.p_error, isect.n, vr.r.d, isect.time);
        vr.medium = medium_for(mi, isect.n, vr.r.d);
    }
}

// What estimate_direct needs to know about the scattering point: a surface with its BSDF, or a point in a medium with its phase function
struct VolVertex {
    bool surface = true;
    InteractionData ref;      // p, p_error, n (n = 0 in a medium), time
    V3 wo, sh_n;
    const BSDF* bsdf = nullptr;
    Float g = 0;              // HenyeyGreenstein
    VolInterface mi;
};

// estimate_direct with handle_media = true, integrator.rs:109-237
// The transmittance loops draw from `sampler` (grid media); `gave_up` (hang guard): the walk that gave up adds nothing.
inline Spectrum vol_estimate_direct(const RenderScene& s, const GridTable& gt, const VolVertex& it, P2 uscatt, int li, P2 ulight, RenderCounters& rc, Sampler& sampler, bool& gave_up) {
    const pbrt_b200_light& light = s.d.lights[li];
    const int flags = BSDF_ALL & ~BSDF_SPECULAR;
    Spectrum Ld(0.0f);
    LightSample ls = light_sample_li(s, li, it.ref, ulight);
    Float lightpdf = ls.pdf, scattpdf = 0.0f;
    V3 wi = ls.wi;
    Spectrum Li = ls.Li;
    if (lightpdf > 0.0f && !Li.is_black()) {
        Spectrum f;
        if (it.surface) { f = it.bsdf->f(it.wo, wi, flags) * abs_dot(wi, it.sh_n); scattpdf = it.bsdf->pdf(it.wo, wi, flags); }
        else { Float p = phase_hg(dot(it.wo, wi), it.g); f = Spectrum(p); scattpdf = p; }
        if (!f.is_black()) {
            Li *= visibility_tr(s, gt, it.ref, it.mi, ls.p1, rc, sampler, gave_up);
            if (gave_up) return Ld;
            if (!Li.is_black()) {
                if (is_delta_light(light)) Ld += f * Li / lightpdf;
                else { Float weight = power_heuristic(1, lightpdf, 1, scattpdf); Ld += f * Li * weight / lightpdf; }
            }
        }
    }
    if (!is_delta_light(light)) {
        Spectrum f;
        bool sampled_specular = false;
        if (it.surface) {
            int sampled_type = 0;
            f = it.bsdf->sample_f(it.wo, &wi, uscatt, &scattpdf, flags, &sampled_type);
            f = f * abs_dot(wi, it.sh_n);
            sampled_specular = (sampled_type & BSDF_SPECULAR) != 0;
        } else {
            Float p = hg_sample_p(it.g, it.wo, &wi, uscatt);
            f = Spectrum(p); scattpdf = p;
        }
        if (!f.is_black() && scattpdf > 0.0f) {
            Float weight = 1.0f;
            if (!sampled_specular) {
                lightpdf = light_pdf_li(s, li, it.ref, wi);
                if (lightpdf == 0.0f) return Ld;
                weight = power_heuristic(1, scattpdf, 1, lightpdf);
            }
            VolRay vr;
            vr.r = spawn_ray(it.ref.p, it.ref.p_error, it.ref.n, wi, it.ref.time);
            vr.medium = medium_for(it.mi, it.ref.n, wi);
            Hit h; Ray r_hit; Spectrum Tr;
            bool found = intersect_tr(s, gt, vr, &h, &r_hit, &Tr, rc, sampler, gave_up);
            if (gave_up) return Ld;
            Spectrum li_(0.0f);
            if (found) {
                if (s.d.prims[h.slot].area_light == li) {
                    SurfaceInteraction lsi = make_interaction(s, r_hit, h);
                    li_ = surface_le(s, lsi, -wi);
                }
            } else li_ = light_le(s, li);
            if (!li_.is_black()) Ld += f * li_ * Tr * weight / scattpdf;
        }
    }
    return Ld;
}

// uniform_sample_onelight(handle_media = true), integrator.rs:81-106
inline Spectrum vol_uniform_sample_onelight(const RenderScene& s, const GridTable& gt, const VolVertex& it, Sampler& sampler, const Distribution1D& distrib, RenderCounters& rc,
                                            bool& gave_up) {
    size_t nlights = s.d.n_lights;
    if (nlights == 0) return Spectrum(0.0f);
    Float lightpdf = 0.0f;
    size_t lightnum = distrib.sample_discrete(sampler.get_1d(), &lightpdf);
    if (lightpdf == 0.0f) return Spectrum(0.0f);
    P2 ulight = sampler.get_2d();
    P2 uscattering = sampler.get_2d();
    return vol_estimate_direct(s, gt, it, uscattering, (int)lightnum, ulight, rc, sampler, gave_up) / lightpdf;
}

// VolPathIntegrator::li, volpath.rs:82-221 (no BSSRDF: none of the five materials has one)
inline Spectrum volpath_li(const RenderScene& s, const GridTable& gt, const IntegratorParams& ip, Ray ray0, int camera_medium, Sampler& sampler, RenderCounters& rc) {
    Spectrum L(0.0f), beta(1.0f);
    VolRay ray; ray.r = ray0; ray.medium = camera_medium;
    bool specular_bounce = false;
    uint64_t bounces = 0;  // usize: `bounces -= 1` at 0 wraps in a release build (see the header note)
    const uint64_t max_depth = (uint64_t)std::max(ip.max_depth, 0);
    Float etascale = 1.0f;
    for (;;) {
        Hit h;
        Ray r0 = ray.r;
        rc.intersection_tests++;
        bool found = scene_intersect(s, ray.r, &h, &rc.trav_closest);
        SurfaceInteraction isect;
        if (found) isect = make_interaction(s, r0, h);
        // HomogeneousMedium::sample, homogeneous.rs:35-72
        bool mi_valid = false, gave_up = false;
        V3 mi_p;
        if (ray.medium >= 0 && s.d.media[ray.medium].grid > 0) {  // GridDensityMedium::sample
            Spectrum w;
            mi_valid = grid_sample(s, gt, s.d.media[ray.medium], ray.r, sampler, &mi_p, &w, gave_up);
            if (gave_up) break;
            beta *= w;
        } else if (ray.medium >= 0) {
            const pbrt_b200_medium& m = s.d.media[ray.medium];
            Spectrum sigma_t = medium_sigma_t(m), sigma_s = spec3(m.sigma_s);
            int channel = (int)std::min<uint64_t>(f2u_sat(sampler.get_1d() * 3.0f), 2);
            Float dist = -std::log(1.0f - sampler.get_1d()) / sigma_t.c[channel];
            Float dlen = length(ray.r.d);
            Float t = std::fmin(dist / dlen, ray.r.t_max);
            bool sampled_medium = t < ray.r.t_max;
            if (sampled_medium) { mi_valid = true; mi_p = ray.r.o + ray.r.d * t; }
            Spectrum Tr = spec_exp(spec_neg(sigma_t) * std::fmin(t, std::numeric_limits<Float>::max()) * dlen);
            Spectrum density = sampled_medium ? sigma_t * Tr : Tr;
            Float pdf = 0.0f;
            for (int i = 0; i < 3; ++i) pdf += density.c[i];
            pdf *= 1.0f / 3.0f;
            if (pdf == 0.0f) pdf = 1.0f;
            beta *= sampled_medium ? Tr * sigma_s / pdf : Tr / pdf;
        }
        if (beta.is_black()) break;
        if (mi_valid) {
            if (bounces >= max_depth) break;
            const Distribution1D& distrib = ip.lookup(mi_p);
            VolVertex v;
            v.surface = false;
            v.ref.p = mi_p; v.ref.p_error = V3(0, 0, 0); v.ref.n = V3(0, 0, 0); v.ref.time = ray.r.time;
            v.wo = -ray.r.d; v.g = s.d.media[ray.medium].g;
            v.mi.inside = v.mi.outside = ray.medium;  // MediumInterface::new(medium)
            Spectrum Ld = beta * vol_uniform_sample_onelight(s, gt, v, sampler, distrib, rc, gave_up);
            if (Ld.is_black()) rc.zero_radiance++;
            L += Ld;
            if (gave_up) break;
            V3 wi;
            hg_sample_p(v.g, v.wo, &wi, sampler.get_2d());
            int med = ray.medium;
            ray.r = spawn_ray(mi_p, V3(0, 0, 0), V3(0, 0, 0), wi, ray.r.time);
            ray.medium = med;
            specular_bounce = false;
        } else {
            if (bounces == 0 || specular_bounce) {
                if (found) L += surface_le(s, isect, -ray.r.d) * beta;
                else for (int li : s.infinite_lights) L += light_le(s, li) * beta;
            }
            if (!found || bounces >= max_depth) break;
            BSDF bsdf;
            int mat = s.d.prims[h.slot].material;
            (void)mat;
            scattering_functions(s, ray.r, h.slot, isect, &bsdf, true);
            VolInterface mif = hit_interface(s, h.slot, ray.medium);
            if (!bsdf.valid) {  // volpath.rs:131-135
                V3 d = ray.r.d;
                ray.r = spawn_ray(isect.p, isect.p_error, isect.n, d, isect.time);
                ray.medium = medium_for(mif, isect.n, d);
                bounces -= 1;   // wraps at 0, and the `continue` skips the increment below
                continue;
            }
            const Distribution1D& distrib = ip.lookup(isect.p);
            VolVertex v;
            v.surface = true;
            v.ref.p = isect.p; v.ref.p_error = isect.p_error; v.ref.n = isect.n; v.ref.time = isect.time;
            v.wo = isect.wo; v.sh_n = isect.sh_n; v.bsdf = &bsdf; v.mi = mif;
            Spectrum Ld = beta * vol_uniform_sample_onelight(s, gt, v, sampler, distrib, rc, gave_up);
            if (Ld.is_black()) rc.zero_radiance++;
            L += Ld;
            if (gave_up) break;
            V3 wo = -ray.r.d, wi;
            Float pdf = 0.0f;
            int flags = 0;
            Spectrum f = bsdf.sample_f(wo, &wi, sampler.get_2d(), &pdf, BSDF_ALL, &flags);
            if (f.is_black() || pdf == 0.0f) break;
            beta *= f * abs_dot(wi, isect.sh_n) / pdf;
            specular_bounce = (flags & BSDF_SPECULAR) != 0;
            if ((flags & BSDF_SPECULAR) && (flags & BSDF_TRANSMISSION)) {
                Float eta = bsdf.eta;
                etascale *= (dot(wo, isect.n) > 0.0f) ? eta * eta : 1.0f / (eta * eta);
            }
            ray.r = spawn_ray(isect.p, isect.p_error, isect.n, wi, isect.time);
            ray.medium = medium_for(mif, isect.n, wi);
        }
        Spectrum rrbeta = beta * etascale;
        if (rrbeta.max_component_value() < ip.rr_threshold && bounces > 3) {
            Float q = std::fmax(1.0f - rrbeta.max_component_value(), 0.05f);
            if (sampler.get_1d() < q) break;
            beta = beta / (1.0f - q);
        }
        bounces += 1;
    }
    return L;
}


// SamplerIntegrator::render of oracle_render.hpp with VolPathIntegrator::li of this file (volpath only)
inline void render(const RenderJob& job, const GridTable& gt, float* rgbw, int nthreads, RenderCounters* total) {
    const pbrt_b200_render_desc& rd = job.rd;
    const int* sb = rd.sampler.sample_bounds;
    const int tilesize = 16;
    int ntx = (sb[2] - sb[0] + tilesize - 1) / tilesize, nty = (sb[3] - sb[1] + tilesize - 1) / tilesize;
    // pbrt_b200_render_desc.tile_order (include/pbrt_b200.h): 0 = the reference's row-major tile numbering; S = S x S-tile super-tiles
    const uint32_t S = rd.tile_order, nstx = S ? (uint32_t)((ntx + (int)S - 1) / (int)S) : 0u, nsty = S ? (uint32_t)((nty + (int)S - 1) / (int)S) : 0u;
    const uint32_t n_positions = S ? nstx * nsty * S * S : (uint32_t)(ntx * nty);
    uint32_t tile_begin = rd.tile_begin, tile_end = rd.tile_end ? rd.tile_end : n_positions;
    uint32_t s_begin = rd.sample_begin, s_end = rd.sample_end ? rd.sample_end : 0xffffffffu;  // 0 => until start_next_sample() says stop
    FilmAccum acc; acc.init(&rd.film);
    std::mutex mu;
    std::atomic<uint32_t> next(tile_begin);
    std::vector<RenderCounters> rcs(nthreads);
    auto worker = [&](int tid) {
        RenderCounters& rc = rcs[tid];
        std::unique_ptr<Sampler> base = make_sampler(rd.sampler, job.tables);
        IntegratorParams ipl = job.ip;
        std::vector<double> local;
        for (;;) {
            uint32_t tile = next.fetch_add(1);
            if (tile >= tile_end) break;
            {   // interleaved tile ownership (pbrt_b200_render_desc.tile_group/mod/rem)
                uint32_t g = rd.tile_group ? rd.tile_group : 1u, m = rd.tile_mod ? rd.tile_mod : 1u;
                if (((tile - tile_begin) / g) % m != rd.tile_rem) continue;
            }
            int tx = tile % ntx, ty = tile / ntx;
            if (S) {
                const uint32_t st = tile / (S * S), w = tile - st * (S * S);
                tx = (int)((st % nstx) * S + w % S); ty = (int)((st / nstx) * S + w / S);
                if (tx >= ntx || ty >= nty) continue;  // position past the image edge
            }
            std::unique_ptr<Sampler> ts = base->clone((int64_t)ty * ntx + tx);
            int x0 = sb[0] + tx * tilesize, x1 = std::min(x0 + tilesize, sb[2]);
            int y0 = sb[1] + ty * tilesize, y1 = std::min(y0 + tilesize, sb[3]);
            struct Contrib { int x, y; Spectrum c; Float w; };
            std::vector<Contrib> contribs;
            for (int y = y0; y < y1; ++y)
                for (int x = x0; x < x1; ++x) {
                    ts->start_pixel(x, y);
                    const int* pb = job.ip.pixel_bounds;
                    if (!(x >= pb[0] && x < pb[2] && y >= pb[1] && y < pb[3])) continue;
                    bool more = true;
                    if (s_begin > 0) more = ts->set_sample_number(s_begin);
                    while (more) {
                        if (ts->current_pixel_sample_index >= s_end) break;
                        CameraSample cs = ts->get_camera_sample(x, y);
                        Ray ray = generate_ray(rd.camera, cs, rd.sampler.samples_per_pixel);
                        rc.camera_rays++;
                        Spectrum L = volpath_li(job.scene, gt, ipl, ray, rd.integrator.camera_medium, *ts, rc);
                        if (L.has_nans()) L = Spectrum(0.0f);                 // integrator.rs:350-368
                        else if (L.y() < -1.0e-5f) L = Spectrum(0.0f);
                        else if (std::isinf(L.y())) L = Spectrum(0.0f);
                        film_add_sample(rd.film, cs.pfilm, L, 1.0f, [&](int px, int py, Spectrum c, Float fw) { contribs.push_back({px, py, c, fw}); });
                        more = ts->start_next_sample();
                    }
                }
            std::lock_guard<std::mutex> g(mu);
            for (auto& c : contribs) {
                size_t o = 4 * ((size_t)(c.y - acc.y0) * acc.width + (c.x - acc.x0));
                acc.sum[o] += c.c.c[0]; acc.sum[o + 1] += c.c.c[1]; acc.sum[o + 2] += c.c.c[2]; acc.sum[o + 3] += c.w;
            }
        }
    };
    std::vector<std::thread> th;
    for (int t = 0; t < nthreads; ++t) th.emplace_back(worker, t);
    for (auto& t : th) t.join();
    for (size_t i = 0; i < acc.sum.size(); ++i) rgbw[i] += (float)acc.sum[i];
    if (total)
        for (auto& rc : rcs) {
            total->camera_rays += rc.camera_rays; total->intersection_tests += rc.intersection_tests; total->shadow_tests += rc.shadow_tests;
            total->zero_radiance += rc.zero_radiance; total->direct_den += rc.direct_den;
            total->trav_closest.nodes_tested += rc.trav_closest.nodes_tested; total->trav_closest.tris_tested += rc.trav_closest.tris_tested;
            total->trav_closest.rays += rc.trav_closest.rays;
            total->trav_any.nodes_tested += rc.trav_any.nodes_tested; total->trav_any.tris_tested += rc.trav_any.tris_tested; total->trav_any.rays += rc.trav_any.rays;
        }
}

}  // namespace grid_media
}  // namespace orc
