// TEST INFRASTRUCTURE -- NOT PRODUCT CODE (see oracle_math.hpp header).
// C entry point of the BDPT oracle (oracle_bdpt.hpp), a library of its own (liboracle_bdpt.so, built by oracle_bdpt.py), loaded with
// ctypes by tests/ only.
#include <thread>
#include <vector>
#include <atomic>
#include <mutex>
#include <cstdio>
#include "oracle_accel.hpp"
#include "oracle_sampling_extra.hpp"
#include "oracle_bdpt.hpp"

using namespace orc;

extern "C" {

// BDPTIntegrator::render (pbrt-v3 bdpt.cpp:318-446) with the tile / sample / interleave windows of orc_render.  rgbw [npix * 4] and
// splat [npix * 3] (RGB, cropped bounds) are ADDED to.  strategies != nullptr: per-(s, t) films (pbrt-v3's visualizestrategies /
// visualizeweights): strategies[k] is a film of npix * 3 RGB sums for strategy k = s + d * (5 + d) / 2 with d = s + t - 2 <= max_depth (pbrt-v3 BufferIndex),
// unweighted (weighted = 0) or multiplied by the MIS weight.  stats_out[12] as orc_render (oracle/capi.cpp).
int orc_bdpt_render(const pbrt_b200_scene_desc* sdesc, const pbrt_b200_render_desc* rd, float* rgbw, float* splat, int nthreads, uint64_t* stats_out,
                    float* strategies, int weighted) {
    if (rd->integrator.kind != PBRT_B200_INTEGRATOR_BDPT || rd->integrator.max_depth < 0) return 1;
    if (rd->sampler.kind == PBRT_B200_SAMPLER_ZEROTWO) return 2;
    RenderJob job;
    setup_job(job, *sdesc, *rd);
    if (nthreads <= 0) nthreads = (int)std::max(1u, std::thread::hardware_concurrency());
    const int max_depth = rd->integrator.max_depth;
    bdpt::CameraImp cam;
    cam.init(rd->camera, rd->film, rd->sampler.sample_bounds);
    const int* sb = rd->sampler.sample_bounds;
    const int tilesize = 16;
    int ntx = (sb[2] - sb[0] + tilesize - 1) / tilesize, nty = (sb[3] - sb[1] + tilesize - 1) / tilesize;
    const uint32_t S = rd->tile_order, nstx = S ? (uint32_t)((ntx + (int)S - 1) / (int)S) : 0u, nsty = S ? (uint32_t)((nty + (int)S - 1) / (int)S) : 0u;
    const uint32_t n_positions = S ? nstx * nsty * S * S : (uint32_t)(ntx * nty);
    uint32_t tile_begin = rd->tile_begin, tile_end = rd->tile_end ? rd->tile_end : n_positions;
    uint32_t s_begin = rd->sample_begin, s_end = rd->sample_end ? rd->sample_end : 0xffffffffu;
    FilmAccum acc; acc.init(&rd->film);
    const size_t npix = (size_t)acc.width * (acc.y1 - acc.y0);
    const int nstrat = (max_depth + 1) * (max_depth + 6) / 2;
    std::vector<double> splat_sum(3 * npix, 0.0), strat_sum(strategies ? (size_t)nstrat * 3 * npix : 0, 0.0);
    std::mutex mu;
    std::atomic<uint32_t> next(tile_begin);
    std::vector<RenderCounters> rcs(nthreads);
    auto worker = [&](int tid) {
        RenderCounters& rc = rcs[tid];
        std::unique_ptr<Sampler> base = make_sampler(rd->sampler, job.tables);
        std::vector<bdpt::Vertex> cv(max_depth + 2), lv(max_depth + 1);
        struct Contrib { int x, y; Spectrum c; Float w; };
        struct Splat { int k; int x, y; Spectrum c; };  // k = -1: the splat film, else a strategy film
        for (;;) {
            uint32_t tile = next.fetch_add(1);
            if (tile >= tile_end) break;
            {
                uint32_t g = rd->tile_group ? rd->tile_group : 1u, m = rd->tile_mod ? rd->tile_mod : 1u;
                if (((tile - tile_begin) / g) % m != rd->tile_rem) continue;
            }
            int tx = tile % ntx, ty = tile / ntx;
            if (S) {
                const uint32_t st = tile / (S * S), w = tile - st * (S * S);
                tx = (int)((st % nstx) * S + w % S); ty = (int)((st / nstx) * S + w / S);
                if (tx >= ntx || ty >= nty) continue;
            }
            std::unique_ptr<Sampler> ts = base->clone((int64_t)ty * ntx + tx);
            int x0 = sb[0] + tx * tilesize, x1 = std::min(x0 + tilesize, sb[2]);
            int y0 = sb[1] + ty * tilesize, y1 = std::min(y0 + tilesize, sb[3]);
            std::vector<Contrib> contribs;
            std::vector<Splat> splats;
            auto add_splat = [&](int k, P2 p, Spectrum v) {  // Film::add_splat (pbrt-v3 film.cpp:126-146)
                if (v.has_nans() || v.y() < 0.0f || std::isinf(v.y())) return;
                int px = (int)std::floor(p.x), py = (int)std::floor(p.y);
                if (!(px >= acc.x0 && px < acc.x1 && py >= acc.y0 && py < acc.y1)) return;
                if (v.y() > rd->film.max_sample_luminance) v *= Spectrum(rd->film.max_sample_luminance / v.y());
                splats.push_back({k, px, py, v});
            };
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
                        Ray ray = generate_ray(rd->camera, cs, rd->sampler.samples_per_pixel);
                        rc.camera_rays++;
                        const Distribution1D* ld = &job.ip.light_distrib;
                        bdpt::Ctx c0{job.scene, job.ip, *ld, cam, rc};
                        int nc = bdpt::camera_subpath(c0, *ts, max_depth + 2, ray, cv.data());
                        ld = &job.ip.lookup(cv[0].p);  // SpatialLightDistribution: looked up at the camera vertex
                        bdpt::Ctx c{job.scene, job.ip, *ld, cam, rc};
                        int nl = job.scene.d.n_lights ? bdpt::light_subpath(c, *ts, max_depth + 1, cv[0].time, lv.data()) : 0;
                        Spectrum L(0.0f);
                        for (int t = 1; t <= nc; ++t)
                            for (int s = 0; s <= nl; ++s) {
                                int depth = t + s - 2;
                                if ((s == 1 && t == 1) || depth < 0 || depth > max_depth) continue;
                                P2 praster = cs.pfilm;
                                Float w = 0.0f;
                                Spectrum Lp = bdpt::connect(c, lv.data(), cv.data(), s, t, *ts, &praster, &w);
                                if (strategies) {
                                    Spectrum v = weighted ? Lp : (w != 0.0f ? Lp / Spectrum(w) : Spectrum(0.0f));
                                    int k = s + depth * (5 + depth) / 2;
                                    add_splat(k, t == 1 ? praster : cs.pfilm, v);
                                }
                                if (t != 1) L += Lp;
                                else add_splat(-1, praster, Lp);
                            }
                        if (L.has_nans()) L = Spectrum(0.0f);
                        else if (L.y() < -1.0e-5f) L = Spectrum(0.0f);
                        else if (std::isinf(L.y())) L = Spectrum(0.0f);
                        film_add_sample(rd->film, cs.pfilm, L, 1.0f, [&](int px, int py, Spectrum cc, Float fw) { contribs.push_back({px, py, cc, fw}); });
                        more = ts->start_next_sample();
                    }
                }
            std::lock_guard<std::mutex> g(mu);
            for (auto& e : contribs) {
                size_t o = 4 * ((size_t)(e.y - acc.y0) * acc.width + (e.x - acc.x0));
                acc.sum[o] += e.c.c[0]; acc.sum[o + 1] += e.c.c[1]; acc.sum[o + 2] += e.c.c[2]; acc.sum[o + 3] += e.w;
            }
            for (auto& e : splats) {
                if (e.x < acc.x0 || e.x >= acc.x1 || e.y < acc.y0 || e.y >= acc.y1) continue;
                size_t o = 3 * ((size_t)(e.y - acc.y0) * acc.width + (e.x - acc.x0));
                double* dst = e.k < 0 ? splat_sum.data() : strat_sum.data() + (size_t)e.k * 3 * npix;
                dst[o] += e.c.c[0]; dst[o + 1] += e.c.c[1]; dst[o + 2] += e.c.c[2];
            }
        }
    };
    std::vector<std::thread> th;
    for (int t = 0; t < nthreads; ++t) th.emplace_back(worker, t);
    for (auto& t : th) t.join();
    for (size_t i = 0; i < acc.sum.size(); ++i) rgbw[i] += (float)acc.sum[i];
    if (splat) for (size_t i = 0; i < splat_sum.size(); ++i) splat[i] += (float)splat_sum[i];
    if (strategies) for (size_t i = 0; i < strat_sum.size(); ++i) strategies[i] += (float)strat_sum[i];
    RenderCounters tot;
    for (auto& r : rcs) {
        tot.camera_rays += r.camera_rays; tot.intersection_tests += r.intersection_tests; tot.shadow_tests += r.shadow_tests;
        tot.trav_closest.nodes_tested += r.trav_closest.nodes_tested; tot.trav_closest.tris_tested += r.trav_closest.tris_tested; tot.trav_closest.rays += r.trav_closest.rays;
    }
    if (stats_out) {
        uint64_t v[12] = {tot.camera_rays, tot.intersection_tests, tot.shadow_tests, 0, 0, tot.trav_closest.nodes_tested, tot.trav_closest.tris_tested,
                          tot.trav_closest.rays, 0, 0, 0, 0};
        std::memcpy(stats_out, v, sizeof v);
    }
    return 0;
}

}  // extern "C"
