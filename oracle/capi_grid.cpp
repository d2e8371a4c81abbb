// TEST INFRASTRUCTURE -- NOT PRODUCT CODE (see oracle_math.hpp header).
// C entry points of the grid-media oracle (oracle_grid.hpp), a library of its own (liboracle_grid.so, built by oracle_grid.py),
// loaded with ctypes by tests/ only.
#include <thread>
#include <vector>
#include <atomic>
#include <cstdio>
#include "oracle_accel.hpp"
#include "oracle_grid.hpp"

using namespace orc;

extern "C" {

// SamplerIntegrator::render with VolPathIntegrator::li for a scene whose media rows may refer to grids[n_grids]
// (pbrt_b200_medium.grid = k > 0: grids[k - 1]).  stats_out[12] as orc_render (oracle/capi.cpp).
int orc_grid_render(const pbrt_b200_scene_desc* sdesc, const pbrt_b200_render_desc* rd, float* rgbw, int nthreads, uint64_t* stats_out,
                    const pbrt_b200_density_grid* grids, uint64_t n_grids) {
    if (rd->integrator.kind != PBRT_B200_INTEGRATOR_VOLPATH) return 1;
    RenderJob job;
    setup_job(job, *sdesc, *rd);
    const grid_media::GridTable gt(grids, n_grids);
    RenderCounters rc;
    grid_media::render(job, gt, rgbw, nthreads <= 0 ? (int)std::max(1u, std::thread::hardware_concurrency()) : nthreads, &rc);
    if (stats_out) {
        uint64_t v[12] = {rc.camera_rays, rc.intersection_tests, rc.shadow_tests, rc.zero_radiance, rc.direct_den,
                          rc.trav_closest.nodes_tested, rc.trav_closest.tris_tested, rc.trav_closest.rays,
                          rc.trav_any.nodes_tested, rc.trav_any.tris_tested, rc.trav_any.rays, 0};
        std::memcpy(stats_out, v, sizeof v);
    }
    return 0;
}

// GridDensityMedium::density (grid.rs) of `grid` at n medium-space points
int orc_grid_density(const pbrt_b200_density_grid* grid, const float* points, uint64_t n, float* out) {
    for (uint64_t i = 0; i < n; ++i) out[i] = grid_media::grid_density(*grid, V3(points[3 * i], points[3 * i + 1], points[3 * i + 2]));
    return 0;
}

}  // extern "C"
