// C-ABI entry points: scene upload and the batch intersect API (include/pbrt_b200.h).
#include <cuda_runtime.h>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <type_traits>

#include "error.h"
#include "pool.h"
#include "scene.cuh"
#include "trace.cuh"
#include "util.cuh"

using namespace pb;

namespace pb {
void render_release_scene_state(pbrt_b200_scene* scene);  // render.cu
}

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
// Persistent warps pull rays from the batch (trace.cuh: trace_queue); rays are 32-byte records
// read as two float4 (128-bit loads), hits are written as one uint4.
struct BatchClosestJob {
    const float4* rays; uint4* hits; const float4* tris;
    PB_D bool load(uint32_t i, f3* o, f3* d, float* t_max) const {
        float4 a = __ldg(rays + 2ull * i), b = __ldg(rays + 2ull * i + 1);
        *o = f3(a.x, a.y, a.z); *d = f3(b.x, b.y, b.z); *t_max = a.w;
        return true;
    }
    PB_D void store(uint32_t i, const TravRay& r) const {
        uint4 out;
        if (r.found) {
            out.x = __float_as_uint(__ldg(tris + 3ull * r.hit.slot).w);  // creation_index
            out.y = __float_as_uint(r.hit.t); out.z = __float_as_uint(r.hit.b0); out.w = __float_as_uint(r.hit.b1);
        } else {
            out.x = PBRT_B200_NO_HIT; out.y = __float_as_uint(r.hit.t); out.z = 0u; out.w = 0u;
        }
        hits[i] = out;
    }
};
struct BatchAnyJob {
    const float4* rays; uint8_t* occluded;
    PB_D bool load(uint32_t i, f3* o, f3* d, float* t_max) const {
        float4 a = __ldg(rays + 2ull * i), b = __ldg(rays + 2ull * i + 1);
        *o = f3(a.x, a.y, a.z); *d = f3(b.x, b.y, b.z); *t_max = a.w;
        return true;
    }
    PB_D void store(uint32_t i, const TravRay& r) const { occluded[i] = r.found ? 1 : 0; }
};

template <bool INST>
__global__ void __launch_bounds__(PB_TRACE_BLOCK) k_intersect_batch(DevScene s, const float4* __restrict__ rays, uint32_t n, uint4* __restrict__ hits,
                                                                   uint32_t* fetch, TraceTune tune) {
    BatchClosestJob job{rays, hits, s.tris};
    trace_queue<false, INST>(s, job, n, fetch, tune);
}
// Packet mode (trace.cuh: trace_queue_packet), scenes without instances, with PBRT_B200_PACKET_TRAVERSAL=2 only: a batch is
// incoherent in general, so the batch API keeps the per-lane walk
__global__ void __launch_bounds__(PB_TRACE_BLOCK) k_intersect_batch_packet(DevScene s, const float4* __restrict__ rays, uint32_t n, uint4* __restrict__ hits,
                                                                          uint32_t* fetch) {
    BatchClosestJob job{rays, hits, s.tris};
    trace_queue_packet<false>(s, job, n, fetch);
}

// A/B variants for tuning (tools/trace_ab.py): one ray per thread, while-while or if-if
template <int VARIANT>
__global__ void __launch_bounds__(PB_TRACE_BLOCK) k_intersect_batch_1rpt(DevScene s, const float4* __restrict__ rays, uint32_t n, uint4* __restrict__ hits) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    BatchClosestJob job{rays, hits, s.tris};
    f3 o, d; float t_max;
    job.load(i, &o, &d, &t_max);
    TravRay r;
    r.found = VARIANT == 0 ? traverse<false>(s, o, d, t_max, &r.hit) : traverse_ifif<false>(s, o, d, t_max, &r.hit);
    job.store(i, r);
}

template <bool INST>
__global__ void __launch_bounds__(PB_TRACE_BLOCK) k_intersect_p_batch(DevScene s, const float4* __restrict__ rays, uint32_t n, uint8_t* __restrict__ occluded,
                                                                     uint32_t* fetch) {
    BatchAnyJob job{rays, occluded};
    trace_queue<true, INST>(s, job, n, fetch);
}
__global__ void __launch_bounds__(PB_TRACE_BLOCK) k_intersect_p_batch_packet(DevScene s, const float4* __restrict__ rays, uint32_t n,
                                                                            uint8_t* __restrict__ occluded, uint32_t* fetch) {
    BatchAnyJob job{rays, occluded};
    trace_queue_packet<true>(s, job, n, fetch);
}

namespace {
// PBRT_B200_PACKET_TRAVERSAL=2 (read per call): the batch entry points walk aligned runs of 32 rays as packets
bool batch_packet() {
    const char* e = getenv("PBRT_B200_PACKET_TRAVERSAL");
    return e && atoi(e) == 2;
}
}  // namespace

// ---------------------------------------------------------------------------
// scene
// ---------------------------------------------------------------------------
// Device-side construction of the traversal layout from the reference's own tables (scene.cuh).
//   k_leaf_records : GeometricPrimitive rows + TriangleMesh SoA -> 48-byte leaf records in BVH slot order
//   k_interior_*   : exclusive scan of "node is interior" -> index of each interior node in the fat-node array
//   k_fat_nodes    : LinearBVHNode[] -> fat nodes (both child boxes in the parent), LAST flags on leaf records
__global__ void __launch_bounds__(256) k_leaf_records(const pbrt_b200_prim* __restrict__ prims, uint32_t n, const uint32_t* __restrict__ tri_indices,
                                                      const float* __restrict__ vertex_p, float4* __restrict__ tris, const float* __restrict__ vertex_n,
                                                      const float* __restrict__ vertex_uv, float4* __restrict__ slot_n, float2* __restrict__ slot_uv) {
    for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < n; s += gridDim.x * blockDim.x) {
        const pbrt_b200_prim p = prims[s];
        uint32_t fl = p.flags & PB_TRI_FLAGS_MASK;
        float4 v[3] = {make_float4(0, 0, 0, 0), make_float4(0, 0, 0, 0), make_float4(0, 0, 0, 0)};
        float4 nn[3] = {make_float4(0, 0, 0, 0), make_float4(0, 0, 0, 0), make_float4(0, 0, 0, 0)};
        float2 uu[3] = {make_float2(0, 0), make_float2(0, 0), make_float2(0, 0)};
        if (p.shape_kind == PBRT_B200_SHAPE_TRIANGLE) {
            const uint32_t* ix = tri_indices + 3ull * p.shape_index;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float* vp = vertex_p + 3ull * ix[k];
                v[k].x = vp[0]; v[k].y = vp[1]; v[k].z = vp[2];
                if (slot_n) { const float* np = vertex_n + 3ull * ix[k]; nn[k] = make_float4(np[0], np[1], np[2], 0.0f); }
                if (slot_uv) { const float* up = vertex_uv + 2ull * ix[k]; uu[k] = make_float2(up[0], up[1]); }
            }
        } else if (p.shape_kind == PBRT_B200_SHAPE_INSTANCE) {
            fl |= PB_TRI_INSTANCE;
        } else {
            fl |= PB_TRI_SPHERE;
        }
        v[0].w = __uint_as_float(p.creation_index);
        v[1].w = __uint_as_float(fl);
        v[2].w = __uint_as_float(p.shape_index);
        tris[3ull * s] = v[0]; tris[3ull * s + 1] = v[1]; tris[3ull * s + 2] = v[2];
        if (slot_n) { slot_n[3ull * s] = nn[0]; slot_n[3ull * s + 1] = nn[1]; slot_n[3ull * s + 2] = nn[2]; }
        if (slot_uv) { slot_uv[3ull * s] = uu[0]; slot_uv[3ull * s + 1] = uu[1]; slot_uv[3ull * s + 2] = uu[2]; }
    }
}
// DevScene::light_tris: vertices and normals of the triangle behind each diffuse area light
__global__ void __launch_bounds__(128) k_light_tris(const pbrt_b200_light* __restrict__ lights, uint32_t n, const uint32_t* __restrict__ tri_indices,
                                                    const float* __restrict__ vertex_p, const float* __restrict__ vertex_n, float4* __restrict__ out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 r[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) r[k] = make_float4(0, 0, 0, 0);
        const pbrt_b200_light l = lights[i];
        if (l.type == PBRT_B200_LIGHT_DIFFUSE && l.shape_kind == PBRT_B200_SHAPE_TRIANGLE) {
            const uint32_t* ix = tri_indices + 3ull * l.shape_index;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float* vp = vertex_p + 3ull * ix[k];
                r[k] = make_float4(vp[0], vp[1], vp[2], 0.0f);
                if (vertex_n) { const float* np = vertex_n + 3ull * ix[k]; r[3 + k] = make_float4(np[0], np[1], np[2], 0.0f); }
            }
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) out[6ull * i + k] = r[k];
    }
}

#define PB_SCAN_BLOCK 1024
PB_D uint32_t node_is_interior(const pbrt_b200_bvh_node* nodes, uint32_t i, uint32_t n) { return (i < n && nodes[i].n_prims == 0) ? 1u : 0u; }
// block-wide exclusive scan of one flag per thread; returns the exclusive prefix, *total = block sum
PB_D uint32_t block_exclusive_scan(uint32_t v, uint32_t* total) {
    __shared__ uint32_t warp_sums[32];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= (unsigned)o) inc += t; }
    if (lane == 31) warp_sums[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < (blockDim.x >> 5) ? warp_sums[lane] : 0u, winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= (unsigned)o) winc += t; }
        warp_sums[lane] = winc - w;  // exclusive
        if (lane == 31) *total = winc;
    }
    __syncthreads();
    uint32_t r = inc - v + warp_sums[warp];
    __syncthreads();
    return r;
}
__global__ void __launch_bounds__(PB_SCAN_BLOCK) k_interior_count(const pbrt_b200_bvh_node* __restrict__ nodes, uint32_t n, uint32_t* __restrict__ block_sums) {
    __shared__ uint32_t total;
    block_exclusive_scan(node_is_interior(nodes, blockIdx.x * PB_SCAN_BLOCK + threadIdx.x, n), &total);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}
__global__ void __launch_bounds__(PB_SCAN_BLOCK) k_interior_scan_blocks(uint32_t* __restrict__ block_sums, uint32_t nb) {
    __shared__ uint32_t total, carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < nb; base += PB_SCAN_BLOCK) {
        uint32_t i = base + threadIdx.x;
        uint32_t v = i < nb ? block_sums[i] : 0u;
        uint32_t ex = block_exclusive_scan(v, &total);
        if (i < nb) block_sums[i] = ex + carry;
        __syncthreads();
        if (threadIdx.x == 0) carry += total;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(PB_SCAN_BLOCK) k_interior_index(const pbrt_b200_bvh_node* __restrict__ nodes, uint32_t n, const uint32_t* __restrict__ block_sums,
                                                                 uint32_t* __restrict__ fat_index) {
    __shared__ uint32_t total;
    uint32_t i = blockIdx.x * PB_SCAN_BLOCK + threadIdx.x;
    uint32_t ex = block_exclusive_scan(node_is_interior(nodes, i, n), &total);
    if (i < n) fat_index[i] = ex + block_sums[blockIdx.x];
}
// One accelerator (the scene's aggregate or one instanced object): nodes [node_base, node_base + n), whose `offset`s are
// relative to node_base (second child) / prim_base (first primitive).  Child refs written to the fat nodes are global.
__global__ void __launch_bounds__(256) k_fat_nodes(const pbrt_b200_bvh_node* __restrict__ nodes, uint32_t node_base, uint32_t n, uint32_t prim_base,
                                                   const uint32_t* __restrict__ fat_index, float4* __restrict__ fat, float4* __restrict__ tris) {
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const uint32_t i = node_base + k;
        const pbrt_b200_bvh_node nd = nodes[i];
        if (nd.n_prims != 0) {  // leaf: the last primitive of the run carries PB_TRI_LAST
            float4* rec = tris + 3ull * (prim_base + nd.offset + nd.n_prims - 1) + 1;
            rec->w = __uint_as_float(__float_as_uint(rec->w) | PB_TRI_LAST);
            continue;
        }
        const uint32_t c0 = i + 1, c1 = node_base + nd.offset;
        const pbrt_b200_bvh_node a = nodes[c0], b = nodes[c1];
        const uint32_t r0 = a.n_prims ? (PB_LEAF_BIT | (prim_base + a.offset)) : fat_index[c0];
        const uint32_t r1 = b.n_prims ? (PB_LEAF_BIT | (prim_base + b.offset)) : fat_index[c1];
        float4* q = fat + 4ull * fat_index[i];
        q[0] = make_float4(a.bounds[0], a.bounds[1], a.bounds[2], a.bounds[3]);
        q[1] = make_float4(a.bounds[4], a.bounds[5], b.bounds[0], b.bounds[1]);
        q[2] = make_float4(b.bounds[2], b.bounds[3], b.bounds[4], b.bounds[5]);
        q[3] = make_float4(__uint_as_float(r0), __uint_as_float(r1), __uint_as_float((uint32_t)nd.axis), 0.0f);
    }
}

// fat nodes -> quad nodes (scene.cuh): quad[i] = the children of fat[i]'s two children
__global__ void __launch_bounds__(256) k_quad_nodes(const float4* __restrict__ fat, uint32_t n_fat, float4* __restrict__ quads) {
    const float INF = __int_as_float(0x7f800000);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_fat; i += gridDim.x * blockDim.x) {
        const float4 p0 = fat[4ull * i], p1 = fat[4ull * i + 1], p2 = fat[4ull * i + 2], p3 = fat[4ull * i + 3];
        const uint32_t cref[2] = {__float_as_uint(p3.x), __float_as_uint(p3.y)};
        const float cbox[2][6] = {{p0.x, p0.y, p0.z, p0.w, p1.x, p1.y}, {p1.z, p1.w, p2.x, p2.y, p2.z, p2.w}};
        float lo[4][3], hi[4][3];
        uint32_t ref[4], axis[2] = {0u, 0u};
        for (int c = 0; c < 2; ++c) {
            if (cref[c] & PB_LEAF_BIT) {  // a leaf child occupies one slot
                for (int a = 0; a < 3; ++a) { lo[2 * c][a] = cbox[c][a]; hi[2 * c][a] = cbox[c][3 + a]; lo[2 * c + 1][a] = INF; hi[2 * c + 1][a] = -INF; }
                ref[2 * c] = cref[c]; ref[2 * c + 1] = PB_REF_NONE;
            } else {
                const float4 g0 = fat[4ull * cref[c]], g1 = fat[4ull * cref[c] + 1], g2 = fat[4ull * cref[c] + 2], g3 = fat[4ull * cref[c] + 3];
                const float gb[2][6] = {{g0.x, g0.y, g0.z, g0.w, g1.x, g1.y}, {g1.z, g1.w, g2.x, g2.y, g2.z, g2.w}};
                for (int k = 0; k < 2; ++k)
                    for (int a = 0; a < 3; ++a) { lo[2 * c + k][a] = gb[k][a]; hi[2 * c + k][a] = gb[k][3 + a]; }
                ref[2 * c] = __float_as_uint(g3.x); ref[2 * c + 1] = __float_as_uint(g3.y);
                axis[c] = __float_as_uint(g3.z);
            }
        }
        float4* q = quads + 8ull * i;
        for (int pr = 0; pr < 2; ++pr) {
            const int a = 2 * pr, b = 2 * pr + 1;
            q[3 * pr + 0] = make_float4(lo[a][0], lo[b][0], lo[a][1], lo[b][1]);
            q[3 * pr + 1] = make_float4(lo[a][2], lo[b][2], hi[a][0], hi[b][0]);
            q[3 * pr + 2] = make_float4(hi[a][1], hi[b][1], hi[a][2], hi[b][2]);
        }
        q[6] = make_float4(__uint_as_float(ref[0]), __uint_as_float(ref[1]), __uint_as_float(ref[2]), __uint_as_float(ref[3]));
        q[7] = make_float4(__uint_as_float(__float_as_uint(p3.z) | (axis[0] << 2) | (axis[1] << 4)), 0.0f, 0.0f, 0.0f);
    }
}

__global__ void k_single_prim_last(const uint32_t* __restrict__ slots, uint32_t n, float4* __restrict__ tris) {
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        float4* rec = tris + 3ull * slots[k] + 1;
        rec->w = __uint_as_float(__float_as_uint(rec->w) | PB_TRI_LAST);
    }
}

namespace {

// The uploader sizes its copies from the mipmap rows, so these are checked before anything is staged.
int validate_mipmaps(const pbrt_b200_scene_desc* d) {
    if (d->n_mipmaps && !d->mipmaps) return fail(PBRT_B200_ERR_INVALID, "scene_create: mipmaps is null");
    if (d->n_mipmaps > 0x7fffffffull) return fail(PBRT_B200_ERR_INVALID, "scene_create: too many mipmaps");
    for (uint64_t i = 0; i < d->n_mipmaps; ++i) {
        const pbrt_b200_mipmap& m = d->mipmaps[i];
        if (!m.texels || (m.channels != 1 && m.channels != 3) || m.width == 0 || m.height == 0 || (m.width & (m.width - 1)) || (m.height & (m.height - 1)) ||
            m.wrap > PBRT_B200_WRAP_CLAMP || !(m.max_anisotropy >= 0.0f))
            return fail(PBRT_B200_ERR_INVALID, "scene_create: malformed mipmap (power-of-two level 0, 1 or 3 channels, max_anisotropy >= 0)");
        uint32_t big = m.width > m.height ? m.width : m.height, levels = 1;
        while (big > 1) { big >>= 1; levels += 1; }
        if (m.n_levels != levels) return fail(PBRT_B200_ERR_INVALID, "scene_create: mipmap n_levels must be 1 + log2(max(width, height))");
    }
    return PBRT_B200_OK;
}

// Grid shapes are checked before anything is staged (the uploader sizes its copies from them); the values are scanned on the
// table-check thread (validate_grid_values).
int validate_grid_shapes(const pbrt_b200_density_grid* grids, uint64_t n_grids) {
    if (n_grids && !grids) return fail(PBRT_B200_ERR_INVALID, "scene_create: grids is null");
    if (n_grids > 0x7fffffffull) return fail(PBRT_B200_ERR_INVALID, "scene_create: too many density grids");
    for (uint64_t i = 0; i < n_grids; ++i) {
        const pbrt_b200_density_grid& g = grids[i];
        if (!g.density) return fail(PBRT_B200_ERR_INVALID, "scene_create: density grid without density values");
        const uint64_t nxy = (uint64_t)g.nx * g.ny;  // < 2^64: both factors are 32-bit
        if (g.nx == 0 || g.ny == 0 || g.nz == 0 || nxy > (1ull << 40) / g.nz)
            return fail(PBRT_B200_ERR_INVALID, "scene_create: density grid nx * ny * nz must be positive and at most 2^40");
        for (int k = 0; k < 16; ++k)
            if (!std::isfinite(g.medium_to_world[k]) || !std::isfinite(g.world_to_medium[k]))
                return fail(PBRT_B200_ERR_INVALID, "scene_create: density grid matrices must be finite");
    }
    return PBRT_B200_OK;
}

// Every medium row's grid index, then every density (finite, >= 0) and each grid's maximum (GridDensityMedium::new).
int validate_grid_values(const pbrt_b200_scene_desc* d, const pbrt_b200_density_grid* grids, uint64_t n_grids, std::vector<float>* max_density) {
    for (uint64_t i = 0; i < d->n_media; ++i)
        if (d->media[i].grid > n_grids) return fail(PBRT_B200_ERR_INVALID, "scene_create: medium grid index out of range");
    max_density->assign(n_grids, 0.0f);
    for (uint64_t i = 0; i < n_grids; ++i) {
        const pbrt_b200_density_grid& g = grids[i];
        const uint64_t n = (uint64_t)g.nx * g.ny * g.nz;
        float m = 0.0f;
        bool ok = true;
        for (uint64_t k = 0; k < n; ++k) {
            const float v = g.density[k];
            ok = ok && v >= 0.0f && v < INFINITY;  // false for NaN
            m = v > m ? v : m;
        }
        if (!ok) return fail(PBRT_B200_ERR_INVALID, "scene_create: densities must be finite and non-negative");
        (*max_density)[i] = m;
    }
    return PBRT_B200_OK;
}

int validate(const pbrt_b200_scene_desc* d) {
    if (d->abi_version != PBRT_B200_ABI_VERSION) return fail(PBRT_B200_ERR_INVALID, "scene_create: abi_version mismatch");
    if (d->n_prims && !d->prims) return fail(PBRT_B200_ERR_INVALID, "scene_create: prims is null");
    if (d->n_nodes && !d->nodes) return fail(PBRT_B200_ERR_INVALID, "scene_create: nodes is null");
    if (d->n_prims && !d->n_nodes) return fail(PBRT_B200_ERR_INVALID, "scene_create: primitives without a BVH (Accelerator \"bvh\" is required)");
    if (d->n_prims > 0x7ffffff0ull) return fail(PBRT_B200_ERR_INVALID, "scene_create: too many primitives");
    if (d->n_nodes > 0x7ffffff0ull) return fail(PBRT_B200_ERR_INVALID, "scene_create: too many BVH nodes");
    // every table whose count is non-zero must be there: the checks below and the uploader dereference them
    if (d->n_triangles && !d->tri_indices) return fail(PBRT_B200_ERR_INVALID, "scene_create: tri_indices is null");
    if (d->n_vertices && !d->vertex_p) return fail(PBRT_B200_ERR_INVALID, "scene_create: vertex_p is null");
    if (d->n_triangles && !d->n_vertices) return fail(PBRT_B200_ERR_INVALID, "scene_create: triangles without vertices");
    if (d->n_spheres && !d->spheres) return fail(PBRT_B200_ERR_INVALID, "scene_create: spheres is null");
    if (d->n_materials && !d->materials) return fail(PBRT_B200_ERR_INVALID, "scene_create: materials is null");
    if (d->n_lights && !d->lights) return fail(PBRT_B200_ERR_INVALID, "scene_create: lights is null");
    {
        // the per-primitive checks are independent: split over a few threads (1 M rows: 3-4 ms on one)
        auto check_rows = [d](uint64_t lo, uint64_t hi) -> const char* {
            for (uint64_t i = lo; i < hi; ++i) {
                const pbrt_b200_prim& p = d->prims[i];
                if (p.shape_kind == PBRT_B200_SHAPE_TRIANGLE) {
                    if (p.shape_index >= d->n_triangles) return "scene_create: triangle index out of range";
                } else if (p.shape_kind == PBRT_B200_SHAPE_SPHERE) {
                    if (p.shape_index >= d->n_spheres) return "scene_create: sphere index out of range";
                } else if (p.shape_kind == PBRT_B200_SHAPE_INSTANCE) {
                    if (p.shape_index >= d->n_instances) return "scene_create: instance index out of range";
                    if (d->n_objects == 0 || i >= d->n_top_prims) return "scene_create: an instance inside an object (ObjectInstance can't be nested, api.rs:1674-1677)";
                } else {
                    return "!scene_create: shape kind outside the hot path (triangle, sphere)";  // '!': ERR_UNSUPPORTED
                }
                if (p.material >= (int64_t)d->n_materials) return "scene_create: material index out of range";
                if (p.area_light >= (int64_t)d->n_lights) return "scene_create: area light index out of range";
            }
            return nullptr;
        };
        const unsigned hw = std::thread::hardware_concurrency();
        const uint64_t nt = d->n_prims < (1u << 16) ? 1 : std::min<uint64_t>(8, std::max(1u, hw / 2));
        std::vector<const char*> res(nt, nullptr);
        std::vector<std::thread> th;
        for (uint64_t t = 1; t < nt; ++t) th.emplace_back([&, t] { res[t] = check_rows(d->n_prims * t / nt, d->n_prims * (t + 1) / nt); });
        res[0] = check_rows(0, d->n_prims / nt);
        // vertex indices: one linear pass over the index buffer (every triangle of the table, referenced by a primitive row or not)
        // instead of a dependent, cache-missing read per primitive row
        const uint64_t n_idx = 3ull * d->n_triangles;
        uint32_t worst = 0;
        for (uint64_t k = 0; k < n_idx; ++k) worst = std::max(worst, d->tri_indices[k]);
        for (auto& x : th) x.join();
        if (n_idx && worst >= d->n_vertices) return fail(PBRT_B200_ERR_INVALID, "scene_create: vertex index out of range");
        for (const char* r : res)
            if (r) return r[0] == '!' ? fail(PBRT_B200_ERR_UNSUPPORTED, r + 1) : fail(PBRT_B200_ERR_INVALID, r);
    }
    if (d->n_objects) {
        if (!d->objects || (d->n_instances && !d->instances)) return fail(PBRT_B200_ERR_INVALID, "scene_create: objects / instances is null");
        if (d->n_top_nodes > d->n_nodes || d->n_top_prims > d->n_prims) return fail(PBRT_B200_ERR_INVALID, "scene_create: n_top_nodes / n_top_prims out of range");
        uint64_t next_node = d->n_top_nodes, next_prim = d->n_top_prims;
        for (uint64_t k = 0; k < d->n_objects; ++k) {
            const pbrt_b200_object& o = d->objects[k];
            if (o.node_offset != next_node || o.prim_offset != next_prim)
                return fail(PBRT_B200_ERR_INVALID, "scene_create: objects must follow the top-level tables back to back, in order");
            next_node += o.n_nodes; next_prim += o.n_prims;
            if (o.node_offset < d->n_top_nodes || o.node_offset + o.n_nodes > d->n_nodes || o.prim_offset < d->n_top_prims || o.n_prims == 0 ||
                o.prim_offset + o.n_prims > d->n_prims || (o.n_nodes == 0 && o.n_prims != 1))
                return fail(PBRT_B200_ERR_INVALID, "scene_create: object table out of range");
        }
        for (uint64_t k = 0; k < d->n_instances; ++k)
            if (d->instances[k].object >= d->n_objects) return fail(PBRT_B200_ERR_INVALID, "scene_create: instance refers to a missing object");
    } else if (d->n_instances) {
        return fail(PBRT_B200_ERR_INVALID, "scene_create: instances without objects");
    }
    if (d->n_media && !d->media) return fail(PBRT_B200_ERR_INVALID, "scene_create: media is null");
    if (d->n_media > 0x7fffffffull) return fail(PBRT_B200_ERR_INVALID, "scene_create: too many media");
    for (uint64_t i = 0; i < d->n_media; ++i) {
        const pbrt_b200_medium& m = d->media[i];
        for (int k = 0; k < 3; ++k)
            if (!(m.sigma_a[k] >= 0.0f) || !(m.sigma_s[k] >= 0.0f) || !(m.sigma_a[k] + m.sigma_s[k] < INFINITY))
                return fail(PBRT_B200_ERR_INVALID, "scene_create: medium coefficients must be finite and non-negative");
        if (!(m.g > -1.0f && m.g < 1.0f)) return fail(PBRT_B200_ERR_INVALID, "scene_create: medium g must lie in (-1, 1)");
    }
    if (d->prim_media)
        for (uint64_t i = 0; i < d->n_prims; ++i) {
            const pbrt_b200_medium_interface& mi = d->prim_media[i];
            if (mi.inside < -1 || mi.outside < -1 || mi.inside >= (int64_t)d->n_media || mi.outside >= (int64_t)d->n_media)
                return fail(PBRT_B200_ERR_INVALID, "scene_create: medium interface index out of range");
        }
    for (uint64_t i = 0; i < d->n_materials; ++i) {
        const pbrt_b200_material& m = d->materials[i];
        if (m.type > PBRT_B200_MAT_SUBSTRATE) return fail(PBRT_B200_ERR_UNSUPPORTED, "scene_create: material outside the device path");
        if (m.type > PBRT_B200_MAT_METAL && !m.textured) return fail(PBRT_B200_ERR_INVALID, "scene_create: uber / substrate rows keep their parameters in material_ext (textured = 1)");
        if (m.textured && !d->material_ext) return fail(PBRT_B200_ERR_INVALID, "scene_create: a textured material without material_ext");
    }
    // textures: every program must be a well-formed postfix expression over existing nodes and images
    if (d->n_textures && !d->textures) return fail(PBRT_B200_ERR_INVALID, "scene_create: textures is null");
    if (d->n_textures > 0x7fffffffull) return fail(PBRT_B200_ERR_INVALID, "scene_create: too many textures");
    for (uint64_t i = 0; i < d->n_textures; ++i) {
        const pbrt_b200_texnode& n = d->textures[i];
        if (n.kind > PBRT_B200_TEX_WINDY || n.mapping > PBRT_B200_MAP_PLANAR) return fail(PBRT_B200_ERR_INVALID, "scene_create: unknown texture kind / mapping");
        if (n.kind == PBRT_B200_TEX_IMAGEMAP && n.image >= d->n_mipmaps) return fail(PBRT_B200_ERR_INVALID, "scene_create: texture image index out of range");
    }
    if (d->material_ext) {
        auto check = [&](const pbrt_b200_texref& r) -> bool {  // stack discipline of one program
            if (r.count == 0) return true;
            if ((uint64_t)r.first + r.count > d->n_textures) return false;
            int depth = 0;
            for (uint32_t k = 0; k < r.count; ++k) {
                const uint32_t kind = d->textures[r.first + k].kind;
                const int pops = kind == PBRT_B200_TEX_MIX ? 3 : (kind == PBRT_B200_TEX_SCALE || kind == PBRT_B200_TEX_CHECKERBOARD2D || kind == PBRT_B200_TEX_CHECKERBOARD3D ||
                                                                  kind == PBRT_B200_TEX_DOTS) ? 2 : 0;
                if (depth < pops) return false;
                depth += 1 - pops;
                if (depth > 8) return false;  // PB_TEX_STACK
            }
            return depth == 1;
        };
        for (uint64_t i = 0; i < d->n_materials; ++i) {
            if (!d->materials[i].textured) continue;
            const pbrt_b200_material_ext& x = d->material_ext[i];
            bool ok = check(x.bump);
            for (int k = 0; k < 5; ++k) ok = ok && check(x.s_tex[k]);
            for (int k = 0; k < 3; ++k) ok = ok && check(x.f_tex[k]);
            if (!ok) return fail(PBRT_B200_ERR_INVALID, "scene_create: malformed texture program (range, operand count or more than 8 stacked operands)");
        }
    }
    for (uint64_t i = 0; i < d->n_lights; ++i) {
        const pbrt_b200_light& l = d->lights[i];
        if (l.type > PBRT_B200_LIGHT_INFINITE) return fail(PBRT_B200_ERR_UNSUPPORTED, "scene_create: light type outside the hot path");
        if (l.type == PBRT_B200_LIGHT_DIFFUSE && l.shape_kind != PBRT_B200_SHAPE_TRIANGLE && l.shape_kind != PBRT_B200_SHAPE_SPHERE)
            return fail(PBRT_B200_ERR_UNSUPPORTED, "scene_create: area lights are triangles or spheres");
        if (l.type == PBRT_B200_LIGHT_DIFFUSE && l.shape_index >= (l.shape_kind == PBRT_B200_SHAPE_SPHERE ? d->n_spheres : d->n_triangles))
            return fail(PBRT_B200_ERR_INVALID, "scene_create: area light shape out of range");
    }
    return PBRT_B200_OK;
}

// One pass over LinearBVHNode[] in array order (parents precede their children: first child at i+1, second at
// `offset` > i, bvh.rs:662-693): structural checks, interior count, and the depth of every node -- the reference
// would panic on a traversal stack deeper than 64 entries (bvh.rs:722).
// The reference's flatten_bvhtree (bvh.rs:662-693) writes the tree in PRE-ORDER: first child at index + 1, second child right after the
// first child's whole sub-tree.  For such an array a scan with a stack of pending second children checks everything the general pass
// below checks (ranges, one parent per node, depth) with sequential memory accesses only, and -- like matching parentheses -- it splits
// into independent segments: a segment that runs out of its own stack records which entry of the (still unknown) incoming stack it
// expects next, and the segments are stitched in order afterwards.  scene_create waits for this check: one thread streams 10^6 nodes
// in ~9 ms, four in ~2.5.  Returns false when the array is not a pre-order tree (the general pass then says what is wrong).
struct PreorderSegment {
    // pops of entries that were pushed BEFORE the segment, in order: the node index each one must hold, and the greatest depth reached
    // (relative to the popped entry's own depth) until the next such pop
    std::vector<uint64_t> ext_expect;
    std::vector<int> ext_max_rel;
    int head_max_rel = 0;       // greatest depth relative to the depth of the segment's first node, before the first external pop
    // what the segment leaves on the stack: second children pushed inside it and not popped, with their depth relative to the last base
    std::vector<uint64_t> left_idx;
    std::vector<int> left_rel;
    int tail_rel = 0;           // depth of the node AFTER the segment relative to the last base (unused when the array ends there)
    uint32_t n_interior = 0;
    bool ok = true, ended = false;  // ended: the scan popped the last pending entry of the WHOLE array at its last node (only legal in the last segment)
};
void preorder_scan_segment(const pbrt_b200_bvh_node* nodes, uint64_t lo, uint64_t hi, uint64_t nn, uint64_t n_prims, PreorderSegment* out) {
    PreorderSegment& S = *out;
    uint64_t pend[PB_STACK_DEPTH];
    int pend_rel[PB_STACK_DEPTH];
    int sp = 0, rel = 0, max_rel = 0;  // rel: depth of node i relative to the current base (segment start, or the last external pop)
    for (uint64_t i = lo; i < hi; ++i) {
        const pbrt_b200_bvh_node& n = nodes[i];
        if (n.n_prims != 0) {
            if ((uint64_t)n.offset + n.n_prims > n_prims) { S.ok = false; return; }
            if (sp > 0) {
                --sp;
                if (pend[sp] != i + 1) { S.ok = false; return; }
                rel = pend_rel[sp];
            } else {  // the entry comes from before the segment (or the tree ends here)
                if (S.ext_expect.empty()) S.head_max_rel = max_rel; else S.ext_max_rel.back() = max_rel;
                if (i + 1 == nn) { S.ended = true; S.n_interior += 0; return; }
                S.ext_expect.push_back(i + 1);
                S.ext_max_rel.push_back(0);
                if (S.ext_expect.size() >= (size_t)PB_STACK_DEPTH) { S.ok = false; return; }  // more pops than any legal stack holds
                rel = 0; max_rel = 0;  // new base: the depth of the popped entry
            }
            continue;
        }
        const uint64_t c1 = n.offset;
        if (n.axis > 2 || c1 <= i + 1 || c1 >= nn || sp + 1 >= PB_STACK_DEPTH) { S.ok = false; return; }
        rel += 1;
        max_rel = std::max(max_rel, rel);
        pend[sp] = c1; pend_rel[sp] = rel;
        ++sp;
        S.n_interior += 1;
    }
    if (S.ext_expect.empty()) S.head_max_rel = max_rel; else S.ext_max_rel.back() = max_rel;
    S.left_idx.assign(pend, pend + sp);
    S.left_rel.assign(pend_rel, pend_rel + sp);
    S.tail_rel = rel;
}
bool check_node_range_preorder(const pbrt_b200_bvh_node* nodes, uint64_t nn, uint64_t n_prims, uint32_t* n_interior) {
    const unsigned hw = std::thread::hardware_concurrency();
    const uint64_t nseg = nn < (1u << 16) ? 1 : std::min<uint64_t>(4, std::max(1u, hw / 2));
    std::vector<PreorderSegment> seg(nseg);
    std::vector<std::thread> th;
    for (uint64_t k = 1; k < nseg; ++k) th.emplace_back([&, k] { preorder_scan_segment(nodes, nn * k / nseg, nn * (k + 1) / nseg, nn, n_prims, &seg[k]); });
    preorder_scan_segment(nodes, 0, nn / nseg, nn, n_prims, &seg[0]);
    for (auto& x : th) x.join();
    // stitch: the global stack of pending second children with their absolute depths
    uint64_t pend[2 * PB_STACK_DEPTH];
    int pend_depth[2 * PB_STACK_DEPTH];
    int sp = 0, base = 0;  // base: absolute depth the next segment's relative depths refer to (the root is at depth 0)
    uint32_t ni = 0;
    for (uint64_t k = 0; k < nseg; ++k) {
        const PreorderSegment& S = seg[k];
        if (!S.ok) return false;
        if (base + S.head_max_rel >= PB_STACK_DEPTH) return false;  // the traversal stacks a far child per level: the bound is on the DEPTH (bvh.rs:722)
        for (size_t e = 0; e < S.ext_expect.size(); ++e) {
            if (sp == 0 || pend[sp - 1] != S.ext_expect[e]) return false;
            base = pend_depth[--sp];
            if (base + S.ext_max_rel[e] >= PB_STACK_DEPTH) return false;
        }
        ni += S.n_interior;
        if (S.ended) {  // legal only as the very end of the array, with nothing left pending
            if (k + 1 != nseg || sp != 0) return false;
            *n_interior = ni;
            return true;
        }
        for (size_t e = 0; e < S.left_idx.size(); ++e) {
            if (sp >= 2 * PB_STACK_DEPTH) return false;
            pend[sp] = S.left_idx[e]; pend_depth[sp] = base + S.left_rel[e];
            ++sp;
        }
        base += S.tail_rel;
    }
    return false;  // the array ended inside a sub-tree
}
int check_node_range(const pbrt_b200_bvh_node* nodes, uint64_t nn, uint64_t n_prims, uint32_t* n_interior) {
    *n_interior = 0;
    if (nn == 0) return PBRT_B200_OK;
    if (check_node_range_preorder(nodes, nn, n_prims, n_interior)) return PBRT_B200_OK;
    if (getenv("PBRT_B200_PROFILE")) fprintf(stderr, "[pbrt_b200] scene_create   (node array is not a pre-order tree: general check)\n");
    *n_interior = 0;
    // per node one byte: depth in bits 0-5, number of parents seen (saturating at 2) in bits 6-7.  Every node but the root must be
    // reached exactly once: a DAG-shaped array (several interior nodes sharing a child) passes the per-node checks but has more
    // interior nodes than a tree of nn nodes, and the device-side layout build sizes its arrays for a tree
    std::vector<uint8_t> info(nn, 0);
    info[0] = 1u << 6;
    uint32_t ni = 0;
    for (uint64_t i = 0; i < nn; ++i) {
        const pbrt_b200_bvh_node& n = nodes[i];
        const uint8_t me = info[i];
        if ((me >> 6) != 1) return fail(PBRT_B200_ERR_INVALID, "scene_create: LinearBVHNode array is not a tree (a node is unreachable or has two parents)");
        if (n.n_prims != 0) {
            if ((uint64_t)n.offset + n.n_prims > n_prims)
                return fail(PBRT_B200_ERR_INVALID, i == 0 ? "scene_create: root node refers past the primitive table" : "scene_create: malformed LinearBVHNode array");
            continue;
        }
        const uint64_t c0 = i + 1, c1 = n.offset;
        if (n.axis > 2 || c1 <= c0 || c1 >= nn) return fail(PBRT_B200_ERR_INVALID, "scene_create: malformed LinearBVHNode array");
        const int dd = (me & 63) + 1;
        if (dd >= PB_STACK_DEPTH) return fail(PBRT_B200_ERR_INVALID, "scene_create: BVH deeper than the reference's 64-entry traversal stack");
        // a child seen for the first time takes this depth and one parent; seen again: the parent count saturates at 2 (caught when reached)
        info[c0] = info[c0] ? (uint8_t)(info[c0] | 0x80u) : (uint8_t)((1u << 6) | dd);
        info[c1] = info[c1] ? (uint8_t)(info[c1] | 0x80u) : (uint8_t)((1u << 6) | dd);
        ++ni;
    }
    *n_interior = ni;
    return PBRT_B200_OK;
}
// the scene's aggregate, then every instanced object's accelerator
int check_nodes(const pbrt_b200_scene_desc* d, uint32_t* n_interior, uint32_t* root_ref, std::vector<uint32_t>* obj_fat_base) {
    *n_interior = 0; *root_ref = PB_REF_NONE;
    obj_fat_base->assign(d->n_objects, 0u);
    const uint64_t top_nodes = d->n_objects ? d->n_top_nodes : d->n_nodes, top_prims = d->n_objects ? d->n_top_prims : d->n_prims;
    if (top_nodes == 0) return PBRT_B200_OK;
    uint32_t ni = 0;
    int rc = check_node_range(d->nodes, top_nodes, top_prims, &ni);
    if (rc) return rc;
    *root_ref = d->nodes[0].n_prims ? (PB_LEAF_BIT | d->nodes[0].offset) : 0u;  // fat index of node 0 is 0 when it is interior
    for (uint64_t k = 0; k < d->n_objects; ++k) {
        const pbrt_b200_object& o = d->objects[k];
        if (o.n_nodes > d->n_nodes || o.node_offset > d->n_nodes - o.n_nodes || o.n_prims > d->n_prims || o.prim_offset > d->n_prims - o.n_prims) continue;  // validate() reports it
        uint32_t no = 0;
        if ((rc = check_node_range(d->nodes + o.node_offset, o.n_nodes, o.n_prims, &no))) return rc;
        (*obj_fat_base)[k] = ni;  // interior nodes are numbered in array order across all accelerators
        ni += no;
    }
    *n_interior = ni;
    return PBRT_B200_OK;
}

}  // namespace

extern "C" int pbrt_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" void pbrt_b200_scene_destroy(pbrt_b200_scene* sc) {
    if (!sc) return;
    cudaSetDevice(sc->device);
    cudaDeviceSynchronize();  // blocks go back to the pool: nothing may still be reading them
    render_release_scene_state(sc);
    pool_free(sc->arena, sc->arena_bytes);
    pool_free(sc->scratch, sc->scratch_bytes);
    if (sc->fetch_counter) pool_free(sc->fetch_counter, 256);
    delete sc;
}

extern "C" int pbrt_b200_scene_create(const pbrt_b200_scene_desc* d, int device, pbrt_b200_scene** out) {
    return pbrt_b200_scene_create_with_grids(d, nullptr, 0, device, out);
}

extern "C" int pbrt_b200_scene_create_with_grids(const pbrt_b200_scene_desc* d, const pbrt_b200_density_grid* grids, uint64_t n_grids, int device,
                                                 pbrt_b200_scene** out) {
    if (!d || !out) return fail(PBRT_B200_ERR_INVALID, "scene_create: null argument");
    *out = nullptr;
    const bool prof = getenv("PBRT_B200_PROFILE") != nullptr;
    auto t0 = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!prof) return;
        auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[pbrt_b200] scene_create %-18s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    };
    if (d->abi_version != PBRT_B200_ABI_VERSION) return fail(PBRT_B200_ERR_INVALID, "scene_create: abi_version mismatch");
    if (d->n_prims && !d->prims) return fail(PBRT_B200_ERR_INVALID, "scene_create: prims is null");
    if (d->n_nodes && !d->nodes) return fail(PBRT_B200_ERR_INVALID, "scene_create: nodes is null");
    if (int rcm = validate_mipmaps(d)) return rcm;
    if (int rcg = validate_grid_shapes(grids, n_grids)) return rcg;
    std::vector<float> max_density;
    // The table checks (index ranges, BVH structure and depth: ~10 ms for 10^6 primitives) run on two worker threads
    // while this thread stages the tables into HBM; nothing on the device dereferences an index before they have passed.
    int rc = PBRT_B200_OK, rc_v = PBRT_B200_OK, rc_n = PBRT_B200_OK;
    std::string err_v, err_n;
    uint32_t n_interior = 0, root_ref = PB_REF_NONE;
    auto timed = [prof](const char* what, auto&& f) {
        auto a = std::chrono::steady_clock::now();
        f();
        if (prof) fprintf(stderr, "[pbrt_b200] scene_create   (%s: %.3f ms)\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a).count());
    };
    std::thread th_v([&] {
        timed("table checks", [&] { rc_v = validate(d); if (!rc_v) rc_v = validate_grid_values(d, grids, n_grids, &max_density); });
        if (rc_v) err_v = pbrt_b200::last_error_cstr();
    });
    std::vector<uint32_t> obj_fat_base;
    std::thread th_n([&] { timed("BVH checks", [&] { rc_n = check_nodes(d, &n_interior, &root_ref, &obj_fat_base); }); if (rc_n) err_n = pbrt_b200::last_error_cstr(); });
    struct Joiner { std::thread &a, &b; ~Joiner() { if (a.joinable()) a.join(); if (b.joinable()) b.join(); } } joiner{th_v, th_n};
    auto join_checks = [&]() -> int {
        th_v.join(); th_n.join();
        if (rc_v) return fail(rc_v, err_v);
        if (rc_n) return fail(rc_n, err_n);
        return PBRT_B200_OK;
    };
    int ndev = pbrt_b200_device_count();
    if (ndev <= 0) {
        if ((rc = join_checks())) return rc;  // malformed tables are reported as such even without a device
        return fail(PBRT_B200_ERR_NO_DEVICE, "scene_create: no CUDA device visible; this library has no CPU fallback");
    }
    if (device < 0 || device >= ndev) return fail(PBRT_B200_ERR_INVALID, "scene_create: device ordinal out of range");
    PB_CUDA_TRY(cudaSetDevice(device));

    const uint64_t nn = d->n_nodes, np = d->n_prims, nv = d->n_vertices, nt = d->n_triangles;
    const uint32_t nb = (uint32_t)((nn + PB_SCAN_BLOCK - 1) / PB_SCAN_BLOCK);
    // resident tables, then build-only temporaries (reference node array, scan scratch) at the tail of the same block
    const uint64_t max_interior = nn / 2 + 1;  // a binary tree has one interior node less than leaves
    size_t need = 0;
    auto add = [&](size_t bytes) { need += Arena::padded(bytes); };
    add(64ull * max_interior); add(128ull * max_interior); add(48ull * np); add(sizeof(pbrt_b200_prim) * np);
    add(12ull * nv); add(d->vertex_n ? 12ull * nv : 0); add(d->vertex_s ? 12ull * nv : 0); add(d->vertex_uv ? 8ull * nv : 0);
    add(12ull * nt); add(sizeof(pbrt_b200_sphere) * d->n_spheres); add(sizeof(pbrt_b200_material) * d->n_materials); add(sizeof(pbrt_b200_light) * d->n_lights);
    add(sizeof(DevInstance) * d->n_instances); add(4ull * d->n_objects); add(sizeof(DevScene));
    add(d->vertex_n ? 48ull * np : 0); add(d->vertex_uv ? 24ull * np : 0); add(96ull * d->n_lights);  // slot_n, slot_uv, light_tris
    add(sizeof(pbrt_b200_medium) * d->n_media); add(d->prim_media ? sizeof(pbrt_b200_medium_interface) * np : 0);
    auto mip_floats = [](const pbrt_b200_mipmap& m) {
        size_t n = 0;
        for (uint32_t l = 0; l < m.n_levels; ++l) n += (size_t)std::max(1u, m.width >> l) * std::max(1u, m.height >> l) * m.channels;
        return n;
    };
    add(sizeof(pbrt_b200_texnode) * d->n_textures); add(sizeof(pbrt_b200_mipmap) * d->n_mipmaps);
    add(d->material_ext ? sizeof(pbrt_b200_material_ext) * d->n_materials : 0);
    for (uint64_t i = 0; i < d->n_mipmaps; ++i) add(4 * mip_floats(d->mipmaps[i]));
    auto grid_floats = [](const pbrt_b200_density_grid& g) { return (size_t)g.nx * g.ny * g.nz; };
    add(sizeof(DevGrid) * n_grids);
    for (uint64_t i = 0; i < n_grids; ++i) add(4 * grid_floats(grids[i]));
    const size_t resident = need;
    add(sizeof(pbrt_b200_bvh_node) * nn); add(4ull * nn); add(4ull * nb);
    need += 4096;

    pbrt_b200_scene* sc = new pbrt_b200_scene();
    sc->device = device;
    sc->n_prims = np; sc->n_nodes = nn;
    std::memset(&sc->dev, 0, sizeof sc->dev);
    sc->arena = pool_alloc(need, &sc->arena_bytes);
    if (!sc->arena) { delete sc; return fail(PBRT_B200_ERR_CUDA, "scene_create: out of device memory"); }
    lap("arena");
    sc->device_bytes = resident;
    Arena A; A.base = reinterpret_cast<char*>(sc->arena); A.size = sc->arena_bytes;
    DevScene& ds = sc->dev;
    ds.n_slots = (uint32_t)np;
    ds.n_lights = (uint32_t)d->n_lights;
    ds.n_materials = (uint32_t)d->n_materials;
    if (nn) {
        std::memcpy(ds.root_box, d->nodes[0].bounds, sizeof ds.root_box);
        // Bounds3f::bounding_sphere (bounds.rs:515-523) on Scene.wb, used by DistantLight::preprocess
        float c[3];
        for (int k = 0; k < 3; ++k) c[k] = (ds.root_box[k] + ds.root_box[3 + k]) * (1.0f / 2.0f);
        bool inside = true;
        for (int k = 0; k < 3; ++k) inside = inside && c[k] >= ds.root_box[k] && c[k] <= ds.root_box[3 + k];
        float dx = ds.root_box[3] - c[0], dy = ds.root_box[4] - c[1], dz = ds.root_box[5] - c[2];
        ds.world_center[0] = c[0]; ds.world_center[1] = c[1]; ds.world_center[2] = c[2];
        ds.world_radius = inside ? sqrtf(dx * dx + dy * dy + dz * dz) : 0.0f;
    }
    cudaStream_t stream = 0;
    cudaError_t err = cudaSuccess;
    // host table -> arena (pageable source: the runtime stages it, the call returns once the source has been read)
    auto up = [&](const void* host, size_t bytes, auto** dev_out) {
        using T = std::remove_pointer_t<std::remove_reference_t<decltype(*dev_out)>>;
        *dev_out = nullptr;
        if (!host || bytes == 0) return;
        char* p = A.take<char>(bytes);
        *dev_out = reinterpret_cast<T*>(p);
        if (err == cudaSuccess) err = cudaMemcpyAsync(p, host, bytes, cudaMemcpyHostToDevice, stream);
    };
    float4* fat = A.take<float4>(4ull * max_interior);
    float4* quads = A.take<float4>(8ull * max_interior);
    float4* tris = A.take<float4>(3ull * np);
    ds.nodes = fat; ds.quads = quads; ds.tris = tris;
    float4* slot_n = (d->vertex_n && np) ? A.take<float4>(3ull * np) : nullptr;
    float2* slot_uv = (d->vertex_uv && np) ? A.take<float2>(3ull * np) : nullptr;
    float4* light_tris = d->n_lights ? A.take<float4>(6ull * d->n_lights) : nullptr;
    ds.slot_n = slot_n; ds.slot_uv = slot_uv; ds.light_tris = light_tris;
    const pbrt_b200_bvh_node* nodes_dev = nullptr;
    up(d->prims, sizeof(pbrt_b200_prim) * np, &ds.prims);
    up(d->vertex_p, 12ull * nv, &ds.vertex_p);
    up(d->tri_indices, 12ull * nt, &ds.tri_indices);
    up(d->nodes, sizeof(pbrt_b200_bvh_node) * nn, &nodes_dev);
    up(d->vertex_n, d->vertex_n ? 12ull * nv : 0, &ds.vertex_n);
    up(d->vertex_s, d->vertex_s ? 12ull * nv : 0, &ds.vertex_s);
    up(d->vertex_uv, d->vertex_uv ? 8ull * nv : 0, &ds.vertex_uv);
    up(d->spheres, sizeof(pbrt_b200_sphere) * d->n_spheres, &ds.spheres);
    up(d->materials, sizeof(pbrt_b200_material) * d->n_materials, &ds.materials);
    up(d->lights, sizeof(pbrt_b200_light) * d->n_lights, &ds.lights);
    up(d->media, sizeof(pbrt_b200_medium) * d->n_media, &ds.media);
    up(d->prim_media, d->prim_media ? sizeof(pbrt_b200_medium_interface) * np : 0, &ds.prim_media);
    ds.n_media = (uint32_t)d->n_media;
    up(d->textures, sizeof(pbrt_b200_texnode) * d->n_textures, &ds.textures);
    up(d->material_ext, d->material_ext ? sizeof(pbrt_b200_material_ext) * d->n_materials : 0, &ds.material_ext);
    ds.n_textures = (uint32_t)d->n_textures; ds.n_mipmaps = (uint32_t)d->n_mipmaps;
    std::vector<pbrt_b200_mipmap> mips(d->mipmaps, d->mipmaps + d->n_mipmaps);  // rows with their texel pointers moved to the device
    for (auto& m : mips) {
        const float* dev_texels = nullptr;
        up(m.texels, 4 * mip_floats(m), &dev_texels);
        m.texels = dev_texels;
    }
    up(mips.data(), sizeof(pbrt_b200_mipmap) * mips.size(), &ds.mipmaps);
    if (err == cudaSuccess && !mips.empty()) err = cudaStreamSynchronize(stream);  // `mips` is a local: its copy must have been read
    std::vector<DevGrid> dev_grids(n_grids);
    for (uint64_t i = 0; i < n_grids; ++i) {
        DevGrid& g = dev_grids[i];
        std::memcpy(g.world_to_medium, grids[i].world_to_medium, sizeof g.world_to_medium);
        g.nx = grids[i].nx; g.ny = grids[i].ny; g.nz = grids[i].nz;
        up(grids[i].density, 4 * grid_floats(grids[i]), &g.density);
    }
    lap("h2d staged");
    if ((rc = join_checks())) { pbrt_b200_scene_destroy(sc); return rc; }
    lap("checks joined");
    bool grid_media = false;  // render.cu runs the grid kernel only for scenes whose media use a grid
    for (uint64_t i = 0; i < d->n_media; ++i) grid_media = grid_media || d->media[i].grid > 0;
    if (grid_media) {  // the maxima come from the table-check thread
        for (uint64_t i = 0; i < n_grids; ++i) {
            dev_grids[i].max_density = max_density[i];
            dev_grids[i].inv_max_density = 1.0f / max_density[i];  // GridDensityMedium::new; +inf for an all-zero grid (vacuum: never used)
        }
        up(dev_grids.data(), sizeof(DevGrid) * n_grids, &sc->grids);
        sc->n_grids = (uint32_t)n_grids;
        if (err == cudaSuccess) err = cudaStreamSynchronize(stream);  // `dev_grids` is a local
    }
    // read on this thread only now: until the table checks have passed, `lights` may be null with a non-zero count
    ds.n_sphere_lights = 0;
    for (uint64_t i = 0; i < d->n_lights; ++i)
        if (d->lights[i].type == PBRT_B200_LIGHT_DIFFUSE && d->lights[i].shape_kind == PBRT_B200_SHAPE_SPHERE) ds.n_sphere_lights += 1;
    ds.root_ref = root_ref;
    ds.n_fat = n_interior;
    if (np && err == cudaSuccess)
        k_leaf_records<<<(unsigned)std::min<uint64_t>((np + 255) / 256, 148 * 16), 256, 0, stream>>>(ds.prims, (uint32_t)np, ds.tri_indices, ds.vertex_p, tris, ds.vertex_n,
                                                                                                       ds.vertex_uv, slot_n, slot_uv);
    if (d->n_lights && err == cudaSuccess)
        k_light_tris<<<(unsigned)std::min<uint64_t>((d->n_lights + 127) / 128, 148 * 8), 128, 0, stream>>>(ds.lights, (uint32_t)d->n_lights, ds.tri_indices, ds.vertex_p, ds.vertex_n,
                                                                                                             light_tris);
    if (nn) {
        uint32_t* fat_index = A.take<uint32_t>(nn);
        uint32_t* block_sums = A.take<uint32_t>(nb);
        if (err == cudaSuccess) {
            k_interior_count<<<nb, PB_SCAN_BLOCK, 0, stream>>>(nodes_dev, (uint32_t)nn, block_sums);
            k_interior_scan_blocks<<<1, PB_SCAN_BLOCK, 0, stream>>>(block_sums, nb);
            k_interior_index<<<nb, PB_SCAN_BLOCK, 0, stream>>>(nodes_dev, (uint32_t)nn, block_sums, fat_index);
            auto fat_launch = [&](uint64_t node_base, uint64_t count, uint64_t prim_base) {
                if (count) k_fat_nodes<<<(unsigned)std::min<uint64_t>((count + 255) / 256, 148 * 16), 256, 0, stream>>>(nodes_dev, (uint32_t)node_base, (uint32_t)count,
                                                                                                                      (uint32_t)prim_base, fat_index, fat, tris);
            };
            fat_launch(0, d->n_objects ? d->n_top_nodes : nn, 0);
            for (uint64_t k = 0; k < d->n_objects; ++k) fat_launch(d->objects[k].node_offset, d->objects[k].n_nodes, d->objects[k].prim_offset);
            if (n_interior) k_quad_nodes<<<(unsigned)std::min<uint64_t>((n_interior + 255) / 256, 148 * 16), 256, 0, stream>>>(fat, n_interior, quads);
        }
    }
    if (d->n_instances && err == cudaSuccess) {
        // TransformedPrimitive table + the LAST flag of one-primitive objects (they have no leaf node to set it)
        std::vector<DevInstance> inst(d->n_instances);
        std::vector<uint32_t> singles;
        for (uint64_t k = 0; k < d->n_objects; ++k)
            if (d->objects[k].n_nodes == 0) singles.push_back((uint32_t)d->objects[k].prim_offset);
        for (uint64_t k = 0; k < d->n_instances; ++k) {
            const pbrt_b200_instance& in = d->instances[k];
            const pbrt_b200_object& o = d->objects[in.object];
            DevInstance& di = inst[k];
            std::memcpy(di.world_to_prim, in.world_to_prim, 64); std::memcpy(di.prim_to_world, in.prim_to_world, 64);
            bool ident = true;
            for (int a = 0; a < 16; ++a) ident = ident && in.prim_to_world[a] == ((a % 5 == 0) ? 1.0f : 0.0f);  // transform.rs:229-238
            di.flags = ident ? PB_INST_IDENTITY : 0u;
            if (o.n_nodes == 0) {
                di.root_ref = PB_LEAF_BIT | (uint32_t)o.prim_offset;
                for (int a = 0; a < 6; ++a) di.root_box[a] = 0.0f;
            } else {
                const pbrt_b200_bvh_node& rn = d->nodes[o.node_offset];
                di.root_ref = rn.n_prims ? (PB_LEAF_BIT | (uint32_t)(o.prim_offset + rn.offset)) : obj_fat_base[in.object];
                di.flags |= PB_INST_HAS_BOX;
                std::memcpy(di.root_box, rn.bounds, sizeof di.root_box);
            }
        }
        up(inst.data(), sizeof(DevInstance) * inst.size(), &ds.instances);
        ds.n_instances = (uint32_t)d->n_instances;
        if (!singles.empty()) {
            const uint32_t* singles_dev = nullptr;
            up(singles.data(), 4ull * singles.size(), &singles_dev);
            if (err == cudaSuccess) k_single_prim_last<<<(unsigned)((singles.size() + 255) / 256), 256, 0, stream>>>(singles_dev, (uint32_t)singles.size(), tris);
        }
        if (err == cudaSuccess) err = cudaStreamSynchronize(stream);  // `inst` / `singles` are stack-owned staging sources
    }
    {
        DevScene* self = A.take<DevScene>(1);
        ds.self_dev = self;
        if (self && err == cudaSuccess) err = cudaMemcpyAsync(self, &ds, sizeof(DevScene), cudaMemcpyHostToDevice, stream);
    }
    lap("enqueue h2d+build");
    if (err == cudaSuccess) err = cudaGetLastError();
    if (err == cudaSuccess) err = cudaStreamSynchronize(stream);
    if (err != cudaSuccess) { pbrt_b200_scene_destroy(sc); PB_CUDA_TRY(err); }
    lap("sync");
    *out = sc;
    return PBRT_B200_OK;
}

extern "C" int pbrt_b200_scene_world_bound(const pbrt_b200_scene* sc, float* b) {
    if (!sc || !b) return fail(PBRT_B200_ERR_INVALID, "scene_world_bound: null argument");
    std::memcpy(b, sc->dev.root_box, 6 * sizeof(float));
    return PBRT_B200_OK;
}

// ---------------------------------------------------------------------------
// batch intersect
// ---------------------------------------------------------------------------
// tunables for A/B measurement of the batch closest-hit kernel: [variant, refill_below, chunk, grid]
static int g_tune[8] = {0, PB_REFILL_BELOW, PB_FETCH_CHUNK, 0, PB_INTERIOR_MIN, 0, 0, 0};
extern "C" void pbrt_b200_debug_tune(int key, int value) { if (key >= 0 && key < 8) g_tune[key] = value; }

namespace {
int ensure_fetch_counter(pbrt_b200_scene* sc) {
    if (sc->fetch_counter) return PBRT_B200_OK;
    size_t got = 0;
    sc->fetch_counter = reinterpret_cast<uint32_t*>(pool_alloc(256, &got));
    if (!sc->fetch_counter) return fail(PBRT_B200_ERR_CUDA, "out of device memory");
    int sm = 148, per_sm = 8;
    cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, sc->device);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sc->dev.n_instances ? k_intersect_batch<true> : k_intersect_batch<false>, PB_TRACE_BLOCK, 0);
    sc->trace_grid = sm * (per_sm > 0 ? per_sm : 1);  // persistent: one resident wave of CTAs
    return PBRT_B200_OK;
}
}  // namespace

extern "C" int pbrt_b200_intersect_dev(pbrt_b200_scene* sc, const pbrt_b200_ray* rays, uint64_t n, pbrt_b200_hit* hits, void* stream) {
    if (!sc || (n && (!rays || !hits))) return fail(PBRT_B200_ERR_INVALID, "intersect_dev: null argument");
    if (n == 0) return PBRT_B200_OK;
    PB_CUDA_TRY(cudaSetDevice(sc->device));
    if (n > 0xfffffff0ull) return fail(PBRT_B200_ERR_INVALID, "intersect_dev: batch too large (split it)");
    int rc = ensure_fetch_counter(sc);
    if (rc) return rc;
    PB_CUDA_TRY(cudaMemsetAsync(sc->fetch_counter, 0, sizeof(uint32_t), (cudaStream_t)stream));
    if (g_tune[0] == 1 || g_tune[0] == 2) {
        unsigned blocks = (unsigned)((n + PB_TRACE_BLOCK - 1) / PB_TRACE_BLOCK);
        if (g_tune[0] == 1) k_intersect_batch_1rpt<0><<<blocks, PB_TRACE_BLOCK, 0, (cudaStream_t)stream>>>(sc->dev, reinterpret_cast<const float4*>(rays), (uint32_t)n, reinterpret_cast<uint4*>(hits));
        else k_intersect_batch_1rpt<1><<<blocks, PB_TRACE_BLOCK, 0, (cudaStream_t)stream>>>(sc->dev, reinterpret_cast<const float4*>(rays), (uint32_t)n, reinterpret_cast<uint4*>(hits));
    } else {
        TraceTune tune{g_tune[1], g_tune[2], g_tune[4]};
        int grid = g_tune[3] > 0 ? g_tune[3] : sc->trace_grid;
        if (sc->dev.n_instances)
            k_intersect_batch<true><<<grid, PB_TRACE_BLOCK, 0, (cudaStream_t)stream>>>(sc->dev, reinterpret_cast<const float4*>(rays), (uint32_t)n,
                                                                                       reinterpret_cast<uint4*>(hits), sc->fetch_counter, tune);
        else if (batch_packet())
            k_intersect_batch_packet<<<grid, PB_TRACE_BLOCK, 0, (cudaStream_t)stream>>>(sc->dev, reinterpret_cast<const float4*>(rays), (uint32_t)n,
                                                                                        reinterpret_cast<uint4*>(hits), sc->fetch_counter);
        else
            k_intersect_batch<false><<<grid, PB_TRACE_BLOCK, 0, (cudaStream_t)stream>>>(sc->dev, reinterpret_cast<const float4*>(rays), (uint32_t)n,
                                                                                        reinterpret_cast<uint4*>(hits), sc->fetch_counter, tune);
    }
    PB_CUDA_TRY(cudaGetLastError());
    return PBRT_B200_OK;
}

extern "C" int pbrt_b200_intersect_p_dev(pbrt_b200_scene* sc, const pbrt_b200_ray* rays, uint64_t n, uint8_t* occluded, void* stream) {
    if (!sc || (n && (!rays || !occluded))) return fail(PBRT_B200_ERR_INVALID, "intersect_p_dev: null argument");
    if (n == 0) return PBRT_B200_OK;
    PB_CUDA_TRY(cudaSetDevice(sc->device));
    if (n > 0xfffffff0ull) return fail(PBRT_B200_ERR_INVALID, "intersect_p_dev: batch too large (split it)");
    int rc = ensure_fetch_counter(sc);
    if (rc) return rc;
    PB_CUDA_TRY(cudaMemsetAsync(sc->fetch_counter, 0, sizeof(uint32_t), (cudaStream_t)stream));
    if (sc->dev.n_instances)
        k_intersect_p_batch<true><<<sc->trace_grid, PB_TRACE_BLOCK, 0, (cudaStream_t)stream>>>(sc->dev, reinterpret_cast<const float4*>(rays), (uint32_t)n, occluded,
                                                                                              sc->fetch_counter);
    else if (batch_packet())
        k_intersect_p_batch_packet<<<sc->trace_grid, PB_TRACE_BLOCK, 0, (cudaStream_t)stream>>>(sc->dev, reinterpret_cast<const float4*>(rays), (uint32_t)n, occluded,
                                                                                               sc->fetch_counter);
    else
        k_intersect_p_batch<false><<<sc->trace_grid, PB_TRACE_BLOCK, 0, (cudaStream_t)stream>>>(sc->dev, reinterpret_cast<const float4*>(rays), (uint32_t)n, occluded,
                                                                                               sc->fetch_counter);
    PB_CUDA_TRY(cudaGetLastError());
    return PBRT_B200_OK;
}

namespace {
int ensure_scratch(pbrt_b200_scene* sc, uint64_t bytes) {
    if (sc->scratch_bytes >= bytes) return PBRT_B200_OK;
    if (sc->scratch) { cudaDeviceSynchronize(); pool_free(sc->scratch, sc->scratch_bytes); }
    sc->scratch = pool_alloc(bytes, &sc->scratch_bytes);
    if (!sc->scratch) { sc->scratch_bytes = 0; return fail(PBRT_B200_ERR_CUDA, "out of device memory"); }
    return PBRT_B200_OK;
}
}  // namespace

extern "C" int pbrt_b200_intersect(pbrt_b200_scene* sc, const pbrt_b200_ray* rays, uint64_t n, pbrt_b200_hit* hits) {
    if (!sc || (n && (!rays || !hits))) return fail(PBRT_B200_ERR_INVALID, "intersect: null argument");
    if (n == 0) return PBRT_B200_OK;
    PB_CUDA_TRY(cudaSetDevice(sc->device));
    int rc = ensure_scratch(sc, n * (sizeof(pbrt_b200_ray) + sizeof(pbrt_b200_hit)));
    if (rc) return rc;
    pbrt_b200_ray* dr = reinterpret_cast<pbrt_b200_ray*>(sc->scratch);
    pbrt_b200_hit* dh = reinterpret_cast<pbrt_b200_hit*>(reinterpret_cast<char*>(sc->scratch) + n * sizeof(pbrt_b200_ray));
    PB_CUDA_TRY(cudaMemcpyAsync(dr, rays, n * sizeof(pbrt_b200_ray), cudaMemcpyHostToDevice, 0));
    rc = pbrt_b200_intersect_dev(sc, dr, n, dh, nullptr);
    if (rc) return rc;
    PB_CUDA_TRY(cudaMemcpyAsync(hits, dh, n * sizeof(pbrt_b200_hit), cudaMemcpyDeviceToHost, 0));
    PB_CUDA_TRY(cudaStreamSynchronize(0));
    return PBRT_B200_OK;
}

extern "C" int pbrt_b200_intersect_p(pbrt_b200_scene* sc, const pbrt_b200_ray* rays, uint64_t n, uint8_t* occluded) {
    if (!sc || (n && (!rays || !occluded))) return fail(PBRT_B200_ERR_INVALID, "intersect_p: null argument");
    if (n == 0) return PBRT_B200_OK;
    PB_CUDA_TRY(cudaSetDevice(sc->device));
    int rc = ensure_scratch(sc, n * (sizeof(pbrt_b200_ray) + 1));
    if (rc) return rc;
    pbrt_b200_ray* dr = reinterpret_cast<pbrt_b200_ray*>(sc->scratch);
    uint8_t* dz = reinterpret_cast<uint8_t*>(sc->scratch) + n * sizeof(pbrt_b200_ray);
    PB_CUDA_TRY(cudaMemcpyAsync(dr, rays, n * sizeof(pbrt_b200_ray), cudaMemcpyHostToDevice, 0));
    rc = pbrt_b200_intersect_p_dev(sc, dr, n, dz, nullptr);
    if (rc) return rc;
    PB_CUDA_TRY(cudaMemcpyAsync(occluded, dz, n, cudaMemcpyDeviceToHost, 0));
    PB_CUDA_TRY(cudaStreamSynchronize(0));
    return PBRT_B200_OK;
}

// Film::write_image arithmetic, core/film.rs:217-264 (host helper; no device work)
extern "C" int pbrt_b200_film_resolve(const float* rgbw, uint64_t npixels, float scale, float* rgb_out) {
    if (npixels && (!rgbw || !rgb_out)) return fail(PBRT_B200_ERR_INVALID, "film_resolve: null argument");
    for (uint64_t i = 0; i < npixels; ++i) {
        const float* p = rgbw + 4 * i;
        // merge_film_tile: tile RGB -> XYZ (spectrum.rs:495-504)
        float X = 0.412453f * p[0] + 0.357580f * p[1] + 0.180423f * p[2];
        float Y = 0.212671f * p[0] + 0.715160f * p[1] + 0.072169f * p[2];
        float Z = 0.019334f * p[0] + 0.119193f * p[1] + 0.950227f * p[2];
        // write_image: XYZ -> RGB (spectrum.rs:484-493)
        float r = 3.240479f * X - 1.537150f * Y - 0.498535f * Z;
        float g = -0.969256f * X + 1.875991f * Y + 0.041556f * Z;
        float b = 0.055648f * X - 0.204043f * Y + 1.057311f * Z;
        float w = p[3];
        if (w != 0.0f) {
            float inv = 1.0f / w;
            r = fmaxf(r * inv, 0.0f); g = fmaxf(g * inv, 0.0f); b = fmaxf(b * inv, 0.0f);
        }
        rgb_out[3 * i] = r * scale; rgb_out[3 * i + 1] = g * scale; rgb_out[3 * i + 2] = b * scale;
    }
    return PBRT_B200_OK;
}

// Film::write_image(splat_scale) (pbrt-v3 film.cpp:148-185): the weighted RGB clamped at 0, plus splat_scale x the splat film
extern "C" int pbrt_b200_film_resolve_splat(const float* rgbw, const float* splat, uint64_t npixels, float splat_scale, float scale, float* rgb_out) {
    if (npixels && (!rgbw || !splat || !rgb_out)) return fail(PBRT_B200_ERR_INVALID, "film_resolve_splat: null argument");
    int rc = pbrt_b200_film_resolve(rgbw, npixels, 1.0f, rgb_out);
    if (rc) return rc;
    for (uint64_t i = 0; i < npixels; ++i) {
        const float* p = splat + 3 * i;
        const float X = 0.412453f * p[0] + 0.357580f * p[1] + 0.180423f * p[2];
        const float Y = 0.212671f * p[0] + 0.715160f * p[1] + 0.072169f * p[2];
        const float Z = 0.019334f * p[0] + 0.119193f * p[1] + 0.950227f * p[2];
        const float c[3] = {3.240479f * X - 1.537150f * Y - 0.498535f * Z, -0.969256f * X + 1.875991f * Y + 0.041556f * Z, 0.055648f * X - 0.204043f * Y + 1.057311f * Z};
        for (int k = 0; k < 3; ++k) rgb_out[3 * i + k] = (rgb_out[3 * i + k] + splat_scale * c[k]) * scale;
    }
    return PBRT_B200_OK;
}
