// Device-resident scene: HBM layout of the flattened pbrt-rust Scene.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/pbrt_b200.h"

namespace pb {

// Child reference inside a fat node / on the traversal stack:
//   bit 31 set  -> leaf, low 31 bits = first BVH slot (run ends at a record with TRI_LAST)
//   bit 31 clear-> interior, low bits = fat-node index
#define PB_LEAF_BIT 0x80000000u
#define PB_REF_NONE 0xffffffffu

// flags in TriRec.v1.w (as uint)
#define PB_TRI_LAST 0x80000000u     /* last primitive of its leaf            */
#define PB_TRI_SPHERE 0x40000000u   /* slot is a sphere, v2.w = sphere index */
#define PB_TRI_INSTANCE 0x20000000u /* slot is a TransformedPrimitive, v2.w = instance index */
#define PB_TRI_FLAGS_MASK 0x000000ffu /* PBRT_B200_PRIM_* of the primitive     */

// TransformedPrimitive (primitive.rs:41-103) as the traversal sees it: both matrices, and where the instanced object's
// accelerator starts in the shared fat-node / leaf-record arrays (child refs are global).
#define PB_INST_IDENTITY 1u /* prim_to_world.is_identity(): the interaction is not transformed back (primitive.rs:75-77) */
#define PB_INST_HAS_BOX 2u
struct DevInstance {
    float world_to_prim[16];
    float prim_to_world[16];
    uint32_t root_ref;     // fat-node index or PB_LEAF_BIT | slot (a BVH whose root is a leaf, or a one-primitive object)
    uint32_t flags;        // PB_INST_IDENTITY | PB_INST_HAS_BOX
    float root_box[6];     // object BVH root bounds; a one-primitive object has no accelerator (api.rs:1691) and no box test
};

// GridDensityMedium (src/media/grid.rs) as the volpath grid kernel reads it: pbrt_b200_density_grid with the density moved to the
// device and max_density found by scene_create (0 for an all-zero grid, which sample and tr treat as vacuum).
struct DevGrid {
    float world_to_medium[16];
    uint32_t nx, ny, nz;
    float max_density;
    float inv_max_density;  // 1 / max_density
    const float* density;   // density[(z * ny + y) * nx + x]
};

struct DevScene {
    // Fat BVH2: per INTERIOR node of the reference's LinearBVHNode array, the exact f32
    // boxes of both children (48 B) + child refs + split axis = 64 B = 4 x float4:
    //  q0 = {c0.min.x, c0.min.y, c0.min.z, c0.max.x}
    //  q1 = {c0.max.y, c0.max.z, c1.min.x, c1.min.y}
    //  q2 = {c1.min.z, c1.max.x, c1.max.y, c1.max.z}
    //  q3 = {ref0, ref1, axis, 0} (bit patterns)
    // c0 = reference child at index+1, c1 = reference child at `offset` (bvh.rs:662-693).
    const float4* nodes;
    // Quad nodes, 128 B = 8 x float4, one per fat node and with the same index: the four GRANDCHILDREN of the reference's
    // interior node (the children of its two children; a child that is a leaf fills one slot and leaves the other empty:
    // lo = +inf, hi = -inf, ref = PB_REF_NONE).  Slots 0,1 = under the first child, 2,3 = under the second child.
    //  pair A (slots 0,1): qa0 = {lo0.x, lo1.x, lo0.y, lo1.y}  qa1 = {lo0.z, lo1.z, hi0.x, hi1.x}  qa2 = {hi0.y, hi1.y, hi0.z, hi1.z}
    //  pair B (slots 2,3): qb0, qb1, qb2 likewise
    //  q6 = {ref0, ref1, ref2, ref3}   q7 = {axis | axis_first << 2 | axis_second << 4, 0, 0, 0}
    // Used by rays without a zero direction component in scenes without instancing (trace.cuh: trav_run_quad).
    const float4* quads;
    uint32_t n_fat;
    uint32_t root_ref;      // PB_REF_NONE when the scene is empty
    float root_box[6];      // LinearBVHNode[0].bounds = Scene.wb
    // Leaf primitives in BVH slot order, vertices pre-gathered (3 x float4 = 48 B):
    //  v0 = {p0.xyz, creation_index}  v1 = {p1.xyz, flags}  v2 = {p2.xyz, shape_index}
    const float4* tris;
    uint32_t n_slots;
    // Shading-side companions of the leaf records, same slot order, so that a hit's normals / uvs are ONE dependent fetch
    // away from the hit record instead of three (slot -> shape_index -> vertex indices -> per-vertex gathers):
    //  slot_n[3 * slot + k] = {n_k.xyz, 0} (only when the scene has per-vertex normals), slot_uv[3 * slot + k] = uv_k
    const float4* slot_n;
    const float2* slot_uv;
    // Triangle area lights: light_tris[6 * light + k] = {p_k.xyz, 0} (k < 3), {n_k.xyz, 0} (k >= 3); zeros for other lights
    const float4* light_tris;
    const pbrt_b200_prim* prims;      // slot order
    const float* vertex_p;
    const float* vertex_n;
    const float* vertex_s;
    const float* vertex_uv;
    const uint32_t* tri_indices;
    const pbrt_b200_sphere* spheres;
    const pbrt_b200_material* materials;
    const pbrt_b200_light* lights;
    const DevInstance* instances;
    uint32_t n_instances;
    // This struct again, resident in HBM.  Kernels get DevScene by value (constant bank); the out-of-line instance code
    // takes this pointer instead, because the address of a kernel parameter would force a local-memory copy of the whole
    // struct into every kernel that might call it.
    const DevScene* self_dev;
    uint32_t n_lights;
    uint32_t n_sphere_lights;  // diffuse area lights whose shape is a sphere: render.cu picks the kernel family that samples them
    uint32_t n_materials;
    // Participating media (volpath): HomogeneousMedium rows and the MediumInterface of every primitive row (nullptr: no media)
    const pbrt_b200_medium* media;
    const pbrt_b200_medium_interface* prim_media;
    uint32_t n_media;
    // Textures (texture.cuh): postfix programs, MIPMap pyramids (texel pointers are device pointers) and the parameter rows of the
    // `textured` materials; all nullptr when the scene has none (render.cu then never launches a Q_TEX kernel)
    const pbrt_b200_texnode* textures;
    const pbrt_b200_mipmap* mipmaps;
    const pbrt_b200_material_ext* material_ext;
    uint32_t n_textures, n_mipmaps;
    // Scene::new preprocessing (scene.rs:32-52, distant.rs:53-60)
    float world_center[3];
    float world_radius;
};

}  // namespace pb

// Host-side owner.  Opaque to C callers.
struct pbrt_b200_scene {
    int device = 0;
    pb::DevScene dev;            // pointers are device pointers
    void* arena = nullptr;       // ONE pooled device block (pool.h) holding every scene table
    size_t arena_bytes = 0;
    uint64_t n_prims = 0, n_nodes = 0;
    uint64_t device_bytes = 0;
    void* scratch = nullptr;     // reusable staging for the host-buffer batch API (pooled)
    size_t scratch_bytes = 0;
    void* light_distrib = nullptr;  // owned by render.cu
    uint32_t* fetch_counter = nullptr;  // device counter of the persistent ray queue (batch API)
    int trace_grid = 0;
    const pb::DevGrid* grids = nullptr;  // density grids of the media rows with grid > 0 (device table of n_grids rows)
    uint32_t n_grids = 0;
};
