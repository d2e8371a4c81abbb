/*
 * pbrt_b200.h -- C ABI of the B200 wavefront path tracer that stands in for
 * pbrt-rust's PathIntegrator hot path.
 *
 * Every entry point names the reference interface (file:line under the
 * pbrt-rust tree) it replaces.  The reference has no FFI today: the binding a
 * maintainer would add (a new `Integrators` variant whose `render` flattens the
 * `Scene` and calls these functions) is shown in INTEGRATION.md.
 *
 * Conventions
 *   - plain C structs, pointers and sizes only; no C++/torch types.
 *   - all input arrays are caller-owned host memory unless a function name ends
 *     in `_dev` (then they are device pointers on the scene's device).
 *   - every function returns 0 on success, non-zero on failure; the message is
 *     available from pbrt_b200_last_error() (thread-local).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point
 *     fails with PBRT_B200_ERR_NO_DEVICE.
 */
#ifndef PBRT_B200_H
#define PBRT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PBRT_B200_ABI_VERSION 5

enum {
    PBRT_B200_OK = 0,
    PBRT_B200_ERR_INVALID = 1,   /* bad argument / inconsistent scene tables      */
    PBRT_B200_ERR_NO_DEVICE = 2, /* no CUDA device (there is no CPU fallback)      */
    PBRT_B200_ERR_CUDA = 3,      /* a CUDA runtime call failed                     */
    PBRT_B200_ERR_UNSUPPORTED = 4/* feature outside the hot path (SURVEY.md s8)    */
};

/* ---- BVH -------------------------------------------------------------- */

/* = LinearBVHNode, src/accelerators/bvh.rs:89-95 (32 bytes, reference order:
 * first child of an interior node is at index+1, second child at `offset`). */
typedef struct pbrt_b200_bvh_node {
    float    bounds[6];  /* p_min.xyz, p_max.xyz                                 */
    uint32_t offset;     /* leaf: first index into prims[]; interior: 2nd child  */
    uint16_t n_prims;    /* 0 => interior                                        */
    uint8_t  axis;       /* interior: split axis                                 */
    uint8_t  pad;
} pbrt_b200_bvh_node;

enum { PBRT_B200_SPLIT_SAH = 0, PBRT_B200_SPLIT_MIDDLE = 2, PBRT_B200_SPLIT_EQUAL = 3 };

/* Host-side mirror of BVHAccel::new + recursive_build + flatten_bvhtree
 * (src/accelerators/bvh.rs:145-375,662-693).  In a real integration the Rust
 * host already owns `BVHAccel.nodes`/`primitives` and skips this call.
 *   prim_bounds : n x 6 floats (world bounds of primitive i)
 *   nodes_out   : capacity >= 2n-1 ; ordered_out : n entries, ordered_out[k] =
 *                 original primitive index stored at BVH slot k
 *   n_nodes_out : number of nodes written                                        */
int pbrt_b200_bvh_build(const float *prim_bounds, uint64_t n, int max_prims_in_node,
                        int split_method, pbrt_b200_bvh_node *nodes_out,
                        uint32_t *ordered_out, uint64_t *n_nodes_out);

/* ---- scene tables ------------------------------------------------------ */

enum {
    PBRT_B200_SHAPE_TRIANGLE = 0,
    PBRT_B200_SHAPE_SPHERE = 1,
    PBRT_B200_SHAPE_INSTANCE = 2 /* the row is a TransformedPrimitive (primitive.rs:41-103): shape_index = instance number,
                                  * material = area_light = -1 (get_material / get_area_light return None, :91-97)   */
};
enum {
    PBRT_B200_PRIM_REVERSE_ORIENTATION = 1u << 0, /* Shape::reverse_orientation          */
    PBRT_B200_PRIM_SWAPS_HANDEDNESS    = 1u << 1, /* Shape::transform_swapshandedness    */
    PBRT_B200_PRIM_HAS_N               = 1u << 2, /* mesh has per-vertex normals         */
    PBRT_B200_PRIM_HAS_S               = 1u << 3, /* mesh has per-vertex tangents        */
    PBRT_B200_PRIM_HAS_UV              = 1u << 4  /* mesh has per-vertex uv              */
};

/* = GeometricPrimitive (src/core/primitive.rs:106-111), in `ordered_prims`
 * order (BVH leaf order).  24 bytes.                                          */
typedef struct pbrt_b200_prim {
    uint32_t shape_kind;     /* PBRT_B200_SHAPE_*                                    */
    uint32_t shape_index;    /* triangle number (into tri_indices/3) or sphere index */
    int32_t  material;       /* index into materials[], -1 = none (pass-through)     */
    int32_t  area_light;     /* index into lights[], -1 = not emissive               */
    uint32_t flags;          /* PBRT_B200_PRIM_*                                     */
    uint32_t creation_index; /* index before BVH reordering (what hit records carry) */
} pbrt_b200_prim;

/* = what an ObjectInstance refers to (src/core/api.rs:1663-1713): the primitives collected between ObjectBegin and
 * ObjectEnd, wrapped in their own BVHAccel when there is more than one (api.rs:1691-1699).  An object's BVH nodes and
 * primitive rows live in the scene's nodes[] / prims[] arrays AFTER the top-level ones; inside an object, node
 * `offset`s (second child / first primitive) are relative to node_offset / prim_offset.  Objects are stored back to
 * back in objects[] order: object 0 starts at n_top_nodes / n_top_prims, object k+1 where object k ends.            */
typedef struct pbrt_b200_object {
    uint64_t node_offset, n_nodes;   /* n_nodes == 0: a single primitive, referenced directly (no accelerator)       */
    uint64_t prim_offset, n_prims;
} pbrt_b200_object;

/* = TransformedPrimitive (src/core/primitive.rs:41-103) with a static AnimatedTransform (start == end,
 * transform.rs:1493-1497).  Per ray: Transform::inverse (m/m_inv swap) + transform_ray (:543-577, origin-error
 * nudge and t_max -= dt), the object's own intersect, r.t_max = ray.t_max, transform_surface_interaction (:607-636). */
typedef struct pbrt_b200_instance {
    float prim_to_world[16];  /* row-major m                                                                          */
    float world_to_prim[16];  /* m_inv                                                                                */
    uint32_t object;          /* index into objects[]                                                                 */
    uint32_t pad[3];
} pbrt_b200_instance; /* 144 bytes */

/* = Sphere (src/shapes/sphere.rs:19-57); full spheres only on the hot path.   */
typedef struct pbrt_b200_sphere {
    float object_to_world[16]; /* row-major m                                        */
    float world_to_object[16];
    float radius;
    uint32_t flags;            /* PBRT_B200_PRIM_REVERSE_ORIENTATION|SWAPS_HANDEDNESS */
    float pad[2];
} pbrt_b200_sphere;

enum {
    PBRT_B200_MAT_MATTE = 0,   /* src/materials/matte.rs:28-52   a=Kd  f0=sigma            */
    PBRT_B200_MAT_PLASTIC = 1, /* src/materials/plastic.rs:34-69 a=Kd b=Ks f0=roughness   */
    PBRT_B200_MAT_MIRROR = 2,  /* src/materials/mirror.rs:23-41  a=Kr                      */
    PBRT_B200_MAT_GLASS = 3,   /* src/materials/glass.rs:35-92   a=Kr b=Kt f0=urough f1=vrough f2=index */
    PBRT_B200_MAT_METAL = 4,   /* src/materials/metal.rs:78-112  a=eta b=k f0=urough f1=vrough */
    /* ABI v5: parameters live in material_ext[] only (the row is always `textured`) */
    PBRT_B200_MAT_UBER = 5,     /* src/materials/uber.rs:41-112      s0..4 = Kd Ks Kr Kt opacity, f0/f1 = u/v roughness, f2 = eta */
    PBRT_B200_MAT_SUBSTRATE = 6 /* src/materials/substrate.rs:34-62  s0 = Kd, s1 = Ks, f0 = nu, f1 = nv (FresnelBlend)           */
};

typedef struct pbrt_b200_material {
    uint32_t type;
    uint32_t remap_roughness;
    float a[3];
    float b[3];
    float f0, f1, f2;
    uint32_t textured;  /* ABI v5: 1 = parameters (texture programs, bump map) come from material_ext[same index] */
} pbrt_b200_material; /* 48 bytes */

/* ---- textures (ABI v5; src/core/texture.rs, src/textures/, src/core/mipmap.rs) ------------------------------------
 * A texture expression (an `Arc<Textures>` tree: scale(mix(imagemap, checkerboard(..)), ..)) is handed over flattened in
 * POSTFIX order: operands first, the operator last; evaluation is a walk over the program with a small value stack.  Texture
 * evaluation has no side effects, so evaluating both operands of a checkerboard and selecting gives the reference's value.
 * Float textures carry their value in all three channels (the arithmetic is channel-wise either way).                     */
enum {
    PBRT_B200_TEX_CONSTANT = 0,       /* textures/constant.rs: v[0..2]                                                   */
    PBRT_B200_TEX_SCALE = 1,          /* textures/scaled.rs: pops tex2, tex1 -> tex1 * tex2                             */
    PBRT_B200_TEX_MIX = 2,            /* textures/mix.rs: pops amount, tex2, tex1 -> tex1 * (1 - amt) + tex2 * amt       */
    PBRT_B200_TEX_BILERP = 3,         /* textures/biler.rs: v = v00 v01 v10 v11 (3 floats each), 2D mapping               */
    PBRT_B200_TEX_IMAGEMAP = 4,       /* textures/imagemap.rs:165-175 -> MIPMap::lookup2 (mipmap.rs:228-269), 2D mapping  */
    PBRT_B200_TEX_UV = 5,             /* textures/uv.rs, 2D mapping                                                       */
    PBRT_B200_TEX_CHECKERBOARD2D = 6, /* textures/checkerboard.rs:28-73: pops tex2, tex1; flags AA_CLOSEDFORM            */
    PBRT_B200_TEX_CHECKERBOARD3D = 7, /* textures/checkerboard.rs:88-100: pops tex2, tex1; m = world_to_texture          */
    PBRT_B200_TEX_DOTS = 8,           /* textures/dots.rs: pops `inside`, `outside` (struct field names), 2D mapping     */
    PBRT_B200_TEX_FBM = 9,            /* textures/fbm.rs: v[0] = omega, v[1] = octaves; m = world_to_texture             */
    PBRT_B200_TEX_WRINKLED = 10,      /* textures/wrinkled.rs: likewise (turbulence)                                      */
    PBRT_B200_TEX_MARBLE = 11,        /* textures/marble.rs: v[0] = omega, v[1] = octaves, v[2] = scale, v[3] = variation */
    PBRT_B200_TEX_WINDY = 12          /* textures/windy.rs                                                                */
};
enum { PBRT_B200_MAP_UV = 0,          /* UVMapping2D, texture.rs:137-162: m[0..3] = su sv du dv                          */
       PBRT_B200_MAP_SPHERICAL = 1,   /* SphericalMapping2D :164-207: m = world_to_texture (row-major Transform.m)        */
       PBRT_B200_MAP_CYLINDRICAL = 2, /* CylindricalMapping2D :209-251: m = world_to_texture                              */
       PBRT_B200_MAP_PLANAR = 3 };    /* PlannarMapping2D :253-283: m[0..2] = vs, m[3..5] = vt, m[6] = ds, m[7] = dt       */
enum { PBRT_B200_TEX_AA_CLOSEDFORM = 1u << 0 }; /* Checkerboard2DTexture AAMethod::ClosedForm                            */

typedef struct pbrt_b200_texnode {
    uint32_t kind;      /* PBRT_B200_TEX_*                                                */
    uint32_t mapping;   /* PBRT_B200_MAP_* for the kinds with a 2D mapping                */
    uint32_t flags;
    uint32_t image;     /* IMAGEMAP: index into mipmaps[]                                 */
    float v[12];
    float m[16];
} pbrt_b200_texnode; /* 128 bytes */

enum { PBRT_B200_WRAP_REPEAT = 0, PBRT_B200_WRAP_BLACK = 1, PBRT_B200_WRAP_CLAMP = 2 };

/* = MIPMap<T> (src/core/mipmap.rs:58-69) after MIPMap::new (:76-198): the pyramid the host built (resampled to a power of two,
 * box-filtered levels), levels back to back, each row-major [t][s] with `channels` floats per texel (1 = ImageTextureFloat,
 * 3 = ImageTextureRGB).  Level l is max(1, width >> l) x max(1, height >> l).                                              */
typedef struct pbrt_b200_mipmap {
    const float *texels;
    uint32_t n_levels;
    uint32_t channels;
    uint32_t width, height;       /* level 0 (a power of two each)                          */
    uint32_t wrap;                /* PBRT_B200_WRAP_*                                       */
    uint32_t do_trilinear;
    float    max_anisotropy;
    uint32_t pad;
} pbrt_b200_mipmap; /* 40 bytes */

/* A texture-valued material parameter: textures[first, first + count) is its postfix program; count == 0: the constant. */
typedef struct pbrt_b200_texref { uint32_t first, count; } pbrt_b200_texref;

/* Parameters of a `textured` material row, by slot (s = spectrum, f = float):
 *   matte s0=Kd f0=sigma | plastic s0=Kd s1=Ks f0=roughness | mirror s0=Kr | glass s0=Kr s1=Kt f0=urough f1=vrough f2=index
 *   metal s0=eta s1=k f0=urough f1=vrough (the host resolves the `roughness` fallback, metal.rs:88-97) | uber, substrate: above.
 * bump.count > 0: Material::bump (src/core/material.rs:46-87) runs first, as in every compute_scattering_functions.        */
typedef struct pbrt_b200_material_ext {
    pbrt_b200_texref s_tex[5];
    float            s_const[5][3];
    pbrt_b200_texref f_tex[3];
    float            f_const[3];
    pbrt_b200_texref bump;
    uint32_t pad[4];
} pbrt_b200_material_ext; /* 160 bytes */

enum {
    PBRT_B200_LIGHT_POINT = 0,    /* src/lights/point.rs:30-97    pos, I=L            */
    PBRT_B200_LIGHT_DISTANT = 1,  /* src/lights/distant.rs:32-122 dir=wlight, L       */
    PBRT_B200_LIGHT_SPOT = 2,     /* src/lights/spot.rs:31-119                        */
    PBRT_B200_LIGHT_DIFFUSE = 3,  /* src/lights/diffuse.rs:20-176 one per emissive shape */
    PBRT_B200_LIGHT_INFINITE = 4  /* src/lights/infinite.rs:120-177, constant radiance */
};

typedef struct pbrt_b200_light {
    uint32_t type;
    uint32_t two_sided;        /* diffuse                                            */
    float L[3];                /* I (point/spot), L (distant), Lemit (diffuse), Lmap*scale (infinite) */
    float pos[3];              /* point/spot: plight (world)                         */
    float dir[3];              /* distant: wlight (world, normalised)                */
    uint32_t shape_kind;       /* diffuse: emitting shape                            */
    uint32_t shape_index;
    uint32_t shape_flags;      /* PBRT_B200_PRIM_* of the emitting shape             */
    float area;                /* diffuse: Shape::area()                             */
    float cos_total_width;     /* spot                                               */
    float cos_falloff_start;   /* spot                                               */
    float world_to_light[16];  /* spot                                               */
    uint32_t n_samples;        /* Light::nsamples() (diffuse / infinite "samples", 1 otherwise; 0 reads as 1): only
                                  DirectLightingIntegrator "all" looks at it (directlighting.rs:61-76)  */
} pbrt_b200_light; /* 136 bytes */

/* = PerspectiveCamera (src/cameras/perspective.rs:22-37); matrices row-major. */
typedef struct pbrt_b200_camera {
    float raster_to_camera[16];
    float camera_to_world[16];
    float lens_radius;
    float focal_distance;
    float shutter_open;
    float shutter_close;
} pbrt_b200_camera;

/* = Film (src/core/film.rs:43-53).  Bounds are [x0,y0,x1,y1), pixels.        */
typedef struct pbrt_b200_film {
    int32_t full_resolution[2];
    int32_t cropped_pixel_bounds[4];
    float   filter_radius[2];
    float   filter_table[256];     /* FILTER_TABLE_WIDTH^2, film.rs:16,77-89        */
    float   scale;
    float   max_sample_luminance;  /* +inf = off                                    */
} pbrt_b200_film;

enum { PBRT_B200_SAMPLER_SOBOL = 0, PBRT_B200_SAMPLER_HALTON = 1, PBRT_B200_SAMPLER_ZEROTWO = 2 };

/* Sampler state the host owns (src/samplers/{sobol,halton,zerotwosequence}.rs).
 * Tables are the reference crate's own constants, passed by pointer.          */
typedef struct pbrt_b200_sampler {
    uint32_t kind;
    uint32_t samples_per_pixel;
    int32_t  sample_bounds[4];       /* Film::get_sample_bounds, film.rs:104-111      */
    uint32_t n_sampled_dimensions;   /* 02-sequence `dimensions` (default 4)          */
    uint32_t pad;
    const uint32_t *sobol_matrices32;/* [1024*52]  sobolmatrices.rs:5                 */
    const uint64_t *vdc_matrices;    /* [25*52]    rows padded, sobolmatrices.rs:26842 */
    const uint64_t *vdc_matrices_inv;/* [26*52]    sobolmatrices.rs:27534             */
} pbrt_b200_sampler;

enum { PBRT_B200_LIGHTS_UNIFORM = 0, PBRT_B200_LIGHTS_POWER = 1, PBRT_B200_LIGHTS_SPATIAL = 2 };

/* Which SamplerIntegrator drives the kernels (api.rs:276-289): `Integrator "path"` (src/integrators/path.rs),
 * `"directlighting"` (src/integrators/directlighting.rs, strategy "one" or "all") or `"whitted"`
 * (src/integrators/whitted.rs).  0 = path keeps descriptors written before the field existed valid.         */
enum { PBRT_B200_INTEGRATOR_PATH = 0, PBRT_B200_INTEGRATOR_DIRECT_ONE = 1, PBRT_B200_INTEGRATOR_DIRECT_ALL = 2,
       PBRT_B200_INTEGRATOR_WHITTED = 3,
       PBRT_B200_INTEGRATOR_VOLPATH = 4 /* `Integrator "volpath"` (src/integrators/volpath.rs:82-262) with homogeneous media */,
       PBRT_B200_INTEGRATOR_BDPT = 5    /* `Integrator "bdpt"` (src/integrators/bdpt.rs) on surfaces; rendered by pbrt_b200_render_splat
                                         * only, since its light-tracing strategies add to a second film                        */ };

/* = PathIntegrator (src/integrators/path.rs:32-40,228-249); max_depth and pixel_bounds mean the same for
 * DirectLightingIntegrator (directlighting.rs:27-39,122-157) and WhittedIntegrator (whitted.rs), which ignore
 * rr_threshold and light_sample_strategy.  A negative max_depth means what path.rs's signed compare makes it:
 * every path ends at its first hit.  Deviation from the reference, which has no upper bound: path and volpath
 * reject max_depth > 65520 (PBRT_B200_ERR_INVALID), since the kernels count bounces in 16 bits.             */
typedef struct pbrt_b200_integrator {
    int32_t  max_depth;
    float    rr_threshold;
    int32_t  pixel_bounds[4];
    uint32_t light_sample_strategy;
    uint32_t kind;                   /* PBRT_B200_INTEGRATOR_*                        */
    int32_t  camera_medium;          /* ABI v4: medium the camera sits in (Camera.medium, camera.rs; index into
                                      * pbrt_b200_scene_desc.media) or -1; only the volpath integrator looks at it   */
    uint32_t reserved;
} pbrt_b200_integrator;

/* = HomogeneousMedium (src/media/homogeneous.rs:10-27) or GridDensityMedium (src/media/grid.rs) with its HenyeyGreenstein phase
 * function (medium.rs:172-200). 32 B. */
typedef struct pbrt_b200_medium {
    float sigma_a[3];
    float sigma_s[3];                /* sigma_t = sigma_a + sigma_s is formed on use, as HomogeneousMedium::new does */
    float g;
    uint32_t grid;                   /* 0: HomogeneousMedium; k > 0: GridDensityMedium whose density grid is grids[k - 1] of
                                      * pbrt_b200_scene_create_with_grids.  A grid medium uses sigma_t = (sigma_a + sigma_s)[0]. */
} pbrt_b200_medium;

/* The density field of a GridDensityMedium (src/media/grid.rs).  medium_to_world maps the unit box [0,1]^3 of the grid onto
 * the world (CTM at MakeNamedMedium x Translate(p0) x Scale(p1 - p0)); world_to_medium is its inverse as the Transform
 * carries it.  Both row-major.  density[(z * ny + y) * nx + x] is the value at voxel (x, y, z), nx * ny * nz floats,
 * finite and >= 0.  152 B. */
typedef struct pbrt_b200_density_grid {
    float medium_to_world[16];
    float world_to_medium[16];
    uint32_t nx, ny, nz, pad;
    const float *density;
} pbrt_b200_density_grid;

/* = MediumInterface of a GeometricPrimitive (src/core/medium.rs:131-160, primitive.rs:105-150): indices into `media`, -1 = none.
 * A row whose two sides differ is a medium transition; other rows inherit the medium of the ray that hits them.        */
typedef struct pbrt_b200_medium_interface {
    int32_t inside;
    int32_t outside;
} pbrt_b200_medium_interface;

/* Flattened Scene (src/core/scene.rs:23-29 + what hangs off it).              */
typedef struct pbrt_b200_scene_desc {
    uint32_t abi_version;            /* PBRT_B200_ABI_VERSION                         */
    uint32_t pad;
    const pbrt_b200_bvh_node *nodes; uint64_t n_nodes;   /* BVHAccel.nodes            */
    const pbrt_b200_prim *prims;     uint64_t n_prims;   /* BVHAccel.primitives order */
    /* TriangleMesh SoA, world space (src/shapes/triangle.rs:21-48) */
    const float *vertex_p;           /* 3*n_vertices                                  */
    const float *vertex_n;           /* 3*n_vertices or NULL                          */
    const float *vertex_s;           /* 3*n_vertices or NULL                          */
    const float *vertex_uv;          /* 2*n_vertices or NULL                          */
    uint64_t n_vertices;
    const uint32_t *tri_indices;     /* 3*n_triangles                                 */
    uint64_t n_triangles;
    const pbrt_b200_sphere *spheres; uint64_t n_spheres;
    const pbrt_b200_material *materials; uint64_t n_materials;
    const pbrt_b200_light *lights;   uint64_t n_lights;  /* Scene.lights order        */
    /* Object instancing.  With n_objects == 0 every node and primitive row belongs to the top-level BVH and
     * n_top_nodes / n_top_prims may be 0 (= n_nodes / n_prims).                                                  */
    const pbrt_b200_object *objects;     uint64_t n_objects;
    const pbrt_b200_instance *instances; uint64_t n_instances;
    uint64_t n_top_nodes, n_top_prims;   /* Scene.aggregate: nodes[0, n_top_nodes), prims[0, n_top_prims)          */
    /* ABI v4: participating media (MakeNamedMedium / MediumInterface, api.rs).  prim_media has one row per `prims` row
     * (same order) or is NULL when no primitive carries a medium interface.                                           */
    const pbrt_b200_medium *media;       uint64_t n_media;
    const pbrt_b200_medium_interface *prim_media;
    /* ABI v5: textures (SURVEY §8 f3).  material_ext has one row per `materials` row or is NULL when no row is `textured`. */
    const pbrt_b200_texnode *textures;   uint64_t n_textures;
    const pbrt_b200_mipmap *mipmaps;     uint64_t n_mipmaps;
    const pbrt_b200_material_ext *material_ext;
} pbrt_b200_scene_desc;

typedef struct pbrt_b200_scene pbrt_b200_scene; /* opaque; owns device memory */

/* ---- rays --------------------------------------------------------------- */

/* Ray as the batch entry points see it (src/core/geometry/ray.rs:9-16). 32 B. */
typedef struct pbrt_b200_ray {
    float o[3];
    float t_max;
    float d[3];
    float time;
} pbrt_b200_ray;

/* Closest-hit record.  prim = creation_index of the hit GeometricPrimitive, or
 * 0xffffffff on a miss; t = r.t_max after the hit (primitive.rs:137);
 * b0,b1 = first two barycentrics (triangle.rs:209-213; b2 = 1-b0-b1 is NOT how
 * the reference computes it, so shading recomputes e2/det from the slot).  16 B. */
typedef struct pbrt_b200_hit {
    uint32_t prim;
    float t;
    float b0;
    float b1;
} pbrt_b200_hit;

#define PBRT_B200_NO_HIT 0xffffffffu

/* ---- entry points -------------------------------------------------------- */

const char *pbrt_b200_last_error(void);
int pbrt_b200_abi_version(void);
/* number of visible CUDA devices (0 => every compute call fails) */
int pbrt_b200_device_count(void);

/* Scene::new (src/core/scene.rs:32-52) + upload.  `device` = CUDA ordinal.     */
int pbrt_b200_scene_create(const pbrt_b200_scene_desc *desc, int device, pbrt_b200_scene **out);
/* The same with the density grids the media rows refer to (pbrt_b200_medium.grid).  scene_create(d, dev, out) is
 * scene_create_with_grids(d, NULL, 0, dev, out).  The densities are copied; a grid is checked before anything reaches the
 * device (index range, non-null density, nx * ny * nz > 0 without overflow, finite non-negative densities, finite matrices). */
int pbrt_b200_scene_create_with_grids(const pbrt_b200_scene_desc *desc, const pbrt_b200_density_grid *grids, uint64_t n_grids, int device,
                                      pbrt_b200_scene **out);
void pbrt_b200_scene_destroy(pbrt_b200_scene *scene);
/* Scene.wb (scene.rs:27): root bounds, 6 floats. */
int pbrt_b200_scene_world_bound(const pbrt_b200_scene *scene, float *bounds6);

/* Scene::intersect (src/core/scene.rs:54-59) over a batch: BVHAccel::intersect
 * (bvh.rs:705-760) + Triangle::intersect (triangle.rs:136-233) / Sphere.        */
int pbrt_b200_intersect(pbrt_b200_scene *scene, const pbrt_b200_ray *rays, uint64_t n,
                        pbrt_b200_hit *hits);
/* Scene::intersect_p (scene.rs:61-66): out[i] = 1 if occluded.                  */
int pbrt_b200_intersect_p(pbrt_b200_scene *scene, const pbrt_b200_ray *rays, uint64_t n,
                          uint8_t *occluded);
/* Same, buffers already resident on the scene's device; asynchronous on
 * `stream` (a cudaStream_t passed as void*, NULL = legacy default stream).      */
int pbrt_b200_intersect_dev(pbrt_b200_scene *scene, const pbrt_b200_ray *rays_dev, uint64_t n,
                            pbrt_b200_hit *hits_dev, void *stream);
int pbrt_b200_intersect_p_dev(pbrt_b200_scene *scene, const pbrt_b200_ray *rays_dev, uint64_t n,
                              uint8_t *occluded_dev, void *stream);

/* Render job = Integrator + Camera + Film + Sampler bound to a scene.          */
typedef struct pbrt_b200_render_desc {
    pbrt_b200_camera camera;
    pbrt_b200_film film;
    pbrt_b200_sampler sampler;
    pbrt_b200_integrator integrator;
    /* Work window for multi-GPU / batched runs: only tiles (16x16 over the sample
     * bounds, integrator.rs:274-279) with index in [tile_begin, tile_end) and
     * pixel samples in [sample_begin, sample_end) are rendered.  0,0 => all.    */
    uint32_t tile_begin, tile_end;
    uint32_t sample_begin, sample_end;
    uint32_t paths_in_flight;   /* 0 => library default                          */
    uint32_t flags;             /* PBRT_B200_RENDER_*                            */
    /* Interleaved ownership inside [tile_begin, tile_end) for static multi-GPU
     * partitioning: tile t is rendered iff ((t - tile_begin) / tile_group) %
     * tile_mod == tile_rem.  0,0,0 => every tile (group 1, mod 1, rem 0).       */
    uint32_t tile_group, tile_mod, tile_rem;
    /* Numbering of the tiles that [tile_begin, tile_end) refers to.  0: the reference's, row-major over the whole image
     * (integrator.rs:274-279).  S > 0: super-tile major -- the image is cut into S x S-tile blocks (S = 8: 128 x 128 pixels),
     * blocks row-major, tiles row-major inside a block, positions past the image edge are empty; the numbering then runs
     * over ceil(ntx/S) * ceil(nty/S) * S * S positions (pbrt_b200_tile_positions).  Consecutive ranges are compact image
     * regions, which is what a multi-GPU scheduler wants to hand out (coherent rays); every tile keeps its own sampler
     * seed and pixels, so the image does not depend on the numbering.                                                  */
    uint32_t tile_order;
} pbrt_b200_render_desc;

enum {
    PBRT_B200_RENDER_KEEP_ON_DEVICE = 1u << 0, /* rgbw_out is a device pointer      */
    PBRT_B200_RENDER_OVERWRITE = 1u << 2,      /* host rgbw_out is overwritten, not added to (Film::set_image, film.rs:172-184,
                                                * instead of merge_film_tile): saves zeroing and re-reading the buffer   */
    PBRT_B200_RENDER_LAZY_SPATIAL = 1u << 1    /* "spatial" light distribution: build voxels on first touch even when
                                                * the whole grid would fit (the mode used automatically for voxels x
                                                * lights > 2^25; results are identical, lightdistrib.rs:231-340)    */
};

/* Number of positions of the tile numbering `tile_order` for a sample-bounds window of w x h pixels (= the number
 * of tiles when tile_order is 0).                                                                                    */
uint32_t pbrt_b200_tile_positions(int w, int h, uint32_t tile_order);

/* ---- work counter shared between the processes that drive the GPUs of one box ------------------------------------
 * The reference hands tiles to its worker threads through one shared queue (integrator.rs:291-296, rayon par_iter).
 * With one process per GPU the queue head is a 64-bit counter in POSIX shared memory: every rank claims the next
 * range of tile positions with one atomic fetch-add on host memory (no network round trip), renders it with
 * pbrt_b200_render(tile_begin, tile_end, tile_order), and the films are summed once at the end.                   */
typedef struct pbrt_b200_work_counter pbrt_b200_work_counter;
/* create != 0: create (or reset) the named counter at 0; otherwise attach to an existing one.                       */
int pbrt_b200_work_counter_open(const char* name, int create, pbrt_b200_work_counter** out);
/* Atomically adds n and returns the PREVIOUS value (the first unit of the caller's claim).                            */
uint64_t pbrt_b200_work_counter_fetch_add(pbrt_b200_work_counter* c, uint64_t n);
/* Raises the counter to at least v (atomic max); returns the previous value.  A rank entering frame f calls it with the
 * frame's base position: whoever arrives first moves the queue head there, nobody waits for anybody.                 */
uint64_t pbrt_b200_work_counter_fetch_max(pbrt_b200_work_counter* c, uint64_t v);
uint64_t pbrt_b200_work_counter_load(const pbrt_b200_work_counter* c);
void pbrt_b200_work_counter_store(pbrt_b200_work_counter* c, uint64_t v);
/* unlink != 0 also removes the name (the creator does that).                                                         */
void pbrt_b200_work_counter_close(pbrt_b200_work_counter* c, int unlink_name);

/* Counters mirroring the reference's stats (integrator.rs:36, scene.rs:14-15,
 * path.rs:24-25).                                                              */
typedef struct pbrt_b200_render_stats {
    uint64_t camera_rays;
    uint64_t intersection_tests;   /* closest-hit rays (path + MIS)                 */
    uint64_t shadow_tests;         /* any-hit rays                                  */
    uint64_t zero_radiance_paths;
    uint64_t kernel_launches;      /* kernels this library launched for the call    */
    double   device_ms;            /* CUDA-event time of the wavefront loop          */
    double   trace_closest_ms;     /* of which: closest-hit traversal kernel         */
    double   trace_any_ms;         /* of which: any-hit traversal kernel             */
    double   shade_ms;             /* of which: classify + shade<material> kernels   */
    double   finish_ms;            /* of which: film accumulation + path regeneration */
    uint64_t iterations;           /* wavefront iterations (one path segment each)   */
} pbrt_b200_render_stats;

/* SamplerIntegrator::render (src/core/integrator.rs:263-403) minus file output:
 * accumulates filter-weighted samples (FilmTile::add_sample, film.rs:292-331)
 * into rgbw_out[4 * width * height] over film.cropped_pixel_bounds as
 * {sum r, sum g, sum b, sum filter weight}; the buffer is ADDED to, so a caller
 * may split a render into several calls (or GPUs) and sum.  `stats` may be NULL.
 * Sample bounds wider or taller than 65535 pixels fail with PBRT_B200_ERR_INVALID. */
int pbrt_b200_render(pbrt_b200_scene *scene, const pbrt_b200_render_desc *desc,
                     float *rgbw_out, pbrt_b200_render_stats *stats);

/* pbrt_b200_render for the PBRT_B200_INTEGRATOR_BDPT kind: BDPTIntegrator::render (pbrt-v3 integrators/bdpt.cpp), whose t = 1
 * strategies (light subpaths connected to the camera) land on arbitrary pixels through Film::add_splat.  rgbw_out is as for
 * pbrt_b200_render; splat_out[3 * width * height] over film.cropped_pixel_bounds receives the splatted RGB sums and follows the
 * same rules (added to, PBRT_B200_RENDER_OVERWRITE and PBRT_B200_RENDER_KEEP_ON_DEVICE apply to both buffers, tile and sample
 * windows sum).  Resolve with pbrt_b200_film_resolve_splat(splat_scale = 1 / samples_per_pixel).  Refused with
 * PBRT_B200_ERR_UNSUPPORTED: scenes with participating media, the 02sequence sampler, and max_depth outside
 * [0, PBRT_B200_BDPT_MAX_DEPTH] (each of the up to 2 * max_depth + 3 subpath vertices of a sample is kept in
 * device memory).  Any other integrator kind is PBRT_B200_ERR_INVALID here.                                                    */
#define PBRT_B200_BDPT_MAX_DEPTH 64
int pbrt_b200_render_splat(pbrt_b200_scene *scene, const pbrt_b200_render_desc *desc,
                           float *rgbw_out, float *splat_out, pbrt_b200_render_stats *stats);

/* Device and pinned-host blocks released by pbrt_b200_scene_destroy are kept in a per-process pool and handed to the
 * next scene (the reference drops its Scene after every WorldEnd, src/core/api.rs:1750-1755; re-allocating ~6 GB of
 * path state per render would dominate short renders).  This returns every cached block to the driver.             */
void pbrt_b200_release_cached_memory(void);

/* LightDistribution::lookup (src/core/lightdistrib.rs:33-36; Uniform :44-61, Power :63-83, Spatial :231-340) for a
 * batch of world-space points: voxel_out[3*n] = SpatialLightDistribution's integer voxel of each point (-1,-1,-1 for
 * the uniform/power strategies), func_out[n * n_lights] = the Distribution1D::func the integrator samples a light from
 * at that point.  Host buffers.  `flags`: PBRT_B200_RENDER_LAZY_SPATIAL or 0.                                        */
int pbrt_b200_light_distribution_lookup(pbrt_b200_scene *scene, uint32_t strategy, uint32_t flags,
                                        const float *points, uint64_t n, int32_t *voxel_out, float *func_out);

/* Film::write_image arithmetic (src/core/film.rs:217-264): RGB->XYZ->RGB,
 * divide by weight, clamp at 0, scale.  rgb_out[3*npixels].  Host buffers.      */
int pbrt_b200_film_resolve(const float *rgbw, uint64_t npixels, float scale, float *rgb_out);

/* Film::write_image(splat_scale) (pbrt-v3 film.cpp:148-185): the weighted RGB of pbrt_b200_film_resolve, clamped at 0, plus
 * splat_scale times the splat film (through the same RGB->XYZ->RGB round trip), times scale.  rgb_out[3*npixels].             */
int pbrt_b200_film_resolve_splat(const float *rgbw, const float *splat, uint64_t npixels, float splat_scale, float scale, float *rgb_out);

#ifdef __cplusplus
}
#endif
#endif /* PBRT_B200_H */
