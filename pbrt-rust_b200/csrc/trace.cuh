// Software BVH traversal + watertight triangle test + sphere quadric (device).
//
// Replaces BVHAccel::intersect / intersect_p (accelerators/bvh.rs:705-814),
// Bounds3f::intersect_p2 (core/geometry/bounds.rs:559-580), Triangle::intersect /
// intersect_p (shapes/triangle.rs:136-233, 400-495) and Sphere::intersect root
// selection (shapes/sphere.rs:59-108).
//
// Exactness contract: the same boxes are tested in the same order with the same f32
// arithmetic as the reference's binary traversal, so primitive IDs, t and the
// barycentrics are bit-identical.  The layout differs (child boxes live in the parent:
// one 64-byte fetch per step, four 128-bit loads): a child box is slab-tested when its
// parent is visited and only the t_max-dependent part of the reference's test
// (`tmin < ray.t_max`) is re-evaluated when the entry is popped -- which is when the
// reference would have tested that node.
// Alternatives that were measured on B200 and lost are recorded in DESIGN.md §4 and profiles/ (r02_cquad.md, r02_trace_lanes.md).
#pragma once
#include "scene.cuh"
#include "vecmath.cuh"

namespace pb {

struct RayHit {
    uint32_t slot;  // BVH slot of the hit primitive or PBRT_B200_NO_HIT
    float t, b0, b1, b2;
    uint32_t inst;  // instance the hit went through (TransformedPrimitive) or PBRT_B200_NO_HIT
};

// --- Triangle::intersect, triangle.rs:136-233 (+ :236-263 rejection for closest hits)
template <bool CLOSEST>
PB_D bool triangle_test(f3 o, f3 dir, float t_max, f3 p0, f3 p1, f3 p2, int kx, int ky, int kz, float Sx, float Sy, float Sz,
                        float* t_out, float* b0_out, float* b1_out, float* b2_out) {
    f3 q0 = p0 - o, q1 = p1 - o, q2 = p2 - o;
    (void)kx; (void)ky;
    f3 p0t = permute_kz(q0, kz), p1t = permute_kz(q1, kz), p2t = permute_kz(q2, kz);
    p0t.x += Sx * p0t.z; p0t.y += Sy * p0t.z;
    p1t.x += Sx * p1t.z; p1t.y += Sy * p1t.z;
    p2t.x += Sx * p2t.z; p2t.y += Sy * p2t.z;
    float e0 = p1t.x * p2t.y - p1t.y * p2t.x;
    float e1 = p2t.x * p0t.y - p2t.y * p0t.x;
    float e2 = p0t.x * p1t.y - p0t.y * p1t.x;
    if (e0 == 0.0f || e1 == 0.0f || e2 == 0.0f) {  // f64 fallback at triangle edges
        e0 = (float)__dsub_rn(__dmul_rn((double)p2t.y, (double)p1t.x), __dmul_rn((double)p2t.x, (double)p1t.y));
        e1 = (float)__dsub_rn(__dmul_rn((double)p0t.y, (double)p2t.x), __dmul_rn((double)p0t.x, (double)p2t.y));
        e2 = (float)__dsub_rn(__dmul_rn((double)p1t.y, (double)p0t.x), __dmul_rn((double)p1t.x, (double)p0t.y));
    }
    if ((e0 < 0.0f || e1 < 0.0f || e2 < 0.0f) && (e0 > 0.0f || e1 > 0.0f || e2 > 0.0f)) return false;
    float det = e0 + e1 + e2;
    if (det == 0.0f) return false;
    p0t.z *= Sz; p1t.z *= Sz; p2t.z *= Sz;
    float tscaled = e0 * p0t.z + e1 * p1t.z + e2 * p2t.z;
    if (det < 0.0f && (tscaled >= 0.0f || tscaled < t_max * det)) return false;
    else if (det > 0.0f && (tscaled <= 0.0f || tscaled >= t_max * det)) return false;
    float invdet = 1.0f / det;
    float b0 = e0 * invdet, b1 = e1 * invdet, b2 = e2 * invdet;
    float t = tscaled * invdet;
    float maxzt = fmaxf(fabsf(p0t.z), fmaxf(fabsf(p1t.z), fabsf(p2t.z)));
    float deltaz = gamma_n(3) * maxzt;
    float maxxt = fmaxf(fabsf(p0t.x), fmaxf(fabsf(p1t.x), fabsf(p2t.x)));
    float maxyt = fmaxf(fabsf(p0t.y), fmaxf(fabsf(p1t.y), fabsf(p2t.y)));
    float deltax = gamma_n(5) * (maxxt + maxzt);
    float deltay = gamma_n(5) * (maxyt + maxzt);
    float deltae = 2.0f * (gamma_n(2) * maxxt * maxyt + deltay * maxxt + deltax * maxyt);
    float maxe = fmaxf(fabsf(e0), fmaxf(fabsf(e1), fabsf(e2)));
    float deltat = 3.0f * (gamma_n(3) * maxe * maxzt + deltae * maxzt + deltaz * maxe) * fabsf(invdet);
    if (t <= deltat) return false;
    *t_out = t; *b0_out = b0; *b1_out = b1; *b2_out = b2;
    return true;
}

// triangle.rs:236-263: after the t tests a closest-hit candidate is still rejected when
// both dpdu x dpdv and the geometric normal vanish.  uv = per-vertex (u,v) or the default
// parameterisation (triangle.rs:109-115).
static __device__ __noinline__ bool triangle_bogus(f3 p0, f3 p1, f3 p2, float2 uv0, float2 uv1, float2 uv2) {
    float2 duv02 = make_float2(uv0.x - uv2.x, uv0.y - uv2.y), duv12 = make_float2(uv1.x - uv2.x, uv1.y - uv2.y);
    f3 dp02 = p0 - p2, dp12 = p1 - p2;
    float determinant = duv02.x * duv12.y - duv02.y * duv12.x;
    bool degenerateuv = fabsf(determinant) < 1.0e-8f;
    f3 dpdu(0.f, 0.f, 0.f), dpdv(0.f, 0.f, 0.f);
    if (!degenerateuv) {
        float inv = 1.0f / determinant;
        dpdu = (dp02 * duv12.y - dp12 * duv02.y) * inv;
        dpdv = (dp02 * -duv12.x + dp12 * duv02.x) * inv;
    }
    if (degenerateuv || len2(cross(dpdu, dpdv)) == 0.0f) {
        f3 ng = cross(p2 - p0, p1 - p0);
        if (len2(ng) == 0.0f) return true;
    }
    return false;
}

#define PB_NO_SLOT 0xffffffffu
// slot != PB_NO_SLOT: the primitive's BVH slot (uvs pre-gathered in slot order, scene.cuh); otherwise through the index buffer
PB_D void fetch_uv(const DevScene& s, uint32_t flags, uint32_t shape_index, float2* uv0, float2* uv1, float2* uv2, uint32_t slot = PB_NO_SLOT) {
    if ((flags & PBRT_B200_PRIM_HAS_UV) && s.vertex_uv) {
        if (slot != PB_NO_SLOT && s.slot_uv) {
            const float2* u = s.slot_uv + 3ull * slot;
            *uv0 = __ldg(u); *uv1 = __ldg(u + 1); *uv2 = __ldg(u + 2);
            return;
        }
        const uint32_t* idx = s.tri_indices + 3ull * shape_index;
        const float2* uv = reinterpret_cast<const float2*>(s.vertex_uv);
        *uv0 = uv[idx[0]]; *uv1 = uv[idx[1]]; *uv2 = uv[idx[2]];
    } else {
        *uv0 = make_float2(0.f, 0.f); *uv1 = make_float2(1.f, 0.f); *uv2 = make_float2(1.f, 1.f);
    }
}

// --- EFloat (core/efloat.rs) ------------------------------------------------
struct EF { float v, lo, hi; };
PB_D EF ef(float v, float err) {
    EF r; r.v = v;
    if (err == 0.0f) { r.lo = v; r.hi = v; } else { r.lo = next_down(v - err); r.hi = next_up(v + err); }
    return r;
}
PB_D EF ef_add(EF a, EF b) { EF r; r.v = a.v + b.v; r.lo = next_down(a.lo + b.lo); r.hi = next_up(a.hi + b.hi); return r; }
PB_D EF ef_sub(EF a, EF b) { EF r; r.v = a.v - b.v; r.lo = next_down(a.lo - b.hi); r.hi = next_up(a.hi - b.lo); return r; }
PB_D EF ef_mul(EF a, EF b) {
    EF r; r.v = a.v * b.v;
    float p0 = a.lo * b.lo, p1 = a.hi * b.lo, p2 = a.lo * b.hi, p3 = a.hi * b.hi;
    r.lo = next_down(fminf(fminf(p0, p1), fminf(p2, p3)));
    r.hi = next_up(fmaxf(fmaxf(p0, p1), fmaxf(p2, p3)));
    return r;
}
PB_D EF ef_div(EF a, EF b) {  // efloat.rs:134-156: the NUMERATOR is tested for straddling zero
    EF r; r.v = a.v / b.v;
    if (a.lo < 0.0f && a.hi > 0.0f) { r.lo = -PB_INF; r.hi = PB_INF; }
    else {
        float q0 = a.lo / b.lo, q1 = a.hi / b.lo, q2 = a.lo / b.hi, q3 = a.hi / b.hi;
        r.lo = next_down(fminf(fminf(q0, q1), fminf(q2, q3)));
        r.hi = next_up(fmaxf(fmaxf(q0, q1), fmaxf(q2, q3)));
    }
    return r;
}

// World ray -> object space with error bounds, transform.rs:579-591
PB_D void sphere_object_ray(const pbrt_b200_sphere& sp, f3 o, f3 d, f3* oo, f3* od, f3* oerr, f3* derr) {
    *oo = xf_point_err(sp.world_to_object, o, oerr);
    *od = xf_vector_err(sp.world_to_object, d, derr);
    float l2 = len2(*od);
    if (l2 > 0.0f) {
        float dt = dot(vabs(*od), *oerr) / l2;
        *oo = *oo + *od * dt;
    }
}

// Sphere::intersect / intersect_p up to the choice of t_shape_hit, sphere.rs:59-108
// (full spheres; the partial-sphere clipping branch cannot trigger).
static __device__ __noinline__ bool sphere_test(const pbrt_b200_sphere* spp, f3 o, f3 d, float t_max, float* t_out) {
    const pbrt_b200_sphere& sp = *spp;
    f3 oo, od, oe, de;
    sphere_object_ray(sp, o, d, &oo, &od, &oe, &de);
    EF ox = ef(oo.x, oe.x), oy = ef(oo.y, oe.y), oz = ef(oo.z, oe.z);
    EF dx = ef(od.x, de.x), dy = ef(od.y, de.y), dz = ef(od.z, de.z);
    EF a = ef_add(ef_add(ef_mul(dx, dx), ef_mul(dy, dy)), ef_mul(dz, dz));
    EF b = ef_mul(ef(2.0f, 0.f), ef_add(ef_add(ef_mul(dx, ox), ef_mul(dy, oy)), ef_mul(dz, oz)));
    EF rr = ef(sp.radius, 0.f);
    EF c = ef_sub(ef_add(ef_add(ef_mul(ox, ox), ef_mul(oy, oy)), ef_mul(oz, oz)), ef_mul(rr, rr));
    // efloat.rs:211-231
    double discrim = __dsub_rn(__dmul_rn((double)b.v, (double)b.v), __dmul_rn(__dmul_rn(4.0, (double)a.v), (double)c.v));
    if (discrim < 0.0) return false;
    double root = sqrt(discrim);
    EF frd = ef((float)root, (float)__dmul_rn((double)PB_MACHINE_EPSILON, root));
    EF q = (b.v < 0.0f) ? ef_mul(ef(-0.5f, 0.f), ef_sub(b, frd)) : ef_mul(ef(-0.5f, 0.f), ef_add(b, frd));
    EF t0 = ef_div(q, a), t1 = ef_div(c, q);
    if (t0.v > t1.v) { EF tmp = t0; t0 = t1; t1 = tmp; }
    if (t0.hi > t_max || t1.lo <= 0.0f) return false;
    EF ts = t0;
    if (ts.lo <= 0.0f) {
        ts = t1;
        if (ts.hi > t_max) return false;
    }
    *t_out = ts.v;
    return true;
}

// --- Bounds3f::intersect_p2, bounds.rs:559-580, minus the final t_max comparison.
// Returns true when the slab tests pass and tmax > 0; *tmin_out is the value the
// reference compares against ray.t_max.
PB_D bool slab_test(float nx, float ny, float nz, float fx, float fy, float fz, f3 o, f3 inv, float* tmin_out) {
    const float widen = 1.0f + 2.0f * gamma_n(3);
    float tmin = (nx - o.x) * inv.x;
    float tmax = (fx - o.x) * inv.x;
    float tymin = (ny - o.y) * inv.y;
    float tymax = (fy - o.y) * inv.y;
    tmax *= widen;
    tymax *= widen;
    bool ok = !(tmin > tymax || tymin > tmax);
    if (tymin > tmin) tmin = tymin;
    if (tymax < tmax) tmax = tymax;
    float tzmin = (nz - o.z) * inv.z;
    float tzmax = (fz - o.z) * inv.z;
    tzmax *= widen;
    ok = ok && !(tmin > tzmax || tzmin > tmax);
    if (tzmin > tmin) tmin = tzmin;
    if (tzmax < tmax) tmax = tzmax;
    *tmin_out = tmin;
    return ok && (tmax > 0.0f);
}

// Same predicate and the same tmin as slab_test for rays whose direction has no zero component: then no
// product (b - o) * inv can be NaN, the reference's compare-and-assign chain equals max/min,
// and its pairwise early-outs equal `tmin <= tmax` (the i == j pairs it skips can only fail
// when that axis' far plane is behind the ray, which `tmax > 0` rejects anyway).
// Two boxes at once with Blackwell's packed f32x2 pipe (FADD2 / FMUL2: two IEEE-rounded f32 results per issue slot; +2-3 %
// on B200 against the scalar form, tools/trace_ab3.py).  Lane .x = child 0, .y = child 1.  Every product and difference is
// rounded exactly as in slab_test (sub -> mul -> mul can never contract), so the results are bit-identical.
struct SlabPair { float tmin0, tmin1; bool ok0, ok1; };
PB_D SlabPair slab_fast2(float2 nx, float2 ny, float2 nz, float2 fx, float2 fy, float2 fz, float2 nox, float2 noy, float2 noz, float2 ix, float2 iy, float2 iz) {
    const float w = 1.0f + 2.0f * gamma_n(3);
    const float2 widen = make_float2(w, w);
    float2 tx0 = __fmul2_rn(__fadd2_rn(nx, nox), ix), ty0 = __fmul2_rn(__fadd2_rn(ny, noy), iy), tz0 = __fmul2_rn(__fadd2_rn(nz, noz), iz);
    float2 tx1 = __fmul2_rn(__fmul2_rn(__fadd2_rn(fx, nox), ix), widen), ty1 = __fmul2_rn(__fmul2_rn(__fadd2_rn(fy, noy), iy), widen),
           tz1 = __fmul2_rn(__fmul2_rn(__fadd2_rn(fz, noz), iz), widen);
    SlabPair r;
    r.tmin0 = fmaxf(fmaxf(tx0.x, ty0.x), tz0.x); r.tmin1 = fmaxf(fmaxf(tx0.y, ty0.y), tz0.y);
    float tmax0 = fminf(fminf(tx1.x, ty1.x), tz1.x), tmax1 = fminf(fminf(tx1.y, ty1.y), tz1.y);
    r.ok0 = (r.tmin0 <= tmax0) && (tmax0 > 0.0f);
    r.ok1 = (r.tmin1 <= tmax1) && (tmax1 > 0.0f);
    return r;
}

#define PB_STACK_DEPTH 64  /* bvh.rs:722 nodes_tovisit = vec![0; 64] */
/* the reference keeps one 64-entry stack per BVHAccel; the unified two-level walk stacks the object's entries on top of the
 * world's, plus the sentinel and the rest-of-leaf entry */
/* the quad walk descends two binary levels per step and can stack three siblings: 3 * 64 / 2 entries for the deepest tree
 * scene_create accepts (depth <= 64) */
#define PB_STACK_SIZE(INST) ((INST) ? 3 * PB_STACK_DEPTH + 2 : 3 * PB_STACK_DEPTH / 2)
#define PB_DONE 0xffffffffu /* traversal finished (has the leaf bit set so the interior loop exits) */

// Per-ray traversal state.  The order of box and primitive tests is the reference's
// (see the exactness contract above); the control flow is "while-while": an inner loop
// that only walks interior nodes, then the leaf run, so that lanes of a warp reconverge
// on the two hot bodies instead of interleaving them.
struct TravRay {
    f3 o, d, inv;
    float t_max, Sx, Sy, Sz;
    uint32_t cur;    // node / leaf reference being visited, or PB_DONE
    int sp;
    int kx, ky, kz;
    bool ngx, ngy, ngz, found;
    uint32_t negmask;   // bit a set: the direction is negative along axis a
    bool nan_possible;  // a zero direction component: 0 * inf can appear in the slab test
    RayHit hit;
    // Inside an instanced object (INST kernels only): the instance being walked, whether it produced a hit, and the world
    // ray to restore when the object's sub-tree has been exhausted (the traversal stack holds a sentinel at that point).
    uint32_t cur_inst;
    bool inst_found;
    float world_t_max;
    f3 wo, wd;
    float2 nox, noy, noz, ivx, ivy, ivz;  // {-o, -o} and {1/d, 1/d} per axis for slab_fast2
};

PB_D bool trav_done(const TravRay& r) { return r.cur == PB_DONE; }

// ray-constant part of the watertight test (triangle.rs:151-165)
PB_D void trav_set_shear(TravRay& r) {
    const f3 d = r.d;
    f3 ad = vabs(d);
    r.kz = (ad.x > ad.y) ? ((ad.x > ad.z) ? 0 : 2) : ((ad.y > ad.z) ? 1 : 2);
    r.kx = (r.kz + 1 == 3) ? 0 : r.kz + 1;
    r.ky = (r.kx + 1 == 3) ? 0 : r.kx + 1;
    const float dpx = comp(d, r.kx), dpy = comp(d, r.ky), dpz = comp(d, r.kz);
    r.Sx = -dpx / dpz; r.Sy = -dpy / dpz; r.Sz = 1.0f / dpz;
}
// everything the box and triangle tests derive from (o, d) alone
PB_D void trav_set_ray(TravRay& r, f3 o, f3 d) {
    r.o = o; r.d = d;
    r.inv = f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
    r.ngx = r.inv.x < 0.0f; r.ngy = r.inv.y < 0.0f; r.ngz = r.inv.z < 0.0f;
    r.negmask = (r.ngx ? 1u : 0u) | (r.ngy ? 2u : 0u) | (r.ngz ? 4u : 0u);
    r.nan_possible = (d.x == 0.0f) || (d.y == 0.0f) || (d.z == 0.0f);
    r.nox = make_float2(-o.x, -o.x); r.noy = make_float2(-o.y, -o.y); r.noz = make_float2(-o.z, -o.z);
    r.ivx = make_float2(r.inv.x, r.inv.x); r.ivy = make_float2(r.inv.y, r.inv.y); r.ivz = make_float2(r.inv.z, r.inv.z);
    trav_set_shear(r);
}
// BVHAccel::intersect's first step: the root node's own bounds test (bvh.rs:724-727).  rb == nullptr: a one-primitive
// object, which the reference intersects directly.
PB_D uint32_t trav_enter_root(const TravRay& r, uint32_t root_ref, const float* rb) {
    if (root_ref == PB_REF_NONE) return PB_DONE;
    if (rb == nullptr) return root_ref;
    float tmin;
    bool ok = slab_test(r.ngx ? rb[3] : rb[0], r.ngy ? rb[4] : rb[1], r.ngz ? rb[5] : rb[2], r.ngx ? rb[0] : rb[3], r.ngy ? rb[1] : rb[4],
                        r.ngz ? rb[2] : rb[5], r.o, r.inv, &tmin);
    return (ok && tmin < r.t_max) ? root_ref : PB_DONE;
}
PB_D void trav_init_at(TravRay& r, f3 o, f3 d, float t_max, uint32_t root_ref, const float* rb) {
    r.t_max = t_max;
    r.hit.slot = PBRT_B200_NO_HIT; r.hit.t = t_max; r.hit.b0 = r.hit.b1 = r.hit.b2 = 0.0f; r.hit.inst = PBRT_B200_NO_HIT;
    r.found = false; r.sp = 0;
    r.cur_inst = PBRT_B200_NO_HIT; r.inst_found = false;
    trav_set_ray(r, o, d);
    r.cur = trav_enter_root(r, root_ref, rb);
}
PB_D void trav_init(const DevScene& s, TravRay& r, f3 o, f3 d, float t_max) { trav_init_at(r, o, d, t_max, s.root_ref, s.root_box); }

// Transform::transform_ray, core/transform.rs:543-577: origin nudged along d by its transform error, t_max -= dt
PB_D void xf_ray(const float* M, f3 o, f3 d, float t_max, f3* o_out, f3* d_out, float* t_max_out) {
    f3 oerr;
    f3 o2 = xf_point_err(M, o, &oerr);
    f3 d2 = xf_vector(M, d);
    float l2 = len2(d2);
    if (l2 > 0.0f) {
        float dt = dot(vabs(d2), oerr) / l2;
        o2 = o2 + d2 * dt;
        t_max -= dt;
    }
    *o_out = o2; *d_out = d2; *t_max_out = t_max;
}

// Traversal stack.  LocalStack: a per-thread array (local memory, served by L1 when it hits).  HybridStack: the first
// PB_SH_STACK levels live in SHARED memory ([level][thread], conflict-free), deeper levels overflow to the local array.
// ncu on k_trace_closest (profiles/r02_ncu_trace.md): local loads -- the pops -- hit L1 only 63 % of the time, as often as the node
// fetches they compete with for the cache, so a third of the pops paid an L2 round trip; a shared-memory level always answers in
// ~29 cycles and takes the stack lines out of the L1 working set.
// Measured on B200 (gpurun_out/r2f_ab.log; hits bit-identical in every variant): inside a frame 16 shared levels give S3 41.1 -> 40.5 ms
// per 16-spp step (closest 16.4 -> 16.1, shadow 8.1 -> 7.8 ms); on isolated 2 M-ray batches the same change LOSES 4-5 % (camera batch
// 4603 -> 4390 Mrays/s: the carve-out shrinks the L1 that a small batch's nodes otherwise fit in).  So the wavefront kernels take the
// hybrid stack and the batch API keeps the local one (trace_queue's SH parameter).
#define PB_SH_STACK 16
#define PB_TRACE_BLOCK 128 /* threads per CTA of every persistent ray-queue kernel */
struct LocalStack {
    uint2* loc;
    PB_D void put(int i, uint2 e) const { loc[i] = e; }
    PB_D uint2 get(int i) const { return loc[i]; }
};
template <int SH, int BLOCK>
struct HybridStack {
    uint2* sh;   // &shared[0][thread]; level l at sh[l * BLOCK]
    uint2* loc;  // levels >= SH
    PB_D void put(int i, uint2 e) const { if (i < SH) sh[i * BLOCK] = e; else loc[i - SH] = e; }
    PB_D uint2 get(int i) const { return i < SH ? sh[i * BLOCK] : loc[i - SH]; }
};

#define PB_INST_EXIT 0xfffffffeu /* stack sentinel (leaf bit set): the instanced object's sub-tree is exhausted */

// pop: the reference tests the popped node's box against the *current* t_max
#define PB_TRAV_POP(r, stack)                                           \
    do {                                                                \
        (r).cur = PB_DONE;                                              \
        while ((r).sp > 0) {                                            \
            --(r).sp;                                                   \
            uint2 e__ = (stack).get((r).sp);                                \
            if (__uint_as_float(e__.y) < (r).t_max) { (r).cur = e__.x; break; } \
        }                                                               \
    } while (0)

template <bool ANY, typename STK> PB_D void quad_step(const DevScene& s, TravRay& r, STK stack);  // defined below (quad nodes)

// Runs the ray until it finishes, or (when `yield_below` > 0) until fewer than `yield_below`
// lanes of the warp are still traversing, so that the caller can refill idle lanes.
// TOP: walking the scene's aggregate (leaf slots may be TransformedPrimitives); false inside an instanced object, where
// ObjectInstance cannot appear (api.rs:1674-1677): one level of instancing, one sentinel on the stack at most.
// Boxes are tested with the literal reference chain (slab_test: exact for rays with a zero direction component); rays without
// one take the quad step at TOP level, chosen per node visit because the ray changes at instance boundaries.
template <bool ANY, bool TOP, typename STK>
PB_D void trav_run_impl(const DevScene& s, TravRay& r, STK stack, int yield_below, int interior_min) {
    while (r.cur != PB_DONE) {
        // ---- interior nodes
        while (!(r.cur & PB_LEAF_BIT)) {
            if (TOP && !r.nan_possible) {
                quad_step<ANY>(s, r, stack);
                if (interior_min > 0 && __popc(__activemask()) < interior_min) break;
                continue;
            }
            const float4* np = s.nodes + 4ull * r.cur;
            float4 q0 = __ldg(np), q1 = __ldg(np + 1), q2 = __ldg(np + 2), q3 = __ldg(np + 3);
            uint32_t ref0 = __float_as_uint(q3.x), ref1 = __float_as_uint(q3.y), axis = __float_as_uint(q3.z);
            float tmin0, tmin1;
            const bool ok0 = slab_test(r.ngx ? q0.w : q0.x, r.ngy ? q1.x : q0.y, r.ngz ? q1.y : q0.z, r.ngx ? q0.x : q0.w, r.ngy ? q0.y : q1.x,
                                       r.ngz ? q0.z : q1.y, r.o, r.inv, &tmin0);
            const bool ok1 = slab_test(r.ngx ? q2.y : q1.z, r.ngy ? q2.z : q1.w, r.ngz ? q2.w : q2.x, r.ngx ? q1.z : q2.y, r.ngy ? q1.w : q2.z,
                                       r.ngz ? q2.x : q2.w, r.o, r.inv, &tmin1);
            // near child = second child when the ray is negative along the split axis (bvh.rs:743-751)
            // a failed slab test becomes tmin = +inf: `tmin < t_max` is then false at the visit and at every later pop, which is
            // all the reference ever asks of that box (an entry whose true tmin is +inf can never pass either).  +3-4 % on B200
            // against separate ok flags and a per-axis select of the near child, bit-identical.
            tmin0 = ok0 ? tmin0 : PB_INF; tmin1 = ok1 ? tmin1 : PB_INF;
            bool second_first = (r.negmask >> axis) & 1u;
            uint32_t nref = second_first ? ref1 : ref0, fref = second_first ? ref0 : ref1;
            float ntmin = second_first ? tmin1 : tmin0, ftmin = second_first ? tmin0 : tmin1;
            bool nhit = ntmin < r.t_max;
            bool fhit = ftmin < r.t_max;
            bool fok = ANY ? fhit : (ftmin < PB_INF);
            if (nhit) {
                if (ANY ? fhit : fok) {
                    stack.put(r.sp, make_uint2(fref, __float_as_uint(ftmin))); ++r.sp;
                }
                r.cur = nref;
            } else if (fhit) {
                r.cur = fref;
            } else {
                PB_TRAV_POP(r, stack);
            }
            // few lanes left descending while the rest of the warp waits at leaves: let the leaves run first
            if (interior_min > 0 && __popc(__activemask()) < interior_min) break;
        }
        if (r.cur == PB_DONE) break;
        // ---- leaf run (bvh.rs:730-736): every primitive of the leaf, in order
        if (TOP && r.cur == PB_INST_EXIT) {
            // back in world space: r.t_max = ray.t_max when the object was hit (primitive.rs:72), the world value otherwise
            if (!r.inst_found) r.t_max = r.world_t_max;
            trav_set_ray(r, r.wo, r.wd);
            r.cur_inst = PBRT_B200_NO_HIT; r.inst_found = false;
            PB_TRAV_POP(r, stack);
            continue;
        }
        if (r.cur & PB_LEAF_BIT) {
            uint32_t slot = r.cur & ~PB_LEAF_BIT;
            uint32_t fl;
            bool entered = false;
            do {
                const float4* tp = s.tris + 3ull * slot;
                float4 v0 = __ldg(tp), v1 = __ldg(tp + 1), v2 = __ldg(tp + 2);
                fl = __float_as_uint(v1.w);
                float t, b0, b1, b2;
                bool h;
                if (fl & (PB_TRI_SPHERE | PB_TRI_INSTANCE)) {
                    if (TOP && (fl & PB_TRI_INSTANCE)) {
                        // TransformedPrimitive::intersect / intersect_p, primitive.rs:58-89: continue the SAME loop inside the
                        // object's accelerator with the ray taken to object space (Transform::transform_ray: origin-error
                        // nudge, t_max -= dt).  Left on the stack, in pop order: the object's nodes, the sentinel that
                        // restores the world ray, then the rest of this leaf.
                        const DevInstance* in = s.instances + __float_as_uint(v2.w);
                        if (!(fl & PB_TRI_LAST)) { stack.put(r.sp, make_uint2(PB_LEAF_BIT | (slot + 1), 0xff800000u)); ++r.sp; }  // tmin = -inf: always resumed
                        stack.put(r.sp, make_uint2(PB_INST_EXIT, 0xff800000u)); ++r.sp;
                        r.wo = r.o; r.wd = r.d; r.world_t_max = r.t_max;
                        r.cur_inst = __float_as_uint(v2.w); r.inst_found = false;
                        f3 o2, d2;
                        float tm2;
                        xf_ray(in->world_to_prim, r.o, r.d, r.t_max, &o2, &d2, &tm2);
                        r.t_max = tm2;
                        trav_set_ray(r, o2, d2);
                        r.cur = trav_enter_root(r, in->root_ref, (in->flags & PB_INST_HAS_BOX) ? in->root_box : nullptr);
                        entered = true;
                        break;
                    }
                    h = sphere_test(s.spheres + __float_as_uint(v2.w), r.o, r.d, r.t_max, &t);
                    b0 = b1 = b2 = 0.0f;
                } else {
                    f3 p0(v0.x, v0.y, v0.z), p1(v1.x, v1.y, v1.z), p2(v2.x, v2.y, v2.z);
                    h = triangle_test<!ANY>(r.o, r.d, r.t_max, p0, p1, p2, r.kx, r.ky, r.kz, r.Sx, r.Sy, r.Sz, &t, &b0, &b1, &b2);
                    if (!ANY && h) {
                        float2 uv0, uv1, uv2;
                        fetch_uv(s, fl, __float_as_uint(v2.w), &uv0, &uv1, &uv2, slot);
                        if (triangle_bogus(p0, p1, p2, uv0, uv1, uv2)) h = false;
                    }
                }
                if (h) {
                    r.found = true;
                    r.hit.slot = slot; r.hit.t = t; r.hit.b0 = b0; r.hit.b1 = b1; r.hit.b2 = b2;
                    if (TOP) { r.hit.inst = r.cur_inst; r.inst_found = r.cur_inst != PBRT_B200_NO_HIT; }
                    if (ANY) { r.cur = PB_DONE; r.sp = 0; break; }
                    r.t_max = t;  // primitive.rs:137
                }
                ++slot;
            } while (!(fl & PB_TRI_LAST));
            if (ANY && r.found) break;
            if (TOP && entered) {
                if (r.cur == PB_DONE) PB_TRAV_POP(r, stack);  // the object's root box was missed: straight to the sentinel
            } else {
                PB_TRAV_POP(r, stack);
            }
        }
        if (yield_below > 0 && __popc(__activemask()) < yield_below) break;
    }
}

// The same walk over QUAD nodes (scene.cuh): one 128-byte fetch tests the four grandchildren of a reference node.
// Exactness: the reference visits a leaf iff the leaf's box passes `tmin < t_max` (and the slab test) when it is reached AND
// every ancestor's box passed when IT was reached.  A child box contains its children's boxes and (x - o) * inv is monotone
// in x in floating point, so a grandchild that passes implies its parent passed (tmin_parent <= tmin_gc <= tmax_gc <=
// tmax_parent, against a t_max that only shrinks): skipping the intermediate box test cannot change the set of leaves
// visited, PROVIDED the leaves are visited in the reference's order -- which is depth-first with the near child first at
// every binary node.  The four slots are therefore walked in exactly that order (near group by the node's axis, near
// slot inside each group by the child's axis), later ones are stacked behind earlier ones, and a stacked entry is
// re-checked against the current t_max when popped, as in the binary walk.  Only for rays without zero direction
// components (slab_fast2's precondition; the others take the binary, NaN-exact walk).
//
// quad_slots: the four slots of quad node `node` in visiting order -- t[k] = the slot's tmin (+inf when its slab test fails), ref[k]
// its reference.  The order depends on the ray only through `negmask` (trav_run_packet passes its warp's shared octant, which
// makes ref[] warp-uniform).
template <bool ANY>
PB_D void quad_slots(const DevScene& s, const TravRay& r, uint32_t node, uint32_t negmask, float* t, uint32_t* ref) {
    const float4* np = s.quads + 8ull * node;
    const float4 a0 = __ldg(np), a1 = __ldg(np + 1), a2 = __ldg(np + 2), b0 = __ldg(np + 3), b1 = __ldg(np + 4), b2 = __ldg(np + 5), q6 = __ldg(np + 6), q7 = __ldg(np + 7);
    SlabPair pa = slab_fast2(r.ngx ? make_float2(a1.z, a1.w) : make_float2(a0.x, a0.y), r.ngy ? make_float2(a2.x, a2.y) : make_float2(a0.z, a0.w),
                             r.ngz ? make_float2(a2.z, a2.w) : make_float2(a1.x, a1.y), r.ngx ? make_float2(a0.x, a0.y) : make_float2(a1.z, a1.w),
                             r.ngy ? make_float2(a0.z, a0.w) : make_float2(a2.x, a2.y), r.ngz ? make_float2(a1.x, a1.y) : make_float2(a2.z, a2.w),
                             r.nox, r.noy, r.noz, r.ivx, r.ivy, r.ivz);
    SlabPair pb = slab_fast2(r.ngx ? make_float2(b1.z, b1.w) : make_float2(b0.x, b0.y), r.ngy ? make_float2(b2.x, b2.y) : make_float2(b0.z, b0.w),
                             r.ngz ? make_float2(b2.z, b2.w) : make_float2(b1.x, b1.y), r.ngx ? make_float2(b0.x, b0.y) : make_float2(b1.z, b1.w),
                             r.ngy ? make_float2(b0.z, b0.w) : make_float2(b2.x, b2.y), r.ngz ? make_float2(b1.x, b1.y) : make_float2(b2.z, b2.w),
                             r.nox, r.noy, r.noz, r.ivx, r.ivy, r.ivz);
    const float tA0 = pa.ok0 ? pa.tmin0 : PB_INF, tA1 = pa.ok1 ? pa.tmin1 : PB_INF, tB0 = pb.ok0 ? pb.tmin0 : PB_INF, tB1 = pb.ok1 ? pb.tmin1 : PB_INF;
    const uint32_t meta = __float_as_uint(q7.x);
    const bool g = (negmask >> (meta & 3u)) & 1u, sA = (negmask >> ((meta >> 2) & 3u)) & 1u, sB = (negmask >> ((meta >> 4) & 3u)) & 1u;
    // reference order inside each group, then of the groups
    const float tAn = sA ? tA1 : tA0, tAf = sA ? tA0 : tA1, tBn = sB ? tB1 : tB0, tBf = sB ? tB0 : tB1;
    const uint32_t rAn = __float_as_uint(sA ? q6.y : q6.x), rAf = __float_as_uint(sA ? q6.x : q6.y);
    const uint32_t rBn = __float_as_uint(sB ? q6.w : q6.z), rBf = __float_as_uint(sB ? q6.z : q6.w);
    // an any-hit ray's answer does not depend on the visiting order (t_max never changes): slots in storage order, no selects (the
    // near / far selects are ~20 % of the node step: shadow batch 4564 -> 4811 Mrays/s on B200, occlusion bits identical)
    const float t0 = ANY ? tA0 : (g ? tBn : tAn), t1 = ANY ? tA1 : (g ? tBf : tAf), t2 = ANY ? tB0 : (g ? tAn : tBn), t3 = ANY ? tB1 : (g ? tAf : tBf);
    const uint32_t r0 = ANY ? __float_as_uint(q6.x) : (g ? rBn : rAn), r1 = ANY ? __float_as_uint(q6.y) : (g ? rBf : rAf),
                   r2 = ANY ? __float_as_uint(q6.z) : (g ? rAn : rBn), r3 = ANY ? __float_as_uint(q6.w) : (g ? rAf : rBf);
    t[0] = t0; t[1] = t1; t[2] = t2; t[3] = t3;
    ref[0] = r0; ref[1] = r1; ref[2] = r2; ref[3] = r3;
}
template <bool ANY, typename STK>
PB_D void quad_step(const DevScene& s, TravRay& r, STK stack) {
    float t[4];
    uint32_t ref[4];
    quad_slots<ANY>(s, r, r.cur, r.negmask, t, ref);
    const float t0 = t[0], t1 = t[1], t2 = t[2], t3 = t[3];
    const uint32_t r0 = ref[0], r1 = ref[1], r2 = ref[2], r3 = ref[3];
    // the first slot that passes is visited now; the others wait on the stack, nearest on top
    uint32_t nref = PB_DONE; float ntm = 0.0f;
#define PB_QPUSH() do { stack.put(r.sp, make_uint2(nref, __float_as_uint(ntm))); ++r.sp; } while (0)
    if (t3 < r.t_max) { nref = r3; ntm = t3; }
    if (t2 < r.t_max) { if (nref != PB_DONE) PB_QPUSH(); nref = r2; ntm = t2; }
    if (t1 < r.t_max) { if (nref != PB_DONE) PB_QPUSH(); nref = r1; ntm = t1; }
    if (t0 < r.t_max) { if (nref != PB_DONE) PB_QPUSH(); nref = r0; ntm = t0; }
#undef PB_QPUSH
    if (nref != PB_DONE) r.cur = nref;
    else PB_TRAV_POP(r, stack);
}
// Every primitive of leaf `first_slot`, in order (bvh.rs:730-736).  Returns true when an any-hit ray is finished.
template <bool ANY>
PB_D bool quad_leaf_run(const DevScene& s, TravRay& r, uint32_t first_slot) {
    uint32_t slot = first_slot;
    uint32_t fl;
    do {
        const float4* tp = s.tris + 3ull * slot;
        float4 v0 = __ldg(tp), v1 = __ldg(tp + 1), v2 = __ldg(tp + 2);
        fl = __float_as_uint(v1.w);
        float t, b0, b1, b2;
        bool h;
        if (fl & PB_TRI_SPHERE) {
            h = sphere_test(s.spheres + __float_as_uint(v2.w), r.o, r.d, r.t_max, &t);
            b0 = b1 = b2 = 0.0f;
        } else {
            f3 p0(v0.x, v0.y, v0.z), p1(v1.x, v1.y, v1.z), p2(v2.x, v2.y, v2.z);
            h = triangle_test<!ANY>(r.o, r.d, r.t_max, p0, p1, p2, r.kx, r.ky, r.kz, r.Sx, r.Sy, r.Sz, &t, &b0, &b1, &b2);
            if (!ANY && h) {
                float2 uv0, uv1, uv2;
                fetch_uv(s, fl, __float_as_uint(v2.w), &uv0, &uv1, &uv2, slot);
                if (triangle_bogus(p0, p1, p2, uv0, uv1, uv2)) h = false;
            }
        }
        if (h) {
            r.found = true;
            r.hit.slot = slot; r.hit.t = t; r.hit.b0 = b0; r.hit.b1 = b1; r.hit.b2 = b2;
            if (ANY) return true;
            r.t_max = t;  // primitive.rs:137
        }
        ++slot;
    } while (!(fl & PB_TRI_LAST));
    return false;
}

// Per-lane form (any subset of a warp may call it: the (0,2) megakernel, the one-ray `traverse`): while-while.
template <bool ANY, typename STK>
PB_D void trav_run_quad(const DevScene& s, TravRay& r, STK stack, int yield_below, int interior_min) {
    while (r.cur != PB_DONE) {
        while (!(r.cur & PB_LEAF_BIT)) {
            quad_step<ANY>(s, r, stack);
            if (interior_min > 0 && __popc(__activemask()) < interior_min) break;
        }
        if (r.cur == PB_DONE) break;
        if (r.cur & PB_LEAF_BIT) {
            if (quad_leaf_run<ANY>(s, r, r.cur & ~PB_LEAF_BIT)) { r.cur = PB_DONE; r.sp = 0; break; }
            PB_TRAV_POP(r, stack);
        }
        if (yield_below > 0 && __popc(__activemask()) < yield_below) break;
    }
}

// PACKET form: ALL 32 lanes call it together and share ONE depth-first walk over the union of the nodes their rays need, so every
// lane is on the same node or leaf at every step and each node / leaf fetch is one broadcast load.  Precondition: every lane that
// has a ray (r.cur != PB_DONE after trav_init) has no zero direction component and the octant `negmask` (trace_queue_packet checks
// it).  The stack is the lanes' own stack at a warp-uniform depth: every lane writes the entry's (warp-uniform) node reference with
// ITS tmin for that slot, or +inf when it does not pass the slot, and a pop's lane mask is the ballot of `tmin < t_max` -- the
// per-lane walk's own pop test.
// Exactness: quad_slots orders the slots by the shared octant, so each lane meets the nodes it passes in the order the per-lane
// walk would (depth-first, near slot first), and a node's mask only holds lanes that passed it.  A slot a lane passes but the warp
// does not visit first waits on the stack behind slots that lane failed; the lane is idle in their sub-trees, so its t_max has not
// changed when the slot is popped and the pop's re-check passes, as the direct visit would have.  Each lane thus runs the same box
// and primitive tests, in the same order, against the same t_max as alone: same tie-breaks, bit-identical hits.
template <bool ANY, typename STK>
PB_D void trav_run_packet(const DevScene& s, TravRay& r, STK stack, uint32_t negmask) {
    const unsigned FULL = 0xffffffffu, lane_bit = 1u << (threadIdx.x & 31u);
    uint32_t mask = __ballot_sync(FULL, r.cur != PB_DONE);  // lanes whose ray passed the root box
    uint32_t cur = mask ? s.root_ref : PB_DONE;
    int sp = 0;  // warp-uniform
#define PB_PACKET_POP()                                                              \
    do {                                                                             \
        cur = PB_DONE;                                                               \
        while (sp > 0) {                                                             \
            --sp;                                                                    \
            const uint2 e__ = stack.get(sp);                                         \
            mask = __ballot_sync(FULL, __uint_as_float(e__.y) < r.t_max);            \
            if (mask) { cur = e__.x; break; }                                        \
        }                                                                            \
    } while (0)
    while (cur != PB_DONE) {
        while (!(cur & PB_LEAF_BIT)) {
            const bool live = mask & lane_bit;
            float t[4];
            uint32_t ref[4];
            quad_slots<ANY>(s, r, cur, negmask, t, ref);
            // the first slot any lane passes is visited now; the others wait on the stack, nearest on top
            uint32_t nref = PB_DONE, nmask = 0;
            float ntm = PB_INF;
#pragma unroll
            for (int k = 3; k >= 0; --k) {
                const bool p = live && t[k] < r.t_max;
                const uint32_t m = __ballot_sync(FULL, p);
                if (m) {
                    if (nref != PB_DONE) { stack.put(sp, make_uint2(nref, __float_as_uint(ntm))); ++sp; }
                    nref = ref[k]; nmask = m; ntm = p ? t[k] : PB_INF;
                }
            }
            cur = nref; mask = nmask;
            if (cur == PB_DONE) PB_PACKET_POP();
        }
        if (cur == PB_DONE) break;
        // an any-hit lane that found an occluder is finished: t_max = -inf fails every later pop
        if ((mask & lane_bit) && quad_leaf_run<ANY>(s, r, cur & ~PB_LEAF_BIT)) r.t_max = -PB_INF;
        PB_PACKET_POP();
    }
#undef PB_PACKET_POP
    r.cur = PB_DONE; r.sp = 0;
}

// INST: the scene contains TransformedPrimitives.  Scenes without instancing run kernels compiled with INST = false, which
// contain no trace of the instance path (measured on S3: the mere presence of the out-of-line call in the leaf loop costs 20%).
template <bool ANY, bool INST, typename STK>
PB_D void trav_run(const DevScene& s, TravRay& r, STK stack, int yield_below, int interior_min = 0) {
    // with instances the ray changes along the way, so the quad walk cannot be chosen once per ray: INST kernels choose it per
    // node visit (trav_run_impl)
    if (INST || r.nan_possible) trav_run_impl<ANY, INST>(s, r, stack, yield_below, interior_min);
    else trav_run_quad<ANY>(s, r, stack, yield_below, interior_min);
}

// Closest-hit (ANY=false) or any-hit (ANY=true) traversal of one ray, run to completion.
template <bool ANY, bool INST = false>
PB_D bool traverse(const DevScene& s, f3 o, f3 d, float t_max, RayHit* hit) {
    uint2 stack_mem[PB_STACK_SIZE(INST)];
    LocalStack stack{stack_mem};
    TravRay r;
    trav_init(s, r, o, d, t_max);
    trav_run<ANY, INST>(s, r, stack, 0);
    *hit = r.hit;
    return r.found;
}

// Variant kept for A/B measurements: single loop with leaf / interior / pop branches ("if-if").
template <bool ANY>
PB_D bool traverse_ifif(const DevScene& s, f3 o, f3 d, float t_max, RayHit* hit) {
    hit->slot = PBRT_B200_NO_HIT; hit->inst = PBRT_B200_NO_HIT;
    hit->t = t_max;
    if (s.root_ref == PB_REF_NONE) return false;
    const f3 inv(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
    const bool ngx = inv.x < 0.0f, ngy = inv.y < 0.0f, ngz = inv.z < 0.0f;
    // ray-constant part of the watertight test (triangle.rs:151-165)
    f3 ad = vabs(d);
    const int kz = (ad.x > ad.y) ? ((ad.x > ad.z) ? 0 : 2) : ((ad.y > ad.z) ? 1 : 2);
    const int kx = (kz + 1 == 3) ? 0 : kz + 1;
    const int ky = (kx + 1 == 3) ? 0 : kx + 1;
    const float dpx = comp(d, kx), dpy = comp(d, ky), dpz = comp(d, kz);
    const float Sx = -dpx / dpz, Sy = -dpy / dpz, Sz = 1.0f / dpz;

    uint2 stack[PB_STACK_DEPTH];
    int sp = 0;
    bool found = false;
    uint32_t cur;
    {
        float tmin;
        const float* rb = s.root_box;
        bool ok = slab_test(ngx ? rb[3] : rb[0], ngy ? rb[4] : rb[1], ngz ? rb[5] : rb[2], ngx ? rb[0] : rb[3], ngy ? rb[1] : rb[4],
                            ngz ? rb[2] : rb[5], o, inv, &tmin);
        if (!(ok && tmin < t_max)) return false;
        cur = s.root_ref;
    }
    for (;;) {
        if (cur & PB_LEAF_BIT) {
            uint32_t slot = cur & ~PB_LEAF_BIT;
            uint32_t fl;
            do {
                const float4* tp = s.tris + 3ull * slot;
                float4 v0 = __ldg(tp), v1 = __ldg(tp + 1), v2 = __ldg(tp + 2);
                fl = __float_as_uint(v1.w);
                float t, b0, b1, b2;
                bool h;
                if (fl & PB_TRI_SPHERE) {
                    h = sphere_test(s.spheres + __float_as_uint(v2.w), o, d, t_max, &t);
                    b0 = b1 = b2 = 0.0f;
                } else {
                    f3 p0(v0.x, v0.y, v0.z), p1(v1.x, v1.y, v1.z), p2(v2.x, v2.y, v2.z);
                    h = triangle_test<!ANY>(o, d, t_max, p0, p1, p2, kx, ky, kz, Sx, Sy, Sz, &t, &b0, &b1, &b2);
                    if (!ANY && h) {
                        float2 uv0, uv1, uv2;
                        fetch_uv(s, fl, __float_as_uint(v2.w), &uv0, &uv1, &uv2, slot);
                        if (triangle_bogus(p0, p1, p2, uv0, uv1, uv2)) h = false;
                    }
                }
                if (h) {
                    if (ANY) { hit->slot = slot; hit->t = t; return true; }
                    t_max = t;  // primitive.rs:137
                    hit->slot = slot; hit->t = t; hit->b0 = b0; hit->b1 = b1; hit->b2 = b2;
                    found = true;
                }
                ++slot;
            } while (!(fl & PB_TRI_LAST));
        } else {
            const float4* np = s.nodes + 4ull * cur;
            float4 q0 = __ldg(np), q1 = __ldg(np + 1), q2 = __ldg(np + 2), q3 = __ldg(np + 3);
            uint32_t ref0 = __float_as_uint(q3.x), ref1 = __float_as_uint(q3.y), axis = __float_as_uint(q3.z);
            float tmin0, tmin1;
            bool ok0 = slab_test(ngx ? q0.w : q0.x, ngy ? q1.x : q0.y, ngz ? q1.y : q0.z, ngx ? q0.x : q0.w, ngy ? q0.y : q1.x,
                                 ngz ? q0.z : q1.y, o, inv, &tmin0);
            bool ok1 = slab_test(ngx ? q2.y : q1.z, ngy ? q2.z : q1.w, ngz ? q2.w : q2.x, ngx ? q1.z : q2.y, ngy ? q1.w : q2.z,
                                 ngz ? q2.x : q2.w, o, inv, &tmin1);
            // near child = second child when the ray is negative along the split axis (bvh.rs:743-751)
            bool second_first = (axis == 0) ? ngx : ((axis == 1) ? ngy : ngz);
            uint32_t nref = second_first ? ref1 : ref0, fref = second_first ? ref0 : ref1;
            float ntmin = second_first ? tmin1 : tmin0, ftmin = second_first ? tmin0 : tmin1;
            bool nok = second_first ? ok1 : ok0, fok = second_first ? ok0 : ok1;
            bool nhit = nok && (ntmin < t_max);
            if (ANY) fok = fok && (ftmin < t_max);  // t_max never changes for any-hit rays
            if (nhit) {
                if (fok) { stack[sp] = make_uint2(fref, __float_as_uint(ftmin)); ++sp; }
                cur = nref;
                continue;
            }
            if (fok && (ftmin < t_max)) { cur = fref; continue; }
        }
        // pop: the reference tests the popped node's box against the *current* t_max
        for (;;) {
            if (sp == 0) return found;
            --sp;
            uint2 e = stack[sp];
            if (__uint_as_float(e.y) < t_max) { cur = e.x; break; }
        }
    }
}


// Persistent-thread ray queue: every warp pulls ray indices [0, n) from a global counter in
// chunks and refills lanes whose ray has finished as soon as fewer than PB_REFILL_BELOW lanes
// are still traversing.  Job provides
//     bool load(uint32_t idx, f3* o, f3* d, float* t_max)
//     void store(uint32_t idx, const TravRay& r)
#define PB_FETCH_CHUNK 32   /* tools/trace_ab.py: larger chunks cost coherent rays 25-45% */
// Refill latency.  A warp's refill is one atomicAdd on a single global counter -- ~1 M of them per 33 M-ray launch, one every ~5 ns
// against the ~4 ns the L2 slice needs per same-address atomic (profiles/r02_ncu_regen.md) -- whose round trip the whole warp waits
// for.  Two ways around it were tried and BOTH measured slower on B200 (hits bit-identical; gpurun_out/r2j_ab.log, r2k_ab.log):
//   * lane 0 reserves the NEXT chunk while the current one is traversed (one chunk of look-ahead per warp):
//     S3 step 35.8 -> 37.2 ms, camera batch 4424 -> 4244 Mrays/s;
//   * reserving 4 / 8 chunks per global atomic and parking the extra ones in shared memory for the sibling warps: 35.8 -> 37.6 / 40.1 ms.
// Both widen the band of the ray queue that is in flight at any moment; the queue is in path order (neighbouring pixels, then
// neighbouring hit points), and the traversal's cache hit rates live off that locality more than they suffer from the refill wait.
#define PB_REFILL_BELOW 24
#define PB_INTERIOR_MIN 16
struct TraceTune { int refill_below; int chunk; int interior_min; };
// The shared levels of the hybrid stack: one array per kernel, which trace_queue and trace_queue_packet both use.
template <int SH>
PB_D uint2* trace_stack_shared() {
    __shared__ uint2 stack_shared[SH > 0 ? SH : 1][PB_TRACE_BLOCK];
    return &stack_shared[0][threadIdx.x];
}
template <bool ANY, bool INST, int SH = 0, typename Job>
PB_D void trace_queue(const DevScene& s, Job& job, uint32_t n, uint32_t* fetch_counter, TraceTune tune = TraceTune{PB_REFILL_BELOW, PB_FETCH_CHUNK, PB_INTERIOR_MIN}) {
    uint2 stack_mem[PB_STACK_SIZE(INST)];
    HybridStack<SH, PB_TRACE_BLOCK> stack{trace_stack_shared<SH>(), stack_mem};  // SH == 0: every level in the local array
    TravRay r;
    r.cur = PB_DONE; r.sp = 0; r.found = false;
    uint32_t ray_idx = 0xffffffffu;
    uint32_t pool_next = 0, pool_end = 0;  // warp-uniform
    bool exhausted = false;                // warp-uniform
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    for (;;) {
        __syncwarp();
        if (trav_done(r) && ray_idx != 0xffffffffu) { job.store(ray_idx, r); ray_idx = 0xffffffffu; }
        __syncwarp();
        unsigned need = __ballot_sync(0xffffffffu, trav_done(r));
        while (need && !exhausted) {
            if (pool_next == pool_end) {
                uint32_t b = 0;
                if (lane == 0) b = atomicAdd(fetch_counter, (uint32_t)tune.chunk);
                b = __shfl_sync(0xffffffffu, b, 0);
                if (b >= n) { exhausted = true; break; }
                pool_next = b; pool_end = min(b + (uint32_t)tune.chunk, n);
            }
            uint32_t avail = pool_end - pool_next;
            bool mine = (need >> lane) & 1u;
            uint32_t rank = __popc(need & lt_mask);
            bool take = mine && rank < avail;
            if (take) {
                ray_idx = pool_next + rank;
                f3 o, d; float t_max = 0.0f;
                if (job.load(ray_idx, &o, &d, &t_max)) trav_init(s, r, o, d, t_max);
                else { r.cur = PB_DONE; r.sp = 0; r.found = false; r.hit.slot = PBRT_B200_NO_HIT; r.hit.t = t_max; r.hit.inst = PBRT_B200_NO_HIT; }
            }
            unsigned took = __ballot_sync(0xffffffffu, take);
            pool_next += __popc(took);
            need &= ~took;
        }
        if (__all_sync(0xffffffffu, ray_idx == 0xffffffffu)) break;
        trav_run<ANY, INST>(s, r, stack, exhausted ? 0 : tune.refill_below, tune.interior_min);
    }
}

// Packet mode of the ray queue (scenes without instances), for queues whose aligned runs of 32 entries are coherent rays: camera
// rays in item order (32 samples of one pixel) and the shadow rays cast from their hits.  A warp takes a whole aligned chunk of 32
// entries -- lane-wise refills would mix pixels -- and walks it as one packet (trav_run_packet) when all its rays share an octant
// and have no zero direction component; any other chunk runs the per-lane walk to completion.
template <bool ANY, int SH = 0, typename Job>
PB_D void trace_queue_packet(const DevScene& s, Job& job, uint32_t n, uint32_t* fetch_counter) {
    uint2 stack_mem[PB_STACK_SIZE(false)];
    HybridStack<SH, PB_TRACE_BLOCK> stack{trace_stack_shared<SH>(), stack_mem};
    const unsigned FULL = 0xffffffffu, lane = threadIdx.x & 31u;
    for (;;) {
        uint32_t b = 0;
        if (lane == 0) b = atomicAdd(fetch_counter, 32u);
        b = __shfl_sync(FULL, b, 0);
        if (b >= n) break;
        const uint32_t idx = b + lane;
        TravRay r;
        r.cur = PB_DONE; r.sp = 0; r.found = false;
        r.hit.slot = PBRT_B200_NO_HIT; r.hit.inst = PBRT_B200_NO_HIT;
        f3 o, d; float t_max = 0.0f;
        if (idx < n) {
            if (job.load(idx, &o, &d, &t_max)) trav_init(s, r, o, d, t_max);
            else r.hit.t = t_max;
        }
        // octant of the chunk: the first lane that traverses; 8 = a zero direction component, never shared
        const bool trav = r.cur != PB_DONE;
        const uint32_t oct = trav ? (r.nan_possible ? 8u : r.negmask) : 0u;
        const uint32_t first = __ffs(__ballot_sync(FULL, trav));
        const uint32_t shared_oct = __shfl_sync(FULL, oct, first ? first - 1 : 0);
        if (__all_sync(FULL, !trav || oct == shared_oct) && shared_oct != 8u) trav_run_packet<ANY>(s, r, stack, shared_oct);
        else if (trav) trav_run<ANY, false>(s, r, stack, 0);
        if (idx < n) job.store(idx, r);
    }
}

}  // namespace pb
