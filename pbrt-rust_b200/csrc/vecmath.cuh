// Device-side scalar/vector helpers.  This translation unit family is compiled with
// --fmad=false: every f32 op is separately rounded, matching Rust (SURVEY.md App. A).
// Reference arithmetic cited per function (paths relative to pbrt-rust/src).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pb {

#define PB_HD __host__ __device__ __forceinline__
#define PB_D __device__ __forceinline__

// core/pbrt.rs:23-34
#define PB_PI 3.14159265358979323846f
#define PB_PI_OVER2 1.57079632679489661923f
#define PB_PI_OVER4 0.78539816339744830961f
#define PB_INV_PI 0.31830988618379067154f
#define PB_INV_4PI 0.07957747154594766788f
#define PB_FLT_MAX 3.402823466e+38f
#define PB_SHADOW_EPSILON 0.0001f
#define PB_MACHINE_EPSILON 5.9604644775390625e-8f /* f32::EPSILON * 0.5 = 2^-24 */
#define PB_ONE_MINUS_EPSILON 0.99999994f          /* 0x1.fffffep-1, core/rng.rs:4 */
#define PB_INF __int_as_float(0x7f800000)

// core/pbrt.rs:206-208  gamma(n) = n*eps / (1 - n*eps)
PB_HD float gamma_n(int n) { return ((float)n * PB_MACHINE_EPSILON) / (1.0f - (float)n * PB_MACHINE_EPSILON); }

// core/pbrt.rs:80-112
PB_D float next_up(float v) {
    if (isinf(v) && v > 0.0f) return v;
    if (v == -0.0f) v = 0.0f;
    uint32_t u = __float_as_uint(v);
    u = (v >= 0.0f) ? u + 1 : u - 1;
    return __uint_as_float(u);
}
PB_D float next_down(float v) {
    if (isinf(v) && v < 0.0f) return v;
    if (v == 0.0f) v = -0.0f;
    uint32_t u = __float_as_uint(v);
    u = (v > 0.0f) ? u - 1 : u + 1;
    return __uint_as_float(u);
}

// compare-based clamp, core/pbrt.rs:172-182
PB_D float clampf(float v, float lo, float hi) { return v < lo ? lo : (v > hi ? hi : v); }

struct f3 {
    float x, y, z;
    PB_HD f3() {}
    PB_HD f3(float a, float b, float c) : x(a), y(b), z(c) {}
};
PB_HD f3 operator+(f3 a, f3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
PB_HD f3 operator-(f3 a, f3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
PB_HD f3 operator-(f3 a) { return f3(-a.x, -a.y, -a.z); }
PB_HD f3 operator*(f3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
// geometry/vector.rs:486-495: v / s == v * (1/s)
PB_D f3 vdiv(f3 a, float s) { float d = 1.0f / s; return f3(a.x * d, a.y * d, a.z * d); }
PB_HD float dot(f3 a, f3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
PB_D float absdot(f3 a, f3 b) { return fabsf(dot(a, b)); }
PB_HD float len2(f3 a) { return a.x * a.x + a.y * a.y + a.z * a.z; }
PB_D float len(f3 a) { return sqrtf(len2(a)); }
PB_D f3 normalize(f3 a) { return vdiv(a, len(a)); }
PB_D f3 vabs(f3 a) { return f3(fabsf(a.x), fabsf(a.y), fabsf(a.z)); }
// geometry/vector.rs:339-353: f64 products, then narrowed
#ifdef PB_TU_SHADE
// shade.cu (tolerance-parity shading, see there): plain f32
PB_D f3 cross(f3 a, f3 b) { return f3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
#else
PB_D f3 cross(f3 a, f3 b) {
    double ax = a.x, ay = a.y, az = a.z, bx = b.x, by = b.y, bz = b.z;
    return f3((float)(__dsub_rn(__dmul_rn(ay, bz), __dmul_rn(az, by))), (float)(__dsub_rn(__dmul_rn(az, bx), __dmul_rn(ax, bz))),
              (float)(__dsub_rn(__dmul_rn(ax, by), __dmul_rn(ay, bx))));
}
#endif
PB_D float maxcomp(f3 a) { return fmaxf(a.x, fmaxf(a.y, a.z)); }
PB_D f3 face_forward(f3 n, f3 v) { return dot(n, v) < 0.0f ? -n : n; }
// c ? a : b as ONE select instruction.  The ternary form of the axis permutations below was compiled to divergent branches
// (BSSY / BRA / BSYNC around predicated moves): ncu attributed 20 % of k_trace_closest's warp instructions to comp()
// (profiles/r02_trace_comp.md); selp keeps the triangle test straight-line.
PB_D float selp(float a, float b, bool c) {
    float r;
    asm("{\n\t.reg .pred p;\n\tsetp.ne.s32 p, %3, 0;\n\tselp.f32 %0, %1, %2, p;\n\t}" : "=f"(r) : "f"(a), "f"(b), "r"((int)c));
    return r;
}
PB_D float comp(f3 a, int i) { return selp(a.x, selp(a.y, a.z, i == 1), i == 0); }
// Triangle::intersect's permutation (triangle.rs:151-160): kz = largest |d| component, kx = kz + 1, ky = kx + 1 (mod 3), i.e. a
// rotation of (x, y, z) chosen by kz alone: kz = 2 -> (x, y, z), kz = 0 -> (y, z, x), kz = 1 -> (z, x, y)
PB_D f3 permute_kz(f3 v, int kz) {
    const bool k0 = kz == 0, k1 = kz == 1;
    return f3(selp(v.y, selp(v.z, v.x, k1), k0), selp(v.z, selp(v.x, v.y, k1), k0), selp(v.x, selp(v.y, v.z, k1), k0));
}
// geometry/vector.rs:589-600
PB_D void coordinate_system(f3 v1, f3* v2, f3* v3) {
    if (fabsf(v1.x) > fabsf(v1.y)) *v2 = vdiv(f3(-v1.z, 0.0f, v1.x), sqrtf(v1.x * v1.x + v1.z * v1.z));
    else *v2 = vdiv(f3(0.0f, v1.z, -v1.y), sqrtf(v1.y * v1.y + v1.z * v1.z));
    *v3 = cross(v1, *v2);
}
// geometry/geometry.rs:6-24
PB_D f3 offset_ray_origin(f3 p, f3 p_error, f3 n, f3 w) {
    float d = dot(vabs(n), p_error);
    f3 off = n * d;
    if (dot(w, n) < 0.0f) off = -off;
    f3 po = p + off;
    if (off.x > 0.0f) po.x = next_up(po.x); else if (off.x < 0.0f) po.x = next_down(po.x);
    if (off.y > 0.0f) po.y = next_up(po.y); else if (off.y < 0.0f) po.y = next_down(po.y);
    if (off.z > 0.0f) po.z = next_up(po.z); else if (off.z < 0.0f) po.z = next_down(po.z);
    return po;
}

// Row-major 4x4 in global memory (core/transform.rs)
struct Mat4 { float m[16]; };
// transform.rs:413-431
PB_D f3 xf_point(const float* M, f3 p) {
    float xp = p.x * M[0] + p.y * M[1] + p.z * M[2] + M[3];
    float yp = p.x * M[4] + p.y * M[5] + p.z * M[6] + M[7];
    float zp = p.x * M[8] + p.y * M[9] + p.z * M[10] + M[11];
    float wp = p.x * M[12] + p.y * M[13] + p.z * M[14] + M[15];
    if (wp == 1.0f) return f3(xp, yp, zp);
    return vdiv(f3(xp, yp, zp), wp);
}
// transform.rs:433-456
PB_D f3 xf_point_err(const float* M, f3 p, f3* err) {
    float xs = fabsf(p.x * M[0]) + fabsf(p.y * M[1]) + fabsf(p.z * M[2]) + fabsf(M[3]);
    float ys = fabsf(p.x * M[4]) + fabsf(p.y * M[5]) + fabsf(p.z * M[6]) + fabsf(M[7]);
    float zs = fabsf(p.x * M[8]) + fabsf(p.y * M[9]) + fabsf(p.z * M[10]) + fabsf(M[11]);
    *err = f3(xs, ys, zs) * gamma_n(3);
    return xf_point(M, p);
}
// transform.rs:458-494
PB_D f3 xf_point_abs_err(const float* M, f3 p, f3 pe, f3* ae) {
    float g = gamma_n(3);
    ae->x = (g + 1.0f) * (fabsf(M[0]) * pe.x + fabsf(M[1]) * pe.y + fabsf(M[2]) * pe.z) +
            g * (fabsf(M[0] * p.x) + fabsf(M[1] * p.y) + fabsf(M[2] * p.z) + fabsf(M[3]));
    ae->y = (g + 1.0f) * (fabsf(M[4]) * pe.x + fabsf(M[5]) * pe.y + fabsf(M[6]) * pe.z) +
            g * (fabsf(M[4] * p.x) + fabsf(M[5] * p.y) + fabsf(M[6] * p.z) + fabsf(M[7]));
    ae->z = (g + 1.0f) * (fabsf(M[8]) * pe.x + fabsf(M[9]) * pe.y + fabsf(M[10]) * pe.z) +
            g * (fabsf(M[8] * p.x) + fabsf(M[9] * p.y) + fabsf(M[10] * p.z) + fabsf(M[11]));
    return xf_point(M, p);
}
// transform.rs:496-508
PB_D f3 xf_vector(const float* M, f3 v) {
    return f3(v.x * M[0] + v.y * M[1] + v.z * M[2], v.x * M[4] + v.y * M[5] + v.z * M[6], v.x * M[8] + v.y * M[9] + v.z * M[10]);
}
// transform.rs:510-527
PB_D f3 xf_vector_err(const float* M, f3 v, f3* ae) {
    float g = gamma_n(3);
    ae->x = g * (fabsf(v.x * M[0]) + fabsf(v.y * M[1]) + fabsf(v.z * M[2]));
    ae->y = g * (fabsf(v.x * M[4]) + fabsf(v.y * M[5]) + fabsf(v.z * M[6]));
    ae->z = g * (fabsf(v.x * M[8]) + fabsf(v.y * M[9]) + fabsf(v.z * M[10]));
    return xf_vector(M, v);
}
// transform.rs:529-541 (pass the INVERSE matrix)
PB_D f3 xf_normal(const float* Mi, f3 n) {
    return f3(n.x * Mi[0] + n.y * Mi[4] + n.z * Mi[8], n.x * Mi[1] + n.y * Mi[5] + n.z * Mi[9], n.x * Mi[2] + n.y * Mi[6] + n.z * Mi[10]);
}

}  // namespace pb
