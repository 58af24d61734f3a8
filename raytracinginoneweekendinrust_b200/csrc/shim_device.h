// shim_device.h — the hot path's arithmetic: intersection, traversal, hit reconstruction,
// textures and scatter.  Every function is __host__ __device__ so that tests/hostsim can
// run the very same code on the CPU against the oracle (a test harness, never a product
// path: the library itself only ever launches the sm_100a kernels in shim_kernels.cu).
//
// Arithmetic policy: this file is compiled with -fmad=false (nvcc) / -ffp-contract=off
// (g++).  Primitive tests and shading follow the reference's IEEE f32/f64 operation order
// (glam 0.22 scalar Vec3) so that they are bit-identical to rustc's output wherever only
// + - * / sqrt are involved; BVH box tests are free to differ because the result of a
// traversal is topology-independent (SURVEY.md §2.2 "BVH traversal").
#pragma once
#include <math.h>
#include "shim_types.h"

namespace shim {

// ---------------------------------------------------------------------------- vec3
SHIM_HD f3 mk3(float x, float y, float z) { f3 r; r.x = x; r.y = y; r.z = z; return r; }
SHIM_HD f3 operator+(f3 a, f3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
SHIM_HD f3 operator-(f3 a, f3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
SHIM_HD f3 operator-(f3 a) { return mk3(-a.x, -a.y, -a.z); }
SHIM_HD f3 operator*(f3 a, f3 b) { return mk3(a.x * b.x, a.y * b.y, a.z * b.z); }
SHIM_HD f3 operator*(f3 a, float s) { return mk3(a.x * s, a.y * s, a.z * s); }
SHIM_HD f3 operator*(float s, f3 a) { return mk3(s * a.x, s * a.y, s * a.z); }
SHIM_HD f3 operator/(f3 a, float s) { return mk3(a.x / s, a.y / s, a.z / s); }
SHIM_HD float dot3(f3 a, f3 b) { return (a.x * b.x) + (a.y * b.y) + (a.z * b.z); }
SHIM_HD f3 cross3(f3 a, f3 b) { return mk3(a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y); }
SHIM_HD float len3(f3 a) { return sqrtf(dot3(a, a)); }
SHIM_HD f3 normalize3(f3 a) { return a * (1.0f / len3(a)); }
SHIM_HD float comp(f3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }
SHIM_HD f3 xyz(f4 v) { return mk3(v.x, v.y, v.z); }
SHIM_HD bool signbit_f(float v) { return f2i(v) < 0; }

#define SHIM_F32_EPS 1.1920929e-07f
#define SHIM_PI 3.14159265358979323846f
#if defined(__CUDA_ARCH__)
#define SHIM_INF __int_as_float(0x7f800000)
#else
#define SHIM_INF INFINITY
#endif

struct Ray { f3 o, d; float time; };
SHIM_HD f3 ray_at(const Ray& r, float t) { return r.o + t * r.d; }
SHIM_HD bool ray_has_nan(const Ray& r) {
    return (r.o.x != r.o.x) | (r.o.y != r.o.y) | (r.o.z != r.o.z) | (r.d.x != r.d.x) | (r.d.y != r.d.y) | (r.d.z != r.d.z);
}

// ---------------------------------------------------------------------------- Philox4x32-10
SHIM_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
#ifndef SHIM_PHILOX_ROUNDS
#define SHIM_PHILOX_ROUNDS 10   // experiment builds only: the stream is defined with 10 rounds (oracle, KATs)
#endif
struct Rng {
    uint32_t pixel, sample, dim, j, k0, k1;
    uint32_t b0, b1, b2, b3;
};
SHIM_HD void rng_init(Rng& r, uint32_t pixel, uint32_t sample, uint64_t seed) {
    r.pixel = pixel; r.sample = sample; r.dim = 0; r.j = 0;
    r.k0 = (uint32_t)seed; r.k1 = (uint32_t)(seed >> 32);
    r.b0 = r.b1 = r.b2 = r.b3 = 0;
}
SHIM_HD void rng_key(Rng& r, uint32_t bounce, uint32_t stage) { r.dim = bounce * 4u + stage; r.j = 0; }
SHIM_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t& o0, uint32_t& o1,
                           uint32_t& o2, uint32_t& o3) {
#pragma unroll
    for (int i = 0; i < SHIM_PHILOX_ROUNDS; ++i) {
        uint32_t h0 = mulhi32(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        uint32_t h1 = mulhi32(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0; c1 = l1; c2 = h0 ^ c3 ^ k1; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    o0 = c0; o1 = c1; o2 = c2; o3 = c3;
}
// counter = (pixel, sample, bounce * 4 + stage, block index), key = seed
SHIM_HD void rng_refill(Rng& r) { philox4x32_10(r.pixel, r.sample, r.dim, r.j >> 2, r.k0, r.k1, r.b0, r.b1, r.b2, r.b3); }
SHIM_HD uint32_t rng_u32(Rng& r) {
    uint32_t lane = r.j & 3u;
    if (lane == 0) rng_refill(r);
    r.j++;
    return lane == 0 ? r.b0 : (lane == 1 ? r.b1 : (lane == 2 ? r.b2 : r.b3));
}
// rand 0.8.5: random::<f32>() keeps 24 bits; gen_range keeps 23 and maps u*(hi-lo)+lo
SHIM_HD float rng_uniform01(Rng& r) { return (float)(rng_u32(r) >> 8) * (1.0f / 16777216.0f); }
SHIM_HD float rng_range(Rng& r, float lo, float hi) {
    float s = hi - lo;
    return (float)(rng_u32(r) >> 9) * (1.0f / 8388608.0f) * s + lo;
}
SHIM_HD float rng_word_pm1(uint32_t w) { return (float)(w >> 9) * (1.0f / 8388608.0f) * 2.0f + -1.0f; }  // rng_range(r, -1, 1) on word w
// utils.rs:9-17
SHIM_HD f3 random_in_unit_disk(Rng& r) {
    for (;;) {
        float a = rng_range(r, -1.0f, 1.0f);
        float b = rng_range(r, -1.0f, 1.0f);
        f3 p = mk3(a, b, 0.0f);
        if (dot3(p, p) < 1.0f) return p;
    }
}
// materials/utils.rs:6-19
SHIM_HD f3 random_in_unit_sphere_stream(Rng& r) {
    for (;;) {
        float a = rng_range(r, -1.0f, 1.0f);
        float b = rng_range(r, -1.0f, 1.0f);
        float c = rng_range(r, -1.0f, 1.0f);
        f3 p = mk3(a, b, c);
        if (dot3(p, p) < 1.0f) return p;
    }
}
// The same draws when the stream is at its start (always the case in scatter: the sphere sample is the first draw of
// its stage).  Try k is words 3k..3k+2 of the stream, so three Philox blocks hold exactly four tries; written out,
// the word-to-try assignment is static and the per-draw refill branch and word select of rng_u32 disappear
// (they were a quarter of wf_shade's instructions).  Leaves the stream where the generic loop would.
SHIM_HD f3 random_in_unit_sphere(Rng& r) {
    if (r.j != 0) return random_in_unit_sphere_stream(r);
    for (uint32_t blk = 0;; blk += 3) {
        uint32_t a0, a1, a2, a3, b0, b1, b2, b3, c0, c1, c2, c3;
        philox4x32_10(r.pixel, r.sample, r.dim, blk, r.k0, r.k1, a0, a1, a2, a3);
        f3 p = mk3(rng_word_pm1(a0), rng_word_pm1(a1), rng_word_pm1(a2));
        if (dot3(p, p) < 1.0f) { r.j = 4u * blk + 3u; r.b0 = a0; r.b1 = a1; r.b2 = a2; r.b3 = a3; return p; }
        philox4x32_10(r.pixel, r.sample, r.dim, blk + 1u, r.k0, r.k1, b0, b1, b2, b3);
        p = mk3(rng_word_pm1(a3), rng_word_pm1(b0), rng_word_pm1(b1));
        if (dot3(p, p) < 1.0f) { r.j = 4u * blk + 6u; r.b0 = b0; r.b1 = b1; r.b2 = b2; r.b3 = b3; return p; }
        philox4x32_10(r.pixel, r.sample, r.dim, blk + 2u, r.k0, r.k1, c0, c1, c2, c3);
        p = mk3(rng_word_pm1(b2), rng_word_pm1(b3), rng_word_pm1(c0));
        if (dot3(p, p) < 1.0f) { r.j = 4u * blk + 9u; r.b0 = c0; r.b1 = c1; r.b2 = c2; r.b3 = c3; return p; }
        p = mk3(rng_word_pm1(c1), rng_word_pm1(c2), rng_word_pm1(c3));
        if (dot3(p, p) < 1.0f) { r.j = 4u * blk + 12u; r.b0 = c0; r.b1 = c1; r.b2 = c2; r.b3 = c3; return p; }
    }
}

// ---------------------------------------------------------------------------- camera.rs:96-106
SHIM_HD Ray camera_get_ray(const CameraPod& c, float s, float t, Rng& rng) {
    f3 rd = c.lens_radius * random_in_unit_disk(rng);
    f3 offset = c.u * rd.x + c.v * rd.y;
    float time = rng_range(rng, c.time0, c.time1);
    Ray r;
    r.o = c.origin + offset;
    r.d = c.llc + s * c.horizontal + t * c.vertical - c.origin - offset;
    r.time = time;
    return r;
}
// renderer.rs:141-143
// renderer.rs:141-143 + camera.rs:96-106 from a stream at its start (the camera stage's first draws), written out
// over Philox blocks like random_in_unit_sphere: words 0,1 jitter the pixel, disk try k is words 2+2k, 3+2k, the word
// after the accepted try is the shutter time.
SHIM_HD Ray camera_sample(const CameraPod& c, int x, int y, int width, int height, Rng& rng) {
    if (rng.j != 0) {
        float u = ((float)x + rng_uniform01(rng)) / (float)(width - 1);
        float v = ((float)y + rng_uniform01(rng)) / (float)(height - 1);
        return camera_get_ray(c, u, v, rng);
    }
    uint32_t w0, w1, w2, w3;
    philox4x32_10(rng.pixel, rng.sample, rng.dim, 0u, rng.k0, rng.k1, w0, w1, w2, w3);
    const float s = ((float)x + (float)(w0 >> 8) * (1.0f / 16777216.0f)) / (float)(width - 1);
    const float t = ((float)y + (float)(w1 >> 8) * (1.0f / 16777216.0f)) / (float)(height - 1);
    f3 p = mk3(rng_word_pm1(w2), rng_word_pm1(w3), 0.0f);
    bool accepted = dot3(p, p) < 1.0f;
    uint32_t time_word;
    for (uint32_t blk = 1;; ++blk) {
        philox4x32_10(rng.pixel, rng.sample, rng.dim, blk, rng.k0, rng.k1, w0, w1, w2, w3);
        if (accepted) { time_word = w0; rng.j = 4u * blk + 1u; break; }
        p = mk3(rng_word_pm1(w0), rng_word_pm1(w1), 0.0f);
        if (dot3(p, p) < 1.0f) { time_word = w2; rng.j = 4u * blk + 3u; break; }
        p = mk3(rng_word_pm1(w2), rng_word_pm1(w3), 0.0f);
        accepted = dot3(p, p) < 1.0f;
    }
    rng.b0 = w0; rng.b1 = w1; rng.b2 = w2; rng.b3 = w3;
    f3 rd = c.lens_radius * p;
    f3 offset = c.u * rd.x + c.v * rd.y;
    Ray r;
    r.o = c.origin + offset;
    r.d = c.llc + s * c.horizontal + t * c.vertical - c.origin - offset;
    r.time = (float)(time_word >> 9) * (1.0f / 8388608.0f) * (c.time1 - c.time0) + c.time0;   // rng_range(rng, time0, time1)
    return r;
}

// ---------------------------------------------------------------------------- object-space ray
struct RayCtx {
    Ray r;      // ray as the shape sees it (after Translate / RotateY, instance.rs)
    f3 inv_d;   // 1/d with |d| clamped away from 0 so that the products below stay finite
    f3 o_inv;   // -o * inv_d: a slab plane distance is one fma(plane, inv_d, o_inv)
    int soff[3]; // SNode walks: byte offset of the ray's {near_l, near_r, far_l, far_r} planes of axis k inside a node
    uint32_t qrot[3]; // QNode walks: rotation (0 / 16 bits) that brings the plane bytes of axis k into that order
};
SHIM_HD f3 rot_y(f3 v, float s, float c) { return mk3(c * v.x - s * v.z, v.y, s * v.x + c * v.z); }       // instance.rs:104-110
SHIM_HD f3 rot_y_back(f3 v, float s, float c) { return mk3(c * v.x + s * v.z, v.y, -s * v.x + c * v.z); } // instance.rs:125-134
SHIM_HD Ray object_ray(const DevObject& ob, const Ray& w) {
    Ray r = w;
    if (ob.flags & OBJ_TRANSLATE) r.o = r.o - mk3(ob.dx, ob.dy, ob.dz);
    if (ob.flags & OBJ_ROTATE) { r.o = rot_y(r.o, ob.sin_t, ob.cos_t); r.d = rot_y(r.d, ob.sin_t, ob.cos_t); }
    return r;
}
SHIM_HD float safe_rcp(float d) {
    // a zero component would make fma(plane, inf, -o*inf) NaN on BOTH planes of a slab the origin lies in
    // (and wrongly cull it); 1e-30 keeps every product finite and the interval (-huge, +huge) or empty
    float a = fabsf(d) < 1e-30f ? copysignf(1e-30f, d) : d;
    return 1.0f / a;
}
SHIM_HD void make_ctx(RayCtx& c, const Ray& r) {
    c.r = r;
    c.inv_d = mk3(safe_rcp(r.d.x), safe_rcp(r.d.y), safe_rcp(r.d.z));
    c.o_inv = mk3(-(r.o.x * c.inv_d.x), -(r.o.y * c.inv_d.y), -(r.o.z * c.inv_d.z));
    c.soff[0] = signbit_f(c.inv_d.x) ? 16 : 0;
    c.soff[1] = signbit_f(c.inv_d.y) ? 48 : 32;
    c.soff[2] = signbit_f(c.inv_d.z) ? 80 : 64;
    c.qrot[0] = signbit_f(c.inv_d.x) ? 16u : 0u;
    c.qrot[1] = signbit_f(c.inv_d.y) ? 16u : 0u;
    c.qrot[2] = signbit_f(c.inv_d.z) ? 16u : 0u;
}

struct TraceCounters { uint32_t nodes, prims, hrpp_tp, hrpp_fp, hrpp_none; };

// per-type table lookup with constant indices only, so a SceneView held in registers is never
// forced into local memory by a dynamic index
SHIM_HD const int* table_of(const int* const* t, int type) {
    return type == PT_SPHERE ? t[0] : (type == PT_MSPHERE ? t[1] : (type == PT_RECT ? t[2] : (type == PT_TRI ? t[3] : t[4])));
}

// ---------------------------------------------------------------------------- primitives
// geometry/sphere.rs:50-89 (f64 quadratic; accepts root == t_max)
SHIM_HD bool hit_sphere(const double* s, const Ray& r, float t_min, float t_max, float& t_out) {
    double dx = (double)r.d.x, dy = (double)r.d.y, dz = (double)r.d.z;
    double ocx = (double)r.o.x - s[0], ocy = (double)r.o.y - s[1], ocz = (double)r.o.z - s[2];
    double a = (dx * dx) + (dy * dy) + (dz * dz);
    double half_b = (ocx * dx) + (ocy * dy) + (ocz * dz);
    double cc = ((ocx * ocx) + (ocy * ocy) + (ocz * ocz)) - s[3];
    double disc = half_b * half_b - a * cc;
#if defined(__CUDA_ARCH__)
    if (__double2hiint(disc) < 0) return false;
#else
    if (signbit(disc)) return false;
#endif
    double sq = sqrt(disc);
    double root = (-half_b - sq) / a;
    if (root < (double)t_min || (double)t_max < root) {
        root = (-half_b + sq) / a;
        if (root < (double)t_min || (double)t_max < root) return false;
    }
    t_out = (float)root;
    return true;
}
// geometry/moving_sphere.rs:47-75 (all f32)
SHIM_HD f3 msphere_center(const f4* m, float time) {
    f3 c0 = xyz(m[0]), c1 = xyz(m[1]);
    float time0 = m[1].w, time1 = m[2].x;
    return c0 + ((time - time0) / (time1 - time0)) * (c1 - c0);
}
SHIM_HD bool hit_msphere(const f4* m, const Ray& r, float t_min, float t_max, float& t_out) {
    float radius = m[0].w;
    f3 oc = r.o - msphere_center(m, r.time);
    float a = dot3(r.d, r.d);
    float half_b = dot3(oc, r.d);
    float c = dot3(oc, oc) - radius * radius;
    float disc = half_b * half_b - a * c;
    if (signbit_f(disc)) return false;
    float sq = sqrtf(disc);
    float root = (-half_b - sq) / a;
    if (root < t_min || t_max < root) {
        root = (-half_b + sq) / a;
        if (root < t_min || t_max < root) return false;
    }
    t_out = root;
    return true;
}
// geometry/rectangle.rs:37-65 / 99-127 / 161-189.  axis: 2 = Xy (a=x,b=y), 1 = Xz (a=x,b=z), 0 = Yz (a=y,b=z)
SHIM_HD bool hit_rect_raw(int axis, float a0, float a1, float b0, float b1, float k, const Ray& r, float t_min, float t_max,
                          float& t_out) {
    int ia = axis == 0 ? 1 : 0, ib = axis == 2 ? 1 : 2;
    float t = (k - comp(r.o, axis)) / comp(r.d, axis);
    if (t < t_min || t > t_max) return false;
    float a = comp(r.o, ia) + t * comp(r.d, ia);
    float b = comp(r.o, ib) + t * comp(r.d, ib);
    if (a < a0 || a > a1 || b < b0 || b > b1) return false;
    t_out = t;
    return true;
}
SHIM_HD bool hit_rect(const f4* q, const Ray& r, float t_min, float t_max, float& t_out) {
    return hit_rect_raw(f2i(q[1].y), q[0].x, q[0].y, q[0].z, q[0].w, q[1].x, r, t_min, t_max, t_out);
}
// geometry/triangle.rs:32-92 (Moller-Trumbore, two-sided); q = {p0, e1, e2}
SHIM_HD bool hit_tri(const f4* q, const Ray& r, float t_min, float t_max, float& t_out) {
    const float epsilon = 0.0000001f;
    f3 p0 = xyz(q[0]), e1 = xyz(q[1]), e2 = xyz(q[2]);
    f3 h = cross3(r.d, e2);
    float a = dot3(e1, h);
    if (a > -epsilon && a < epsilon) return false;
    float f = 1.0f / a;
    f3 s = r.o - p0;
    float u = f * dot3(s, h);
    if (u < 0.0f || u > 1.0f) return false;
    f3 qq = cross3(s, e1);
    float v = f * dot3(r.d, qq);
    if (v < 0.0f || u + v > 1.0f) return false;
    float t = f * dot3(e2, qq);
    if (t < t_min || t > t_max) return false;
    if (t > epsilon) { t_out = t; return true; }
    return false;
}
// geometry/cube.rs:23-93: list of six rects (z-min, z-max, y-min, y-max, x-min, x-max), later wins ties
SHIM_HD void cube_side(const f4* q, int face, int& axis, float& a0, float& a1, float& b0, float& b1, float& k) {
    f3 mn = xyz(q[0]), mx = xyz(q[1]);
    if (face < 2) { axis = 2; a0 = mn.x; a1 = mx.x; b0 = mn.y; b1 = mx.y; k = face == 0 ? mn.z : mx.z; }
    else if (face < 4) { axis = 1; a0 = mn.x; a1 = mx.x; b0 = mn.z; b1 = mx.z; k = face == 2 ? mn.y : mx.y; }
    else { axis = 0; a0 = mn.y; a1 = mx.y; b0 = mn.z; b1 = mx.z; k = face == 4 ? mn.x : mx.x; }
}
SHIM_HD bool hit_cube(const f4* q, const Ray& r, float t_min, float t_max, float& t_out, int& face_out) {
    float closest = t_max;
    bool any = false;
#pragma unroll
    for (int f = 0; f < 6; ++f) {
        int axis; float a0, a1, b0, b1, k, t;
        cube_side(q, f, axis, a0, a1, b0, b1, k);
        if (hit_rect_raw(axis, a0, a1, b0, b1, k, r, t_min, closest, t)) { closest = t; face_out = f; any = true; }
    }
    t_out = closest;
    return any;
}

// ONLY >= 0: the caller knows every primitive it can meet is of that type (a Bvh of spheres only): no dispatch
template <int ONLY = -1>
SHIM_HD bool hit_prim(const SceneView& sv, uint32_t ref, const RayCtx& c, float t_min, float t_max, float& t, int& face) {
    uint32_t i = prim_index(ref);
    if (ONLY == PT_SPHERE) return hit_sphere(sv.sph + 4 * (size_t)i, c.r, t_min, t_max, t);
    if (ONLY == PT_TRI) return hit_tri(sv.tri + 3 * (size_t)i, c.r, t_min, t_max, t);
    switch (prim_type(ref)) {
    case PT_SPHERE: return hit_sphere(sv.sph + 4 * (size_t)i, c.r, t_min, t_max, t);
    case PT_MSPHERE: return hit_msphere(sv.msph + 3 * (size_t)i, c.r, t_min, t_max, t);
    case PT_RECT: return hit_rect(sv.rect + 2 * (size_t)i, c.r, t_min, t_max, t);
    case PT_TRI: return hit_tri(sv.tri + 3 * (size_t)i, c.r, t_min, t_max, t);
    case PT_CUBE: return hit_cube(sv.cube + 2 * (size_t)i, c.r, t_min, t_max, t, face);
    default: return false;
    }
}

// ---------------------------------------------------------------------------- BVH traversal
// Result contract (bvh.rs:363-417): the brute-force closest hit over the subtree's
// primitives, each tested as Hittable::hit(ray, t_min, t_max); among primitives with exactly
// equal t the one latest in left-to-right leaf order wins (`left.t < right.t` else right).
// Any visiting order satisfies it as long as ties are resolved by leaf rank (sv.rank[]).
//
// The walk is a while-while loop with a short stack: phase 1 descends inner nodes (one 64-byte
// node = both child boxes, four 16-byte loads, two fused-multiply-add slab tests, near child
// first) until the lane's next entry is a primitive; phase 2 tests that primitive.  Lanes of a
// warp therefore run their primitive tests (the f64 sphere quadratic) together.
SHIM_HD float slab_plane(float plane, float inv, float o_inv) {
#if defined(__CUDA_ARCH__)
    return __fmaf_rn(plane, inv, o_inv);
#else
    return fmaf(plane, inv, o_inv);
#endif
}
SHIM_HD bool slab(float mnx, float mny, float mnz, float mxx, float mxy, float mxz, const RayCtx& c, float t_min, float t_max,
                  float& t_near) {
    float x0 = slab_plane(mnx, c.inv_d.x, c.o_inv.x), x1 = slab_plane(mxx, c.inv_d.x, c.o_inv.x);
    float y0 = slab_plane(mny, c.inv_d.y, c.o_inv.y), y1 = slab_plane(mxy, c.inv_d.y, c.o_inv.y);
    float z0 = slab_plane(mnz, c.inv_d.z, c.o_inv.z), z1 = slab_plane(mxz, c.inv_d.z, c.o_inv.z);
    float tn = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), t_min));
    float tf = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), t_max));
    t_near = tn;
    return !(tf < tn);  // aabb.rs:36 rejects only when t_max < t_min
}

struct BvhBest { float t; uint32_t prim; int face; bool any; };

// One 64-byte DevNode.  A divergent walk out of global memory is bound by the L1 data pipe (one wavefront per lane and
// load instruction: 74 % of its peak in the mesh walk with four 16-byte loads per node), so a node in global memory is
// fetched with two 32-byte loads (LDG.E.ENL2.256, sm_100a) - half the wavefronts.  Nodes staged in shared memory keep
// the 16-byte loads.
SHIM_HD void load_node(const DevNode* nodes, int cur, f4& a, f4& b, f4& c, i4& d) {
    const DevNode* n = nodes + cur;
#if defined(__CUDA_ARCH__) && !defined(SHIM_NO_LDG256)
    if (__isGlobal(nodes)) {
        asm("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
            : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "l"(n));
        asm("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8+32];"
            : "=f"(c.x), "=f"(c.y), "=f"(c.z), "=f"(c.w), "=r"(d.x), "=r"(d.y), "=r"(d.z), "=r"(d.w) : "l"(n));
        return;
    }
#endif
    a = n->a; b = n->b; c = n->c; d = n->d;
}

#define SHIM_BVH_STACK 40
// An exact f32 tie between two primitives of one BVH (bvh.rs:396-415).  Across leaves the reference compares the two
// f32 t's and the later leaf wins.  Inside one recorded two-primitive leaf it tests the right child against the LEFT
// child's f32 t, which an f64 sphere root can exceed by the rounding: the right one wins only if it is still a hit
// under that bound.  Returns whether the candidate replaces the current best.
template <int ONLY = -1>
SHIM_HD bool tie_goes_to_candidate(const SceneView& sv, const RayCtx& c, float t_min, uint32_t cand, uint32_t best, float t) {
    const bool later = table_of(sv.rank, prim_type(cand))[prim_index(cand)] > table_of(sv.rank, prim_type(best))[prim_index(best)];
    if (table_of(sv.sibling, prim_type(cand))[prim_index(cand)] != (int)best) return later;
    float t2; int f2 = 0;
    const bool right_survives = hit_prim<ONLY>(sv, later ? cand : best, c, t_min, t, t2, f2);
    return later ? right_survives : !right_survives;
}

#define SHIM_STACK_END 0x7fffffff
SHIM_HD float max3f(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }   // FMNMX3 on sm_100a
SHIM_HD float min3f(float a, float b, float c) { return fminf(fminf(a, b), c); }
// Both child boxes of an SNode against one ray: X, Y, Z are the ray's {near_l, near_r, far_l, far_r} plane quadruples
// (SNode::ax[2 * axis + sign]); same result as two slab() calls on the plain node.
SHIM_HD void slab_pair_signed(const f4& X, const f4& Y, const f4& Z, const RayCtx& c, float t_min, float t_cull, float& tl, float& tr,
                              bool& hl, bool& hr) {
    tl = fmaxf(max3f(slab_plane(X.x, c.inv_d.x, c.o_inv.x), slab_plane(Y.x, c.inv_d.y, c.o_inv.y), slab_plane(Z.x, c.inv_d.z, c.o_inv.z)), t_min);
    tr = fmaxf(max3f(slab_plane(X.y, c.inv_d.x, c.o_inv.x), slab_plane(Y.y, c.inv_d.y, c.o_inv.y), slab_plane(Z.y, c.inv_d.z, c.o_inv.z)), t_min);
    const float fl = fminf(min3f(slab_plane(X.z, c.inv_d.x, c.o_inv.x), slab_plane(Y.z, c.inv_d.y, c.o_inv.y), slab_plane(Z.z, c.inv_d.z, c.o_inv.z)), t_cull);
    const float fr = fminf(min3f(slab_plane(X.w, c.inv_d.x, c.o_inv.x), slab_plane(Y.w, c.inv_d.y, c.o_inv.y), slab_plane(Z.w, c.inv_d.z, c.o_inv.z)), t_cull);
    hl = !(fl < tl);   // aabb.rs:36 rejects only when t_max < t_min
    hr = !(fr < tr);
}
// ---- QNode (shim_types.h): the eight words of a node and the slab test of both child boxes on the quantised planes
SHIM_HD uint32_t byte_perm32(uint32_t x, uint32_t y, uint32_t sel) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, y, sel);
#else
    const uint64_t v = ((uint64_t)y << 32) | x;
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i) r |= (uint32_t)((v >> (8 * ((sel >> (4 * i)) & 7u))) & 0xffu) << (8 * i);
    return r;
#endif
}
SHIM_HD uint32_t rotl32(uint32_t w, uint32_t r) {   // r = 0 or 16
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(w, w, r);
#else
    return r ? ((w << r) | (w >> (32u - r))) : w;
#endif
}
SHIM_HD void load_qnode(const QNode* nodes, int cur, uint32_t* w) {
    const QNode* n = nodes + cur;
#if defined(__CUDA_ARCH__)
    if (__isGlobal(nodes)) {
        asm("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
            : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]) : "l"(n));
        return;
    }
#endif
    w[0] = n->o[0]; w[1] = n->o[1]; w[2] = n->o[2]; w[3] = n->q[0]; w[4] = n->q[1]; w[5] = n->q[2];
    w[6] = (uint32_t)n->left; w[7] = (uint32_t)n->right;
}
// A plane is origin + q * S.  With f = the float 1 + q * 2^-15 (the byte dropped into the mantissa of 1.0 by one PRMT)
// and a = 2^15 * S / d:  (origin + q * S - o) / d  =  f * a + ((origin - o) / d - a): two instructions per plane.
// The rounding of these f32 operations is far below the grid step the builder added as margin (2^-9 of a step for
// the cancellation in b; an ulp of the distances otherwise, as in slab()).
SHIM_HD void slab_pair_q(const uint32_t* w, const RayCtx& c, float t_min, float t_cull, float& tl, float& tr, bool& hl, bool& hr) {
    float nl[3], nr[3], fl[3], fr[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float inv = k == 0 ? c.inv_d.x : (k == 1 ? c.inv_d.y : c.inv_d.z), oinv = k == 0 ? c.o_inv.x : (k == 1 ? c.o_inv.y : c.o_inv.z);
        const float a = i2f((int)(w[k] << 23)) * inv;   // bits 0-7 = exponent byte, bit 8 = 0 (sign)
        const float b = slab_plane(i2f((int)w[k]), inv, oinv) - a;
        const uint32_t q = rotl32(w[3 + k], c.qrot[k]);   // bytes {near_l, near_r, far_l, far_r}
        nl[k] = slab_plane(i2f((int)byte_perm32(q, 0x3F800000u, 0x7604u)), a, b);
        nr[k] = slab_plane(i2f((int)byte_perm32(q, 0x3F800000u, 0x7614u)), a, b);
        fl[k] = slab_plane(i2f((int)byte_perm32(q, 0x3F800000u, 0x7624u)), a, b);
        fr[k] = slab_plane(i2f((int)byte_perm32(q, 0x3F800000u, 0x7634u)), a, b);
    }
    tl = fmaxf(max3f(nl[0], nl[1], nl[2]), t_min);
    tr = fmaxf(max3f(nr[0], nr[1], nr[2]), t_min);
    const float el = fminf(min3f(fl[0], fl[1], fl[2]), t_cull);
    const float er = fminf(min3f(fr[0], fr[1], fr[2]), t_cull);
    hl = !(el < tl);
    hr = !(er < tr);
}
// SIGNED: node layout.  1 = walk sv.snodes (SNode, see shim_types.h); start_node and every non-negative reference are
// then byte offsets.  2 = walk sv.qnodes (QNode: larger boxes, so more nodes may be visited; the hit is the same).
// Both layouts visit the same nodes in the same order and return the same hit: for a box with min <= max and a finite
// reciprocal the plane the sign picks IS the smaller of the two products (fma is monotonic), and max/min are
// associative.
// ANY: an any-hit query.  It returns at the first primitive the closest-hit walk would accept (best holds it), so it is
// a prefix of that walk: until a first hit, t_cull == t_max in both and they test the same boxes and primitives.
template <bool COUNT, int ONLY = -1, int SIGNED = 0, bool ANY = false>
SHIM_HD bool bvh_closest(const SceneView& sv, int start_node, const RayCtx& c, float t_min, float t_max, BvhBest& best,
                         TraceCounters* cnt) {
    best.t = t_max; best.prim = 0; best.face = 0; best.any = false;
    // Boxes are culled against the closest hit so far (the reference never does: BvhNode::hit passes the caller's
    // t_max down unchanged, bvh.rs:385-394).  A primitive that TIES the current best often touches its own box
    // (a cube face is its box face), and the box entry is computed by different arithmetic than the primitive's
    // t, so the cull uses best.t widened by 2^-18 relative: ties are always tested and the tie rule decides.
    float t_cull = t_max;
    int stack[SHIM_BVH_STACK];
    int sp = 0;
    int cur = start_node;  // >= 0 inner node, < 0 ~prim_ref, SHIM_STACK_END when done
#if defined(__CUDA_ARCH__)
    uint32_t p0 = 0, px = 0, py = 0, pz = 0;
    if (SIGNED == 1) {   // the SNode walk lives in shared memory (wf_extend_solo / wf_trace_solo stage sv.snodes there)
        p0 = (uint32_t)__cvta_generic_to_shared(sv.snodes);
        px = p0 + (uint32_t)c.soff[0]; py = p0 + (uint32_t)c.soff[1]; pz = p0 + (uint32_t)c.soff[2];
        // opaque to the optimiser: otherwise it re-derives the three offsets from the direction signs in every
        // iteration (ten address instructions per node) instead of keeping three registers
        asm volatile("" : "+r"(px), "+r"(py), "+r"(pz));
    }
#endif
    for (;;) {
        while (cur >= 0 && cur != SHIM_STACK_END) {
            float tl, tr;
            bool hl, hr;
            int left, right;
            if (SIGNED == 2) {
                uint32_t w[8];
                load_qnode(sv.qnodes, cur, w);
                slab_pair_q(w, c, t_min, t_cull, tl, tr, hl, hr);
                left = (int)w[6]; right = (int)w[7];
                hr = hr && right != CHILD_NONE;
            } else if (SIGNED == 1) {
                f4 X, Y, Z;
                i4 nd;
#if defined(__CUDA_ARCH__)
                // shared-memory addresses of the ray's plane quadruples: one add per load (px, py, pz are per-ray)
                asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(X.x), "=f"(X.y), "=f"(X.z), "=f"(X.w) : "r"(px + (uint32_t)cur));
                asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(Y.x), "=f"(Y.y), "=f"(Y.z), "=f"(Y.w) : "r"(py + (uint32_t)cur));
                asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(Z.x), "=f"(Z.y), "=f"(Z.z), "=f"(Z.w) : "r"(pz + (uint32_t)cur));
                asm("ld.shared.v2.s32 {%0, %1}, [%2+96];" : "=r"(nd.x), "=r"(nd.y) : "r"(p0 + (uint32_t)cur));
#else
                const char* nb = reinterpret_cast<const char*>(sv.snodes) + cur;
                X = *reinterpret_cast<const f4*>(nb + c.soff[0]);
                Y = *reinterpret_cast<const f4*>(nb + c.soff[1]);
                Z = *reinterpret_cast<const f4*>(nb + c.soff[2]);
                nd = *reinterpret_cast<const i4*>(nb + 96);
#endif
                slab_pair_signed(X, Y, Z, c, t_min, t_cull, tl, tr, hl, hr);
                hr = hr && nd.y != CHILD_NONE;
                left = nd.x; right = nd.y;
            } else {
                f4 na, nb, nc;
                i4 nd;
                load_node(sv.nodes, cur, na, nb, nc, nd);
                hl = slab(na.x, na.y, na.z, na.w, nb.x, nb.y, c, t_min, t_cull, tl);
                hr = slab(nb.z, nb.w, nc.x, nc.y, nc.z, nc.w, c, t_min, t_cull, tr);
                hr = hr && nd.y != CHILD_NONE;
                left = nd.x; right = nd.y;
            }
            if (COUNT) cnt->nodes++;
            if (hl && hr) {
                bool swap = tr < tl;
                cur = swap ? right : left;
                if (sp < SHIM_BVH_STACK) stack[sp++] = swap ? left : right;
            } else if (hl) {
                cur = left;
            } else if (hr) {
                cur = right;
            } else {
                cur = sp > 0 ? stack[--sp] : SHIM_STACK_END;
            }
        }
        if (cur == SHIM_STACK_END) break;
        {
            uint32_t ref = ~(uint32_t)cur;
            float t; int face = 0;
            if (COUNT) cnt->prims++;
            // the primitive sees the widened bound too (an identical sphere's f64 root can lie just above the
            // f32-rounded best.t); what counts is its f32 t: closer wins, an exact tie goes to the later leaf
            // of the recorded tree (bvh.rs:409-415), anything beyond best.t is not a hit
            if (hit_prim<ONLY>(sv, ref, c, t_min, t_cull, t, face) && !(t > best.t)) {
                if constexpr (ANY) { best.t = t; best.prim = ref; best.face = face; best.any = true; return true; }
                bool take = !best.any || t < best.t;
                if (!take) take = tie_goes_to_candidate<ONLY>(sv, c, t_min, ref, best.prim, t);
                if (take) { best.t = t; best.prim = ref; best.face = face; best.any = true; t_cull = t + fabsf(t) * 3.8146973e-06f; }
            }
            cur = sp > 0 ? stack[--sp] : SHIM_STACK_END;
        }
    }
    return best.any;
}

// ---------------------------------------------------------------------------- hrpp.rs:132-193
SHIM_HD uint32_t hrpp_map_float(float v) {
    uint32_t bits = (uint32_t)f2i(v);
    uint32_t sign = (bits >> 31) & 1u, expo = (bits >> 25) & 0x3fu, mant = (bits >> 17) & 0x3fu;
    return (sign << 15) | (expo << 7) | mant;
}
SHIM_HD uint64_t hrpp_hash(const Ray& r) {
    uint64_t h0 = hrpp_map_float(r.o.x) ^ hrpp_map_float(r.d.z);
    uint64_t h1 = hrpp_map_float(r.o.y) ^ hrpp_map_float(r.d.y);
    uint64_t h2 = hrpp_map_float(r.o.z) ^ hrpp_map_float(r.d.x);
    return h0 | (h1 << 16) | (h2 << 32);
}


// The predictor table (Predictor, hrpp.rs:33-83) as a lock-free open-addressing table.  The reference keeps
// an unbounded AHashSet of leaf indices per key behind a Mutex; here a slot holds up to HRPP_LEAVES leaves
// (the cap the reference's own TODO proposes, hrpp.rs:65) and probing is bounded, so an insert into a full
// neighbourhood is dropped — the table is a cache either way.
#define SHIM_HRPP_EMPTY 0xFFFFFFFFu
SHIM_HD unsigned long long hrpp_cas64(unsigned long long* p, unsigned long long expect, unsigned long long val) {
#if defined(__CUDA_ARCH__)
    return atomicCAS(p, expect, val);
#else
    unsigned long long old = *p; if (old == expect) *p = val; return old;
#endif
}
SHIM_HD uint32_t hrpp_cas32(uint32_t* p, uint32_t expect, uint32_t val) {
#if defined(__CUDA_ARCH__)
    return atomicCAS(p, expect, val);
#else
    uint32_t old = *p; if (old == expect) *p = val; return old;
#endif
}
SHIM_HD size_t hrpp_home(const SceneView& sv, int table, unsigned long long key) {
    unsigned long long h = (key * 0x9E3779B97F4A7C15ull) >> (64 - sv.hrpp_log2);
    return (size_t)table * ((size_t)sv.hrpp_mask + 1) + (size_t)h;
}
#define SHIM_HRPP_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull
// One probe of the neighbourhood serves the lookup (Predictor::get_predictions, hrpp.rs:59-62) and, after a miss,
// the insert (Predictor::insert, hrpp.rs:64-82): `found` = the slot that holds the key, `empty` = the first empty
// slot before the end of the probe sequence (where the key would be inserted), -1 = none.  All HRPP_PROBES keys are
// fetched before any is looked at, so a lookup costs one memory latency, not one per probe (a full table of other
// rays' keys - the steady state of a render - made every miss a chain of eight dependent loads).
struct HrppProbe { long long found, empty; };
SHIM_HD HrppProbe hrpp_probe(const SceneView& sv, int table, unsigned long long key) {
    const unsigned long long tag = key | (1ull << 63);
    const size_t base = (size_t)table * ((size_t)sv.hrpp_mask + 1), home = hrpp_home(sv, table, key) - base;
    unsigned long long k[HRPP_PROBES];
#pragma unroll
    for (int p = 0; p < HRPP_PROBES; ++p) k[p] = sv.hrpp_slots[base + ((home + (size_t)p) & sv.hrpp_mask)].key;
    HrppProbe r; r.found = -1; r.empty = -1;
#pragma unroll
    for (int p = 0; p < HRPP_PROBES; ++p) {
        if (r.found < 0 && r.empty < 0) {
            if (k[p] == tag) r.found = (long long)(base + ((home + (size_t)p) & sv.hrpp_mask));
            else if (k[p] == SHIM_HRPP_EMPTY_KEY) r.empty = (long long)(base + ((home + (size_t)p) & sv.hrpp_mask));
        }
    }
    return r;
}
// adds `leaf` to the predictions of `slot` (which holds the ray's key); a full leaf list drops it (the cap, hrpp.rs:65)
SHIM_HD void hrpp_add_leaf(const SceneView& sv, long long slot, uint32_t leaf) {
    uint32_t* l = sv.hrpp_slots[slot].leaf;
    for (int j = 0; j < HRPP_LEAVES; ++j) {
        uint32_t v = l[j];
        if (v == SHIM_HRPP_EMPTY) v = hrpp_cas32(l + j, SHIM_HRPP_EMPTY, leaf), v = (v == SHIM_HRPP_EMPTY) ? leaf : v;
        if (v == leaf) return;
    }
}
// Predictor::insert after a probe: into the slot that holds the key, else claim the empty slot the probe saw (if another
// ray claimed it for another key in the meantime the prediction is dropped - the table is a cache); a neighbourhood
// without an empty slot drops it too
SHIM_HD void hrpp_insert(const SceneView& sv, const HrppProbe& pr, unsigned long long key, uint32_t leaf) {
    long long slot = pr.found;
    if (slot < 0) {
        if (pr.empty < 0) return;
        const unsigned long long tag = key | (1ull << 63);
        const unsigned long long old = hrpp_cas64(&sv.hrpp_slots[pr.empty].key, SHIM_HRPP_EMPTY_KEY, tag);
        if (old != SHIM_HRPP_EMPTY_KEY && old != tag) return;
        slot = pr.empty;
    }
    hrpp_add_leaf(sv, slot, leaf);
}

// Bvh::hit with a predictor, bvh.rs:107-211 (GO_UP_LEVEL = 0: predictions are leaf nodes).  A hit found in the
// predicted nodes is returned as the answer even if a closer one exists elsewhere (bvh.rs:145-156).
template <bool COUNT>
SHIM_HD bool bvh_closest_predicted(const SceneView& sv, const DevObject& ob, const RayCtx& c, float t_min, float t_max, BvhBest& best,
                                   TraceCounters* cnt) {
    const unsigned long long key = hrpp_hash(c.r);
    const HrppProbe pr = hrpp_probe(sv, ob.predictor, key);
    if (pr.found >= 0) {
        float closest = t_max;
        bool any = false;
        for (int j = 0; j < HRPP_LEAVES; ++j) {
            uint32_t node = sv.hrpp_slots[pr.found].leaf[j];
            if (node == SHIM_HRPP_EMPTY) break;
            BvhBest b;
            if (bvh_closest<COUNT>(sv, (int)node, c, t_min, closest, b, cnt)) { closest = b.t; best = b; any = true; }
        }
        if (any) { cnt->hrpp_tp++; return true; }
        cnt->hrpp_fp++;
    } else {
        cnt->hrpp_none++;
    }
    if (!bvh_closest<COUNT>(sv, ob.ref, c, t_min, t_max, best, cnt)) return false;
    int leaf = table_of(sv.leaf, prim_type(best.prim))[prim_index(best.prim)];
    hrpp_insert(sv, pr, key, (uint32_t)leaf);
    return true;
}

// shape of one top-level object against its object-space ray
// HASBVH = false: the caller knows the world holds no Bvh object (a flat list like the Cornell scenes)
// QN: the Bvh object sv.q_object is walked on its quantised nodes (same hit; tests/hostsim pins that)
// ANY: a Bvh object answers with its first accepted primitive (bvh_closest<..., ANY>), not the closest one
template <bool COUNT, bool HRPP, bool HASBVH = true, bool QN = false, bool ANY = false>
SHIM_HD bool shape_hit(const SceneView& sv, const DevObject& ob, const RayCtx& c, float t_min, float t_max, float& t, uint32_t& prim,
                       int& face, TraceCounters* cnt) {
    if (!HASBVH || ob.kind == OBJ_PRIM) {
        face = 0;
        if (COUNT) cnt->prims++;
        if (hit_prim(sv, (uint32_t)ob.ref, c, t_min, t_max, t, face)) { prim = (uint32_t)ob.ref; return true; }
        return false;
    }
    BvhBest best;
    bool hit;
    if (QN && sv.qnodes && ob.ref == sv.objects[sv.q_object].ref) hit = bvh_closest<COUNT, -1, 2, ANY>(sv, 0, c, t_min, t_max, best, cnt);
    else hit = (HRPP && (ob.flags & OBJ_PREDICTOR)) ? bvh_closest_predicted<COUNT>(sv, ob, c, t_min, t_max, best, cnt)
                                                    : bvh_closest<COUNT, -1, 0, ANY>(sv, ob.ref, c, t_min, t_max, best, cnt);
    if (hit) { t = best.t; prim = best.prim; face = best.face; return true; }
    return false;
}

// HittableList::hit over the flattened world (hittable.rs:100-118), with ConstantMedium::hit
// (hittable.rs:177-233) for medium objects.  `rng` must be keyed to STAGE_INTERSECT.
// ANY: the occlusion query - returns at the first object that has a hit (for a medium: once its free path is accepted).
// Until that object `closest` is t_max, so it makes the closest-hit query's tests and Philox draws, a prefix of them;
// h.obj >= 0 exactly when the closest-hit query's does.  h is then that first hit, not the closest one.
template <bool COUNT, bool HRPP = false, bool HASBVH = true, bool QN = false, bool ANY = false>
SHIM_HD Hit closest_hit(const SceneView& sv, const Ray& ray, float t_min, float t_max, Rng& rng, TraceCounters* cnt) {
    Hit h; h.t = t_max; h.obj = -1; h.prim = 0; h.face = 0;
    float closest = t_max;
    for (int oi = 0; oi < sv.n_objects; ++oi) {
        const DevObject& ob = sv.objects[oi];
        RayCtx c;
        c.r = object_ray(ob, ray);
        if (HASBVH && ob.kind == OBJ_BVH) make_ctx(c, c.r);  // reciprocals are only needed for box tests
        float t; uint32_t prim; int face;
        // One copy of the shape code serves all three calls (a medium asks its boundary twice, hittable.rs:190-199):
        // with shape_hit inlined three times the generic kernel was 7 100 instructions and 18 % of its stall samples
        // were instruction fetches.
        const bool medium = (ob.flags & OBJ_MEDIUM) != 0;
        float lo = medium ? -SHIM_INF : t_min, hi = medium ? SHIM_INF : closest, t1 = 0.0f;
        bool found = true;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int pass = 0; pass < 2; ++pass) {
            // a medium's boundary stays a closest-hit query: the free path needs its entry and exit t
            if constexpr (ANY) found = medium ? shape_hit<COUNT, HRPP, HASBVH, QN>(sv, ob, c, lo, hi, t, prim, face, cnt)
                                              : shape_hit<COUNT, HRPP, HASBVH, QN, true>(sv, ob, c, lo, hi, t, prim, face, cnt);
            else found = shape_hit<COUNT, HRPP, HASBVH, QN>(sv, ob, c, lo, hi, t, prim, face, cnt);
            if (!found || !medium || pass == 1) break;
            t1 = t; lo = t1 + 0.0001f;
        }
        if (!found) continue;
        if (medium) {
            float t2 = t;
            if (t1 < t_min) t1 = t_min;
            if (t2 > closest) t2 = closest;
            if (t1 >= t2) continue;
            if (t1 < 0.0f) t1 = 0.0f;
            float ray_length = len3(ray.d);
            float dist_inside = (t2 - t1) * ray_length;
            float hit_distance = ob.neg_inv_density * logf(rng_uniform01(rng));
            if (hit_distance > dist_inside) continue;
            t = t1 + hit_distance / ray_length;
            closest = t;
            h.t = t; h.obj = oi; h.prim = 0; h.face = 0;
        } else {
            closest = t;
            h.t = t; h.obj = oi; h.prim = prim; h.face = face;
        }
        if constexpr (ANY) break;
    }
    return h;
}

// closest_hit for a world that is exactly one plain Bvh (no Translate / RotateY / medium / predictor), e.g. the
// Book-1 scene (main.rs:185-251): no object loop, no object-space ray, fewer live registers in wf_extend_solo.
template <bool COUNT, int ONLY = -1, bool SIGNED = false>
SHIM_HD Hit closest_hit_solo(const SceneView& sv, const Ray& ray, float t_min, float t_max, TraceCounters* cnt) {
    Hit h; h.t = t_max; h.obj = -1; h.prim = 0; h.face = 0;
    RayCtx c;
    make_ctx(c, ray);
    BvhBest best;
    const int root = SIGNED ? sv.objects[0].ref * (int)sizeof(SNode) : sv.objects[0].ref;
    if (bvh_closest<COUNT, ONLY, SIGNED>(sv, root, c, t_min, t_max, best, cnt)) { h.t = best.t; h.obj = 0; h.prim = best.prim; h.face = best.face; }
    return h;
}

// Every stored material reference is a word: material index | kind << 28 (the flattener packs the kind in, so the
// closest-hit stage learns which material queue a hit goes to from the primitive record it already holds in
// shared memory instead of a second, dependent load from the material table).
SHIM_HD int mat_word_index(int w) { return w & 0x0fffffff; }
SHIM_HD int mat_word_kind(int w) { return (int)((uint32_t)w >> 28); }
SHIM_HD int prim_material_word(const SceneView& sv, uint32_t ref) {
    uint32_t i = prim_index(ref);
    switch (prim_type(ref)) {
    case PT_SPHERE: return sv.sph_mat[i];
    case PT_MSPHERE: return f2i(sv.msph[3 * (size_t)i + 2].y);
    case PT_RECT: return f2i(sv.rect[2 * (size_t)i + 1].z);
    case PT_TRI: return f2i(sv.tri[3 * (size_t)i].w);
    default: return f2i(sv.cube[2 * (size_t)i].w);
    }
}
SHIM_HD int prim_material(const SceneView& sv, uint32_t ref) { return mat_word_index(prim_material_word(sv, ref)); }
SHIM_HD int hit_material_word(const SceneView& sv, const Hit& h) {
    const DevObject& ob = sv.objects[h.obj];
    return (ob.flags & OBJ_MEDIUM) ? ob.phase_mat : prim_material_word(sv, h.prim);
}
SHIM_HD int hit_material(const SceneView& sv, const Hit& h) { return mat_word_index(hit_material_word(sv, h)); }
SHIM_HD int hit_handle(const SceneView& sv, const Hit& h) {
    if (h.obj < 0) return -1;
    const DevObject& ob = sv.objects[h.obj];
    if (ob.flags & OBJ_MEDIUM) return ob.handle;
    return table_of(sv.handle, prim_type(h.prim))[prim_index(h.prim)];
}

// ---------------------------------------------------------------------------- hit record
struct HitRec { f3 point, normal; float t, u, v; bool front_face; int material; };

// geometry/sphere.rs:41-46
SHIM_HD void sphere_uv(f3 p, float& u, float& v) {
    float theta = acosf(-p.y);
    float phi = atan2f(-p.z, p.x) + SHIM_PI;
    u = phi / (2.0f * SHIM_PI);
    v = theta / SHIM_PI;
}
// HitRecord::new, hittable.rs:28-52
SHIM_HD void rec_new(HitRec& rec, const Ray& r, f3 outward, float t, float u, float v, int material) {
    rec.point = ray_at(r, t);
    rec.front_face = signbit_f(dot3(r.d, outward));
    rec.normal = rec.front_face ? outward : -outward;
    rec.t = t; rec.u = u; rec.v = v; rec.material = material;
}
// Rebuilds the HitRecord the reference's hit() chain would have returned for this hit.
// `need_uv`: the sphere uv (acos/atan2) is only evaluated when the material's texture reads it.
SHIM_HD void reconstruct_hit(const SceneView& sv, const Ray& ray, const Hit& h, bool need_uv, HitRec& rec) {
    const DevObject& ob = sv.objects[h.obj];
    if (ob.flags & OBJ_MEDIUM) {  // hittable.rs:216-231
        rec.point = ray_at(ray, h.t);
        rec.normal = mk3(1.0f, 0.0f, 0.0f);
        rec.t = h.t; rec.u = 0.0f; rec.v = 0.0f; rec.front_face = true; rec.material = mat_word_index(ob.phase_mat);
        return;
    }
    Ray r = object_ray(ob, ray);
    uint32_t i = prim_index(h.prim);
    switch (prim_type(h.prim)) {
    case PT_SPHERE: {
        f4 s = sv.sph_s[i];
        f3 point = ray_at(r, h.t);
        f3 n = (point - xyz(s)) / s.w;
        float u = 0.0f, v = 0.0f;
        if (need_uv) sphere_uv(n, u, v);
        rec_new(rec, r, n, h.t, u, v, mat_word_index(sv.sph_mat[i]));
        break;
    }
    case PT_MSPHERE: {
        const f4* m = sv.msph + 3 * (size_t)i;
        f3 point = ray_at(r, h.t);
        f3 n = (point - msphere_center(m, r.time)) / m[0].w;
        float u = 0.0f, v = 0.0f;
        if (need_uv) sphere_uv(n, u, v);
        rec_new(rec, r, n, h.t, u, v, f2i(m[2].y));
        break;
    }
    case PT_TRI: {
        const f4* q = sv.tri + 3 * (size_t)i;
        f3 n = normalize3(cross3(xyz(q[1]), xyz(q[2])));
        rec_new(rec, r, n, h.t, 0.0f, 0.0f, f2i(q[0].w));
        break;
    }
    default: {  // PT_RECT, PT_CUBE
        int axis, mat; float a0, a1, b0, b1, k;
        if (prim_type(h.prim) == PT_RECT) {
            const f4* q = sv.rect + 2 * (size_t)i;
            axis = f2i(q[1].y); a0 = q[0].x; a1 = q[0].y; b0 = q[0].z; b1 = q[0].w; k = q[1].x; mat = f2i(q[1].z);
        } else {
            const f4* q = sv.cube + 2 * (size_t)i;
            cube_side(q, h.face, axis, a0, a1, b0, b1, k);
            mat = f2i(q[0].w);
        }
        int ia = axis == 0 ? 1 : 0, ib = axis == 2 ? 1 : 2;
        float a = comp(r.o, ia) + h.t * comp(r.d, ia);
        float b = comp(r.o, ib) + h.t * comp(r.d, ib);
        float u = (a - a0) / (a1 - a0);
        float v = (b - b0) / (b1 - b0);
        f3 n = axis == 0 ? mk3(1, 0, 0) : (axis == 1 ? mk3(0, 1, 0) : mk3(0, 0, 1));
        rec_new(rec, r, n, h.t, u, v, mat);
        break;
    }
    }
    if (ob.flags & OBJ_ROTATE) {  // instance.rs:124-141
        f3 p = rot_y_back(rec.point, ob.sin_t, ob.cos_t);
        f3 n = rot_y_back(rec.normal, ob.sin_t, ob.cos_t);
        rec.point = p;
        bool front = dot3(r.d, n) < 0.0f;  // set_face_normal with the rotated ray; front_face is left untouched
        rec.normal = front ? n : -n;
    }
    if (ob.flags & OBJ_TRANSLATE) rec.point = rec.point + mk3(ob.dx, ob.dy, ob.dz);  // instance.rs:40-42
}

// shim_hit_record (include/shimmer_b200.h) of a closest_hit result as three 16-byte words: {point, normal.x},
// {normal.yz, t, u}, {v, front_face, material, hittable}.  uv is always evaluated, as the reference's hit() does;
// material and hittable are the ids hit_material / hit_handle give.  A miss: t = +inf, ids -1, the rest 0.
SHIM_HD void hit_record_words(const SceneView& sv, const Ray& ray, const Hit& h, f4& w0, f4& w1, f4& w2) {
    if (h.obj < 0) {
        w0 = f4{0.0f, 0.0f, 0.0f, 0.0f};
        w1 = f4{0.0f, 0.0f, SHIM_INF, 0.0f};
        w2 = f4{0.0f, i2f(0), i2f(-1), i2f(-1)};
        return;
    }
    HitRec rec;
    reconstruct_hit(sv, ray, h, true, rec);
    w0 = f4{rec.point.x, rec.point.y, rec.point.z, rec.normal.x};
    w1 = f4{rec.normal.y, rec.normal.z, rec.t, rec.u};
    w2 = f4{rec.v, i2f(rec.front_face ? 1 : 0), i2f(hit_material(sv, h)), i2f(hit_handle(sv, h))};
}

// ---------------------------------------------------------------------------- ray-batch queries
// Ray i of a batch (7 floats: origin, direction, time) and its Philox stream: pixel i, sample 0, bounce 0 of
// STAGE_INTERSECT.  The batch kernels (trace_batch in shim_kernels.cuh) and the CPU harness both read rays this way.
SHIM_HD void batch_ray(const float* rays, long long i, uint64_t seed, Ray& r, Rng& rng) {
    const float* q = rays + i * 7;
    r.o = mk3(q[0], q[1], q[2]); r.d = mk3(q[3], q[4], q[5]); r.time = q[6];
    rng_init(rng, (uint32_t)i, 0, seed);
    rng_key(rng, 0, STAGE_INTERSECT);
}

// What each query stores for ray i.  shim_trace_closest: the hittable id and t (+inf on a miss).
struct StoreClosest {
    int* prim_id; float* t_out;
    SHIM_HD void operator()(const SceneView& sv, long long i, const Ray&, const Hit& h) const {
        prim_id[i] = hit_handle(sv, h);
        t_out[i] = h.obj < 0 ? SHIM_INF : h.t;
    }
};
// shim_trace_hit: the record as three 16-byte stores (out: 3 f4 per ray).
struct StoreRecord {
    f4* out;
    SHIM_HD void operator()(const SceneView& sv, long long i, const Ray& r, const Hit& h) const {
        f4 w0, w1, w2;
        hit_record_words(sv, r, h, w0, w1, w2);
        out[3 * i] = w0;
        out[3 * i + 1] = w1;
        out[3 * i + 2] = w2;
    }
};
// shim_trace_occluded: 1 where the walk accepted a hit.
struct StoreOccluded {
    uint8_t* occluded;
    SHIM_HD void operator()(const SceneView&, long long i, const Ray&, const Hit& h) const { occluded[i] = h.obj >= 0 ? 1 : 0; }
};

// ---------------------------------------------------------------------------- textures
// Perlin / Turbulence standing in for the `noise` crate (see DESIGN.md); f64 like the crate.
SHIM_HD double perlin_fade(double t) { return t * t * t * (t * (t * 6.0 - 15.0) + 10.0); }
SHIM_HD double perlin_lerp(double t, double a, double b) { return a + t * (b - a); }
SHIM_HD double perlin_grad(int h, double x, double y, double z) {
    h &= 15;
    double u = h < 8 ? x : y;
    double v = h < 4 ? y : ((h == 12 || h == 14) ? x : z);
    return ((h & 1) == 0 ? u : -u) + ((h & 2) == 0 ? v : -v);
}
SHIM_HD double perlin_get(const uint8_t* perm, double x, double y, double z) {
    double fx = floor(x), fy = floor(y), fz = floor(z);
    int X = (int)((long long)fx & 255), Y = (int)((long long)fy & 255), Z = (int)((long long)fz & 255);
    x -= fx; y -= fy; z -= fz;
    double u = perlin_fade(x), v = perlin_fade(y), w = perlin_fade(z);
#define SHIM_P(i) ((int)perm[(i) & 255])
    int A = SHIM_P(X) + Y, AA = SHIM_P(A) + Z, AB = SHIM_P(A + 1) + Z;
    int B = SHIM_P(X + 1) + Y, BA = SHIM_P(B) + Z, BB = SHIM_P(B + 1) + Z;
    double r = perlin_lerp(
        w,
        perlin_lerp(v, perlin_lerp(u, perlin_grad(SHIM_P(AA), x, y, z), perlin_grad(SHIM_P(BA), x - 1, y, z)),
                    perlin_lerp(u, perlin_grad(SHIM_P(AB), x, y - 1, z), perlin_grad(SHIM_P(BB), x - 1, y - 1, z))),
        perlin_lerp(v, perlin_lerp(u, perlin_grad(SHIM_P(AA + 1), x, y, z - 1), perlin_grad(SHIM_P(BA + 1), x - 1, y, z - 1)),
                    perlin_lerp(u, perlin_grad(SHIM_P(AB + 1), x, y - 1, z - 1), perlin_grad(SHIM_P(BB + 1), x - 1, y - 1, z - 1))));
#undef SHIM_P
    return r;
}
#define SHIM_FBM_OCTAVES 6
SHIM_HD double fbm_get(const uint8_t* tables, double x, double y, double z) {
    const double lac = 2.0943951023931953, pers = 0.5;
    double result = 0.0, att = pers, denom = 0.0;
    for (int i = 0; i < SHIM_FBM_OCTAVES; ++i) {
        double s = perlin_get(tables + 256 * i, x, y, z) * att;
        denom += att;
        att *= pers;
        result += s;
        x *= lac; y *= lac; z *= lac;
    }
    return result * (1.0 / denom);
}
// tables: [0] source, [1..6] x-distort octaves, [7..12] y, [13..18] z
SHIM_HD double turbulence_get(const uint8_t* t, double x, double y, double z) {
    double x0 = x + 12414.0 / 65536.0, y0 = y + 65124.0 / 65536.0, z0 = z + 31337.0 / 65536.0;
    double x1 = x + 26519.0 / 65536.0, y1 = y + 18128.0 / 65536.0, z1 = z + 60493.0 / 65536.0;
    double x2 = x + 53820.0 / 65536.0, y2 = y + 11213.0 / 65536.0, z2 = z + 44845.0 / 65536.0;
    double xd = x + fbm_get(t + 256 * 1, x0, y0, z0) * 1.0;
    double yd = y + fbm_get(t + 256 * 7, x1, y1, z1) * 1.0;
    double zd = z + fbm_get(t + 256 * 13, x2, y2, z2) * 1.0;
    return perlin_get(t, xd, yd, zd);
}

// texture record: a = {kind, even|w, odd|h, blob offset}, b = {r, g, b, scale}
SHIM_HD f3 tex_value(const SceneView& sv, int ti, float u, float v, f3 p) {
    for (int guard = 0; guard < 16; ++guard) {
        f4 a = sv.textures[2 * (size_t)ti], b = sv.textures[2 * (size_t)ti + 1];
        int kind = f2i(a.x);
        if (kind == TEX_SOLID) return mk3(b.x, b.y, b.z);
        if (kind == TEX_CHECKER) {  // checker.rs:27-37
            float sines = sinf(b.w * p.x) * sinf(b.w * p.y) * sinf(b.w * p.z);
            ti = signbit_f(sines) ? f2i(a.z) : f2i(a.y);
            continue;
        }
        if (kind == TEX_MARBLE) {   // marble.rs:23-29
            float n = (float)turbulence_get(sv.perlin + (size_t)(uint32_t)f2i(a.w), (double)p.x, (double)p.y, (double)p.z);
            float g = 0.5f * (1.0f + sinf(b.w * p.z + 10.0f * n));
            return mk3(1.0f * g, 1.0f * g, 1.0f * g);
        }
        {                           // image_texture.rs:21-52
            uint32_t w = (uint32_t)f2i(a.y), hgt = (uint32_t)f2i(a.z);
            float uu = fminf(fmaxf(u, 0.0f), 1.0f);
            float vv = fminf(fmaxf(v, 0.0f), 1.0f);
            vv = 1.0f - vv;
            uint32_t i = (uint32_t)(uu * (float)w), j = (uint32_t)(vv * (float)hgt);
            if (i >= w) i = w - 1;
            if (j >= hgt) j = hgt - 1;
            const uint8_t* px = sv.images + (size_t)(uint32_t)f2i(a.w) + ((size_t)j * w + i) * 3;
            const float s = 1.0f / 255.0f;
            return mk3((float)px[0] * s, (float)px[1] * s, (float)px[2] * s);
        }
    }
    return mk3(0, 0, 0);
}
// does evaluating this texture read (u, v)?  (only image textures do)
SHIM_HD bool tex_needs_uv(const SceneView& sv, int ti) {
    // checker children may be images; walk both branches iteratively with a tiny stack
    int stack[8]; int sp = 0; stack[sp++] = ti;
    while (sp > 0) {
        int t = stack[--sp];
        f4 a = sv.textures[2 * (size_t)t];
        int kind = f2i(a.x);
        if (kind == TEX_IMAGE) return true;
        if (kind == TEX_CHECKER && sp + 2 <= 8) { stack[sp++] = f2i(a.y); stack[sp++] = f2i(a.z); }
    }
    return false;
}

// ---------------------------------------------------------------------------- materials
// material record: a = {kind, tex, fuzz, ior}, b = {albedo rgb, needs_uv}
SHIM_HD f3 reflect3(f3 v, f3 n) { return v - 2.0f * dot3(v, n) * n; }  // materials/utils.rs:37-39
SHIM_HD f3 refract3(f3 uv, f3 n, float eta) {                          // materials/utils.rs:41-46
    float cos_theta = fminf(dot3(-uv, n), 1.0f);
    f3 perp = eta * (uv + cos_theta * n);
    f3 par = -sqrtf(fabsf(1.0f - dot3(perp, perp))) * n;
    return par + perp;
}
SHIM_HD float schlick(float cosine, float ref_idx) {                   // dialectric.rs:26-29
    float r0 = (1.0f - ref_idx) / (1.0f + ref_idx);
    r0 = r0 * r0;
    float x = 1.0f - cosine;
    float x2 = x * x;
    return r0 + (1.0f - r0) * (x * (x2 * x2));
}
SHIM_HD f3 mat_emit(const SceneView& sv, int mi, const HitRec& rec) {  // material.rs:20-22, diffuse_light.rs:34-36
    f4 a = sv.materials[2 * (size_t)mi];
    if (f2i(a.x) == MAT_DIFFUSE_LIGHT) return tex_value(sv, f2i(a.y), rec.u, rec.v, rec.point);
    return mk3(0, 0, 0);
}
// `rng` must be keyed to STAGE_SCATTER
// `kind` is the material's kind (a compile-time constant in the material-sorted shade kernels)
SHIM_HD bool mat_scatter(const SceneView& sv, int kind, int mi, const Ray& ray, const HitRec& rec, Rng& rng, f3& att, Ray& out) {
    f4 a = sv.materials[2 * (size_t)mi], b = sv.materials[2 * (size_t)mi + 1];
    switch (kind) {
    case MAT_LAMBERTIAN: {  // lambertian.rs:35-52
        f3 dir = rec.normal + normalize3(random_in_unit_sphere(rng));
        if (fabsf(dir.x) < SHIM_F32_EPS && fabsf(dir.y) < SHIM_F32_EPS && fabsf(dir.z) < SHIM_F32_EPS) dir = rec.normal;
        out.o = rec.point; out.d = dir; out.time = ray.time;
        att = tex_value(sv, f2i(a.y), rec.u, rec.v, rec.point);
        return true;
    }
    case MAT_METAL: {       // metal.rs:26-42
        f3 reflected = reflect3(normalize3(ray.d), rec.normal);
        out.o = rec.point; out.d = reflected + a.z * random_in_unit_sphere(rng); out.time = ray.time;
        att = mk3(b.x, b.y, b.z);
        return dot3(out.d, rec.normal) > 0.0f;
    }
    case MAT_DIELECTRIC: {  // dialectric.rs:33-60
        att = mk3(1, 1, 1);
        float ratio = rec.front_face ? 1.0f / a.w : a.w;
        f3 unit = normalize3(ray.d);
        float cos_theta = fminf(dot3(-unit, rec.normal), 1.0f);
        float sin_theta = sqrtf(1.0f - cos_theta * cos_theta);
        bool cannot = ratio * sin_theta > 1.0f;
        f3 dir;
        if (cannot || schlick(cos_theta, ratio) > rng_uniform01(rng)) dir = reflect3(unit, rec.normal);
        else dir = refract3(unit, rec.normal, ratio);
        out.o = rec.point; out.d = dir; out.time = ray.time;
        return true;
    }
    case MAT_DIFFUSE_LIGHT: return false;  // diffuse_light.rs:25-32
    default: {              // isotropic.rs:32-42
        out.o = rec.point; out.d = random_in_unit_sphere(rng); out.time = ray.time;
        att = tex_value(sv, f2i(a.y), rec.u, rec.v, rec.point);
        return true;
    }
    }
}
SHIM_HD int mat_kind(const SceneView& sv, int mi) { return f2i(sv.materials[2 * (size_t)mi].x); }
SHIM_HD bool mat_needs_uv(const SceneView& sv, int mi) { return sv.materials[2 * (size_t)mi + 1].w != 0.0f; }

}  // namespace shim
