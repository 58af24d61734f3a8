// shimmer_oracle.cpp — CPU restatement of the `shimmer` hot path.  TEST INFRASTRUCTURE ONLY.
//
// This file is the ORACLE for the B200 backend: a plain C++17 restatement of what
// jalberse/RayTracingInOneWeekendInRust computes under `Renderer::render`
// (reference src/renderer.rs:42-149).  Nothing in the product path may include,
// link or call it; only tests/, __graft_entry__.smoke() and bench.py's
// cpu_baseline / --impl reference legs use it (as the checker / the CPU arm).
//
// PARITY PINNING.  The reference is Rust and cannot be compiled in this image
// (no cargo/rustc), so the oracle is pinned against what the reference's own
// tests hold for this path: the two Aabb::hit rays and four Aabb::union cases
// (aabb.rs:65-141), the two Tile::tile layouts (renderer.rs:307-378), the
// get_uv prose table (geometry/sphere.rs:37-40) and HRPP key known answers
// derived from hrpp.rs:132-193 (tests/test_oracle_kat.py).  Everything else on
// the path has NO test or golden vector in the reference: for those functions
// this oracle is "parity unpinned" — a line-by-line restatement, cited below.
//
// Third-party arithmetic that is not under /root/reference (glam 0.22.0 Vec3,
// rand 0.8.5 distributions, noise 0.8.2 Perlin/Turbulence) is restated from the
// published algorithms; see DESIGN.md "Third-party arithmetic".  The random
// STREAM is ours by necessity (the reference uses OS-seeded thread_rng and is
// irreproducible): Philox4x32-10 keyed (pixel, sample, bounce*4+stage), the
// same keying the device uses, so sample k of pixel p follows the same path
// on both sides.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -fPIC -shared -pthread
//        (no -ffast-math: IEEE f32/f64 op-for-op like rustc emits).

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

namespace orc {

// ---------------------------------------------------------------------------
// glam 0.22 scalar Vec3 / DVec3 (operation order as published: dot is
// x*x + y*y + z*z left to right, normalize multiplies by 1/length, Vec3/f32
// divides per component).
// ---------------------------------------------------------------------------
struct V3 {
    float x, y, z;
    float operator[](int i) const { return i == 0 ? x : (i == 1 ? y : z); }
    float& at(int i) { return i == 0 ? x : (i == 1 ? y : z); }
};
static inline V3 v3(float x, float y, float z) { return V3{x, y, z}; }
static inline V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
static inline V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
static inline V3 operator-(V3 a) { return {-a.x, -a.y, -a.z}; }
static inline V3 operator*(V3 a, V3 b) { return {a.x * b.x, a.y * b.y, a.z * b.z}; }
static inline V3 operator*(V3 a, float s) { return {a.x * s, a.y * s, a.z * s}; }
static inline V3 operator*(float s, V3 a) { return {s * a.x, s * a.y, s * a.z}; }
static inline V3 operator/(V3 a, float s) { return {a.x / s, a.y / s, a.z / s}; }
static inline float dot(V3 a, V3 b) { return (a.x * b.x) + (a.y * b.y) + (a.z * b.z); }
static inline V3 cross(V3 a, V3 b) {
    return {a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y};
}
static inline float length_squared(V3 a) { return dot(a, a); }
static inline float length(V3 a) { return std::sqrt(dot(a, a)); }
static inline V3 normalize(V3 a) { return a * (1.0f / length(a)); }

struct D3 { double x, y, z; };
static inline D3 operator-(D3 a, D3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
static inline double dot(D3 a, D3 b) { return (a.x * b.x) + (a.y * b.y) + (a.z * b.z); }

static const float F32_EPS = 1.1920929e-07f;  // f32::EPSILON
static const float F32_INF = std::numeric_limits<float>::infinity();
static const float PI_F = 3.14159265358979323846f;  // std::f32::consts::PI

static inline bool sign_negative(float v) { return std::signbit(v); }
static inline bool sign_negative(double v) { return std::signbit(v); }

// ---------------------------------------------------------------------------
// Random numbers.  Distributions follow rand 0.8.5: random::<f32>() is a 24-bit
// uniform in [0,1); gen_range(a..b) is a 23-bit uniform u in [0,1) mapped as
// u*(b-a)+a.  Two generators: keyed Philox4x32-10 (parity) and xorshift32
// (CPU-baseline timing, stands in for thread_rng).
// ---------------------------------------------------------------------------
static inline void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                 uint32_t k0, uint32_t k1, uint32_t out[4]) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

enum { STAGE_CAMERA = 0, STAGE_INTERSECT = 1, STAGE_SCATTER = 2 };

struct Rng {
    // keyed mode
    bool keyed = true;
    uint32_t pixel = 0, sample = 0, dim = 0, j = 0, k0 = 0, k1 = 0;
    uint32_t buf[4] = {0, 0, 0, 0};
    // fast mode
    uint32_t xs = 0x9E3779B9u;
    void key(uint32_t bounce, uint32_t stage) { dim = bounce * 4u + stage; j = 0; }
    uint32_t next_u32() {
        if (!keyed) {
            xs ^= xs << 13; xs ^= xs >> 17; xs ^= xs << 5;
            return xs * 0x9E3779B1u;
        }
        if ((j & 3u) == 0) philox4x32_10(pixel, sample, dim, j >> 2, k0, k1, buf);
        uint32_t v = buf[j & 3u];
        ++j;
        return v;
    }
    float uniform01() { return (float)(next_u32() >> 8) * (1.0f / 16777216.0f); }
    float uniform23() { return (float)(next_u32() >> 9) * (1.0f / 8388608.0f); }
    float range(float lo, float hi) { float s = hi - lo; return uniform23() * s + lo; }
};

// utils.rs:9-17
static V3 random_in_unit_disk(Rng& rng) {
    for (;;) {
        float a = rng.range(-1.0f, 1.0f);
        float b = rng.range(-1.0f, 1.0f);
        V3 p = v3(a, b, 0.0f);
        if (length_squared(p) < 1.0f) return p;
    }
}
// materials/utils.rs:6-19
static V3 random_in_unit_sphere(Rng& rng) {
    for (;;) {
        float a = rng.range(-1.0f, 1.0f);
        float b = rng.range(-1.0f, 1.0f);
        float c = rng.range(-1.0f, 1.0f);
        V3 p = v3(a, b, c);
        if (length_squared(p) < 1.0f) return p;
    }
}
// materials/utils.rs:22-24
static V3 random_unit_vector(Rng& rng) { return normalize(random_in_unit_sphere(rng)); }
// utils.rs:5-7
static bool near_zero(V3 v) {
    return std::fabs(v.x) < F32_EPS && std::fabs(v.y) < F32_EPS && std::fabs(v.z) < F32_EPS;
}
// materials/utils.rs:37-46
static V3 reflect(V3 v, V3 n) { return v - 2.0f * dot(v, n) * n; }
static V3 refract(V3 uv, V3 n, float eta) {
    float cos_theta = std::fmin(dot(-uv, n), 1.0f);
    V3 perp = eta * (uv + cos_theta * n);
    V3 par = -std::sqrt(std::fabs(1.0f - length_squared(perp))) * n;
    return par + perp;
}

// ---------------------------------------------------------------------------
// ray.rs:12-30
// ---------------------------------------------------------------------------
struct Ray {
    V3 origin, direction;
    float time;
    V3 at(float t) const { return origin + t * direction; }
};

// ---------------------------------------------------------------------------
// aabb.rs:8-62
// ---------------------------------------------------------------------------
struct Aabb {
    V3 min, max;
    bool hit(const Ray& ray, float t_min, float t_max) const {
        for (int i = 0; i < 3; ++i) {
            float inv_d = 1.0f / ray.direction[i];
            float t0 = (min[i] - ray.origin[i]) * inv_d;
            float t1 = (max[i] - ray.origin[i]) * inv_d;
            if (inv_d < 0.0f) std::swap(t0, t1);
            t_min = t0 > t_min ? t0 : t_min;
            t_max = t1 < t_max ? t1 : t_max;
            if (t_max < t_min) return false;
        }
        return true;
    }
};
// f32::min / f32::max (NaN-ignoring like fminf/fmaxf)
static Aabb aabb_union(const Aabb& a, const Aabb& b) {
    return Aabb{v3(std::fmin(a.min.x, b.min.x), std::fmin(a.min.y, b.min.y), std::fmin(a.min.z, b.min.z)),
                v3(std::fmax(a.max.x, b.max.x), std::fmax(a.max.y, b.max.y), std::fmax(a.max.z, b.max.z))};
}

// ---------------------------------------------------------------------------
// Perlin / Turbulence standing in for noise 0.8.2 (source not vendored; the
// contract is the formula at textures/marble.rs:23-29).  Same structure as the
// crate: Turbulence = source Perlin sampled at a point displaced by three
// Fbm<Perlin> (seeds 0,1,2; 6 octaves; lacunarity 2*pi/3; persistence 0.5).
// The permutation table comes from splitmix64(seed) Fisher-Yates.  f64.
// ---------------------------------------------------------------------------
static inline uint64_t splitmix64(uint64_t& s) {
    s += 0x9E3779B97F4A7C15ull;
    uint64_t z = s;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
struct Perlin {
    uint8_t perm[256];
    void init(uint32_t seed) {
        for (int i = 0; i < 256; ++i) perm[i] = (uint8_t)i;
        uint64_t s = 0x5851F42D4C957F2Dull ^ (uint64_t)seed;
        for (int i = 255; i > 0; --i) {
            uint32_t jx = (uint32_t)(splitmix64(s) % (uint64_t)(i + 1));
            std::swap(perm[i], perm[jx]);
        }
    }
    static double fade(double t) { return t * t * t * (t * (t * 6.0 - 15.0) + 10.0); }
    static double lerp(double t, double a, double b) { return a + t * (b - a); }
    static double grad(int h, double x, double y, double z) {
        h &= 15;
        double u = h < 8 ? x : y;
        double v = h < 4 ? y : ((h == 12 || h == 14) ? x : z);
        return ((h & 1) == 0 ? u : -u) + ((h & 2) == 0 ? v : -v);
    }
    int p(int i) const { return perm[i & 255]; }
    double get(double x, double y, double z) const {
        double fx = std::floor(x), fy = std::floor(y), fz = std::floor(z);
        int X = (int)((long long)fx & 255), Y = (int)((long long)fy & 255), Z = (int)((long long)fz & 255);
        x -= fx; y -= fy; z -= fz;
        double u = fade(x), v = fade(y), w = fade(z);
        int A = p(X) + Y, AA = p(A) + Z, AB = p(A + 1) + Z;
        int B = p(X + 1) + Y, BA = p(B) + Z, BB = p(B + 1) + Z;
        return lerp(w,
                    lerp(v, lerp(u, grad(p(AA), x, y, z), grad(p(BA), x - 1, y, z)),
                         lerp(u, grad(p(AB), x, y - 1, z), grad(p(BB), x - 1, y - 1, z))),
                    lerp(v, lerp(u, grad(p(AA + 1), x, y, z - 1), grad(p(BA + 1), x - 1, y, z - 1)),
                         lerp(u, grad(p(AB + 1), x, y - 1, z - 1), grad(p(BB + 1), x - 1, y - 1, z - 1))));
    }
};
static const int FBM_OCTAVES = 6;
static const double FBM_LACUNARITY = 2.0943951023931953;  // 2*pi/3
static const double FBM_PERSISTENCE = 0.5;
struct Fbm {
    Perlin oct[FBM_OCTAVES];
    double scale;
    void init(uint32_t seed) {
        double denom = 0.0, a = FBM_PERSISTENCE;
        for (int i = 0; i < FBM_OCTAVES; ++i) { oct[i].init(seed + (uint32_t)i); denom += a; a *= FBM_PERSISTENCE; }
        scale = 1.0 / denom;
    }
    double get(double x, double y, double z) const {
        double result = 0.0, att = FBM_PERSISTENCE;
        for (int i = 0; i < FBM_OCTAVES; ++i) {
            double s = oct[i].get(x, y, z) * att;
            att *= FBM_PERSISTENCE;
            result += s;
            x *= FBM_LACUNARITY; y *= FBM_LACUNARITY; z *= FBM_LACUNARITY;
        }
        return result * scale;
    }
};
struct Turbulence {
    Perlin source;
    Fbm dx, dy, dz;
    void init(uint32_t seed) { source.init(seed); dx.init(0); dy.init(1); dz.init(2); }
    double get(double x, double y, double z) const {
        const double power = 1.0;
        double x0 = x + 12414.0 / 65536.0, y0 = y + 65124.0 / 65536.0, z0 = z + 31337.0 / 65536.0;
        double x1 = x + 26519.0 / 65536.0, y1 = y + 18128.0 / 65536.0, z1 = z + 60493.0 / 65536.0;
        double x2 = x + 53820.0 / 65536.0, y2 = y + 11213.0 / 65536.0, z2 = z + 44845.0 / 65536.0;
        double xd = x + dx.get(x0, y0, z0) * power;
        double yd = y + dy.get(x1, y1, z1) * power;
        double zd = z + dz.get(x2, y2, z2) * power;
        return source.get(xd, yd, zd);
    }
};

// ---------------------------------------------------------------------------
// textures/*.rs
// ---------------------------------------------------------------------------
enum TexKind { TEX_SOLID = 0, TEX_CHECKER = 1, TEX_MARBLE = 2, TEX_IMAGE = 3 };
struct Texture {
    int kind = TEX_SOLID;
    V3 color{0, 0, 0};
    float scale = 0;
    int even = -1, odd = -1;
    std::shared_ptr<Turbulence> turb;
    std::vector<uint8_t> rgb;
    uint32_t w = 0, h = 0;
};

// ---------------------------------------------------------------------------
// materials/*.rs
// ---------------------------------------------------------------------------
enum MatKind { MAT_LAMBERTIAN = 0, MAT_METAL = 1, MAT_DIELECTRIC = 2, MAT_DIFFUSE_LIGHT = 3, MAT_ISOTROPIC = 4 };
struct Material {
    int kind = MAT_LAMBERTIAN;
    int tex = -1;
    V3 albedo{0, 0, 0};
    float fuzz = 0, ior = 1;
};

// hittable.rs:15-62
struct HitRecord {
    V3 point{0, 0, 0}, normal{0, 0, 0};
    float t = 0, u = 0, v = 0;
    bool front_face = false;
    int material = -1;
    // not in the reference: identity of what was hit, for gate 1 and HRPP
    int prim_id = -1;
    int face = 0;
};
static HitRecord make_hit(const Ray& ray, V3 outward, float t, float u, float v, int material, int prim_id) {
    HitRecord r;
    r.point = ray.at(t);
    r.front_face = sign_negative(dot(ray.direction, outward));
    r.normal = r.front_face ? outward : -outward;
    r.t = t; r.u = u; r.v = v; r.material = material; r.prim_id = prim_id;
    return r;
}
static void set_face_normal(HitRecord& rec, const Ray& ray, V3 outward) {
    bool front = dot(ray.direction, outward) < 0.0f;
    rec.normal = front ? outward : -outward;
}

struct Counters {
    uint64_t rays = 0, node_visits = 0, prim_tests = 0, hrpp_tp = 0, hrpp_fp = 0, hrpp_none = 0;
    void add(const Counters& o) {
        rays += o.rays; node_visits += o.node_visits; prim_tests += o.prim_tests;
        hrpp_tp += o.hrpp_tp; hrpp_fp += o.hrpp_fp; hrpp_none += o.hrpp_none;
    }
};

struct Scene;
struct Ctx {
    const Scene* scene = nullptr;
    Rng* rng = nullptr;        // stage-keyed by the caller
    bool use_predictors = false;
    Counters cnt;
};

struct Hittable {
    int id = -1;
    virtual ~Hittable() {}
    virtual bool hit(const Ray& ray, float t_min, float t_max, Ctx& ctx, HitRecord& out) const = 0;
    virtual bool bounding_box(float t0, float t1, Aabb& out) const = 0;
    virtual bool is_list() const { return false; }
};
typedef std::shared_ptr<Hittable> HPtr;

// geometry/sphere.rs:41-109
static void sphere_uv(V3 p, float& u, float& v) {
    float theta = std::acos(-p.y);
    float phi = std::atan2(-p.z, p.x) + PI_F;
    u = phi / (2.0f * PI_F);
    v = theta / PI_F;
}
struct Sphere : Hittable {
    V3 center; float radius; int material;
    bool hit(const Ray& ray, float t_min, float t_max, Ctx& ctx, HitRecord& out) const override {
        ctx.cnt.prim_tests++;
        D3 direction{(double)ray.direction.x, (double)ray.direction.y, (double)ray.direction.z};
        D3 origin{(double)ray.origin.x, (double)ray.origin.y, (double)ray.origin.z};
        D3 c{(double)center.x, (double)center.y, (double)center.z};
        double r = (double)radius;
        D3 oc = origin - c;
        double a = dot(direction, direction);
        double half_b = dot(oc, direction);
        double cc = dot(oc, oc) - r * r;
        double disc = half_b * half_b - a * cc;
        if (sign_negative(disc)) return false;
        double sq = std::sqrt(disc);
        double root = (-half_b - sq) / a;
        if (root < (double)t_min || (double)t_max < root) {
            root = (-half_b + sq) / a;
            if (root < (double)t_min || (double)t_max < root) return false;
        }
        V3 point = ray.at((float)root);
        V3 normal = (point - center) / radius;
        float u, v;
        sphere_uv(normal, u, v);
        out = make_hit(ray, normal, (float)root, u, v, material, id);
        return true;
    }
    bool bounding_box(float, float, Aabb& out) const override {
        V3 rad = v3(radius, radius, radius);
        out = Aabb{center - rad, center + rad};
        return true;
    }
};

// geometry/moving_sphere.rs:47-93 (all f32; bounding box keeps the reference's
// end-box typo: its min uses center(time_0))
struct MovingSphere : Hittable {
    V3 c0, c1; float time0, time1, radius; int material;
    V3 center(float time) const { return c0 + ((time - time0) / (time1 - time0)) * (c1 - c0); }
    bool hit(const Ray& ray, float t_min, float t_max, Ctx& ctx, HitRecord& out) const override {
        ctx.cnt.prim_tests++;
        V3 oc = ray.origin - center(ray.time);
        float a = length_squared(ray.direction);
        float half_b = dot(oc, ray.direction);
        float c = length_squared(oc) - radius * radius;
        float disc = half_b * half_b - a * c;
        if (sign_negative(disc)) return false;
        float sq = std::sqrt(disc);
        float root = (-half_b - sq) / a;
        if (root < t_min || t_max < root) {
            root = (-half_b + sq) / a;
            if (root < t_min || t_max < root) return false;
        }
        V3 point = ray.at(root);
        V3 normal = (point - center(ray.time)) / radius;
        float u, v;
        sphere_uv(normal, u, v);
        out = make_hit(ray, normal, root, u, v, material, id);
        return true;
    }
    bool bounding_box(float t0, float t1, Aabb& out) const override {
        V3 rad = v3(radius, radius, radius);
        Aabb start{center(t0) - rad, center(t0) + rad};
        Aabb end{center(t0) - rad, center(t1) + rad};
        out = aabb_union(start, end);
        return true;
    }
};

// geometry/rectangle.rs — axis 2 = XyRect (a=x,b=y,k=z), 1 = XzRect (a=x,b=z,k=y), 0 = YzRect (a=y,b=z,k=x)
struct Rect : Hittable {
    int axis; float a0, a1, b0, b1, k; int material;
    bool hit(const Ray& ray, float t_min, float t_max, Ctx& ctx, HitRecord& out) const override {
        ctx.cnt.prim_tests++;
        int ia = axis == 0 ? 1 : 0, ib = axis == 2 ? 1 : 2;
        float t = (k - ray.origin[axis]) / ray.direction[axis];
        if (t < t_min || t > t_max) return false;
        float a = ray.origin[ia] + t * ray.direction[ia];
        float b = ray.origin[ib] + t * ray.direction[ib];
        if (a < a0 || a > a1 || b < b0 || b > b1) return false;
        float u = (a - a0) / (a1 - a0);
        float v = (b - b0) / (b1 - b0);
        V3 n = axis == 0 ? v3(1, 0, 0) : (axis == 1 ? v3(0, 1, 0) : v3(0, 0, 1));
        out = make_hit(ray, n, t, u, v, material, id);
        return true;
    }
    bool bounding_box(float, float, Aabb& out) const override {
        if (axis == 2) out = Aabb{v3(a0, b0, k - F32_EPS), v3(a1, b1, k + F32_EPS)};
        else if (axis == 1) out = Aabb{v3(a0, k - F32_EPS, b0), v3(a1, k + F32_EPS, b1)};
        else out = Aabb{v3(k - F32_EPS, a0, b0), v3(k + F32_EPS, a1, b1)};
        return true;
    }
};

// geometry/triangle.rs:32-107
struct Tri : Hittable {
    V3 p0, p1, p2; int material;
    bool hit(const Ray& ray, float t_min, float t_max, Ctx& ctx, HitRecord& out) const override {
        ctx.cnt.prim_tests++;
        const float epsilon = 0.0000001f;
        V3 edge1 = p1 - p0, edge2 = p2 - p0;
        V3 h = cross(ray.direction, edge2);
        float a = dot(edge1, h);
        if (a > -epsilon && a < epsilon) return false;
        float f = 1.0f / a;
        V3 s = ray.origin - p0;
        float u = f * dot(s, h);
        if (u < 0.0f || u > 1.0f) return false;
        V3 q = cross(s, edge1);
        float v = f * dot(ray.direction, q);
        if (v < 0.0f || u + v > 1.0f) return false;
        float t = f * dot(edge2, q);
        if (t < t_min || t > t_max) return false;
        if (t > epsilon) {
            V3 n = normalize(cross(edge1, edge2));
            out = make_hit(ray, n, t, 0.0f, 0.0f, material, id);
            return true;
        }
        return false;
    }
    bool bounding_box(float, float, Aabb& out) const override {
        out = Aabb{v3(std::fmin(p0.x, std::fmin(p1.x, p2.x)) - F32_EPS, std::fmin(p0.y, std::fmin(p1.y, p2.y)) - F32_EPS,
                      std::fmin(p0.z, std::fmin(p1.z, p2.z)) - F32_EPS),
                   v3(std::fmax(p0.x, std::fmax(p1.x, p2.x)) + F32_EPS, std::fmax(p0.y, std::fmax(p1.y, p2.y)) + F32_EPS,
                      std::fmax(p0.z, std::fmax(p1.z, p2.z)) + F32_EPS)};
        return true;
    }
};

// hittable.rs:84-141
struct HittableList : Hittable {
    std::vector<HPtr> objects;
    bool is_list() const override { return true; }
    bool hit(const Ray& ray, float t_min, float t_max, Ctx& ctx, HitRecord& out) const override {
        float closest = t_max;
        bool any = false;
        HitRecord rec;
        for (const HPtr& o : objects) {
            if (o->hit(ray, t_min, closest, ctx, rec)) {
                closest = rec.t;
                out = rec;
                any = true;
            }
        }
        return any;
    }
    bool bounding_box(float t0, float t1, Aabb& out) const override {
        if (objects.empty()) return false;
        bool have = false;
        Aabb acc{};
        for (const HPtr& o : objects) {
            Aabb b;
            if (!o->bounding_box(t0, t1, b)) return false;
            acc = have ? aabb_union(acc, b) : b;
            have = true;
        }
        out = acc;
        return true;
    }
};

// geometry/cube.rs:23-97 — a HittableList of six rects: z-min, z-max, y-min, y-max, x-min, x-max
struct Cube : Hittable {
    V3 pmin, pmax;
    HittableList sides;
    void build(int material) {
        auto mk = [&](int axis, float a0, float a1, float b0, float b1, float k) {
            auto r = std::make_shared<Rect>();
            r->axis = axis; r->a0 = a0; r->a1 = a1; r->b0 = b0; r->b1 = b1; r->k = k; r->material = material; r->id = id;
            sides.objects.push_back(r);
        };
        mk(2, pmin.x, pmax.x, pmin.y, pmax.y, pmin.z);
        mk(2, pmin.x, pmax.x, pmin.y, pmax.y, pmax.z);
        mk(1, pmin.x, pmax.x, pmin.z, pmax.z, pmin.y);
        mk(1, pmin.x, pmax.x, pmin.z, pmax.z, pmax.y);
        mk(0, pmin.y, pmax.y, pmin.z, pmax.z, pmin.x);
        mk(0, pmin.y, pmax.y, pmin.z, pmax.z, pmax.x);
    }
    bool hit(const Ray& ray, float t_min, float t_max, Ctx& ctx, HitRecord& out) const override {
        // list semantics; record which side answered (face) for diagnostics
        float closest = t_max;
        bool any = false;
        HitRecord rec;
        for (int f = 0; f < 6; ++f) {
            if (sides.objects[f]->hit(ray, t_min, closest, ctx, rec)) {
                closest = rec.t;
                out = rec;
                out.face = f;
                any = true;
            }
        }
        return any;
    }
    bool bounding_box(float, float, Aabb& out) const override { out = Aabb{pmin, pmax}; return true; }
};

// geometry/instance.rs:14-52
struct Translate : Hittable {
    HPtr inner; V3 disp;
    bool hit(const Ray& ray, float t_min, float t_max, Ctx& ctx, HitRecord& out) const override {
        Ray moved{ray.origin - disp, ray.direction, ray.time};
        if (!inner->hit(moved, t_min, t_max, ctx, out)) return false;
        out.point = out.point + disp;
        return true;
    }
    bool bounding_box(float t0, float t1, Aabb& out) const override {
        Aabb b;
        if (!inner->bounding_box(t0, t1, b)) return false;
        out = Aabb{b.min + disp, b.max + disp};
        return true;
    }
};
// geometry/instance.rs:54-147 (bbox keeps the reference's `for c in 0..2` loop)
struct RotateY : Hittable {
    HPtr inner; float sin_t, cos_t; bool has_box = false; Aabb box{};
    void init(float degrees) {
        float radians = degrees * (PI_F / 180.0f);  // f32::to_radians
        sin_t = std::sin(radians);
        cos_t = std::cos(radians);
        Aabb b;
        if (inner->bounding_box(0.0f, 1.0f, b)) {
            V3 mn = v3(F32_INF, F32_INF, F32_INF), mx = v3(-F32_INF, -F32_INF, -F32_INF);
            for (int i = 0; i < 2; ++i) for (int j = 0; j < 2; ++j) for (int k = 0; k < 2; ++k) {
                float fi = (float)i, fj = (float)j, fk = (float)k;
                float x = fi * b.max.x + (1.0f - fi) * b.min.x;
                float y = fj * b.max.y + (1.0f - fj) * b.min.y;
                float z = fk * b.max.z + (1.0f - fk) * b.min.z;
                float nx = cos_t * x + sin_t * z;
                float nz = -sin_t * x + cos_t * z;
                V3 tester = v3(nx, y, nz);
                for (int c = 0; c < 2; ++c) {
                    mn.at(c) = std::fmin(mn[c], tester[c]);
                    mx.at(c) = std::fmax(mx[c], tester[c]);
                }
            }
            box = Aabb{mn, mx};
            has_box = true;
        }
    }
    V3 rot(V3 v) const { return v3(cos_t * v.x - sin_t * v.z, v.y, sin_t * v.x + cos_t * v.z); }
    bool hit(const Ray& ray, float t_min, float t_max, Ctx& ctx, HitRecord& out) const override {
        Ray rr{rot(ray.origin), rot(ray.direction), ray.time};
        if (!inner->hit(rr, t_min, t_max, ctx, out)) return false;
        V3 p = v3(cos_t * out.point.x + sin_t * out.point.z, out.point.y, -sin_t * out.point.x + cos_t * out.point.z);
        V3 n = v3(cos_t * out.normal.x + sin_t * out.normal.z, out.normal.y, -sin_t * out.normal.x + cos_t * out.normal.z);
        out.point = p;
        set_face_normal(out, rr, n);
        return true;
    }
    bool bounding_box(float, float, Aabb& out) const override { if (has_box) out = box; return has_box; }
};

// hittable.rs:143-238
struct ConstantMedium : Hittable {
    HPtr boundary; int phase_material; float neg_inv_density;
    bool hit(const Ray& ray, float t_min, float t_max, Ctx& ctx, HitRecord& out) const override {
        HitRecord h1, h2;
        if (!boundary->hit(ray, -F32_INF, F32_INF, ctx, h1)) return false;
        if (!boundary->hit(ray, h1.t + 0.0001f, F32_INF, ctx, h2)) return false;
        if (h1.t < t_min) h1.t = t_min;
        if (h2.t > t_max) h2.t = t_max;
        if (h1.t >= h2.t) return false;
        if (h1.t < 0.0f) h1.t = 0.0f;
        float ray_length = length(ray.direction);
        float dist_inside = (h2.t - h1.t) * ray_length;
        float hit_distance = neg_inv_density * std::log(ctx.rng->uniform01());
        if (hit_distance > dist_inside) return false;
        float t = h1.t + hit_distance / ray_length;
        HitRecord r;
        r.point = ray.at(t);
        r.normal = v3(1, 0, 0);
        r.t = t; r.u = 0; r.v = 0; r.front_face = true;
        r.material = phase_material;
        r.prim_id = id;
        out = r;
        return true;
    }
    bool bounding_box(float t0, float t1, Aabb& out) const override { return boundary->bounding_box(t0, t1, out); }
};

// ---------------------------------------------------------------------------
// hrpp.rs:33-83, 132-193
// ---------------------------------------------------------------------------
static uint16_t map_float_to_hash(float val) {
    uint32_t bits;
    std::memcpy(&bits, &val, 4);
    uint16_t sign = (uint16_t)(bits >> 31) & 0x1;
    uint16_t expo = (uint16_t)(bits >> 25) & 0x3f;   // BitPrecision::Six
    uint16_t mant = (uint16_t)(bits >> 17) & 0x3f;
    return (uint16_t)((sign << 15) | (expo << 7) | mant);
}
static uint64_t hrpp_hash(const Ray& ray) {
    uint64_t ox = map_float_to_hash(ray.origin.x), oy = map_float_to_hash(ray.origin.y), oz = map_float_to_hash(ray.origin.z);
    uint64_t dx = map_float_to_hash(ray.direction.x), dy = map_float_to_hash(ray.direction.y), dz = map_float_to_hash(ray.direction.z);
    uint64_t h0 = ox ^ dz, h1 = oy ^ dy, h2 = oz ^ dx;
    return (h0 << 0) | (h1 << 16) | (h2 << 32);
}
struct Predictor {
    std::mutex mtx;
    std::unordered_map<uint64_t, std::vector<int>> table;  // set semantics, insertion order
    uint32_t tp = 0, fp = 0, none = 0;
    bool get(const Ray& ray, std::vector<int>& out) {
        std::lock_guard<std::mutex> g(mtx);
        auto it = table.find(hrpp_hash(ray));
        if (it == table.end()) return false;
        out = it->second;  // the reference clones the set
        return true;
    }
    void insert(const Ray& ray, int node) {
        std::lock_guard<std::mutex> g(mtx);
        auto& v = table[hrpp_hash(ray)];
        if (std::find(v.begin(), v.end(), node) == v.end()) v.push_back(node);
    }
};

// ---------------------------------------------------------------------------
// bvh.rs:31-440
// ---------------------------------------------------------------------------
struct BvhChild { int index = -1; HPtr hittable; };
struct BvhNode { int parent = -1; int idx = 0; BvhChild left, right; Aabb box; };

static int total_cmp(float a, float b) {  // f32::total_cmp
    int32_t l, r;
    std::memcpy(&l, &a, 4); std::memcpy(&r, &b, 4);
    l ^= (int32_t)(((uint32_t)(l >> 31)) >> 1);
    r ^= (int32_t)(((uint32_t)(r >> 31)) >> 1);
    return l < r ? -1 : (l > r ? 1 : 0);
}

struct Bvh : Hittable {
    std::vector<BvhNode> nodes;
    int root = -1;
    uint32_t max_depth = 0;
    std::shared_ptr<Predictor> predictor;  // Bvh::with_predictor
    uint64_t axis_state = 0;

    int next_axis() { return (int)(splitmix64(axis_state) % 3ull); }  // stands in for rng.gen_range(0..=2)

    static int box_compare(const HPtr& a, const HPtr& b, int axis) {
        Aabb ba, bb;
        a->bounding_box(0.0f, 0.0f, ba); b->bounding_box(0.0f, 0.0f, bb);
        return total_cmp(ba.min[axis], bb.min[axis]);
    }
    int build(HPtr* objs, size_t n, float t0, float t1) {
        int axis = next_axis();
        BvhChild left, right;
        if (n == 1) {
            left.hittable = objs[0]; right.hittable = objs[0];
        } else if (n == 2) {
            if (box_compare(objs[0], objs[1], axis) < 0) { left.hittable = objs[0]; right.hittable = objs[1]; }
            else { left.hittable = objs[1]; right.hittable = objs[0]; }
        } else {
            std::stable_sort(objs, objs + n, [axis](const HPtr& a, const HPtr& b) { return box_compare(a, b, axis) < 0; });
            size_t mid = n / 2;
            left.index = build(objs, mid, t0, t1);
            right.index = build(objs + mid, n - mid, t0, t1);
        }
        Aabb lb, rb;
        if (left.index >= 0) lb = nodes[left.index].box; else left.hittable->bounding_box(t0, t1, lb);
        if (right.index >= 0) rb = nodes[right.index].box; else right.hittable->bounding_box(t0, t1, rb);
        BvhNode node;
        node.box = aabb_union(lb, rb);
        node.idx = (int)nodes.size();
        if (left.index >= 0) nodes[left.index].parent = node.idx;
        if (right.index >= 0) nodes[right.index].parent = node.idx;
        node.left = left; node.right = right;
        nodes.push_back(node);
        return node.idx;
    }
    uint32_t depth_of(int i) const {
        const BvhNode& n = nodes[i];
        uint32_t l = n.left.index >= 0 ? depth_of(n.left.index) : 0;
        uint32_t r = n.right.index >= 0 ? depth_of(n.right.index) : 0;
        return (l > r ? l : r) + 1;
    }
    // BvhNode::hit, bvh.rs:363-417
    bool node_hit(int ni, const Ray& ray, float t_min, float t_max, Ctx& ctx, HitRecord& out, int& leaf) const {
        const BvhNode& n = nodes[ni];
        ctx.cnt.node_visits++;
        if (!n.box.hit(ray, t_min, t_max)) return false;
        HitRecord hl, hr;
        int ll = -1, lr = -1;
        bool got_l, got_r;
        if (n.left.index >= 0) got_l = node_hit(n.left.index, ray, t_min, t_max, ctx, hl, ll);
        else { got_l = n.left.hittable->hit(ray, t_min, t_max, ctx, hl); ll = n.idx; }
        float t_max_right = got_l ? hl.t : t_max;
        if (n.right.index >= 0) got_r = node_hit(n.right.index, ray, t_min, t_max, ctx, hr, lr);
        else { got_r = n.right.hittable->hit(ray, t_min, t_max_right, ctx, hr); lr = n.idx; }
        if (!got_l && !got_r) return false;
        if (got_l && !got_r) { out = hl; leaf = ll; return true; }
        if (!got_l && got_r) { out = hr; leaf = lr; return true; }
        if (hl.t < hr.t) { out = hl; leaf = ll; } else { out = hr; leaf = lr; }
        return true;
    }
    // Bvh::hit, bvh.rs:107-218 (GO_UP_LEVEL = 0)
    bool hit(const Ray& ray, float t_min, float t_max, Ctx& ctx, HitRecord& out) const override {
        int leaf = -1;
        if (predictor && ctx.use_predictors) {
            std::vector<int> pred;
            if (predictor->get(ray, pred)) {
                float closest = t_max;
                bool any = false;
                HitRecord rec; int lf;
                for (int ni : pred) {
                    if (node_hit(ni, ray, t_min, closest, ctx, rec, lf)) { closest = rec.t; out = rec; any = true; }
                }
                if (any) { ctx.cnt.hrpp_tp++; return true; }
                ctx.cnt.hrpp_fp++;
                if (!node_hit(root, ray, t_min, t_max, ctx, out, leaf)) return false;
                predictor->insert(ray, leaf);
                return true;
            }
            ctx.cnt.hrpp_none++;
            if (!node_hit(root, ray, t_min, t_max, ctx, out, leaf)) return false;
            predictor->insert(ray, leaf);
            return true;
        }
        return node_hit(root, ray, t_min, t_max, ctx, out, leaf);
    }
    bool bounding_box(float, float, Aabb& out) const override { out = nodes[root].box; return true; }
};

// ---------------------------------------------------------------------------
// Scene container (the oracle's side of the builder vocabulary)
// ---------------------------------------------------------------------------
struct Scene {
    std::vector<Texture> textures;
    std::vector<Material> materials;
    std::vector<HPtr> hittables;
    HittableList world;
    std::string err;

    V3 tex_value(int ti, float u, float v, V3 p) const {
        const Texture& t = textures[ti];
        switch (t.kind) {
        case TEX_SOLID: return t.color;
        case TEX_CHECKER: {  // checker.rs:27-37
            float sines = std::sin(t.scale * p.x) * std::sin(t.scale * p.y) * std::sin(t.scale * p.z);
            return sign_negative(sines) ? tex_value(t.odd, u, v, p) : tex_value(t.even, u, v, p);
        }
        case TEX_MARBLE: {   // marble.rs:23-29
            float n = (float)t.turb->get((double)p.x, (double)p.y, (double)p.z);
            return v3(1, 1, 1) * 0.5f * (1.0f + std::sin(t.scale * p.z + 10.0f * n));
        }
        default: {           // image_texture.rs:21-52
            float uu = std::fmin(std::fmax(u, 0.0f), 1.0f);
            float vv = std::fmin(std::fmax(v, 0.0f), 1.0f);
            vv = 1.0f - vv;
            uint32_t i = (uint32_t)(uu * (float)t.w), j = (uint32_t)(vv * (float)t.h);
            if (i >= t.w) i = t.w - 1;
            if (j >= t.h) j = t.h - 1;
            const uint8_t* px = &t.rgb[((size_t)j * t.w + i) * 3];
            const float s = 1.0f / 255.0f;
            return v3((float)px[0] * s, (float)px[1] * s, (float)px[2] * s);
        }
        }
    }
    V3 emit(int mi, float u, float v, V3 p) const {
        const Material& m = materials[mi];
        if (m.kind == MAT_DIFFUSE_LIGHT) return tex_value(m.tex, u, v, p);
        return v3(0, 0, 0);
    }
    static float reflectance(float cosine, float ref_idx) {
        float r0 = (1.0f - ref_idx) / (1.0f + ref_idx);
        r0 = r0 * r0;
        float x = 1.0f - cosine;
        float x2 = x * x;
        return r0 + (1.0f - r0) * (x * (x2 * x2));  // powi(5) as llvm expands it
    }
    bool scatter(int mi, const Ray& ray, const HitRecord& rec, Rng& rng, V3& att, Ray& out) const {
        const Material& m = materials[mi];
        switch (m.kind) {
        case MAT_LAMBERTIAN: {  // lambertian.rs:35-52
            V3 dir = rec.normal + random_unit_vector(rng);
            if (near_zero(dir)) dir = rec.normal;
            out = Ray{rec.point, dir, ray.time};
            att = tex_value(m.tex, rec.u, rec.v, rec.point);
            return true;
        }
        case MAT_METAL: {       // metal.rs:26-42
            V3 reflected = reflect(normalize(ray.direction), rec.normal);
            out = Ray{rec.point, reflected + m.fuzz * random_in_unit_sphere(rng), ray.time};
            att = m.albedo;
            return dot(out.direction, rec.normal) > 0.0f;
        }
        case MAT_DIELECTRIC: {  // dialectric.rs:33-60
            att = v3(1, 1, 1);
            float ratio = rec.front_face ? 1.0f / m.ior : m.ior;
            V3 unit = normalize(ray.direction);
            float cos_theta = std::fmin(dot(-unit, rec.normal), 1.0f);
            float sin_theta = std::sqrt(1.0f - cos_theta * cos_theta);
            bool cannot = ratio * sin_theta > 1.0f;
            V3 dir;
            if (cannot || reflectance(cos_theta, ratio) > rng.uniform01()) dir = reflect(unit, rec.normal);
            else dir = refract(unit, rec.normal, ratio);
            out = Ray{rec.point, dir, ray.time};
            return true;
        }
        case MAT_DIFFUSE_LIGHT: return false;  // diffuse_light.rs:25-37
        default: {              // isotropic.rs:32-42
            out = Ray{rec.point, random_in_unit_sphere(rng), ray.time};
            att = tex_value(m.tex, rec.u, rec.v, rec.point);
            return true;
        }
        }
    }
};

// ---------------------------------------------------------------------------
// camera.rs:44-106
// ---------------------------------------------------------------------------
struct Camera {
    V3 origin, horizontal, vertical, llc, u, v;
    float lens_radius, time0, time1;
    void init(V3 from, V3 at, V3 vup, float vfov, float aspect, float aperture, float focus, float t0, float t1) {
        float theta = vfov * (PI_F / 180.0f);
        float h = std::tan(theta / 2.0f);
        float vh = 2.0f * h, vw = aspect * vh;
        V3 w = normalize(from - at);
        u = normalize(cross(vup, w));
        v = cross(w, u);
        origin = from;
        horizontal = focus * vw * u;
        vertical = focus * vh * v;
        llc = origin - horizontal / 2.0f - vertical / 2.0f - focus * w;
        lens_radius = aperture / 2.0f;
        time0 = t0; time1 = t1;
    }
    Ray get_ray(float s, float t, Rng& rng) const {
        V3 rd = lens_radius * random_in_unit_disk(rng);
        V3 offset = u * rd.x + v * rd.y;
        float time = rng.range(time0, time1);  // gen_range(t0..=t1); see DESIGN.md on the closed end
        return Ray{origin + offset, llc + s * horizontal + t * vertical - origin - offset, time};
    }
};

// ---------------------------------------------------------------------------
// ray.rs:32-62 — recursive, as written; plus the iterative equivalent the
// wavefront uses (same samples, association of the products differs).
// ---------------------------------------------------------------------------
static V3 ray_color_recursive(const Scene& sc, const Ray& ray, uint32_t depth, uint32_t max_depth, V3 background, Rng& rng, Ctx& ctx) {
    if (depth == 0) return v3(0, 0, 0);
    uint32_t bounce = max_depth - depth;
    HitRecord rec;
    rng.key(bounce, STAGE_INTERSECT);
    ctx.cnt.rays++;
    if (sc.world.hit(ray, 0.001f, F32_INF, ctx, rec)) {
        V3 emitted = sc.emit(rec.material, rec.u, rec.v, rec.point);
        V3 att; Ray next;
        rng.key(bounce, STAGE_SCATTER);
        if (sc.scatter(rec.material, ray, rec, rng, att, next))
            return emitted + att * ray_color_recursive(sc, next, depth - 1, max_depth, background, rng, ctx);
        return emitted;
    }
    return background;
}
static V3 ray_color_iterative(const Scene& sc, Ray ray, uint32_t max_depth, V3 background, Rng& rng, Ctx& ctx) {
    V3 L = v3(0, 0, 0), thr = v3(1, 1, 1);
    for (uint32_t bounce = 0; bounce < max_depth; ++bounce) {
        HitRecord rec;
        rng.key(bounce, STAGE_INTERSECT);
        ctx.cnt.rays++;
        if (!sc.world.hit(ray, 0.001f, F32_INF, ctx, rec)) { L = L + thr * background; break; }
        V3 emitted = sc.emit(rec.material, rec.u, rec.v, rec.point);
        L = L + thr * emitted;
        V3 att; Ray next;
        rng.key(bounce, STAGE_SCATTER);
        if (!sc.scatter(rec.material, ray, rec, rng, att, next)) break;
        thr = thr * att;
        ray = next;
    }
    return L;
}

// renderer.rs:242-296
struct Tile { int width, height, x0, y0; };
static std::vector<Tile> tile_layout(int W, int H, int tw, int th) {
    int nx = W / tw, rx = W % tw, ny = H / th, ry = H % th;
    std::vector<Tile> tiles;
    for (int ty = 0; ty < ny; ++ty) {
        for (int tx = 0; tx < nx; ++tx) tiles.push_back({tw, th, tx * tw, ty * th});
        if (rx > 0) tiles.push_back({rx, th, nx * tw, ty * th});
    }
    if (ry > 0) for (int tx = 0; tx < nx; ++tx) tiles.push_back({tw, ry, tx * tw, ny * th});
    if (rx > 0 && ry > 0) tiles.push_back({rx, ry, nx * tw, ny * th});
    return tiles;
}

}  // namespace orc

// ===========================================================================
// C API (ctypes).  Same builder vocabulary and id semantics as include/shimmer_b200.h
// so one Python scene description drives both.
// ===========================================================================
using namespace orc;

#define ORC_API extern "C" __attribute__((visibility("default")))

static thread_local std::string g_err;
static thread_local Counters g_last;
static int fail(const std::string& m) { g_err = m; return -1; }

ORC_API const char* orc_last_error() { return g_err.c_str(); }
ORC_API void* orc_scene_create() { return new Scene(); }
ORC_API void orc_scene_destroy(void* s) { delete (Scene*)s; }

static bool ok_tex(Scene* s, int t) { return t >= 0 && t < (int)s->textures.size(); }
static bool ok_mat(Scene* s, int m) { return m >= 0 && m < (int)s->materials.size(); }
static bool ok_hit(Scene* s, int h) { return h >= 0 && h < (int)s->hittables.size(); }

ORC_API int orc_texture_solid(void* sp, float r, float g, float b) {
    Scene* s = (Scene*)sp; Texture t; t.kind = TEX_SOLID; t.color = v3(r, g, b);
    s->textures.push_back(t); return (int)s->textures.size() - 1;
}
ORC_API int orc_texture_checker(void* sp, float scale, int even, int odd) {
    Scene* s = (Scene*)sp; if (!ok_tex(s, even) || !ok_tex(s, odd)) return fail("bad texture id");
    Texture t; t.kind = TEX_CHECKER; t.scale = scale; t.even = even; t.odd = odd;
    s->textures.push_back(t); return (int)s->textures.size() - 1;
}
ORC_API int orc_texture_marble(void* sp, float scale, uint32_t seed) {
    Scene* s = (Scene*)sp; Texture t; t.kind = TEX_MARBLE; t.scale = scale;
    t.turb = std::make_shared<Turbulence>(); t.turb->init(seed);
    s->textures.push_back(t); return (int)s->textures.size() - 1;
}
ORC_API int orc_texture_image(void* sp, const uint8_t* rgb, int w, int h) {
    Scene* s = (Scene*)sp; if (!rgb || w <= 0 || h <= 0) return fail("bad image");
    Texture t; t.kind = TEX_IMAGE; t.w = (uint32_t)w; t.h = (uint32_t)h; t.rgb.assign(rgb, rgb + (size_t)w * h * 3);
    s->textures.push_back(t); return (int)s->textures.size() - 1;
}
static int push_mat(Scene* s, const Material& m) { s->materials.push_back(m); return (int)s->materials.size() - 1; }
ORC_API int orc_material_lambertian(void* sp, int tex) {
    Scene* s = (Scene*)sp; if (!ok_tex(s, tex)) return fail("bad texture id");
    Material m; m.kind = MAT_LAMBERTIAN; m.tex = tex; return push_mat(s, m);
}
ORC_API int orc_material_metal(void* sp, float r, float g, float b, float fuzz) {
    Scene* s = (Scene*)sp; Material m; m.kind = MAT_METAL; m.albedo = v3(r, g, b);
    m.fuzz = fuzz < 0.0f ? 0.0f : (fuzz > 1.0f ? 1.0f : fuzz);  // metal.rs:17-22
    return push_mat(s, m);
}
ORC_API int orc_material_dielectric(void* sp, float ior) {
    Scene* s = (Scene*)sp; Material m; m.kind = MAT_DIELECTRIC; m.ior = ior; return push_mat(s, m);
}
ORC_API int orc_material_diffuse_light(void* sp, int tex) {
    Scene* s = (Scene*)sp; if (!ok_tex(s, tex)) return fail("bad texture id");
    Material m; m.kind = MAT_DIFFUSE_LIGHT; m.tex = tex; return push_mat(s, m);
}
ORC_API int orc_material_isotropic(void* sp, int tex) {
    Scene* s = (Scene*)sp; if (!ok_tex(s, tex)) return fail("bad texture id");
    Material m; m.kind = MAT_ISOTROPIC; m.tex = tex; return push_mat(s, m);
}
static int push_hit(Scene* s, HPtr h) { h->id = (int)s->hittables.size(); s->hittables.push_back(h); return h->id; }
ORC_API int orc_sphere(void* sp, float cx, float cy, float cz, float r, int mat) {
    Scene* s = (Scene*)sp; if (!ok_mat(s, mat)) return fail("bad material id");
    auto h = std::make_shared<Sphere>(); h->center = v3(cx, cy, cz); h->radius = r; h->material = mat; return push_hit(s, h);
}
ORC_API int orc_moving_sphere(void* sp, float c0x, float c0y, float c0z, float c1x, float c1y, float c1z,
                              float t0, float t1, float r, int mat) {
    Scene* s = (Scene*)sp; if (!ok_mat(s, mat)) return fail("bad material id");
    auto h = std::make_shared<MovingSphere>(); h->c0 = v3(c0x, c0y, c0z); h->c1 = v3(c1x, c1y, c1z);
    h->time0 = t0; h->time1 = t1; h->radius = r; h->material = mat; return push_hit(s, h);
}
static int add_rect(Scene* s, int axis, float a0, float a1, float b0, float b1, float k, int mat) {
    if (!ok_mat(s, mat)) return fail("bad material id");
    auto h = std::make_shared<Rect>(); h->axis = axis; h->a0 = a0; h->a1 = a1; h->b0 = b0; h->b1 = b1; h->k = k; h->material = mat;
    return push_hit(s, h);
}
ORC_API int orc_xy_rect(void* sp, float x0, float x1, float y0, float y1, float k, int mat) { return add_rect((Scene*)sp, 2, x0, x1, y0, y1, k, mat); }
ORC_API int orc_xz_rect(void* sp, float x0, float x1, float z0, float z1, float k, int mat) { return add_rect((Scene*)sp, 1, x0, x1, z0, z1, k, mat); }
ORC_API int orc_yz_rect(void* sp, float y0, float y1, float z0, float z1, float k, int mat) { return add_rect((Scene*)sp, 0, y0, y1, z0, z1, k, mat); }
ORC_API int orc_tri(void* sp, const float* p, int mat) {
    Scene* s = (Scene*)sp; if (!ok_mat(s, mat)) return fail("bad material id");
    auto h = std::make_shared<Tri>(); h->p0 = v3(p[0], p[1], p[2]); h->p1 = v3(p[3], p[4], p[5]); h->p2 = v3(p[6], p[7], p[8]); h->material = mat;
    return push_hit(s, h);
}
ORC_API int orc_list_create(void* sp) { Scene* s = (Scene*)sp; return push_hit(s, std::make_shared<HittableList>()); }
ORC_API int orc_list_add(void* sp, int list, int h) {
    Scene* s = (Scene*)sp; if (!ok_hit(s, list) || !ok_hit(s, h) || !s->hittables[list]->is_list()) return fail("bad list/hittable id");
    static_cast<HittableList*>(s->hittables[list].get())->objects.push_back(s->hittables[h]); return 0;
}
ORC_API int orc_tris_bulk(void* sp, const float* xyz, int n, int mat, int list) {
    Scene* s = (Scene*)sp; int first = -1;
    for (int i = 0; i < n; ++i) {
        int id = orc_tri(sp, xyz + (size_t)i * 9, mat); if (id < 0) return id;
        if (i == 0) first = id;
        if (orc_list_add(sp, list, id) < 0) return -1;
    }
    (void)s; return first;
}
ORC_API int orc_cube(void* sp, float x0, float y0, float z0, float x1, float y1, float z1, int mat) {
    Scene* s = (Scene*)sp; if (!ok_mat(s, mat)) return fail("bad material id");
    auto h = std::make_shared<Cube>(); h->pmin = v3(x0, y0, z0); h->pmax = v3(x1, y1, z1);
    int id = push_hit(s, h); h->build(mat); return id;
}
ORC_API int orc_bvh(void* sp, int list, float t0, float t1, uint64_t seed, int with_predictor) {
    Scene* s = (Scene*)sp; if (!ok_hit(s, list) || !s->hittables[list]->is_list()) return fail("bvh needs a list");
    auto* l = static_cast<HittableList*>(s->hittables[list].get());
    if (l->objects.empty()) return fail("bvh over an empty list");
    auto h = std::make_shared<Bvh>();
    h->axis_state = seed;
    std::vector<HPtr> objs = l->objects;  // Bvh::new consumes the list
    h->nodes.reserve(objs.size() * 2 + 1);
    h->root = h->build(objs.data(), objs.size(), t0, t1);
    h->max_depth = h->depth_of(h->root);
    if (with_predictor) h->predictor = std::make_shared<Predictor>();
    return push_hit(s, h);
}
ORC_API int orc_translate(void* sp, int h, float dx, float dy, float dz) {
    Scene* s = (Scene*)sp; if (!ok_hit(s, h)) return fail("bad hittable id");
    auto t = std::make_shared<Translate>(); t->inner = s->hittables[h]; t->disp = v3(dx, dy, dz); return push_hit(s, t);
}
ORC_API int orc_rotate_y(void* sp, int h, float degrees) {
    Scene* s = (Scene*)sp; if (!ok_hit(s, h)) return fail("bad hittable id");
    auto r = std::make_shared<RotateY>(); r->inner = s->hittables[h]; r->init(degrees); return push_hit(s, r);
}
ORC_API int orc_constant_medium(void* sp, int boundary, float density, int tex) {
    Scene* s = (Scene*)sp; if (!ok_hit(s, boundary) || !ok_tex(s, tex)) return fail("bad id");
    Material m; m.kind = MAT_ISOTROPIC; m.tex = tex; int pm = push_mat(s, m);
    auto c = std::make_shared<ConstantMedium>(); c->boundary = s->hittables[boundary]; c->phase_material = pm;
    c->neg_inv_density = -1.0f / density; return push_hit(s, c);
}
ORC_API int orc_world_add(void* sp, int h) {
    Scene* s = (Scene*)sp; if (!ok_hit(s, h)) return fail("bad hittable id");
    s->world.objects.push_back(s->hittables[h]); return 0;
}
ORC_API int orc_commit(void*) { return 0; }

// ---- introspection used by tests -------------------------------------------------------
ORC_API int orc_bvh_info(void* sp, int h, int* n_nodes, int* root, int* height) {
    Scene* s = (Scene*)sp; if (!ok_hit(s, h)) return fail("bad hittable id");
    Bvh* b = dynamic_cast<Bvh*>(s->hittables[h].get()); if (!b) return fail("not a bvh");
    *n_nodes = (int)b->nodes.size(); *root = b->root; *height = (int)b->max_depth; return 0;
}
// per node: left, right (>=0 node index, <0 ~hittable id), parent, and the 6 box floats
ORC_API int orc_bvh_nodes(void* sp, int h, int* left, int* right, int* parent, float* boxes) {
    Scene* s = (Scene*)sp; if (!ok_hit(s, h)) return fail("bad hittable id");
    Bvh* b = dynamic_cast<Bvh*>(s->hittables[h].get()); if (!b) return fail("not a bvh");
    for (size_t i = 0; i < b->nodes.size(); ++i) {
        const BvhNode& n = b->nodes[i];
        left[i] = n.left.index >= 0 ? n.left.index : ~n.left.hittable->id;
        right[i] = n.right.index >= 0 ? n.right.index : ~n.right.hittable->id;
        parent[i] = n.parent;
        const float bx[6] = {n.box.min.x, n.box.min.y, n.box.min.z, n.box.max.x, n.box.max.y, n.box.max.z};
        std::memcpy(boxes + i * 6, bx, sizeof bx);
    }
    return 0;
}

// ---- known-answer helpers ---------------------------------------------------------------
ORC_API int orc_aabb_hit(const float* mn, const float* mx, const float* o, const float* d, float t_min, float t_max) {
    Aabb b{v3(mn[0], mn[1], mn[2]), v3(mx[0], mx[1], mx[2])};
    Ray r{v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2]), 0.0f};
    return b.hit(r, t_min, t_max) ? 1 : 0;
}
ORC_API void orc_aabb_union(const float* a, const float* b, float* out) {
    Aabb r = aabb_union(Aabb{v3(a[0], a[1], a[2]), v3(a[3], a[4], a[5])}, Aabb{v3(b[0], b[1], b[2]), v3(b[3], b[4], b[5])});
    out[0] = r.min.x; out[1] = r.min.y; out[2] = r.min.z; out[3] = r.max.x; out[4] = r.max.y; out[5] = r.max.z;
}
ORC_API int orc_tile_layout(int W, int H, int tw, int th, int* out, int cap) {
    auto t = tile_layout(W, H, tw, th);
    for (size_t i = 0; i < t.size() && (int)i < cap; ++i) {
        out[i * 4 + 0] = t[i].width; out[i * 4 + 1] = t[i].height; out[i * 4 + 2] = t[i].x0; out[i * 4 + 3] = t[i].y0;
    }
    return (int)t.size();
}
ORC_API void orc_sphere_uv(float x, float y, float z, float* uv) { sphere_uv(v3(x, y, z), uv[0], uv[1]); }
ORC_API uint32_t orc_map_float_to_hash(float v) { return map_float_to_hash(v); }
ORC_API uint64_t orc_hrpp_hash(const float* o, const float* d) {
    return hrpp_hash(Ray{v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2]), 0.0f});
}
ORC_API void orc_philox(const uint32_t* ctr, const uint32_t* key, uint32_t* out) {
    philox4x32_10(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1], out);
}
ORC_API void orc_camera_fields(const float* c, float* out) {
    Camera cam; cam.init(v3(c[0], c[1], c[2]), v3(c[3], c[4], c[5]), v3(c[6], c[7], c[8]), c[9], c[10], c[11], c[12], c[13], c[14]);
    const V3* f[6] = {&cam.origin, &cam.horizontal, &cam.vertical, &cam.llc, &cam.u, &cam.v};
    for (int i = 0; i < 6; ++i) { out[i * 3] = f[i]->x; out[i * 3 + 1] = f[i]->y; out[i * 3 + 2] = f[i]->z; }
    out[18] = cam.lens_radius; out[19] = cam.time0; out[20] = cam.time1;
}
ORC_API void orc_texture_value(void* sp, int tex, float u, float v, const float* p, float* out) {
    V3 c = ((Scene*)sp)->tex_value(tex, u, v, v3(p[0], p[1], p[2])); out[0] = c.x; out[1] = c.y; out[2] = c.z;
}

// ---- gate 1: closest hit on a ray batch -------------------------------------------------
// rays: N x 7 (origin, direction, time).  Medium draws use the stream keyed
// (pixel = ray index, sample = 0, bounce 0, STAGE_INTERSECT) under `seed`.
// counters (optional, 3 x u64): rays, node visits, primitive tests.
ORC_API int orc_trace_closest(void* sp, const float* rays, int64_t n, float t_min, float t_max, uint64_t seed,
                              int use_predictors, int32_t* prim_id, float* t_out, uint64_t* counters) {
    Scene* s = (Scene*)sp;
    Ctx ctx; ctx.scene = s; ctx.use_predictors = use_predictors != 0;
    for (int64_t i = 0; i < n; ++i) {
        const float* r = rays + i * 7;
        Ray ray{v3(r[0], r[1], r[2]), v3(r[3], r[4], r[5]), r[6]};
        Rng rng; rng.keyed = true; rng.pixel = (uint32_t)i; rng.sample = 0; rng.k0 = (uint32_t)seed; rng.k1 = (uint32_t)(seed >> 32);
        rng.key(0, STAGE_INTERSECT);
        ctx.rng = &rng;
        HitRecord rec;
        ctx.cnt.rays++;
        if (s->world.hit(ray, t_min, t_max, ctx, rec)) { prim_id[i] = rec.prim_id; t_out[i] = rec.t; }
        else { prim_id[i] = -1; t_out[i] = F32_INF; }
    }
    if (counters) { counters[0] = ctx.cnt.rays; counters[1] = ctx.cnt.node_visits; counters[2] = ctx.cnt.prim_tests; }
    return 0;
}

// world.hit for each ray with the whole record, the stream keyed as in orc_trace_closest.  out: 12 words per ray in the
// layout of shim_hit_record: point[3], normal[3], t, u, v (f32), front_face, material, hittable id (i32).
// A miss: t = +inf, material = hittable = -1, everything else 0.  counters as in orc_trace_closest.
ORC_API int orc_trace_record(void* sp, const float* rays, int64_t n, float t_min, float t_max, uint64_t seed, uint32_t* out,
                             uint64_t* counters) {
    Scene* s = (Scene*)sp;
    Ctx ctx; ctx.scene = s;
    for (int64_t i = 0; i < n; ++i) {
        const float* r = rays + i * 7;
        Ray ray{v3(r[0], r[1], r[2]), v3(r[3], r[4], r[5]), r[6]};
        Rng rng; rng.keyed = true; rng.pixel = (uint32_t)i; rng.sample = 0; rng.k0 = (uint32_t)seed; rng.k1 = (uint32_t)(seed >> 32);
        rng.key(0, STAGE_INTERSECT);
        ctx.rng = &rng;
        HitRecord rec;
        ctx.cnt.rays++;
        float f[9] = {0, 0, 0, 0, 0, 0, F32_INF, 0, 0};
        int32_t w[3] = {0, -1, -1};
        if (s->world.hit(ray, t_min, t_max, ctx, rec)) {
            float g[9] = {rec.point.x, rec.point.y, rec.point.z, rec.normal.x, rec.normal.y, rec.normal.z, rec.t, rec.u, rec.v};
            memcpy(f, g, sizeof f);
            w[0] = rec.front_face ? 1 : 0; w[1] = rec.material; w[2] = rec.prim_id;
        }
        memcpy(out + i * 12, f, sizeof f);
        memcpy(out + i * 12 + 9, w, sizeof w);
    }
    if (counters) { counters[0] = ctx.cnt.rays; counters[1] = ctx.cnt.node_visits; counters[2] = ctx.cnt.prim_tests; }
    return 0;
}

// ---- render --------------------------------------------------------------------------------
struct OrcRenderParams {
    int32_t width, height, spp, max_depth, tile_w, tile_h;
    float background[3];
    uint64_t seed;
    int32_t sample_begin;   // first absolute sample index (sample-range sharding)
    int32_t sample_count;   // samples rendered per pixel by this call (0 = spp)
    int32_t rng_fast;       // 0 = keyed Philox (parity), 1 = xorshift (CPU baseline timing)
    int32_t iterative;      // 0 = recursion as in ray.rs, 1 = iterative equivalent
    int32_t threads;        // 0 = hardware_concurrency
    int32_t use_predictors; // predictors Some / None
    int32_t raw_sum;        // 1 = leave per-pixel sums (no division by spp)
};
struct OrcStats { uint64_t rays, samples, node_visits, prim_tests, hrpp_tp, hrpp_fp, hrpp_none; double seconds; int32_t threads; };

// One sample of one pixel (renderer.rs:140-146), exposed for per-sample parity checks.
static V3 sample_radiance(const Scene& sc, const Camera& cam, const OrcRenderParams& p, int x, int y, uint32_t sample, Rng& rng, Ctx& ctx) {
    if (rng.keyed) { rng.pixel = (uint32_t)(y * p.width + x); rng.sample = sample; rng.key(0, STAGE_CAMERA); }
    float u = ((float)x + rng.uniform01()) / (float)(p.width - 1);
    float v = ((float)y + rng.uniform01()) / (float)(p.height - 1);
    Ray ray = cam.get_ray(u, v, rng);
    V3 bg = v3(p.background[0], p.background[1], p.background[2]);
    ctx.rng = &rng;
    if (p.iterative) return ray_color_iterative(sc, ray, (uint32_t)p.max_depth, bg, rng, ctx);
    return ray_color_recursive(sc, ray, (uint32_t)p.max_depth, (uint32_t)p.max_depth, bg, rng, ctx);
}

ORC_API int orc_render(void* sp, const float* cam15, const OrcRenderParams* pp, float* out_rgb, OrcStats* stats) {
    Scene* s = (Scene*)sp;
    OrcRenderParams p = *pp;
    if (p.width < 2 || p.height < 2 || p.spp < 1 || p.tile_w < 1 || p.tile_h < 1) return fail("bad render params");
    Camera cam; cam.init(v3(cam15[0], cam15[1], cam15[2]), v3(cam15[3], cam15[4], cam15[5]), v3(cam15[6], cam15[7], cam15[8]),
                         cam15[9], cam15[10], cam15[11], cam15[12], cam15[13], cam15[14]);
    int count = p.sample_count > 0 ? p.sample_count : p.spp;
    std::vector<Tile> tiles = tile_layout(p.width, p.height, p.tile_w, p.tile_h);
    int nthreads = p.threads > 0 ? p.threads : (int)std::thread::hardware_concurrency();
    if (nthreads < 1) nthreads = 1;
    std::atomic<size_t> next{0};
    std::mutex stat_mtx;
    Counters total;
    auto t_start = std::chrono::steady_clock::now();
    auto worker = [&](int tid) {
        Ctx ctx; ctx.scene = s; ctx.use_predictors = p.use_predictors != 0;
        Rng rng; rng.keyed = !p.rng_fast; rng.k0 = (uint32_t)p.seed; rng.k1 = (uint32_t)(p.seed >> 32);
        rng.xs = 0x9E3779B9u * (uint32_t)(tid + 1) + (uint32_t)p.seed;
        for (;;) {
            size_t ti = next.fetch_add(1);
            if (ti >= tiles.size()) break;
            const Tile& tl = tiles[ti];
            for (int ty = 0; ty < tl.height; ++ty) for (int tx = 0; tx < tl.width; ++tx) {
                int x = tl.x0 + tx, y = tl.y0 + ty;
                V3 acc = v3(0, 0, 0);
                for (int k = 0; k < count; ++k) acc = acc + sample_radiance(*s, cam, p, x, y, (uint32_t)(p.sample_begin + k), rng, ctx);
                if (!p.raw_sum) acc = acc / (float)p.spp;
                float* o = out_rgb + ((size_t)y * p.width + x) * 3;
                o[0] = acc.x; o[1] = acc.y; o[2] = acc.z;
            }
        }
        std::lock_guard<std::mutex> g(stat_mtx);
        total.add(ctx.cnt);
    };
    std::vector<std::thread> pool;
    for (int i = 0; i < nthreads; ++i) pool.emplace_back(worker, i);
    for (auto& t : pool) t.join();
    double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
    if (stats) {
        stats->rays = total.rays; stats->samples = (uint64_t)p.width * p.height * count;
        stats->node_visits = total.node_visits; stats->prim_tests = total.prim_tests;
        stats->hrpp_tp = total.hrpp_tp; stats->hrpp_fp = total.hrpp_fp; stats->hrpp_none = total.hrpp_none;
        stats->seconds = secs; stats->threads = nthreads;
    }
    return 0;
}

// Per-sample radiance for a list of (x, y, sample) triples — used to compare the device
// path sample by sample.  Optionally records the rays traced along each path
// (origin, direction, time; 7 floats each) up to ray_cap, for the gate-1 batch.
ORC_API int orc_sample_radiance(void* sp, const float* cam15, const OrcRenderParams* pp, const int32_t* xys, int64_t n,
                                float* out_rgb, uint64_t* rays_out) {
    Scene* s = (Scene*)sp;
    OrcRenderParams p = *pp;
    Camera cam; cam.init(v3(cam15[0], cam15[1], cam15[2]), v3(cam15[3], cam15[4], cam15[5]), v3(cam15[6], cam15[7], cam15[8]),
                         cam15[9], cam15[10], cam15[11], cam15[12], cam15[13], cam15[14]);
    Ctx ctx; ctx.scene = s; ctx.use_predictors = p.use_predictors != 0;
    Rng rng; rng.keyed = true; rng.k0 = (uint32_t)p.seed; rng.k1 = (uint32_t)(p.seed >> 32);
    for (int64_t i = 0; i < n; ++i) {
        V3 c = sample_radiance(*s, cam, p, xys[i * 3], xys[i * 3 + 1], (uint32_t)xys[i * 3 + 2], rng, ctx);
        out_rgb[i * 3] = c.x; out_rgb[i * 3 + 1] = c.y; out_rgb[i * 3 + 2] = c.z;
    }
    if (rays_out) *rays_out = ctx.cnt.rays;
    g_last = ctx.cnt;
    return 0;
}
// counters of the calling thread's last orc_sample_radiance: rays, node visits, prim tests, hrpp tp / fp / none
ORC_API void orc_last_counters(uint64_t* out6) {
    out6[0] = g_last.rays; out6[1] = g_last.node_visits; out6[2] = g_last.prim_tests;
    out6[3] = g_last.hrpp_tp; out6[4] = g_last.hrpp_fp; out6[5] = g_last.hrpp_none;
}

// Records every ray the integrator traces (camera + bounce rays) for the given samples,
// iterative integrator; returns the number written (<= cap).  Gate-1 ray batches come from here.
ORC_API int64_t orc_record_path_rays(void* sp, const float* cam15, const OrcRenderParams* pp, const int32_t* xys, int64_t n,
                                     float* rays7, int64_t cap) {
    Scene* s = (Scene*)sp;
    OrcRenderParams p = *pp;
    Camera cam; cam.init(v3(cam15[0], cam15[1], cam15[2]), v3(cam15[3], cam15[4], cam15[5]), v3(cam15[6], cam15[7], cam15[8]),
                         cam15[9], cam15[10], cam15[11], cam15[12], cam15[13], cam15[14]);
    Ctx ctx; ctx.scene = s; ctx.use_predictors = false;
    Rng rng; rng.keyed = true; rng.k0 = (uint32_t)p.seed; rng.k1 = (uint32_t)(p.seed >> 32);
    int64_t w = 0;
    for (int64_t i = 0; i < n && w < cap; ++i) {
        int x = xys[i * 3], y = xys[i * 3 + 1];
        rng.pixel = (uint32_t)(y * p.width + x); rng.sample = (uint32_t)xys[i * 3 + 2]; rng.key(0, STAGE_CAMERA);
        float u = ((float)x + rng.uniform01()) / (float)(p.width - 1);
        float v = ((float)y + rng.uniform01()) / (float)(p.height - 1);
        Ray ray = cam.get_ray(u, v, rng);
        ctx.rng = &rng;
        for (uint32_t bounce = 0; bounce < (uint32_t)p.max_depth && w < cap; ++bounce) {
            float* o = rays7 + w * 7;
            o[0] = ray.origin.x; o[1] = ray.origin.y; o[2] = ray.origin.z;
            o[3] = ray.direction.x; o[4] = ray.direction.y; o[5] = ray.direction.z; o[6] = ray.time;
            ++w;
            HitRecord rec;
            rng.key(bounce, STAGE_INTERSECT);
            if (!s->world.hit(ray, 0.001f, F32_INF, ctx, rec)) break;
            V3 att; Ray next;
            rng.key(bounce, STAGE_SCATTER);
            if (!s->scatter(rec.material, ray, rec, rng, att, next)) break;
            ray = next;
        }
    }
    return w;
}

// HRPP table statistics of one BVH (hrpp.rs:85-130): entries, total leaves stored.
ORC_API int orc_predictor_stats(void* sp, int h, uint64_t* entries, uint64_t* leaves) {
    Scene* s = (Scene*)sp; if (!ok_hit(s, h)) return fail("bad hittable id");
    Bvh* b = dynamic_cast<Bvh*>(s->hittables[h].get()); if (!b || !b->predictor) return fail("no predictor");
    *entries = b->predictor->table.size(); uint64_t l = 0;
    for (auto& kv : b->predictor->table) l += kv.second.size();
    *leaves = l; return 0;
}
