// oracle.cpp — TEST INFRASTRUCTURE: CPU oracle for the per-pixel Monte Carlo sample loop
// of hatoo/raytracing-1w (master).  NEVER linked, imported or executed by the product
// (librt1w.so); only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
// `--impl reference` legs may load it.
//
// It restates the reference algorithm in C++17 with f64 arithmetic, recursion, per-node
// virtual dispatch, ref-counted material handles, one heap-allocated PDF per Lambertian
// bounce and a per-pixel RNG stream — the cost model of the Rust original — and doubles
// as the CPU baseline because the Rust crate cannot be built in this image (no rustc, no
// cargo, crates not vendored; SURVEY.md §8c).  Each function cites the reference
// file:line it follows (paths relative to /root/reference/src).
//
// PARITY STATUS: the reference has no tests, golden vectors or fixtures.  The oracle is
// pinned by (a) the known-answer table derived from the reference formulas (SURVEY.md §4,
// tests/test_oracle_known_answers.py) and (b) region means of the reference's published
// rest_of_your_life.png (tests/golden/rest_of_your_life_regions.json, made by
// tests/golden/make_reference_regions.py).  RNG bit streams are "parity unpinned"
// (see chacha_rng.hpp); image parity is statistical by construction.
#include "oracle.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <limits>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#ifdef _OPENMP
#include <omp.h>
#endif

#include "chacha_rng.hpp"

namespace oracle {

using Float = double; // main.rs:1
using MyRng = StdRng; // main.rs:2
static const Float PI = 3.14159265358979323846264338327950288;
static const Float INF = std::numeric_limits<Float>::infinity();

// ------------------------------------------------------------------ vectors (cgmath)
struct V3 {
    Float x, y, z;
    Float operator[](int i) const { return i == 0 ? x : (i == 1 ? y : z); }
    Float &at(int i) { return i == 0 ? x : (i == 1 ? y : z); }
};
static inline V3 v3(Float x, Float y, Float z) { return V3{x, y, z}; }
static inline V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
static inline V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
static inline V3 operator-(V3 a) { return {-a.x, -a.y, -a.z}; }
static inline V3 operator*(Float s, V3 a) { return {s * a.x, s * a.y, s * a.z}; }
static inline V3 operator*(V3 a, Float s) { return {a.x * s, a.y * s, a.z * s}; }
static inline V3 operator/(V3 a, Float s) { return {a.x / s, a.y / s, a.z / s}; }
static inline Float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static inline V3 cross(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
static inline Float magnitude2(V3 a) { return dot(a, a); }
static inline Float magnitude(V3 a) { return std::sqrt(dot(a, a)); }
static inline V3 normalize(V3 a) { return a * (1.0 / magnitude(a)); } // cgmath: self * (1/magnitude)
static inline V3 mul_element_wise(V3 a, V3 b) { return {a.x * b.x, a.y * b.y, a.z * b.z}; }

// ------------------------------------------------------------------ ray.rs:5-15
struct Ray {
    V3 origin, direction;
    Float time;
    V3 at(Float t) const { return origin + t * direction; }
};

// ------------------------------------------------------------------ aabb.rs
struct AABB {
    V3 minimum, maximum;
    bool hit(const Ray &ray, Float t_min, Float t_max) const { // aabb.rs:13-32
        for (int a = 0; a < 3; ++a) {
            Float inv_d = 1.0 / ray.direction[a];
            Float t0 = (minimum[a] - ray.origin[a]) * inv_d;
            Float t1 = (maximum[a] - ray.origin[a]) * inv_d;
            if (inv_d < 0.0) std::swap(t0, t1);
            t_min = t0 > t_min ? t0 : t_min;
            t_max = t1 < t_max ? t1 : t_max;
            if (t_max <= t_min) return false;
        }
        return true;
    }
};
// closed-interval variant used only by the tie sweep of oracle_trace_closest (not in the reference)
inline bool aabb_hit_closed(const AABB &b, const Ray &ray, Float t_min, Float t_max) {
    for (int a = 0; a < 3; ++a) {
        Float inv_d = 1.0 / ray.direction[a];
        Float t0 = (b.minimum[a] - ray.origin[a]) * inv_d, t1 = (b.maximum[a] - ray.origin[a]) * inv_d;
        if (inv_d < 0.0) std::swap(t0, t1);
        if (t0 > t_min) t_min = t0;
        if (t1 < t_max) t_max = t1;
        if (t_max < t_min) return false;
    }
    return true;
}
static AABB surrounding_box(AABB a, AABB b) { // aabb.rs:35-52
    return AABB{v3(std::fmin(a.minimum.x, b.minimum.x), std::fmin(a.minimum.y, b.minimum.y), std::fmin(a.minimum.z, b.minimum.z)),
                v3(std::fmax(a.maximum.x, b.maximum.x), std::fmax(a.maximum.y, b.maximum.y), std::fmax(a.maximum.z, b.maximum.z))};
}

// ------------------------------------------------------------------ onb.rs
struct Onb {
    V3 u, v, w;
    static Onb from_w(V3 n) { // onb.rs:13-24
        V3 w = normalize(n);
        V3 a = std::fabs(w.x) > 0.9 ? v3(0.0, 1.0, 0.0) : v3(1.0, 0.0, 0.0);
        V3 v = normalize(cross(w, a));
        V3 u = cross(w, v);
        return Onb{u, v, w};
    }
    V3 local(V3 a) const { return u * a.x + v * a.y + w * a.z; } // onb.rs:26-28
};

// ------------------------------------------------------------------ math.rs
static V3 random_in_unit_sphere(MyRng &rng) { // math.rs:6-18
    for (;;) {
        Float x = rng.gen_range(-1.0, 1.0), y = rng.gen_range(-1.0, 1.0), z = rng.gen_range(-1.0, 1.0);
        V3 v = v3(x, y, z);
        if (magnitude2(v) < 1.0) return v;
    }
}
static V3 random_in_unit_disk(MyRng &rng) { // math.rs:30-37
    for (;;) {
        Float x = rng.gen_range(-1.0, 1.0), y = rng.gen_range(-1.0, 1.0);
        V3 p = v3(x, y, 0.0);
        if (magnitude2(p) < 1.0) return p;
    }
}
static V3 random_cosine_direction(MyRng &rng) { // math.rs:39-49
    Float r1 = rng.gen_f64(), r2 = rng.gen_f64();
    Float z = std::sqrt(1.0 - r2);
    Float phi = 2.0 * PI * r1;
    return v3(std::cos(phi) * std::sqrt(r2), std::sin(phi) * std::sqrt(r2), z);
}
static V3 random_to_sphere(Float radius, Float distance_squared, MyRng &rng) { // math.rs:51-65
    Float r1 = rng.gen_f64(), r2 = rng.gen_f64();
    Float z = 1.0 + r2 * (std::sqrt(1.0 - radius * radius / distance_squared) - 1.0);
    Float phi = 2.0 * PI * r1;
    Float s = std::sqrt(1.0 - z * z);
    return v3(std::cos(phi) * s, std::sin(phi) * s, z);
}
static void sphere_uv(V3 p, Float &u, Float &v) { // math.rs:67-71
    Float theta = std::acos(-p.y);
    Float phi = std::atan2(-p.z, p.x) + PI;
    u = phi / (2.0 * PI), v = theta / PI;
}

// ------------------------------------------------------------------ perlin.rs
struct Perlin {
    V3 ranvec[256];
    int perm_x[256], perm_y[256], perm_z[256];
    static Float perlin_interp(const V3 c[2][2][2], Float u, Float v, Float w) { // perlin.rs:88-106
        Float uu = u * u * (3.0 - 2.0 * u), vv = v * v * (3.0 - 2.0 * v), ww = w * w * (3.0 - 2.0 * w);
        Float accum = 0.0;
        for (int i = 0; i < 2; ++i)
            for (int j = 0; j < 2; ++j)
                for (int k = 0; k < 2; ++k) {
                    V3 weight_v = v3(u - i, v - j, w - k);
                    accum += (i * uu + (1 - i) * (1.0 - uu)) * (j * vv + (1 - j) * (1.0 - vv)) * (k * ww + (1 - k) * (1.0 - ww)) *
                             dot(c[i][j][k], weight_v);
                }
        return accum;
    }
    Float noise(V3 p) const { // perlin.rs:46-72
        Float u = p.x - std::floor(p.x), v = p.y - std::floor(p.y), w = p.z - std::floor(p.z);
        long i = long(std::floor(p.x)), j = long(std::floor(p.y)), k = long(std::floor(p.z));
        V3 c[2][2][2];
        for (int di = 0; di < 2; ++di)
            for (int dj = 0; dj < 2; ++dj)
                for (int dk = 0; dk < 2; ++dk)
                    c[di][dj][dk] = ranvec[perm_x[(i + di) & 255] ^ perm_y[(j + dj) & 255] ^ perm_z[(k + dk) & 255]];
        return perlin_interp(c, u, v, w);
    }
    Float turb(V3 p, int depth) const { // perlin.rs:74-86
        Float accum = 0.0, weight = 1.0;
        V3 temp_p = p;
        for (int i = 0; i < depth; ++i) {
            accum += weight * noise(temp_p);
            weight *= 0.5;
            temp_p = temp_p * 2.0;
        }
        return std::fabs(accum);
    }
};

// ------------------------------------------------------------------ texture.rs
struct Texture {
    virtual ~Texture() = default;
    virtual V3 value(Float u, Float v, V3 p) const = 0;
};
struct SolidColor : Texture { // texture.rs:40-44
    V3 color_value;
    V3 value(Float, Float, V3) const override { return color_value; }
};
struct CheckerTexture : Texture { // texture.rs:46-55
    std::shared_ptr<Texture> odd, even;
    V3 value(Float u, Float v, V3 p) const override {
        Float sines = std::sin(10.0 * p.x) * std::sin(10.0 * p.y) * std::sin(10.0 * p.z);
        return sines < 0.0 ? odd->value(u, v, p) : even->value(u, v, p);
    }
};
struct NoiseTexture : Texture { // texture.rs:57-65
    std::shared_ptr<Perlin> perlin;
    Float scale;
    V3 value(Float, Float, V3 p) const override {
        return v3(1.0, 1.0, 1.0) * 0.5 * (1.0 + std::sin(scale * p.z + 10.0 * perlin->turb(p, 7)));
    }
};
struct PerlinTexture : Texture { // perlin.rs:109-113
    std::shared_ptr<Perlin> perlin;
    V3 value(Float, Float, V3 p) const override { return perlin->noise(p) * v3(1.0, 1.0, 1.0); }
};
struct ImageTexture : Texture { // texture.rs:67-89
    std::vector<uint8_t> rgb8;
    uint32_t width = 0, height = 0;
    V3 value(Float u, Float v, V3) const override {
        u = std::fmin(std::fmax(u, 0.0), 1.0);
        v = 1.0 - std::fmin(std::fmax(v, 0.0), 1.0);
        uint32_t i = uint32_t(u * Float(width)), j = uint32_t(v * Float(height));
        i = std::min(i, width - 1), j = std::min(j, height - 1);
        const uint8_t *px = &rgb8[(size_t(j) * width + i) * 3];
        const Float COLOR_SCALE = 1.0 / 255.0;
        return v3(px[0] * COLOR_SCALE, px[1] * COLOR_SCALE, px[2] * COLOR_SCALE);
    }
};

// ------------------------------------------------------------------ hittable.rs:10-47
struct Material;
using MaterialArc = std::shared_ptr<Material>; // Arc<Box<dyn Material>> (atomic refcount, hittable.rs:17)

struct HitRecord {
    V3 position, normal;
    Float t, u, v;
    bool front_face;
    MaterialArc material;
    int prim = -1; // leaf primitive id (not in the reference; parity bookkeeping only)
    static HitRecord make(V3 position, V3 outward_normal, Float t, Float u, Float v, const Ray &ray, MaterialArc material, int prim) {
        bool front_face = dot(ray.direction, outward_normal) < 0.0; // hittable.rs:30
        V3 normal = front_face ? outward_normal : -outward_normal;
        return HitRecord{position, normal, t, u, v, front_face, std::move(material), prim};
    }
};
using Hit = std::optional<HitRecord>;

struct PathReplay; // oracle_replay_paths: one path's Philox stream (below)

// per-thread context for the closest-hit parity replay (ConstantMedium free-flight draw)
struct TraceReplay {
    bool active = false;
    uint64_t seed = 0, ray_index = 0;
    PathReplay *path = nullptr; // non-null inside oracle_replay_paths: media draw from the path's own stream
    // tie bookkeeping (parity only): every leaf hit that was accepted at some point of the walk, and
    // whether a leaf rejected a candidate that lies within 1e-9 relative of the range end
    int n_cand = 0;
    int cand_prim[32];
    double cand_t[32];
    bool near_reject = false;
    void reset() { n_cand = 0, near_reject = false; }
    void accept(int prim, double t) {
        if (!active || prim < 0) return;
        if (n_cand < 32) cand_prim[n_cand] = prim, cand_t[n_cand] = t, ++n_cand;
        else near_reject = true;
    }
    void reject(int prim, double t, double t_min, double t_max) {
        if (!active || prim < 0) return;
        const double tol = 1e-9;
        if ((t > t_max && t <= t_max + tol * std::fmax(1.0, std::fabs(t_max))) || (t < t_min && t >= t_min - tol)) near_reject = true;
    }
};
static thread_local TraceReplay g_replay;

// One path of oracle_replay_paths: its Philox key and counter words (oracle.h: the draw map) and what the replay
// records about it.  `depth` is the depth of the ray being traced or scattered (0 = the camera ray).
struct PathReplay {
    uint32_t k0 = 0, k1 = 0; // pixel seed j*w+i, seed lo
    uint32_t s = 0, hi = 0;  // global sample index, seed hi
    uint32_t depth = 0;
    int mutation = 0;
    const int32_t *leaf_of_prim = nullptr; // device leaf index of each oracle primitive id (media only)
    int n_map = 0;
    uint32_t flags = 0;
    void block(uint32_t d, uint32_t purpose, uint32_t b, uint32_t out[4]) const {
        const uint32_t word = purpose ^ (mutation == 2 ? 0u : hi << 4);
        const uint32_t ctr[4] = {s, d, word, b}, key[2] = {k0, k1};
        philox4x32_10(ctr, key, out);
    }
};
static const uint32_t RNG_CAMERA = 0, RNG_SCATTER = 1, RNG_MEDIUM = 2;
static const uint32_t FLAG_HIT = 1, FLAG_DRAW = 2, FLAG_RANGE = 4;
static const double NEAR = 1e-4; // a draw decision this close to its threshold is flagged (FLAG_DRAW)
static inline float u01f(uint32_t x) { return float(x >> 8) * (1.0f / 16777216.0f); }
static inline void path_near(PathReplay &p, double value, double threshold) {
    if (std::fabs(value - threshold) <= NEAR * std::fmax(1.0, std::fabs(threshold))) p.flags |= FLAG_DRAW;
}
// free flight: counter (s, depth, RNG_MEDIUM, leaf index of the medium), u01 of the first word
static Float path_medium_xi(const PathReplay &p, int prim) {
    uint32_t block = uint32_t(prim);
    if (p.mutation != 5 && p.leaf_of_prim) {
        if (prim < 0 || prim >= p.n_map) throw std::runtime_error("medium primitive outside leaf_of_prim");
        block = uint32_t(p.leaf_of_prim[prim]);
    }
    uint32_t x[4];
    p.block(p.depth, RNG_MEDIUM, block, x);
    return Float(u01f(x[0]));
}
static void path_near_threshold(PathReplay &p, Float hit_distance, Float inside) {
    if (std::fabs(hit_distance - inside) <= NEAR * std::fmax(std::fabs(inside), 1e-3)) p.flags |= FLAG_DRAW;
}

struct Hittable { // hittable.rs:63-72
    virtual ~Hittable() = default;
    virtual Hit hit(const Ray &ray, Float t_min, Float t_max, MyRng &rng) const = 0;
    virtual AABB bounding_box(Float time0, Float time1) const = 0;
    virtual Float pdf_value(V3, V3, MyRng &) const { return 0.0; }
    virtual V3 random(V3, MyRng &) const { return v3(1.0, 0.0, 0.0); }
};
using HittableBox = std::unique_ptr<Hittable>;

// ------------------------------------------------------------------ pdf.rs
struct Pdf {
    virtual ~Pdf() = default;
    virtual Float value(V3 direction, MyRng &rng) const = 0;
    virtual V3 generate(MyRng &rng) const = 0;
};
struct CosinePdf : Pdf { // pdf.rs:36-45
    Onb uvw;
    explicit CosinePdf(Onb o) : uvw(o) {}
    Float value(V3 direction, MyRng &) const override {
        Float cosine = dot(normalize(direction), uvw.w);
        return std::fmax(cosine / PI, 0.0);
    }
    V3 generate(MyRng &rng) const override { return uvw.local(random_cosine_direction(rng)); }
};
struct HittablePdf : Pdf { // pdf.rs:47-55
    V3 o;
    const Hittable *hittable;
    Float value(V3 direction, MyRng &rng) const override { return hittable->pdf_value(o, direction, rng); }
    V3 generate(MyRng &rng) const override { return hittable->random(o, rng); }
};
struct MixturePdf : Pdf { // pdf.rs:57-69
    const Pdf *p0, *p1;
    Float value(V3 direction, MyRng &rng) const override { return 0.5 * p0->value(direction, rng) + 0.5 * p1->value(direction, rng); }
    V3 generate(MyRng &rng) const override { return rng.gen_bool() ? p0->generate(rng) : p1->generate(rng); }
};

// ------------------------------------------------------------------ material.rs
struct Scatter { // material.rs:15-23
    bool specular;
    Ray specular_ray{};
    std::unique_ptr<Pdf> pdf; // Box<dyn Pdf>
    V3 attenuation;
};
struct Material { // material.rs:25-50
    virtual ~Material() = default;
    virtual std::optional<Scatter> scatter(const Ray &, const HitRecord &, MyRng &) const { return std::nullopt; }
    virtual Float scattering_pdf(const Ray &, const HitRecord &, const Ray &, MyRng &) const { return 0.0; }
    virtual V3 emitted(const Ray &, const HitRecord &, Float, Float, V3) const { return v3(0.0, 0.0, 0.0); }
};
struct NullMaterial : Material {}; // material.rs:68
struct Lambertian : Material {     // material.rs:70-92
    std::shared_ptr<Texture> albedo;
    std::optional<Scatter> scatter(const Ray &, const HitRecord &rec, MyRng &) const override {
        Scatter s;
        s.specular = false;
        s.attenuation = albedo->value(rec.u, rec.v, rec.position);
        s.pdf = std::make_unique<CosinePdf>(Onb::from_w(rec.normal)); // heap allocation per bounce, material.rs:76
        return s;
    }
    Float scattering_pdf(const Ray &, const HitRecord &rec, const Ray &scattered, MyRng &) const override {
        Float cosine = dot(rec.normal, normalize(scattered.direction));
        return std::fmax(cosine / PI, 0.0);
    }
};
static V3 reflect(V3 v, V3 n) { return v - 2.0 * dot(v, n) * n; } // material.rs:94-96
struct Metal : Material {                                          // material.rs:98-112
    V3 albedo;
    Float fuzz;
    std::optional<Scatter> scatter(const Ray &ray, const HitRecord &rec, MyRng &rng) const override {
        V3 reflected = reflect(normalize(ray.direction), rec.normal);
        Scatter s;
        s.specular = true;
        s.specular_ray = Ray{rec.position, reflected + fuzz * random_in_unit_sphere(rng), ray.time};
        s.attenuation = albedo;
        return s;
    }
};
static V3 refract(V3 uv, V3 n, Float etai_over_etat) { // material.rs:114-119
    Float cos_theta = std::fmin(dot(-uv, n), 1.0);
    V3 r_out_perp = etai_over_etat * (uv + cos_theta * n);
    V3 r_out_parallel = -std::sqrt(std::fabs(1.0 - magnitude2(r_out_perp))) * n;
    return r_out_perp + r_out_parallel;
}
static Float reflectance(Float cosine, Float ref_idx) { // material.rs:121-125
    Float r0 = (1.0 - ref_idx) / (1.0 + ref_idx);
    r0 = r0 * r0;
    return r0 + (1.0 - r0) * std::pow(1.0 - cosine, 5.0);
}
struct Dielectric : Material { // material.rs:132-161
    Float ir;
    std::optional<Scatter> scatter(const Ray &ray, const HitRecord &rec, MyRng &rng) const override {
        Float refraction_ratio = rec.front_face ? 1.0 / ir : ir;
        V3 unit_direction = normalize(ray.direction);
        Float cos_theta = std::fmin(dot(-unit_direction, rec.normal), 1.0);
        Float sin_theta = std::sqrt(1.0 - cos_theta * cos_theta);
        bool cannot_refract = refraction_ratio * sin_theta > 1.0;
        V3 direction = (cannot_refract || reflectance(cos_theta, refraction_ratio) > rng.gen_f64())
                           ? reflect(unit_direction, rec.normal)
                           : refract(unit_direction, rec.normal, refraction_ratio);
        Scatter s;
        s.specular = true;
        s.specular_ray = Ray{rec.position, direction, ray.time};
        s.attenuation = v3(1.0, 1.0, 1.0);
        return s;
    }
};
struct DiffuseLight : Material { // material.rs:163-182
    std::shared_ptr<Texture> emit;
    V3 emitted(const Ray &, const HitRecord &rec, Float u, Float v, V3 p) const override {
        return rec.front_face ? emit->value(u, v, p) : v3(0.0, 0.0, 0.0);
    }
};
struct Isotropic : Material { // constant_medium.rs:31-51
    std::shared_ptr<Texture> albedo;
    std::optional<Scatter> scatter(const Ray &ray, const HitRecord &rec, MyRng &rng) const override {
        Scatter s;
        s.attenuation = albedo->value(rec.u, rec.v, rec.position);
        s.specular = true;
        s.specular_ray = Ray{rec.position, random_in_unit_sphere(rng), ray.time};
        return s;
    }
};

// ------------------------------------------------------------------ sphere.rs
struct Sphere : Hittable {
    V3 center;
    Float radius;
    MaterialArc material;
    int prim = -1;
    Hit hit(const Ray &ray, Float t_min, Float t_max, MyRng &) const override { // sphere.rs:24-63
        V3 oc = ray.origin - center;
        Float a = magnitude2(ray.direction);
        Float half_b = dot(oc, ray.direction);
        Float c = magnitude2(oc) - radius * radius;
        Float discriminant = half_b * half_b - a * c;
        if (discriminant < 0.0) return std::nullopt;
        Float sqrtd = std::sqrt(discriminant);
        Float root = (-half_b - sqrtd) / a;
        if (root < t_min || t_max < root) {
            g_replay.reject(prim, root, t_min, t_max);
            root = (-half_b + sqrtd) / a;
            if (root < t_min || t_max < root) {
                g_replay.reject(prim, root, t_min, t_max);
                return std::nullopt;
            }
        }
        g_replay.accept(prim, root);
        V3 position = ray.at(root);
        V3 outward_normal = (position - center) / radius;
        Float u, v;
        sphere_uv(outward_normal, u, v);
        return HitRecord::make(position, outward_normal, root, u, v, ray, material, prim);
    }
    AABB bounding_box(Float, Float) const override { // sphere.rs:65-70
        return AABB{center - v3(radius, radius, radius), center + v3(radius, radius, radius)};
    }
    Float pdf_value(V3 o, V3 v, MyRng &rng) const override { // sphere.rs:72-90
        if (!hit(Ray{o, v, 0.0}, 0.001, INF, rng)) return 0.0;
        Float cos_theta_max = std::sqrt(1.0 - radius * radius / magnitude2(center - o));
        Float solid_angle = 2.0 * PI * (1.0 - cos_theta_max);
        return 1.0 / solid_angle;
    }
    V3 random(V3 o, MyRng &rng) const override { // sphere.rs:92-99
        V3 direction = center - o;
        Float distance_squared = magnitude2(direction);
        Onb uvw = Onb::from_w(direction);
        return uvw.local(random_to_sphere(radius, distance_squared, rng));
    }
};

// ------------------------------------------------------------------ moving_sphere.rs
struct MovingSphere : Hittable {
    V3 center0, center1;
    Float time0, time1, radius;
    MaterialArc material;
    int prim = -1;
    V3 center(Float time) const { return center0 + ((time - time0) / (time1 - time0)) * (center1 - center0); } // :23-26
    Hit hit(const Ray &ray, Float t_min, Float t_max, MyRng &) const override {                                // :31-70
        V3 oc = ray.origin - center(ray.time);
        Float a = magnitude2(ray.direction);
        Float half_b = dot(oc, ray.direction);
        Float c = magnitude2(oc) - radius * radius;
        Float discriminant = half_b * half_b - a * c;
        if (discriminant < 0.0) return std::nullopt;
        Float sqrtd = std::sqrt(discriminant);
        Float root = (-half_b - sqrtd) / a;
        if (root < t_min || t_max < root) {
            g_replay.reject(prim, root, t_min, t_max);
            root = (-half_b + sqrtd) / a;
            if (root < t_min || t_max < root) {
                g_replay.reject(prim, root, t_min, t_max);
                return std::nullopt;
            }
        }
        g_replay.accept(prim, root);
        V3 position = ray.at(root);
        V3 outward_normal = (position - center(ray.time)) / radius;
        Float u, v;
        sphere_uv(outward_normal, u, v);
        return HitRecord::make(position, outward_normal, root, u, v, ray, material, prim);
    }
    AABB bounding_box(Float t0, Float t1) const override { // :72-84
        V3 r = v3(radius, radius, radius);
        return surrounding_box(AABB{center(t0) - r, center(t0) + r}, AABB{center(t1) - r, center(t1) + r});
    }
};

// ------------------------------------------------------------------ aarect.rs
// axis = the constant axis (2: XYRect, 1: XZRect, 0: YZRect); (a,b) = the two in-plane axes in
// the reference's field order (x,y) / (x,z) / (y,z).
template <int AXIS> struct AARect : Hittable {
    static constexpr int A = AXIS == 0 ? 1 : 0;
    static constexpr int B = AXIS == 2 ? 1 : 2;
    Float a0, a1, b0, b1, k;
    MaterialArc material;
    int prim = -1;
    Hit hit(const Ray &ray, Float t_min, Float t_max, MyRng &) const override { // aarect.rs:46-72, 84-110, 152-178
        Float t = (k - ray.origin[AXIS]) / ray.direction[AXIS];
        if (t < t_min || t > t_max) {
            if (g_replay.active) {
                Float ra = ray.origin[A] + t * ray.direction[A], rb = ray.origin[B] + t * ray.direction[B];
                if (!(ra < a0 || ra > a1 || rb < b0 || rb > b1)) g_replay.reject(prim, t, t_min, t_max);
            }
            return std::nullopt;
        }
        Float a = ray.origin[A] + t * ray.direction[A];
        Float b = ray.origin[B] + t * ray.direction[B];
        if (a < a0 || a > a1 || b < b0 || b > b1) return std::nullopt;
        g_replay.accept(prim, t);
        Float u = (a - a0) / (a1 - a0), v = (b - b0) / (b1 - b0);
        V3 outward_normal = v3(AXIS == 0 ? 1.0 : 0.0, AXIS == 1 ? 1.0 : 0.0, AXIS == 2 ? 1.0 : 0.0);
        return HitRecord::make(ray.at(t), outward_normal, t, u, v, ray, material, prim);
    }
    AABB bounding_box(Float, Float) const override { // aarect.rs:74-79, 112-117, 180-185
        V3 lo, hi;
        lo.at(AXIS) = k - 0.0001, hi.at(AXIS) = k + 0.0001;
        lo.at(A) = a0, hi.at(A) = a1, lo.at(B) = b0, hi.at(B) = b1;
        return AABB{lo, hi};
    }
    Float pdf_value(V3 origin, V3 v, MyRng &rng) const override { // only XZRect overrides, aarect.rs:119-138
        if (AXIS != 1) return 0.0;
        Hit rec = hit(Ray{origin, v, 0.0}, 0.001, INF, rng);
        if (!rec) return 0.0;
        Float area = (a1 - a0) * (b1 - b0);
        Float distance_squared = rec->t * rec->t * magnitude2(v);
        Float cosine = std::fabs(dot(v, rec->normal) / magnitude(v));
        return distance_squared / (cosine * area);
    }
    V3 random(V3 origin, MyRng &rng) const override { // aarect.rs:140-147
        if (AXIS != 1) return v3(1.0, 0.0, 0.0);
        Float x = rng.gen_range(a0, a1);
        Float z = rng.gen_range(b0, b1);
        return v3(x, k, z) - origin;
    }
};
using XYRect = AARect<2>;
using XZRect = AARect<1>;
using YZRect = AARect<0>;

// ------------------------------------------------------------------ bvh.rs
struct BVHNode : Hittable {
    HittableBox left, right; // BVHChild::One => right == nullptr
    AABB aabb;
    AABB bounding_box(Float, Float) const override { return aabb; }
    Hit hit(const Ray &ray, Float t_min, Float t_max, MyRng &rng) const override { // bvh.rs:25-50
        if (!aabb.hit(ray, t_min, t_max)) return std::nullopt;
        if (!right) return left->hit(ray, t_min, t_max, rng);
        Hit hit_left = left->hit(ray, t_min, t_max, rng);
        if (hit_left) {
            Hit hit_right = right->hit(ray, t_min, hit_left->t, rng);
            return hit_right ? hit_right : hit_left;
        }
        return right->hit(ray, t_min, t_max, rng);
    }
    static std::unique_ptr<BVHNode> make(std::vector<HittableBox> objects, Float time0, Float time1, MyRng &rng) { // bvh.rs:54-103
        auto node = std::make_unique<BVHNode>();
        size_t len = objects.size();
        if (len == 0) throw std::runtime_error("objects mut not be empty");
        if (len == 1) {
            node->left = std::move(objects.back());
            node->aabb = node->left->bounding_box(time0, time1);
        } else if (len == 2) {
            node->left = std::move(objects[1]); // objects.pop() twice: last, then first
            node->right = std::move(objects[0]);
            node->aabb = surrounding_box(node->left->bounding_box(time0, time1), node->right->bounding_box(time0, time1));
        } else {
            int axis = int(rng.gen_range_inclusive_u64(2));
            std::stable_sort(objects.begin(), objects.end(), [&](const HittableBox &a, const HittableBox &b) {
                return a->bounding_box(time0, time1).minimum[axis] < b->bounding_box(time0, time1).minimum[axis];
            });
            std::vector<HittableBox> right_half;
            for (size_t i = len / 2; i < len; ++i) right_half.push_back(std::move(objects[i]));
            objects.resize(len / 2);
            auto l = make(std::move(objects), time0, time1, rng);
            auto r = make(std::move(right_half), time0, time1, rng);
            node->aabb = surrounding_box(l->aabb, r->aabb);
            node->left = std::move(l), node->right = std::move(r);
        }
        return node;
    }
    void release_leaves(std::vector<HittableBox> &out) { // parity bookkeeping: dismantles the tree
        for (HittableBox *c : {&left, &right}) {
            if (!*c) continue;
            if (auto *b = dynamic_cast<BVHNode *>(c->get())) b->release_leaves(out);
            else out.push_back(std::move(*c));
        }
    }
    void shape(int depth, int &n_nodes, int &max_depth) const {
        ++n_nodes;
        max_depth = std::max(max_depth, depth);
        if (auto *l = dynamic_cast<const BVHNode *>(left.get())) l->shape(depth + 1, n_nodes, max_depth);
        if (auto *r = dynamic_cast<const BVHNode *>(right.get())) r->shape(depth + 1, n_nodes, max_depth);
    }
};

// ------------------------------------------------------------------ aabox.rs
struct AABox : Hittable {
    V3 box_min, box_max;
    std::unique_ptr<BVHNode> sides;
    static std::unique_ptr<AABox> make(V3 p0, V3 p1, const MaterialArc &material, MyRng &rng, int first_prim) { // aabox.rs:22-84
        auto rect_xy = [&](Float k, int id) { auto r = std::make_unique<XYRect>(); r->a0 = p0.x, r->a1 = p1.x, r->b0 = p0.y, r->b1 = p1.y, r->k = k, r->material = material, r->prim = id; return r; };
        auto rect_xz = [&](Float k, int id) { auto r = std::make_unique<XZRect>(); r->a0 = p0.x, r->a1 = p1.x, r->b0 = p0.z, r->b1 = p1.z, r->k = k, r->material = material, r->prim = id; return r; };
        auto rect_yz = [&](Float k, int id) { auto r = std::make_unique<YZRect>(); r->a0 = p0.y, r->a1 = p1.y, r->b0 = p0.z, r->b1 = p1.z, r->k = k, r->material = material, r->prim = id; return r; };
        std::vector<HittableBox> sides;
        sides.push_back(rect_xy(p1.z, first_prim + 0));
        sides.push_back(rect_xy(p0.z, first_prim + 1));
        sides.push_back(rect_xz(p1.y, first_prim + 2));
        sides.push_back(rect_xz(p0.y, first_prim + 3));
        sides.push_back(rect_yz(p1.x, first_prim + 4));
        sides.push_back(rect_yz(p0.x, first_prim + 5));
        auto b = std::make_unique<AABox>();
        b->box_min = p0, b->box_max = p1;
        b->sides = BVHNode::make(std::move(sides), 0.0, 1.0, rng);
        return b;
    }
    Hit hit(const Ray &ray, Float t_min, Float t_max, MyRng &rng) const override { return sides->hit(ray, t_min, t_max, rng); } // :88-96
    AABB bounding_box(Float, Float) const override { return AABB{box_min, box_max}; }                                            // :98-103
};

// ------------------------------------------------------------------ hittable.rs wrappers
struct Translate : Hittable { // hittable.rs:205-234
    HittableBox hittable;
    V3 offset;
    Hit hit(const Ray &ray, Float t_min, Float t_max, MyRng &rng) const override {
        Ray moved{ray.origin - offset, ray.direction, ray.time};
        Hit h = hittable->hit(moved, t_min, t_max, rng);
        if (!h) return std::nullopt;
        return HitRecord::make(h->position + offset, h->normal, h->t, h->u, h->v, moved, h->material, h->prim);
    }
    AABB bounding_box(Float t0, Float t1) const override {
        AABB b = hittable->bounding_box(t0, t1);
        return AABB{b.minimum + offset, b.maximum + offset};
    }
};
static AABB rotate_y_bbox(AABB bbox, Float sin_theta, Float cos_theta) { // hittable.rs:164-194
    V3 mn = v3(INF, INF, INF), mx = v3(-INF, -INF, -INF);
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2; ++j)
            for (int k = 0; k < 2; ++k) {
                Float x = i * bbox.maximum.x + (1.0 - i) * bbox.minimum.x;
                Float y = j * bbox.maximum.y + (1.0 - j) * bbox.minimum.y;
                Float z = k * bbox.maximum.z + (1.0 - k) * bbox.minimum.z;
                Float newx = cos_theta * x + sin_theta * z;
                Float newz = -sin_theta * x + cos_theta * z;
                V3 tester = v3(newx, y, newz);
                for (int c = 0; c < 3; ++c) {
                    mn.at(c) = std::fmin(mn[c], tester[c]);
                    mx.at(c) = std::fmax(mx[c], tester[c]);
                }
            }
    return AABB{mn, mx};
}
struct RotateY : Hittable { // hittable.rs:157-203, 236-284
    HittableBox hittable;
    Float sin_theta, cos_theta;
    AABB aabb;
    static std::unique_ptr<RotateY> make(HittableBox h, Float time0, Float time1, Float degrees) {
        auto r = std::make_unique<RotateY>();
        Float radians = degrees * (PI / 180.0);
        r->sin_theta = std::sin(radians), r->cos_theta = std::cos(radians);
        r->aabb = rotate_y_bbox(h->bounding_box(time0, time1), r->sin_theta, r->cos_theta);
        r->hittable = std::move(h);
        return r;
    }
    Hit hit(const Ray &ray, Float t_min, Float t_max, MyRng &rng) const override {
        V3 origin = ray.origin, direction = ray.direction;
        origin.x = cos_theta * ray.origin.x - sin_theta * ray.origin.z;
        origin.z = sin_theta * ray.origin.x + cos_theta * ray.origin.z;
        direction.x = cos_theta * ray.direction.x - sin_theta * ray.direction.z;
        direction.z = sin_theta * ray.direction.x + cos_theta * ray.direction.z;
        Ray rotated_r{origin, direction, ray.time};
        Hit h = hittable->hit(rotated_r, t_min, t_max, rng);
        if (!h) return std::nullopt;
        V3 p = h->position, normal = h->normal;
        p.x = cos_theta * h->position.x + sin_theta * h->position.z;
        p.z = -sin_theta * h->position.x + cos_theta * h->position.z;
        normal.x = cos_theta * h->normal.x + sin_theta * h->normal.z;
        normal.z = -sin_theta * h->normal.x + cos_theta * h->normal.z;
        return HitRecord::make(p, normal, h->t, h->u, h->v, rotated_r, h->material, h->prim); // note: object-space ray, :269-277
    }
    AABB bounding_box(Float, Float) const override { return aabb; }
};
struct FlipFace : Hittable { // hittable.rs:286-297
    HittableBox inner;
    Hit hit(const Ray &ray, Float t_min, Float t_max, MyRng &rng) const override {
        Hit h = inner->hit(ray, t_min, t_max, rng);
        if (h) h->front_face = !h->front_face;
        return h;
    }
    AABB bounding_box(Float t0, Float t1) const override { return inner->bounding_box(t0, t1); }
};

// `impl Hittable for [T]` — the light list (hittable.rs:112-155)
struct HittableList : Hittable {
    std::vector<HittableBox> items;
    Hit hit(const Ray &ray, Float t_min, Float t_max, MyRng &rng) const override {
        Hit best;
        Float closest = t_max;
        for (auto &h : items) {
            Hit r = h->hit(ray, t_min, closest, rng);
            if (r) closest = r->t, best = std::move(r);
        }
        return best;
    }
    AABB bounding_box(Float t0, Float t1) const override {
        AABB b = items.at(0)->bounding_box(t0, t1);
        for (size_t i = 1; i < items.size(); ++i) b = surrounding_box(b, items[i]->bounding_box(t0, t1));
        return b;
    }
    Float pdf_value(V3 o, V3 v, MyRng &rng) const override { // :144-150
        Float weight = 1.0 / Float(items.size());
        Float sum = 0.0;
        for (auto &h : items) sum += weight * h->pdf_value(o, v, rng);
        return sum;
    }
    V3 random(V3 o, MyRng &rng) const override { // :152-154 (panics on an empty list)
        if (items.empty()) throw std::runtime_error("called `Option::unwrap()` on a `None` value");
        return items[rng.gen_index(uint32_t(items.size()))]->random(o, rng);
    }
};

// ------------------------------------------------------------------ constant_medium.rs
struct ConstantMedium : Hittable {
    HittableBox boundary;
    MaterialArc phase_function;
    Float neg_inv_density;
    int prim = -1;
    AABB bounding_box(Float t0, Float t1) const override { return boundary->bounding_box(t0, t1); }
    Hit hit(const Ray &ray, Float t_min, Float t_max, MyRng &rng) const override { // constant_medium.rs:58-113
        Hit rec1 = boundary->hit(ray, -INF, INF, rng);
        if (!rec1) return std::nullopt;
        Hit rec2 = boundary->hit(ray, rec1->t + 0.0001, INF, rng);
        if (!rec2) return std::nullopt;
        rec1->t = std::fmax(rec1->t, t_min);
        rec2->t = std::fmin(rec2->t, t_max);
        if (rec1->t >= rec2->t) return std::nullopt;
        rec1->t = std::fmax(rec1->t, 0.0);
        Float ray_length = magnitude(ray.direction);
        Float distance_inside_boundary = (rec2->t - rec1->t) * ray_length;
        Float xi;
        if (g_replay.path) { // path replay: the render's free-flight draw (oracle.h: oracle_replay_paths)
            xi = path_medium_xi(*g_replay.path, prim);
        } else if (g_replay.active) { // parity replay of the device's keyed draw (rt1w.h: rt1w_trace_closest)
            uint32_t ctr[4] = {uint32_t(g_replay.ray_index), uint32_t(g_replay.ray_index >> 32), 0x4d454449u, uint32_t(prim)};
            uint32_t key[2] = {uint32_t(g_replay.seed), uint32_t(g_replay.seed >> 32)};
            uint32_t out[4];
            philox4x32_10(ctr, key, out);
            xi = Float(float(out[0] >> 8) * (1.0f / 16777216.0f));
        } else {
            xi = rng.gen_f64();
        }
        Float hit_distance = neg_inv_density * std::log(xi);
        if (g_replay.path) path_near_threshold(*g_replay.path, hit_distance, distance_inside_boundary);
        if (hit_distance > distance_inside_boundary) return std::nullopt;
        Float t = rec1->t + hit_distance / ray_length;
        g_replay.accept(prim, t);
        HitRecord rec{ray.at(t), v3(1.0, 0.0, 0.0), t, 0.0, 0.0, true, phase_function, prim};
        return rec;
    }
};

// ------------------------------------------------------------------ main.rs:51-190
struct RayCounter {
    uint64_t rays = 0;
};

static V3 ray_color(const Ray &ray, V3 background, const Hittable &world, const Hittable &lights, int depth, MyRng &rng, RayCounter &rc) {
    if (depth == 0) return v3(0.0, 0.0, 0.0);
    ++rc.rays;
    Hit rec = world.hit(ray, 0.001, INF, rng);
    if (!rec) return background;
    V3 emitted = rec->material->emitted(ray, *rec, rec->u, rec->v, rec->position);
    std::optional<Scatter> sc = rec->material->scatter(ray, *rec, rng);
    if (!sc) return emitted;
    if (sc->specular) return mul_element_wise(sc->attenuation, ray_color(sc->specular_ray, background, world, lights, depth - 1, rng, rc));
    HittablePdf p0;
    p0.o = rec->position, p0.hittable = &lights;
    MixturePdf mixed;
    mixed.p0 = &p0, mixed.p1 = sc->pdf.get();
    Ray scattered{rec->position, mixed.generate(rng), rec->t}; // time = hit t, main.rs:86
    Float pdf = mixed.value(scattered.direction, rng);
    Float spdf = rec->material->scattering_pdf(ray, *rec, scattered, rng);
    V3 li = ray_color(scattered, background, world, lights, depth - 1, rng, rc);
    return emitted + mul_element_wise(sc->attenuation * spdf, li / pdf); // main.rs:91-104
}

static V3 ray_color_without_light_objects(const Ray &ray, V3 background, const Hittable &world, int depth, MyRng &rng, RayCounter &rc) {
    if (depth == 0) return v3(0.0, 0.0, 0.0);
    ++rc.rays;
    Hit rec = world.hit(ray, 0.001, INF, rng);
    if (!rec) return background;
    V3 emitted = rec->material->emitted(ray, *rec, rec->u, rec->v, rec->position);
    std::optional<Scatter> sc = rec->material->scatter(ray, *rec, rng);
    if (!sc) return emitted;
    if (sc->specular) return mul_element_wise(sc->attenuation, ray_color_without_light_objects(sc->specular_ray, background, world, depth - 1, rng, rc));
    Ray scattered{rec->position, sc->pdf->generate(rng), rec->t}; // main.rs:142-146
    Float pdf_value = sc->pdf->value(scattered.direction, rng);
    Float spdf = rec->material->scattering_pdf(ray, *rec, scattered, rng);
    V3 li = ray_color_without_light_objects(scattered, background, world, depth - 1, rng, rc);
    return emitted + mul_element_wise(sc->attenuation * spdf, li / pdf_value);
}

// ------------------------------------------------------------------ camera.rs:61-73
static Ray camera_get_ray(const rt1w_camera &c, Float s, Float t, MyRng &rng) {
    V3 rd = c.lens_radius * random_in_unit_disk(rng); // runs even when lens_radius == 0
    V3 cu = v3(c.u[0], c.u[1], c.u[2]), cv = v3(c.v[0], c.v[1], c.v[2]);
    V3 offset = cu * rd.x + cv * rd.y;
    V3 origin = v3(c.origin[0], c.origin[1], c.origin[2]);
    V3 llc = v3(c.lower_left_corner[0], c.lower_left_corner[1], c.lower_left_corner[2]);
    V3 hor = v3(c.horizontal[0], c.horizontal[1], c.horizontal[2]), ver = v3(c.vertical[0], c.vertical[1], c.vertical[2]);
    Ray r;
    r.origin = origin + offset;
    r.direction = llc + s * hor + t * ver - origin - offset;
    r.time = rng.gen_range(c.time0, c.time1);
    return r;
}

// ------------------------------------------------------------------ scene loading
struct Scene {
    std::vector<MaterialArc> materials;
    std::vector<std::shared_ptr<Texture>> textures;
    std::vector<std::shared_ptr<Perlin>> perlins;
    HittableBox world;
    HittableList lights;
    bool has_lights = false;
    int n_prims = 0;
    // parity bookkeeping only: every numbered leaf once more, standing alone under a copy of its
    // wrapper chain, so that ties can be found independently of any BVH order
    std::vector<HittableBox> flat;
    std::vector<const MovingSphere *> moving; // the flat twins of the moving spheres outside wrappers (path replay)
};

struct Loader {
    const rt1w_scene_desc &d;
    Scene &scene;
    MyRng rng;
    int next_prim = 0;
    bool number_prims = true;
    std::vector<int> wrappers; // node ids of the Translate / RotateY / FlipFace wrappers above the current node

    void add_flat(int prim, HittableBox leaf) {
        if (prim < 0) return;
        for (size_t i = wrappers.size(); i-- > 0;) {
            const rt1w_node &w = d.nodes[wrappers[i]];
            if (w.type == RT1W_NODE_TRANSLATE) {
                auto t = std::make_unique<Translate>();
                t->hittable = std::move(leaf), t->offset = v3(w.p[0], w.p[1], w.p[2]);
                leaf = std::move(t);
            } else if (w.type == RT1W_NODE_ROTATE_Y) {
                leaf = RotateY::make(std::move(leaf), w.p[1], w.p[2], w.p[0]);
            } else {
                auto f = std::make_unique<FlipFace>();
                f->inner = std::move(leaf);
                leaf = std::move(f);
            }
        }
        if (scene.flat.size() <= size_t(prim)) scene.flat.resize(size_t(prim) + 1);
        scene.flat[size_t(prim)] = std::move(leaf);
    }

    std::shared_ptr<Texture> texture(int id) {
        if (id < 0 || id >= d.n_textures) throw std::runtime_error("texture id out of range");
        if (scene.textures[id]) return scene.textures[id];
        const rt1w_texture &t = d.textures[id];
        std::shared_ptr<Texture> out;
        switch (t.type) {
        case RT1W_TEX_SOLID: {
            auto s = std::make_shared<SolidColor>();
            s->color_value = v3(t.color[0], t.color[1], t.color[2]);
            out = s;
            break;
        }
        case RT1W_TEX_CHECKER: {
            auto c = std::make_shared<CheckerTexture>();
            c->odd = texture(t.odd), c->even = texture(t.even);
            out = c;
            break;
        }
        case RT1W_TEX_NOISE: {
            auto n = std::make_shared<NoiseTexture>();
            n->perlin = scene.perlins.at(t.table), n->scale = t.scale;
            out = n;
            break;
        }
        case RT1W_TEX_PERLIN: {
            auto n = std::make_shared<PerlinTexture>();
            n->perlin = scene.perlins.at(t.table);
            out = n;
            break;
        }
        case RT1W_TEX_IMAGE: {
            if (t.table < 0 || t.table >= d.n_images) throw std::runtime_error("image id out of range");
            const rt1w_image &im = d.images[t.table];
            auto i = std::make_shared<ImageTexture>();
            i->width = uint32_t(im.width), i->height = uint32_t(im.height);
            i->rgb8.assign(im.rgb8, im.rgb8 + size_t(im.width) * im.height * 3);
            out = i;
            break;
        }
        default: throw std::runtime_error("unknown texture type");
        }
        scene.textures[id] = out;
        return out;
    }
    MaterialArc material(int id) {
        if (id < 0 || id >= d.n_materials) throw std::runtime_error("material id out of range");
        if (scene.materials[id]) return scene.materials[id];
        const rt1w_material &m = d.materials[id];
        MaterialArc out;
        switch (m.type) {
        case RT1W_MAT_LAMBERTIAN: { auto x = std::make_shared<Lambertian>(); x->albedo = texture(m.texture); out = x; break; }
        case RT1W_MAT_METAL: { auto x = std::make_shared<Metal>(); x->albedo = v3(m.albedo[0], m.albedo[1], m.albedo[2]); x->fuzz = m.fuzz; out = x; break; }
        case RT1W_MAT_DIELECTRIC: { auto x = std::make_shared<Dielectric>(); x->ir = m.ir; out = x; break; }
        case RT1W_MAT_DIFFUSE_LIGHT: { auto x = std::make_shared<DiffuseLight>(); x->emit = texture(m.texture); out = x; break; }
        case RT1W_MAT_ISOTROPIC: { auto x = std::make_shared<Isotropic>(); x->albedo = texture(m.texture); out = x; break; }
        case RT1W_MAT_NONE: out = std::make_shared<NullMaterial>(); break;
        default: throw std::runtime_error("unknown material type");
        }
        scene.materials[id] = out;
        return out;
    }
    int take_prims(int n) {
        if (!number_prims) return -1000000; // boundary leaves / light copies carry no primitive id
        int first = next_prim;
        next_prim += n;
        return first;
    }
    HittableBox node(int id) {
        if (id < 0 || id >= d.n_nodes) throw std::runtime_error("node id out of range");
        const rt1w_node &n = d.nodes[id];
        auto child = [&](int i) {
            if (i >= n.child_count) throw std::runtime_error("node is missing a child");
            return node(d.children[n.child_begin + i]);
        };
        const double *p = n.p;
        switch (n.type) {
        case RT1W_NODE_SPHERE: {
            auto s = std::make_unique<Sphere>();
            s->center = v3(p[0], p[1], p[2]), s->radius = p[3], s->material = material(n.material), s->prim = take_prims(1);
            add_flat(s->prim, std::make_unique<Sphere>(*s));
            return s;
        }
        case RT1W_NODE_MOVING_SPHERE: {
            auto s = std::make_unique<MovingSphere>();
            s->center0 = v3(p[0], p[1], p[2]), s->center1 = v3(p[3], p[4], p[5]), s->time0 = p[6], s->time1 = p[7], s->radius = p[8];
            s->material = material(n.material), s->prim = take_prims(1);
            if (s->prim >= 0 && wrappers.empty()) {
                auto twin = std::make_unique<MovingSphere>(*s);
                scene.moving.push_back(twin.get());
                add_flat(s->prim, std::move(twin));
            } else {
                add_flat(s->prim, std::make_unique<MovingSphere>(*s));
            }
            return s;
        }
        case RT1W_NODE_XY_RECT: { auto r = std::make_unique<XYRect>(); r->a0 = p[0], r->a1 = p[1], r->b0 = p[2], r->b1 = p[3], r->k = p[4], r->material = material(n.material), r->prim = take_prims(1); add_flat(r->prim, std::make_unique<XYRect>(*r)); return r; }
        case RT1W_NODE_XZ_RECT: { auto r = std::make_unique<XZRect>(); r->a0 = p[0], r->a1 = p[1], r->b0 = p[2], r->b1 = p[3], r->k = p[4], r->material = material(n.material), r->prim = take_prims(1); add_flat(r->prim, std::make_unique<XZRect>(*r)); return r; }
        case RT1W_NODE_YZ_RECT: { auto r = std::make_unique<YZRect>(); r->a0 = p[0], r->a1 = p[1], r->b0 = p[2], r->b1 = p[3], r->k = p[4], r->material = material(n.material), r->prim = take_prims(1); add_flat(r->prim, std::make_unique<YZRect>(*r)); return r; }
        case RT1W_NODE_AABOX: {
            MaterialArc m = material(n.material);
            int first = take_prims(6);
            if (first >= 0) { // the six sides again, one by one (same order as AABox::make)
                MyRng scratch = MyRng::seed_from_u64(0);
                auto twin = AABox::make(v3(p[0], p[1], p[2]), v3(p[3], p[4], p[5]), m, scratch, first);
                std::vector<HittableBox> sides;
                twin->sides->release_leaves(sides);
                for (auto &side : sides) {
                    int id = -1;
                    if (auto *r = dynamic_cast<XYRect *>(side.get())) id = r->prim;
                    else if (auto *r = dynamic_cast<XZRect *>(side.get())) id = r->prim;
                    else if (auto *r = dynamic_cast<YZRect *>(side.get())) id = r->prim;
                    add_flat(id, std::move(side));
                }
            }
            return AABox::make(v3(p[0], p[1], p[2]), v3(p[3], p[4], p[5]), m, rng, first);
        }
        case RT1W_NODE_TRANSLATE: {
            auto t = std::make_unique<Translate>();
            wrappers.push_back(id);
            t->hittable = child(0), t->offset = v3(p[0], p[1], p[2]);
            wrappers.pop_back();
            return t;
        }
        case RT1W_NODE_ROTATE_Y: {
            wrappers.push_back(id);
            HittableBox c = child(0);
            wrappers.pop_back();
            return RotateY::make(std::move(c), p[1], p[2], p[0]);
        }
        case RT1W_NODE_FLIP_FACE: {
            auto f = std::make_unique<FlipFace>();
            wrappers.push_back(id);
            f->inner = child(0);
            wrappers.pop_back();
            return f;
        }
        case RT1W_NODE_CONSTANT_MEDIUM: {
            auto m = std::make_unique<ConstantMedium>();
            m->prim = take_prims(1);
            bool saved = number_prims;
            number_prims = false;
            m->boundary = child(0);
            number_prims = saved;
            m->phase_function = material(n.material);
            m->neg_inv_density = -1.0 / p[0];
            if (m->prim >= 0) {
                auto twin = std::make_unique<ConstantMedium>();
                twin->prim = m->prim, twin->phase_function = m->phase_function, twin->neg_inv_density = m->neg_inv_density;
                number_prims = false;
                twin->boundary = child(0);
                number_prims = saved;
                add_flat(m->prim, std::move(twin));
            }
            return m;
        }
        case RT1W_NODE_BVH: {
            std::vector<HittableBox> objs;
            for (int i = 0; i < n.child_count; ++i) objs.push_back(child(i));
            return BVHNode::make(std::move(objs), p[0], p[1], rng);
        }
        default: throw std::runtime_error("unknown node type");
        }
    }
};

// ------------------------------------------------------------------ path replay (oracle_replay_paths)
// ray_color / ray_color_without_light_objects (main.rs:51-190) with every random number taken from the product's
// Philox stream at the counter the device uses for it (oracle.h: the draw map).  The reference's call order is not the
// device's field order, so each draw site names its block and field instead of consuming a sequential stream.
struct ReplayBounce {
    int prim, material;
    double t;
    V3 weight;
    uint32_t flags;
};

// The replay's own copies of the small helpers it shares with ray_color (material.rs:94-125, onb.rs:13-28): a second caller
// changes how the compiler inlines and contracts them there, and oracle_render must stay bit for bit what it was.
__attribute__((noinline)) static V3 replay_reflect(V3 v, V3 n) { return v - 2.0 * dot(v, n) * n; }
__attribute__((noinline)) static V3 replay_refract(V3 uv, V3 n, Float etai_over_etat) {
    Float cos_theta = std::fmin(dot(-uv, n), 1.0);
    V3 r_out_perp = etai_over_etat * (uv + cos_theta * n);
    V3 r_out_parallel = -std::sqrt(std::fabs(1.0 - magnitude2(r_out_perp))) * n;
    return r_out_perp + r_out_parallel;
}
__attribute__((noinline)) static Float replay_reflectance(Float cosine, Float ref_idx) {
    Float r0 = (1.0 - ref_idx) / (1.0 + ref_idx);
    r0 = r0 * r0;
    return r0 + (1.0 - r0) * std::pow(1.0 - cosine, 5.0);
}
__attribute__((noinline)) static Onb replay_onb(V3 n) {
    V3 w = normalize(n);
    V3 a = std::fabs(w.x) > 0.9 ? v3(0.0, 1.0, 0.0) : v3(1.0, 0.0, 0.0);
    V3 v = normalize(cross(w, a));
    return Onb{cross(w, v), v, w};
}
__attribute__((noinline)) static V3 replay_local(const Onb &o, V3 a) { return o.u * a.x + o.v * a.y + o.w * a.z; }

struct PathTracer {
    const Scene &sc;
    V3 background;
    int max_depth;
    PathReplay &p;
    std::vector<ReplayBounce> *log;
    uint64_t rays = 0;
    MyRng unused = MyRng::seed_from_u64(0); // the Hittable interface takes an RNG; no draw is taken from it here

    // the device's random_in_unit_sphere (kernels.cuh): block 0 of (s, depth, RNG_SCATTER), then 1, 2, ...; f32 test
    V3 unit_sphere(const uint32_t x0[4]) {
        uint32_t x[4] = {x0[0], x0[1], x0[2], x0[3]};
        for (uint32_t b = 1;; ++b) {
            const float px = 2.0f * u01f(x[0]) - 1.0f, py = 2.0f * u01f(x[1]) - 1.0f, pz = 2.0f * u01f(x[2]) - 1.0f;
            const float l2 = px * px + py * py + pz * pz;
            path_near(p, l2, 1.0);
            if (l2 < 1.0f) return v3(px, py, pz);
            p.block(scatter_depth(), RNG_SCATTER, p.mutation == 4 ? 0u : b, x);
            if (p.mutation == 4 && b > 64) return v3(px, py, pz); // the reused block never passes
        }
    }
    uint32_t scatter_depth() const { return p.mutation == 1 ? p.depth + 1 : p.depth; }

    // closest hit, flagged (FLAG_HIT) when the winner is not robust: a tie the oracle_trace_closest bookkeeping sees, a
    // winner within 1e-9 of t_min, or a winner that changes when the direction moves by 1e-5 relative
    Hit closest(const Ray &ray) {
        g_replay.active = true;
        g_replay.reset();
        Hit h = sc.world->hit(ray, 0.001, INF, unused);
        bool amb = g_replay.near_reject;
        if (h) {
            const double tol = 1e-9 * std::fmax(1.0, std::fabs(h->t));
            for (int c = 0; c < g_replay.n_cand; ++c)
                if (g_replay.cand_prim[c] != h->prim && std::fabs(g_replay.cand_t[c] - h->t) <= tol) amb = true;
            if (std::fabs(h->t - 0.001) < 1e-9) amb = true;
            if (sc.flat.size() <= 8192) // BVH-independent sweep for coplanar ties (as oracle_trace_closest; skipped on huge scenes)
                for (size_t k = 0; k < sc.flat.size() && !amb; ++k) {
                    if (int(k) == h->prim || !sc.flat[k]) continue;
                    if (!aabb_hit_closed(sc.flat[k]->bounding_box(0.0, 1.0), ray, h->t - 2.0 * tol, h->t + 2.0 * tol)) continue;
                    const bool medium = dynamic_cast<const ConstantMedium *>(sc.flat[k].get()) != nullptr;
                    Hit o = medium ? sc.flat[k]->hit(ray, 0.001, INF, unused) : sc.flat[k]->hit(ray, std::fmax(0.001, h->t - tol), h->t + tol, unused);
                    if (o && std::fabs(o->t - h->t) <= tol) amb = true;
                }
        }
        // a moving sphere at a time outside [time0, time1] has left the box every tree bounds it by, so whether a ray finds it
        // depends on the tree (DESIGN.md section 3, quirk 1): flagged wherever a direct test meets one before the winner
        for (const MovingSphere *ms : sc.moving)
            if (!amb && (ray.time < ms->time0 || ray.time > ms->time1)) {
                const double t_end = h ? h->t + 1e-9 * std::fmax(1.0, std::fabs(h->t)) : INF;
                if (ms->hit(ray, 0.001, t_end, unused)) amb = true;
            }
        g_replay.active = false;
        const int id = h ? h->prim : -1;
        const double ed = 1e-5 * magnitude(ray.direction);
        for (int k : {0, 3, 5, 6}) {
            if (amb) break;
            Ray q = ray;
            q.direction = q.direction + v3((k & 1) ? ed : -ed, (k & 2) ? ed : -ed, (k & 4) ? ed : -ed);
            Hit hq = sc.world->hit(q, 0.001, INF, unused);
            if ((hq ? hq->prim : -1) != id) amb = true;
            else if (hq && std::fabs(hq->t - h->t) > 1e-3 * std::fmax(1e-3, std::fabs(h->t))) amb = true; // root switch
        }
        if (amb) p.flags |= FLAG_HIT;
        return h;
    }

    // A textured attenuation the device cannot reproduce to 1e-3: its ray lands within ~5e-7 of the path length of the f64
    // hit after a diffuse bounce (MUFU sin / cos in the azimuth, 2^-21), 1.2e-7 for a camera ray (f32 direction), stretched
    // by 1 / cos at grazing incidence, and it evaluates the texture in f32 (2^-23 of the coordinates).  A Perlin or checker
    // value that moves by more than 1e-3 relative within that distance is flagged (FLAG_RANGE).
    void fragile_texture(const Texture *tex, const Ray &ray, const HitRecord &rec, V3 c0) {
        if (dynamic_cast<const SolidColor *>(tex)) return;
        const Float len = magnitude(ray.direction);
        const Float cosi = std::fabs(dot(ray.direction, rec.normal)) / len;
        const V3 q = rec.position;
        const Float delta = (p.depth == 0 ? 1.2e-7 : 5e-7) * rec.t * len / std::fmax(cosi, 1e-3) +
                            std::ldexp(std::fmax(std::fmax(std::fabs(q.x), std::fabs(q.y)), std::fmax(std::fabs(q.z), 1.0)), -23);
        for (int k = 0; k < 6; ++k) {
            V3 e = v3(k / 2 == 0 ? 1.0 : 0.0, k / 2 == 1 ? 1.0 : 0.0, k / 2 == 2 ? 1.0 : 0.0) * ((k & 1) ? -delta : delta);
            V3 c = tex->value(rec.u, rec.v, q + e);
            for (int ch = 0; ch < 3; ++ch)
                if (std::fabs(c[ch] - c0[ch]) > 1e-3 * std::fabs(c0[ch]) + 1e-9) {
                    p.flags |= FLAG_RANGE;
                    return;
                }
        }
    }

    // HittableList::random for the light the device picks, with the device's r1 = u01(x.z), r2 = u01(x.w) (aarect.rs:140-147,
    // sphere.rs:92-99, math.rs:51-65; other kinds keep the trait default (1, 0, 0), hittable.rs:69-71)
    static V3 light_random(const Hittable *L, V3 o, Float r1, Float r2) {
        if (auto *r = dynamic_cast<const XZRect *>(L)) return v3(r->a0 + (r->a1 - r->a0) * r1, r->k, r->b0 + (r->b1 - r->b0) * r2) - o;
        if (auto *s = dynamic_cast<const Sphere *>(L)) {
            V3 direction = s->center - o;
            Float distance_squared = magnitude2(direction);
            Float z = 1.0 + r2 * (std::sqrt(1.0 - s->radius * s->radius / distance_squared) - 1.0);
            Float phi = 2.0 * PI * r1, q = std::sqrt(1.0 - z * z);
            return replay_onb(direction).local(v3(std::cos(phi) * q, std::sin(phi) * q, z));
        }
        return v3(1.0, 0.0, 0.0);
    }

    V3 color(const Ray &ray, uint32_t d) {
        const uint32_t limit = uint32_t(max_depth) + (p.mutation == 8 ? 1u : 0u);
        if (d >= limit) return v3(0.0, 0.0, 0.0); // main.rs:59-61
        ++rays;
        p.depth = d;
        Hit rec = closest(ray);
        if (!rec) {
            if (log) log->push_back(ReplayBounce{-1, -1, INF, background, p.flags});
            return background;
        }
        const Material *m = rec->material.get();
        V3 emitted = m->emitted(ray, *rec, rec->u, rec->v, rec->position);
        if (p.mutation == 6)
            if (auto *l = dynamic_cast<const DiffuseLight *>(m)) emitted = l->emit->value(rec->u, rec->v, rec->position);
        uint32_t x[4];
        p.depth = d;
        p.block(scatter_depth(), RNG_SCATTER, 0, x);
        int kind = -1;
        V3 att = v3(1.0, 1.0, 1.0);
        if (dynamic_cast<const Lambertian *>(m)) kind = RT1W_MAT_LAMBERTIAN;
        else if (dynamic_cast<const Metal *>(m)) kind = RT1W_MAT_METAL;
        else if (dynamic_cast<const Dielectric *>(m)) kind = RT1W_MAT_DIELECTRIC;
        else if (dynamic_cast<const Isotropic *>(m)) kind = RT1W_MAT_ISOTROPIC;
        else kind = dynamic_cast<const DiffuseLight *>(m) ? RT1W_MAT_DIFFUSE_LIGHT : RT1W_MAT_NONE;
        if (kind == RT1W_MAT_DIFFUSE_LIGHT || kind == RT1W_MAT_NONE) {
            if (log) log->push_back(ReplayBounce{rec->prim, kind, rec->t, emitted, p.flags});
            return emitted;
        }
        if (kind != RT1W_MAT_LAMBERTIAN) { // specular: attenuation * ray_color(specular_ray) (main.rs:73)
            Ray out{rec->position, v3(0, 0, 0), ray.time};
            if (kind == RT1W_MAT_METAL) { // material.rs:98-112
                const Metal *mm = static_cast<const Metal *>(m);
                V3 reflected = replay_reflect(normalize(ray.direction), rec->normal);
                out.direction = mm->fuzz == 0.0 ? reflected : reflected + mm->fuzz * unit_sphere(x);
                att = mm->albedo;
            } else if (kind == RT1W_MAT_DIELECTRIC) { // material.rs:132-161, xi = u01(x.x)
                const Dielectric *dm = static_cast<const Dielectric *>(m);
                Float ratio = rec->front_face ? 1.0 / dm->ir : dm->ir;
                V3 unit = normalize(ray.direction);
                Float cos_theta = std::fmin(dot(-unit, rec->normal), 1.0);
                Float sin_theta = std::sqrt(1.0 - cos_theta * cos_theta);
                path_near(p, ratio * sin_theta, 1.0);
                bool reflects = ratio * sin_theta > 1.0;
                if (!reflects) {
                    const Float xi = u01f(x[0]), f = replay_reflectance(cos_theta, ratio);
                    path_near(p, f, xi);
                    reflects = f > xi;
                }
                out.direction = reflects ? replay_reflect(unit, rec->normal) : replay_refract(unit, rec->normal, ratio);
            } else { // Isotropic, constant_medium.rs:36-51
                const Texture *tex = static_cast<const Isotropic *>(m)->albedo.get();
                att = tex->value(rec->u, rec->v, rec->position);
                fragile_texture(tex, ray, *rec, att);
                out.direction = unit_sphere(x);
            }
            if (log) log->push_back(ReplayBounce{rec->prim, kind, rec->t, att, p.flags});
            return mul_element_wise(att, color(out, d + 1));
        }
        // Lambertian: MixturePdf(HittablePdf(lights), CosinePdf) (main.rs:75-104) or the CosinePdf alone (main.rs:142-160)
        const Texture *tex = static_cast<const Lambertian *>(m)->albedo.get();
        att = tex->value(rec->u, rec->v, rec->position);
        fragile_texture(tex, ray, *rec, att);
        const Onb uvw = replay_onb(rec->normal);
        const Float r1 = u01f(x[2]), r2 = u01f(x[3]);
        const auto &lights = sc.lights.items;
        const int n = sc.has_lights ? int(lights.size()) : 0;
        V3 dir;
        if (n > 0 && (x[0] >> 31)) { // rng.gen::<bool>() (pdf.rs:63-64), then slice.choose (hittable.rs:153)
            const int idx = std::min(int(u01f(p.mutation == 3 ? x[0] : x[1]) * float(n)), n - 1);
            dir = light_random(lights[size_t(idx)].get(), rec->position, r1, r2);
        } else { // math.rs:39-49
            Float z = std::sqrt(1.0 - r2), phi = 2.0 * PI * r1;
            dir = replay_local(uvw, v3(std::cos(phi) * std::sqrt(r2), std::sin(phi) * std::sqrt(r2), z));
        }
        Ray scattered{rec->position, dir, p.mutation == 7 ? ray.time : rec->t}; // time = hit t, main.rs:86
        Float pdf = std::fmax(dot(normalize(dir), uvw.w) / PI, 0.0); // pdf.rs:36-45
        if (n > 0) pdf = 0.5 * sc.lights.pdf_value(rec->position, dir, unused) + 0.5 * pdf; // pdf.rs:58-60
        const Float spdf = std::fmax(dot(rec->normal, normalize(dir)) / PI, 0.0); // material.rs:82-91
        const Float wgt = spdf / pdf;
        if (!(pdf >= double(std::numeric_limits<float>::min())) || !(std::fabs(wgt) <= double(std::numeric_limits<float>::max())) ||
            (wgt != 0.0 && std::fabs(wgt) < double(std::numeric_limits<float>::min())))
            p.flags |= FLAG_RANGE;
        if (log) log->push_back(ReplayBounce{rec->prim, kind, rec->t, att * wgt, p.flags});
        V3 li = color(scattered, d + 1);
        return emitted + mul_element_wise(att * spdf, li / pdf); // main.rs:91-104
    }
};

// The render's camera ray (render.cu: camera_ray) as the product's f32 ray: counter (s, 0, RNG_CAMERA, 0) gives the s / t
// jitters and the shutter time, blocks 1, 2, ... the lens sample (two tries per block, f32 test).
static Ray replay_camera_ray(const rt1w_camera &c, int w, int h, PathReplay &p) {
    const uint32_t j = p.k0 / uint32_t(w), i = p.k0 - j * uint32_t(w);
    uint32_t x[4];
    p.block(0, RNG_CAMERA, 0, x);
    const Float us = u01f(p.mutation == 9 ? x[1] : x[0]), ut = u01f(p.mutation == 9 ? x[0] : x[1]);
    const Float s = (Float(i) + us) / Float(w - 1), t = (Float(j) + ut) / Float(h - 1); // main.rs:968-969
    Float rx = 0.0, ry = 0.0;
    if (c.lens_radius != 0.0) {
        float px = 0.0f, py = 0.0f;
        for (uint32_t b = 1;; ++b) {
            uint32_t y[4];
            p.block(0, RNG_CAMERA, b, y);
            px = 2.0f * u01f(y[0]) - 1.0f, py = 2.0f * u01f(y[1]) - 1.0f;
            path_near(p, px * px + py * py, 1.0);
            if (px * px + py * py < 1.0f) break;
            px = 2.0f * u01f(y[2]) - 1.0f, py = 2.0f * u01f(y[3]) - 1.0f;
            path_near(p, px * px + py * py, 1.0);
            if (px * px + py * py < 1.0f) break;
        }
        rx = c.lens_radius * Float(px), ry = c.lens_radius * Float(py);
    }
    const V3 cu = v3(c.u[0], c.u[1], c.u[2]), cv = v3(c.v[0], c.v[1], c.v[2]);
    const V3 offset = cu * rx + cv * ry; // camera.rs:62-66
    const V3 origin = v3(c.origin[0], c.origin[1], c.origin[2]);
    const V3 llc = v3(c.lower_left_corner[0], c.lower_left_corner[1], c.lower_left_corner[2]);
    const V3 hor = v3(c.horizontal[0], c.horizontal[1], c.horizontal[2]), ver = v3(c.vertical[0], c.vertical[1], c.vertical[2]);
    const V3 dir = llc + s * hor + t * ver - origin - offset; // camera.rs:67-70
    Ray r;
    r.origin = origin + offset;
    r.direction = v3(float(dir.x), float(dir.y), float(dir.z)); // the product's rays carry f32 directions and time
    r.time = float(c.time0 + (c.time1 - c.time0) * Float(u01f(x[2]))); // camera.rs:71
    return r;
}

} // namespace oracle

// ===================================================================== C interface
using namespace oracle;

struct oracle_scene {
    Scene scene;
};

static thread_local std::string g_error;

extern "C" {

const char *oracle_last_error(void) { return g_error.c_str(); }

oracle_scene *oracle_scene_load(const rt1w_scene_desc *desc, uint64_t bvh_seed) {
    try {
        if (!desc) throw std::runtime_error("null description");
        auto s = std::make_unique<oracle_scene>();
        Scene &sc = s->scene;
        sc.materials.resize(desc->n_materials);
        sc.textures.resize(desc->n_textures);
        for (int i = 0; i < desc->n_perlins; ++i) {
            auto p = std::make_shared<Perlin>();
            for (int k = 0; k < 256; ++k) {
                p->ranvec[k] = v3(desc->perlins[i].ranvec[k][0], desc->perlins[i].ranvec[k][1], desc->perlins[i].ranvec[k][2]);
                p->perm_x[k] = desc->perlins[i].perm_x[k], p->perm_y[k] = desc->perlins[i].perm_y[k], p->perm_z[k] = desc->perlins[i].perm_z[k];
            }
            sc.perlins.push_back(p);
        }
        Loader ld{*desc, sc, MyRng::seed_from_u64(bvh_seed), 0, true, {}};
        sc.world = ld.node(desc->world);
        sc.n_prims = ld.next_prim;
        sc.has_lights = desc->has_lights != 0;
        ld.number_prims = false;
        for (int i = 0; i < desc->n_lights; ++i) sc.lights.items.push_back(ld.node(desc->lights[i]));
        return s.release();
    } catch (const std::exception &e) {
        g_error = e.what();
        return nullptr;
    }
}
void oracle_scene_free(oracle_scene *s) { delete s; }
int32_t oracle_scene_num_prims(const oracle_scene *s) { return s ? s->scene.n_prims : -1; }
void oracle_scene_bvh_shape(const oracle_scene *s, int32_t *n_nodes, int32_t *depth) {
    int n = 0, dmax = 0;
    if (auto *b = dynamic_cast<const BVHNode *>(s->scene.world.get())) b->shape(1, n, dmax);
    if (n_nodes) *n_nodes = n;
    if (depth) *depth = dmax;
}

static void set_threads(int32_t threads) {
#ifdef _OPENMP
    if (threads > 0) omp_set_num_threads(threads);
    else omp_set_num_threads(omp_get_num_procs());
#else
    (void)threads;
#endif
}

int32_t oracle_trace_closest(const oracle_scene *s, const rt1w_ray *rays, size_t n, uint64_t seed, int32_t *prim_id, double *t,
                             double *normal3, uint8_t *front_face, double *uv2, uint8_t *ambiguous, int32_t threads) {
    if (!s || !rays) return 1;
    set_threads(threads);
    const Hittable &world = *s->scene.world;
    AABB wb = world.bounding_box(0.0, 1.0);
    const double extent = std::fmax(std::fmax(wb.maximum.x - wb.minimum.x, wb.maximum.y - wb.minimum.y), wb.maximum.z - wb.minimum.z);
    // The product solves ray/primitive intersections in f64 from the same f32 inputs, so only genuine
    // (near-)ties are excluded: two leaves within 1e-9 relative of the winning t, a candidate within
    // 1e-9 of the range ends, or a winner that changes under a 1e-9-relative perturbation of the ray.
    const double rel = 1e-9;
#pragma omp parallel for schedule(dynamic, 1024)
    for (long long i = 0; i < (long long)n; ++i) {
        MyRng rng = MyRng::seed_from_u64(uint64_t(i));
        g_replay.active = true, g_replay.seed = seed, g_replay.ray_index = uint64_t(i);
        Ray r{v3(rays[i].origin[0], rays[i].origin[1], rays[i].origin[2]), v3(rays[i].direction[0], rays[i].direction[1], rays[i].direction[2]),
              double(rays[i].time)};
        g_replay.reset();
        Hit h = world.hit(r, 0.001, INF, rng);
        int id = h ? h->prim : -1;
        bool tie = g_replay.near_reject;
        if (h) {
            const double tol = 1e-9 * std::fmax(1.0, std::fabs(h->t));
            for (int c = 0; c < g_replay.n_cand; ++c)
                if (g_replay.cand_prim[c] != id && std::fabs(g_replay.cand_t[c] - h->t) <= tol) tie = true;
            // BVH-independent sweep: any other leaf whose own hit lands within tol of the winner
            // (the reference may never reach it: an un-padded AABox bound culls exact ties, aabb.rs:26)
            const auto &flat = s->scene.flat;
            for (size_t k = 0; k < flat.size() && !tie; ++k) {
                if (int(k) == id || !flat[k]) continue;
                if (!aabb_hit_closed(flat[k]->bounding_box(0.0, 1.0), r, h->t - 2.0 * tol, h->t + 2.0 * tol)) continue;
                const bool medium = dynamic_cast<const ConstantMedium *>(flat[k].get()) != nullptr;
                Hit o = medium ? flat[k]->hit(r, 0.001, INF, rng) : flat[k]->hit(r, std::fmax(0.001, h->t - tol), h->t + tol, rng);
                if (o && std::fabs(o->t - h->t) <= tol) tie = true;
            }
        }
        if (prim_id) prim_id[i] = id;
        if (t) t[i] = h ? h->t : INF;
        if (normal3) {
            normal3[3 * i] = h ? h->normal.x : 0.0, normal3[3 * i + 1] = h ? h->normal.y : 0.0, normal3[3 * i + 2] = h ? h->normal.z : 0.0;
        }
        if (front_face) front_face[i] = h ? uint8_t(h->front_face) : 0;
        if (uv2) uv2[2 * i] = h ? h->u : 0.0, uv2[2 * i + 1] = h ? h->v : 0.0;
        if (ambiguous) {
            bool amb = tie || (h && std::fabs(h->t - 0.001) < 1e-9);
            double dlen = magnitude(r.direction);
            const double eo = rel * std::fmax(extent, 1.0), ed = rel * dlen;
            for (int k = 0; k < 8 && !amb; ++k) {
                Ray q = r;
                q.origin = q.origin + v3((k & 1) ? eo : -eo, (k & 2) ? eo : -eo, (k & 4) ? eo : -eo);
                q.direction = q.direction + v3((k & 4) ? ed : -ed, (k & 1) ? ed : -ed, (k & 2) ? ed : -ed);
                Hit hq = world.hit(q, 0.001, INF, rng);
                int idq = hq ? hq->prim : -1;
                if (idq != id) amb = true;
                else if (hq && std::fabs(hq->t - h->t) > 1e-3 * std::fmax(1e-3, std::fabs(h->t))) amb = true; // root switch on the same primitive
            }
            ambiguous[i] = amb ? 1 : 0;
        }
        g_replay.active = false;
    }
    return 0;
}

int32_t oracle_render(const oracle_scene *s, const rt1w_camera *camera, const rt1w_render_params *params, int32_t threads,
                      double *rgb_sum, double *stat, oracle_render_stats *stats) {
    if (!s || !camera || !params || !rgb_sum) return 1;
    set_threads(threads);
    const int w = params->width, h = params->height;
    const int s0 = params->sample_begin, s1 = params->sample_end;
    const V3 background = v3(params->background[0], params->background[1], params->background[2]);
    const Hittable &world = *s->scene.world;
    const HittableList &lights = s->scene.lights;
    const bool has_lights = s->scene.has_lights;
    const double clamp = params->stat_clamp > 0 ? params->stat_clamp : INF;
    uint64_t total_rays = 0;
    int used_threads = 1;
    auto t_begin = std::chrono::steady_clock::now();
    // rows j = h-1 .. 0 (main.rs:957-959); dynamic scheduling stands in for rayon's work stealing
#pragma omp parallel reduction(+ : total_rays)
    {
#ifdef _OPENMP
#pragma omp single
        used_threads = omp_get_num_threads();
#endif
        RayCounter rc;
#pragma omp for schedule(dynamic, 1)
        for (int row = 0; row < h; ++row) {
            const int j = h - 1 - row;
            for (int i = 0; i < w; ++i) {
                uint64_t pixel_seed = uint64_t(j) * uint64_t(w) + uint64_t(i); // main.rs:964
                if (s0 != 0) pixel_seed ^= 0x9E3779B97F4A7C15ull * uint64_t(s0 + 1); // disjoint stream for a later sample range
                MyRng rng = MyRng::seed_from_u64(pixel_seed);
                V3 pixel = v3(0.0, 0.0, 0.0);
                double st[6] = {0, 0, 0, 0, 0, 0};
                for (int sidx = s0; sidx < s1; ++sidx) {
                    Float u = (Float(i) + rng.gen_f64()) / Float(w - 1); // main.rs:968-969
                    Float v = (Float(j) + rng.gen_f64()) / Float(h - 1);
                    Ray ray = camera_get_ray(*camera, u, v, rng);
                    V3 c = has_lights ? ray_color(ray, background, world, lights, params->max_depth, rng, rc)
                                      : ray_color_without_light_objects(ray, background, world, params->max_depth, rng, rc);
                    pixel = pixel + c;
                    if (stat) {
                        for (int ch = 0; ch < 3; ++ch) {
                            double x = c[ch];
                            if (std::isnan(x)) x = 0.0;
                            x = std::fmin(x, clamp);
                            st[ch] += x, st[3 + ch] += x * x;
                        }
                    }
                }
                size_t px = size_t(row) * w + i;
                rgb_sum[3 * px] = pixel.x, rgb_sum[3 * px + 1] = pixel.y, rgb_sum[3 * px + 2] = pixel.z;
                if (stat)
                    for (int k = 0; k < 6; ++k) stat[6 * px + k] = st[k];
            }
        }
        total_rays += rc.rays;
    }
    auto t_end = std::chrono::steady_clock::now();
    if (stats) {
        stats->paths = uint64_t(w) * h * uint64_t(s1 - s0);
        stats->rays = total_rays;
        stats->seconds = std::chrono::duration<double>(t_end - t_begin).count();
        stats->threads = used_threads;
    }
    return 0;
}

static PathReplay replay_key(const oracle_scene *s, const rt1w_render_params *params, const int32_t *leaf_of_prim, uint32_t pixel_seed,
                             int32_t sample, int32_t mutation) {
    PathReplay p;
    p.k0 = pixel_seed, p.k1 = uint32_t(params->seed), p.hi = uint32_t(params->seed >> 32), p.s = uint32_t(sample);
    p.mutation = mutation, p.leaf_of_prim = leaf_of_prim, p.n_map = s->scene.n_prims;
    return p;
}

static V3 replay_one(const oracle_scene *s, const rt1w_camera *camera, const rt1w_render_params *params, PathReplay &p,
                     std::vector<ReplayBounce> *log, uint64_t &rays) {
    const V3 background = v3(params->background[0], params->background[1], params->background[2]);
    PathTracer tr{s->scene, background, params->max_depth, p, log};
    g_replay.path = &p;
    Ray r = replay_camera_ray(*camera, params->width, params->height, p);
    V3 c = tr.color(r, 0);
    g_replay.path = nullptr;
    rays = tr.rays;
    return c;
}

int32_t oracle_replay_paths(const oracle_scene *s, const rt1w_camera *camera, const rt1w_render_params *params, const int32_t *leaf_of_prim,
                            size_t n, const uint32_t *pixel_seed, const int32_t *sample, int32_t mutation, int32_t threads, double *out_rgb,
                            uint32_t *out_rays, uint8_t *out_flags) {
    if (!s || !camera || !params || !pixel_seed || !sample || !out_rgb) return 1;
    if (params->width < 2 || params->height < 2 || params->max_depth < 1) return 2;
    set_threads(threads);
    bool failed = false;
    std::string message;
#pragma omp parallel for schedule(dynamic, 256)
    for (long long i = 0; i < (long long)n; ++i) {
        try {
            PathReplay p = replay_key(s, params, leaf_of_prim, pixel_seed[i], sample[i], mutation);
            uint64_t rays = 0;
            V3 c = replay_one(s, camera, params, p, nullptr, rays);
            out_rgb[3 * i] = c.x, out_rgb[3 * i + 1] = c.y, out_rgb[3 * i + 2] = c.z;
            if (out_rays) out_rays[i] = uint32_t(rays);
            if (out_flags) out_flags[i] = uint8_t(p.flags);
        } catch (const std::exception &e) {
            g_replay.path = nullptr;
#pragma omp critical
            {
                message = e.what();
                failed = true;
            }
        }
    }
    if (failed) g_error = message;
    return failed ? 3 : 0;
}

int32_t oracle_replay_path_log(const oracle_scene *s, const rt1w_camera *camera, const rt1w_render_params *params, const int32_t *leaf_of_prim,
                               uint32_t pixel_seed, int32_t sample, int32_t mutation, char *buf, size_t capacity) {
    if (!s || !camera || !params || !buf || capacity == 0) return 1;
    std::vector<ReplayBounce> log;
    PathReplay p = replay_key(s, params, leaf_of_prim, pixel_seed, sample, mutation);
    uint64_t rays = 0;
    V3 c;
    try {
        c = replay_one(s, camera, params, p, &log, rays);
    } catch (const std::exception &e) {
        g_replay.path = nullptr;
        g_error = e.what();
        return 3;
    }
    std::string out;
    char line[256];
    std::snprintf(line, sizeof line, "pixel seed %u sample %d: L = (%.9g, %.9g, %.9g), %llu rays, flags %u\n", pixel_seed, sample, c.x, c.y, c.z,
                  (unsigned long long)rays, p.flags);
    out += line;
    for (size_t d = 0; d < log.size(); ++d) {
        const ReplayBounce &b = log[d];
        std::snprintf(line, sizeof line, "  depth %zu: prim %d material %d t %.9g weight (%.6g, %.6g, %.6g) flags %u\n", d, b.prim, b.material, b.t,
                      b.weight.x, b.weight.y, b.weight.z, b.flags);
        out += line;
    }
    std::snprintf(buf, capacity, "%s", out.c_str());
    return 0;
}

void oracle_replay_camera_rays(const oracle_scene *s, const rt1w_camera *camera, const rt1w_render_params *params, size_t n,
                               const uint32_t *pixel_seed, const int32_t *sample, int32_t mutation, double *origin3, double *dir3, double *time) {
    for (size_t i = 0; i < n; ++i) {
        PathReplay p = replay_key(s, params, nullptr, pixel_seed[i], sample[i], mutation);
        Ray r = replay_camera_ray(*camera, params->width, params->height, p);
        origin3[3 * i] = r.origin.x, origin3[3 * i + 1] = r.origin.y, origin3[3 * i + 2] = r.origin.z;
        dir3[3 * i] = r.direction.x, dir3[3 * i + 1] = r.direction.y, dir3[3 * i + 2] = r.direction.z;
        time[i] = r.time;
    }
}

// ---- known-answer probes
static MyRng &probe_rng() {
    static thread_local MyRng r = MyRng::seed_from_u64(0);
    return r;
}
double oracle_xz_rect_pdf_value(const double rect[5], const double o[3], const double v[3]) {
    XZRect r;
    r.a0 = rect[0], r.a1 = rect[1], r.b0 = rect[2], r.b1 = rect[3], r.k = rect[4], r.material = std::make_shared<NullMaterial>();
    return r.pdf_value(v3(o[0], o[1], o[2]), v3(v[0], v[1], v[2]), probe_rng());
}
double oracle_sphere_pdf_value(const double c[3], double radius, const double o[3], const double v[3]) {
    Sphere s;
    s.center = v3(c[0], c[1], c[2]), s.radius = radius, s.material = std::make_shared<NullMaterial>();
    return s.pdf_value(v3(o[0], o[1], o[2]), v3(v[0], v[1], v[2]), probe_rng());
}
double oracle_sphere_hit_t(const double c[3], double radius, const double o[3], const double d[3], double t_min, double t_max) {
    Sphere s;
    s.center = v3(c[0], c[1], c[2]), s.radius = radius, s.material = std::make_shared<NullMaterial>();
    Hit h = s.hit(Ray{v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2]), 0.0}, t_min, t_max, probe_rng());
    return h ? h->t : std::numeric_limits<double>::quiet_NaN();
}
double oracle_reflectance(double cosine, double ref_idx) { return reflectance(cosine, ref_idx); }
void oracle_refract(const double uv[3], const double n[3], double eta, double out[3]) {
    V3 r = refract(v3(uv[0], uv[1], uv[2]), v3(n[0], n[1], n[2]), eta);
    out[0] = r.x, out[1] = r.y, out[2] = r.z;
}
void oracle_sphere_uv(const double p[3], double out_uv[2]) { sphere_uv(v3(p[0], p[1], p[2]), out_uv[0], out_uv[1]); }
void oracle_onb_from_w(const double n[3], double o[9]) {
    Onb b = Onb::from_w(v3(n[0], n[1], n[2]));
    o[0] = b.u.x, o[1] = b.u.y, o[2] = b.u.z, o[3] = b.v.x, o[4] = b.v.y, o[5] = b.v.z, o[6] = b.w.x, o[7] = b.w.y, o[8] = b.w.z;
}
void oracle_quantise(const double rgb_sum[3], int32_t spp, int32_t out[3]) { // color.rs:14-21,56-65
    double scale = 1.0 / double(spp);
    for (int c = 0; c < 3; ++c) {
        double x = std::isnan(rgb_sum[c]) ? 0.0 : rgb_sum[c];
        x *= scale;
        double g = std::sqrt(x);
        g = g < 0.0 ? 0.0 : (g > 0.999 ? 0.999 : g); // f64::clamp (NaN stays NaN -> `as usize` gives 0)
        double q = 256.0 * g;
        out[c] = std::isnan(q) ? 0 : int32_t(q);
    }
}
void oracle_camera_ray(const rt1w_camera *cam, double s, double t, double o[3], double d[3]) {
    rt1w_camera c = *cam;
    c.lens_radius = 0.0;
    MyRng rng = MyRng::seed_from_u64(0);
    Ray r = camera_get_ray(c, s, t, rng);
    o[0] = r.origin.x, o[1] = r.origin.y, o[2] = r.origin.z, d[0] = r.direction.x, d[1] = r.direction.y, d[2] = r.direction.z;
}
void oracle_rotate_y_bbox(const double bmin[3], const double bmax[3], double deg, double omin[3], double omax[3]) {
    double rad = deg * (PI / 180.0);
    AABB b = rotate_y_bbox(AABB{v3(bmin[0], bmin[1], bmin[2]), v3(bmax[0], bmax[1], bmax[2])}, std::sin(rad), std::cos(rad));
    omin[0] = b.minimum.x, omin[1] = b.minimum.y, omin[2] = b.minimum.z, omax[0] = b.maximum.x, omax[1] = b.maximum.y, omax[2] = b.maximum.z;
}
int32_t oracle_hit_one(const oracle_scene *s, const double o[3], const double d[3], double time, double *t, double p[3], double n[3],
                       int32_t *front_face) {
    MyRng rng = MyRng::seed_from_u64(0);
    Hit h = s->scene.world->hit(Ray{v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2]), time}, 0.001, INF, rng);
    if (!h) return -1;
    if (t) *t = h->t;
    if (p) p[0] = h->position.x, p[1] = h->position.y, p[2] = h->position.z;
    if (n) n[0] = h->normal.x, n[1] = h->normal.y, n[2] = h->normal.z;
    if (front_face) *front_face = h->front_face;
    return h->prim;
}
static Perlin perlin_from(const rt1w_perlin *tab) {
    Perlin p;
    for (int k = 0; k < 256; ++k) {
        p.ranvec[k] = v3(tab->ranvec[k][0], tab->ranvec[k][1], tab->ranvec[k][2]);
        p.perm_x[k] = tab->perm_x[k], p.perm_y[k] = tab->perm_y[k], p.perm_z[k] = tab->perm_z[k];
    }
    return p;
}
double oracle_perlin_noise(const rt1w_perlin *tab, const double p[3]) { return perlin_from(tab).noise(v3(p[0], p[1], p[2])); }
double oracle_perlin_turb(const rt1w_perlin *tab, const double p[3], int32_t depth) { return perlin_from(tab).turb(v3(p[0], p[1], p[2]), depth); }
void oracle_texture_value(const oracle_scene *s, int32_t texture, double u, double v, const double p[3], double out[3]) {
    V3 c = s->scene.textures.at(texture)->value(u, v, v3(p[0], p[1], p[2]));
    out[0] = c.x, out[1] = c.y, out[2] = c.z;
}
void oracle_bvh_count(int32_t n_objects, uint64_t seed, int32_t *n_nodes, int32_t *depth) {
    MyRng rng = MyRng::seed_from_u64(seed);
    MyRng pos = MyRng::seed_from_u64(seed + 1);
    std::vector<HittableBox> objs;
    auto m = std::make_shared<NullMaterial>();
    for (int i = 0; i < n_objects; ++i) {
        auto s = std::make_unique<Sphere>();
        s->center = v3(pos.gen_f64(), pos.gen_f64(), pos.gen_f64()), s->radius = 0.01, s->material = m;
        objs.push_back(std::move(s));
    }
    auto root = BVHNode::make(std::move(objs), 0.0, 1.0, rng);
    int n = 0, dmax = 0;
    root->shape(1, n, dmax);
    *n_nodes = n, *depth = dmax;
}
void oracle_chacha_block(const uint32_t state[16], int32_t rounds, uint32_t out[16]) { chacha_block(state, rounds, out); }
void oracle_stdrng_u32(uint64_t seed, int32_t n, uint32_t *out) {
    MyRng r = MyRng::seed_from_u64(seed);
    for (int i = 0; i < n; ++i) out[i] = r.next_u32();
}
void oracle_stdrng_from_seed_u32(const uint8_t seed[32], int32_t n, uint32_t *out) {
    MyRng r = MyRng::from_seed(seed);
    for (int i = 0; i < n; ++i) out[i] = r.next_u32();
}
void oracle_stdrng_f64(uint64_t seed, int32_t n, double *out) {
    MyRng r = MyRng::seed_from_u64(seed);
    for (int i = 0; i < n; ++i) out[i] = r.gen_f64();
}
void oracle_philox(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) { philox4x32_10(ctr, key, out); }
}
