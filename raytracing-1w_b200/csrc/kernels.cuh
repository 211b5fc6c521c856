// kernels.cuh — device code of the wavefront path tracer (sm_100a).
//
// Everything the reference does per ray inside `ray_color` (main.rs:51-190) lives here as
// __device__ functions; render.cu wraps them into the fused wave kernels (scatter / start paths,
// closest hit, regroup per material) and the closest-hit parity kernel.
//
// Precision policy (DESIGN.md "Precision"): the reference is f64 throughout (main.rs:1).
//   * BVH node slab tests: f32 on conservatively padded boxes (bvh.cpp store_box).
//   * primitive intersection, hit position, wrapper transforms: f64 (B200 issues DFMA at half the
//     FFMA rate; this keeps hit distances bit-close to the reference and removes every f32
//     self-intersection artefact of 555-unit scenes with t_min = 0.001).
//   * directions, normals, pdfs, throughput, textures, radiance sums: f32.
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>
#include <stddef.h>
#include <stdint.h>

#include "device_types.h"
#include "flat_plans.h"
#include "philox.h"

namespace rt1w {

#define RT1W_DEV __device__ __forceinline__

constexpr double kTMin = 0.001;      // main.rs:62
constexpr float kPiF = 3.14159265358979323846f;
#ifndef RT1W_STACK_SMEM
#define RT1W_STACK_SMEM 16 // 16 KB of stacks per 128-thread CTA; 24 entries were 1-2 % slower (less L1 left for the nodes)
#endif
constexpr int kStackSmem = RT1W_STACK_SMEM;       // per-thread short stack entries kept in shared memory
constexpr int kStackLocal = 64 - RT1W_STACK_SMEM; // overflow entries (local memory; the builder caps the depth at 62)

struct SceneView {
    const float4 *nodes;       // 2 x float4 per node
    const uint4 *wide_nodes;   // 5 x uint4 per node of the compressed 8-wide tree (bvh8.h), or nullptr
    const DPrim *prims;        // leaf order
    const float4 *prim_boxes;  // flat scenes: 2 x float4 per primitive in SCAN order (see flat_stage), else nullptr
    const FlatGroups *flat_groups; // flat scenes: the scan-order groups of prim_boxes (flat_plans.h), else nullptr
    const int32_t *prim_id;    // leaf index -> primitive id (DFS order of the description)
    const DFrame *frames;
    const DMaterial *materials;
    const DTexture *textures;
    const DPerlin *perlins;
    const cudaTextureObject_t *images;
    const int2 *image_dims;
    const DLight *lights;
    int32_t n_lights, has_lights;
    int32_t n_prims, n_nodes, n_wide, n_perlins, n_frames;
    int32_t n_global; // the last n_global primitives are in no tree: every ray tests them (hit_globals)
    int32_t flat; // scan the primitive list (closest_hit_flat) instead of walking the BVH
    int32_t wide; // BVH scenes: walk the 8-wide tree by default (render flags may force either layout)
    int32_t rich_textures; // some texture is not a SolidColor
    int32_t flat_plan; // flat scenes: the plan (flat_plans.h) of flat_groups' layout, or -1
};

struct f3 {
    float x, y, z;
};
struct d3 {
    double x, y, z;
};
// Explicit rounding.  The code of a bounce is inlined into the wave kernels and into the tail kernel (render.cu), and a path
// must come out bit for bit the same whichever of them runs its bounce.  A plain multiply and add (PTX mul / add without a
// rounding modifier) may be contracted into an FMA by ptxas in one kernel and not in the other - it was, in the scatters - so
// the shading arithmetic (these helpers, materials, light pdfs, finalize_hit, textures) is written with fmaf / __fmul_rn /
// __fadd_rn and __fma_rn / __dmul_rn / __dadd_rn, which are never re-fused: the FMA form where one is wanted, one rounding per
// step elsewhere.  The primitive solves are left to the compiler (pinning the sphere quadratic cost one_weekend 0.9 %);
// tests/test_gpu_schedule_invariance.py checks that the kernels agree on them.
RT1W_DEV f3 mk3(float x, float y, float z) { return f3{x, y, z}; }
RT1W_DEV f3 operator+(f3 a, f3 b) { return f3{__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z)}; }
RT1W_DEV f3 operator-(f3 a, f3 b) { return f3{__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y), __fsub_rn(a.z, b.z)}; }
RT1W_DEV f3 operator-(f3 a) { return f3{-a.x, -a.y, -a.z}; }
RT1W_DEV f3 operator*(float s, f3 a) { return f3{__fmul_rn(s, a.x), __fmul_rn(s, a.y), __fmul_rn(s, a.z)}; }
RT1W_DEV f3 operator*(f3 a, f3 b) { return f3{__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y), __fmul_rn(a.z, b.z)}; }
RT1W_DEV f3 fma3(float s, f3 a, f3 b) { return f3{fmaf(s, a.x, b.x), fmaf(s, a.y, b.y), fmaf(s, a.z, b.z)}; } // s * a + b
RT1W_DEV float dot(f3 a, f3 b) { return fmaf(a.z, b.z, fmaf(a.y, b.y, __fmul_rn(a.x, b.x))); }
RT1W_DEV f3 cross(f3 a, f3 b) {
    return f3{fmaf(a.y, b.z, -__fmul_rn(a.z, b.y)), fmaf(a.z, b.x, -__fmul_rn(a.x, b.z)), fmaf(a.x, b.y, -__fmul_rn(a.y, b.x))};
}
RT1W_DEV f3 normalize(f3 a) { return rsqrtf(dot(a, a)) * a; }

// ------------------------------------------------------------------------------------------
// Ray + path state as the kernels see them (SoA in HBM, see Pool in render.cu)
// ------------------------------------------------------------------------------------------
struct Ray {
    double ox, oy, oz;
    float dx, dy, dz;
    float time;
};

struct __align__(16) RayB { // second 16-byte word of a ray slot
    double oz;
    float dx, dy;
};
struct __align__(16) RayC { // third word: rest of the ray + the path bookkeeping
    float dz, time;
    uint32_t state; // (sample - sample_begin) << 8 | depth
    uint32_t pixel; // the reference's pixel seed j * width + i, row j counted from the bottom (main.rs:964)
};
struct __align__(16) HitRec {
    double t;
    int32_t leaf;  // index into SceneView::prims (leaf order)
    uint32_t meta; // the primitive's meta word (material id / type), so shading need not wait for the primitive record
};

// How ConstantMedium candidates draw their free-flight number (constant_medium.rs:85).
// counter = (c0, c1, c2, id), key = (k0, k1); `exact` selects the f64 logarithm and the
// primitive-id keyed counter that the CPU checker replays (rt1w.h: rt1w_trace_closest).
struct MediumRng {
    uint32_t c0, c1, c2, k0, k1;
};

// ------------------------------------------------------------------------------------------
// Wrapper chains
// ------------------------------------------------------------------------------------------
struct LocalRay {
    double ox, oy, oz, dx, dy, dz;
};

// The rigid part of a wrapper chain: the first 40 bytes of a DFrame (global memory) or its shared-memory copy.
struct FrameXf {
    double sin_t, cos_t, bx, by, bz;
};
static_assert(offsetof(DFrame, bz) == 32, "FrameXf must alias the head of DFrame");

RT1W_DEV const FrameXf *frame_xf(const DFrame *frames, int frame) { return reinterpret_cast<const FrameXf *>(frames + frame); }

RT1W_DEV LocalRay to_local(const FrameXf *f, const Ray &r) { // f == nullptr: no wrapper chain
    LocalRay l;
    if (f == nullptr) {
        l.ox = r.ox, l.oy = r.oy, l.oz = r.oz, l.dx = r.dx, l.dy = r.dy, l.dz = r.dz;
        return l;
    }
    // hittable.rs:207 and :241-245, composed on the host
    const double s = f->sin_t, c = f->cos_t;
    l.ox = c * r.ox - s * r.oz + f->bx;
    l.oy = r.oy + f->by;
    l.oz = s * r.ox + c * r.oz + f->bz;
    l.dx = c * double(r.dx) - s * double(r.dz);
    l.dy = r.dy;
    l.dz = s * double(r.dx) + c * double(r.dz);
    return l;
}

// ------------------------------------------------------------------------------------------
// Primitive tests (f64).  Each returns the accepted root in [tmin, tmax] like the reference.
// ------------------------------------------------------------------------------------------

RT1W_DEV bool sphere_roots(const LocalRay &l, double cx, double cy, double cz, double radius, double &r0, double &r1) {
    // sphere.rs:31-41
    const double ocx = l.ox - cx, ocy = l.oy - cy, ocz = l.oz - cz;
    const double a = l.dx * l.dx + l.dy * l.dy + l.dz * l.dz;
    const double half_b = ocx * l.dx + ocy * l.dy + ocz * l.dz;
    const double c = ocx * ocx + ocy * ocy + ocz * ocz - radius * radius;
    const double disc = half_b * half_b - a * c;
    if (disc < 0.0) return false;
    const double sqrtd = sqrt(disc);
    const double inv_a = 1.0 / a;
    r0 = (-half_b - sqrtd) * inv_a;
    r1 = (-half_b + sqrtd) * inv_a;
    return true;
}

RT1W_DEV bool hit_sphere(const LocalRay &l, double cx, double cy, double cz, double radius, double tmin, double tmax, double &t) {
    double r0, r1;
    if (!sphere_roots(l, cx, cy, cz, radius, r0, r1)) return false;
    double root = r0; // sphere.rs:43-48: near root first, then far
    if (root < tmin || tmax < root) {
        root = r1;
        if (root < tmin || tmax < root) return false;
    }
    t = root;
    return true;
}

// num / den for a denominator inside the f32 exponent range: f32 reciprocal seed + two f64 Newton corrections
// (relative error ~1e-16; the IEEE division sequence costs three times as many issue slots).
RT1W_DEV double div_newton(double num, double den) {
    float rf;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rf) : "f"(__double2float_rn(den)));
    const double r0 = double(rf);
    double q = num * r0;
    q = fma(fma(-q, den, num), r0, q);
    q = fma(fma(-q, den, num), r0, q);
    return q;
}

// rect with constant axis ax (0: YZRect, 1: XZRect, 2: XYRect); aarect.rs:46-72,84-110,152-178.
// The axis is data, not a template parameter: lanes of a warp that test different rectangles
// (walls, box sides) run the same instruction stream.
RT1W_DEV bool hit_rect(const LocalRay &l, int ax, double a0, double a1, double b0, double b1, double k, double tmin, double tmax, double &t) {
    const double oc = ax == 0 ? l.ox : (ax == 1 ? l.oy : l.oz);
    const double dc = ax == 0 ? l.dx : (ax == 1 ? l.dy : l.dz);
    const double oa = ax == 0 ? l.oy : l.ox, da = ax == 0 ? l.dy : l.dx;
    const double ob = ax == 2 ? l.oy : l.oz, db = ax == 2 ? l.dy : l.dz;
    // t = (k - oc) / dc must land in [tmin, tmax].  Compare before dividing: planes behind the origin,
    // beyond the current best hit, and the plane the ray starts on leave without paying for the division.
    const double num = k - oc;
    if (dc > 0.0 ? (num < tmin * dc || num > tmax * dc) : (dc < 0.0 && (num > tmin * dc || num < tmax * dc))) return false;
    // |dc| tiny or zero: the reference's inf / NaN results (aarect.rs:85-88) come out of the real division
    const double tt = fabs(dc) > 1e-30 ? div_newton(num, dc) : num / dc;
    if (tt < tmin || tt > tmax) return false;
    const double a = oa + tt * da, b = ob + tt * db;
    if (a < a0 || a > a1 || b < b0 || b > b1) return false;
    t = tt;
    return true;
}

// 1 / d with |1/d| capped at 1e18: slab distances of an axis the ray is parallel to stay finite and keep their sign
RT1W_DEV float rcp_capped(float d) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(copysignf(fmaxf(fabsf(d), 1e-18f), d)));
    return r;
}

// three-input min / max (sm_100: FMNMX3, one issue slot)
RT1W_DEV float max3(float a, float b, float c) {
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}
RT1W_DEV float min3(float a, float b, float c) {
    float r;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

// AABox (aabox.rs:22-103) = six rectangles, tested for the closest accepted root.  The device keeps the box
// as one primitive and runs the rectangle test (hit_rect, shared with the plain rectangles so that a warp
// mixing walls and box sides stays on one code path) on ONE side in the common case: the side an f32 slab
// computation names as the entry (origin outside: an accepted entry is the closest root of the six) or, when
// the entry lies before t_min, the exit; then the other of the two.  If both fail - f32 picked the wrong
// neighbour at an edge, or the ray misses the box - the remaining sides are tested like the reference does,
// closest root wins.
// Sides are numbered as aabox.rs:29-76 lists them: XY@z1, XY@z0, XZ@y1, XZ@y0, YZ@x1, YZ@x0.
// returns the first side to test | the second one << 4
RT1W_DEV int box_first_sides(const LocalRay &l, double x0, double y0, double z0, double x1, double y1, double z1, bool &leaves_before_tmin) {
    const float ix = rcp_capped(float(l.dx)), iy = rcp_capped(float(l.dy)), iz = rcp_capped(float(l.dz));
    const float ax = float(x0 - l.ox) * ix, bx = float(x1 - l.ox) * ix;
    const float ay = float(y0 - l.oy) * iy, by = float(y1 - l.oy) * iy;
    const float az = float(z0 - l.oz) * iz, bz = float(z1 - l.oz) * iz;
    const float fx = fminf(ax, bx), fy = fminf(ay, by), fz = fminf(az, bz); // front planes
    const float kx = fmaxf(ax, bx), ky = fmaxf(ay, by), kz = fmaxf(az, bz); // back planes
    const int a_in = fx >= fy ? (fx >= fz ? 0 : 2) : (fy >= fz ? 1 : 2);    // entry: the front plane crossed last
    const int a_out = kx <= ky ? (kx <= kz ? 0 : 2) : (ky <= kz ? 1 : 2);   // exit: the back plane crossed first
    // entering a positive-going axis happens at the box minimum, leaving it at the maximum
    const int s_in = (2 - a_in) * 2 + ((a_in == 0 ? ix : (a_in == 1 ? iy : iz)) > 0.0f ? 1 : 0);
    const int s_out = (2 - a_out) * 2 + ((a_out == 0 ? ix : (a_out == 1 ? iy : iz)) > 0.0f ? 0 : 1);
    const bool entry_first = fmaxf(fmaxf(fx, fy), fz) >= float(kTMin);
    // The ray leaves the box well before t_min (typically: it starts ON the box, scattered off one of its sides): beyond
    // t_min it is outside the box by at least 1e-4 |d_exit|, so no side can hold an accepted root (aabox.rs:84-103
    // would test six rectangles and find nothing).  Only claimed when the exit axis is not grazing, so that this margin
    // dwarfs the f64 rounding of the rectangle tests (1e-16 of the coordinates).
    leaves_before_tmin = fminf(fminf(kx, ky), kz) < 0.0009f && fabsf(a_out == 0 ? ix : (a_out == 1 ? iy : iz)) < 1e4f;
    return entry_first ? (s_in | (s_out << 4)) : (s_out | (s_in << 4));
}

template <bool EXACT>
RT1W_DEV bool medium_sample(double t_in, double t_out, double neg_inv_density, double ray_length, double tmin, double tmax,
                            const MediumRng &mr, uint32_t id, double &t) {
    // constant_medium.rs:74-104 given the two boundary hits
    double t1 = fmax(t_in, tmin), t2 = fmin(t_out, tmax);
    if (t1 >= t2) return false;
    t1 = fmax(t1, 0.0);
    const double inside = (t2 - t1) * ray_length;
    const Philox4 x = philox4x32_10(mr.c0, mr.c1, mr.c2, id, mr.k0, mr.k1);
    const float xi = u01(x.x);
    const double hit_distance = EXACT ? neg_inv_density * log(double(xi)) : neg_inv_density * double(__logf(xi));
    if (hit_distance > inside) return false;
    t = t1 + hit_distance / ray_length;
    return true;
}

// One candidate primitive (record at `P`: global memory, or the shared-memory copy of the flat-scan
// path).  Returns true and the hit parameter when it lands in [t_min, tmax].
// `frames`: the wrapper frames (global memory, or the flat scan's shared-memory copies).
// MEDIA = false compiles the ConstantMedium cases out (scenes without media: no Philox, no f64 slabs in the loop).
// `box_sides`: for a P_BOX the caller passes 0 on the first call and calls again while it comes back non-zero
// (sides still to test); `side` is written with the side tested by this call.
// BOXES = false compiles the P_BOX case out (the flat scan keeps the six rectangles, api.cu).
// ROUND = true compiles everything but the sphere kinds out (hit_globals: its copy of this function is a sixth the size).
template <bool EXACT, bool MEDIA, bool BOXES, bool ROUND = false>
RT1W_DEV bool hit_prim(const SceneView &sc, const DFrame *frames, const DPrim *P, int leaf, const Ray &r, double tmax, const MediumRng &mr, double &t,
                       uint32_t &box_sides, int &side) {
    const double2 *w = reinterpret_cast<const double2 *>(P);
    const int4 tail = *reinterpret_cast<const int4 *>(w + 3); // q2 | meta | frame
    const uint32_t meta = uint32_t(tail.z);
    const int type = int(meta & 15u);
    const double2 p01 = w[0], p23 = w[1];
    const LocalRay l = to_local(tail.w < 0 ? nullptr : frame_xf(frames, tail.w), r);
    if (!ROUND && (type == P_XY_RECT || type == P_XZ_RECT || type == P_YZ_RECT || (BOXES && type == P_BOX))) { // one rectangle test
        int ax = P_YZ_RECT - type;
        double a0 = p01.x, a1 = p01.y, b0 = p23.x, b1 = p23.y, k = w[2].x;
        bool box_first = false;
        if (BOXES && type == P_BOX) {
            const double2 q01 = w[2];
            const double x0 = p01.x, y0 = p01.y, z0 = p23.x, x1 = q01.x, y1 = q01.y, z1 = __hiloint2double(tail.y, tail.x);
            const bool first = box_sides == 0u;
            if (first) { // sides left to test in bits 0..5, the one to test second in bits 8..10
                bool gone;
                const int two = box_first_sides(l, x0, y0, z0, x1, y1, z1, gone);
                if (gone) return false; // box_sides is still 0: the caller's loop over the sides ends
                side = two & 15;
                box_sides = 0x3fu | (uint32_t((two >> 4) | 8) << 8);
            } else if (box_sides >> 8) {
                side = int(box_sides >> 8) & 7;
                box_sides &= 0x3fu;
            } else {
                side = __ffs(int(box_sides)) - 1;
            }
            box_sides &= ~(1u << side);
            ax = 2 - (side >> 1);
            const bool low_plane = (side & 1) != 0;
            k = ax == 0 ? (low_plane ? x0 : x1) : (ax == 1 ? (low_plane ? y0 : y1) : (low_plane ? z0 : z1));
            a0 = ax == 0 ? y0 : x0, a1 = ax == 0 ? y1 : x1;
            b0 = ax == 2 ? y0 : z0, b1 = ax == 2 ? y1 : z1;
            box_first = first;
        }
        // ONE call site for plain rectangles and box sides, ONE sphere solve for the three sphere kinds below: lanes on
        // different primitive kinds share the instruction stream, and the kernel's hot code stays near the 32 KB the
        // instruction cache holds
        const bool hit = hit_rect(l, ax, a0, a1, b0, b1, k, kTMin, tmax, t);
        if (BOXES && type == P_BOX) {
            if (box_first && hit) box_sides = 0u; // the side f32 named was right: nothing closer on this box
            if ((box_sides & 0x3fu) == 0u) box_sides = 0u;
        }
        return hit;
    }
    if (!MEDIA) { // medium-free kernels (random_scene, one_weekend): one inlined solve per sphere kind is 1 % faster there
        if (type == P_SPHERE) return hit_sphere(l, p01.x, p01.y, p23.x, p23.y, kTMin, tmax, t);
        if (type == P_MOVING_SPHERE) { // moving_sphere.rs:23-26,31-48
            const float4 f = *reinterpret_cast<const float4 *>(w + 2);
            const double s = double((r.time - f.w) * __int_as_float(tail.x));
            return hit_sphere(l, p01.x + s * double(f.x), p01.y + s * double(f.y), p23.x + s * double(f.z), p23.y, kTMin, tmax, t);
        }
        return false;
    }
    if (type == P_SPHERE || type == P_MOVING_SPHERE || (MEDIA && type == P_MEDIUM_SPHERE)) {
        double cx = p01.x, cy = p01.y, cz = p23.x;
        if (type == P_MOVING_SPHERE) { // moving_sphere.rs:23-26,31-48
            const float4 f = *reinterpret_cast<const float4 *>(w + 2);
            const double s = double((r.time - f.w) * __int_as_float(tail.x));
            cx += s * double(f.x), cy += s * double(f.y), cz += s * double(f.z);
        }
        double r0, r1;
        if (!sphere_roots(l, cx, cy, cz, p23.y, r0, r1)) return false;
        if (!MEDIA || type != P_MEDIUM_SPHERE) { // sphere.rs:43-48: near root first, then far
            double root = r0;
            if (root < kTMin || tmax < root) {
                root = r1;
                if (root < kTMin || tmax < root) return false;
            }
            t = root;
            return true;
        }
        // boundary.hit(-inf, inf) then boundary.hit(t1 + 0.0001, inf), constant_medium.rs:58-72
        if (r1 < r0 + 0.0001) return false;
        const double nid = w[2].x;
        const double len = sqrt(l.dx * l.dx + l.dy * l.dy + l.dz * l.dz);
        const uint32_t id = EXACT ? uint32_t(__ldg(sc.prim_id + leaf)) : uint32_t(leaf);
        return medium_sample<EXACT>(r0, r1, nid, len, kTMin, tmax, mr, id, t);
    }
    switch (type) {
    case P_MEDIUM_BOX: { // the six sides of aabox.rs:29-76 as three slabs
        if (!MEDIA || ROUND) return false;
        const double2 q01 = w[2];
        const double q2 = __hiloint2double(tail.y, tail.x);
        const double ix = 1.0 / l.dx, iy = 1.0 / l.dy, iz = 1.0 / l.dz;
        double ax = (p01.x - l.ox) * ix, bx = (q01.x - l.ox) * ix;
        double ay = (p01.y - l.oy) * iy, by = (q01.y - l.oy) * iy;
        double az = (p23.x - l.oz) * iz, bz = (q2 - l.oz) * iz;
        const double t_in = fmax(fmax(fmin(ax, bx), fmin(ay, by)), fmin(az, bz));
        const double t_out = fmin(fmin(fmax(ax, bx), fmax(ay, by)), fmax(az, bz));
        if (!(t_in <= t_out)) return false;
        if (t_out < t_in + 0.0001) return false;
        const double len = sqrt(l.dx * l.dx + l.dy * l.dy + l.dz * l.dz);
        const uint32_t id = EXACT ? uint32_t(__ldg(sc.prim_id + leaf)) : uint32_t(leaf);
        return medium_sample<EXACT>(t_in, t_out, p23.y, len, kTMin, tmax, mr, id, t);
    }
    default: return false;
    }
}

// ------------------------------------------------------------------------------------------
// extend: closest hit over the flat SAH BVH (replaces BVHNode::hit, bvh.rs:25-50)
// ------------------------------------------------------------------------------------------
// The node test in the FMA form t = plane * (1/d) - o * (1/d), |1/d| capped at 1e18 (rcp_capped) so that an axis the ray
// is parallel to yields finite distances of the right sign.  The rounding of the form - 2^-24 (|o| + |plane - o|) in space
// units - is covered by the padding of the node boxes (bvh.cpp: conservative_box with 1e-6 of the scene's reach on top).
struct SlabRay {
    float ix, iy, iz, ox, oy, oz; // 1/d and -o/d
};

RT1W_DEV bool slab(const float4 lo, const float4 hi, const SlabRay &s, float tmax, float &tnear) {
    const float ax = fmaf(lo.x, s.ix, s.ox), bx = fmaf(hi.x, s.ix, s.ox);
    const float ay = fmaf(lo.y, s.iy, s.oy), by = fmaf(hi.y, s.iy, s.oy);
    const float az = fmaf(lo.z, s.iz, s.oz), bz = fmaf(hi.z, s.iz, s.oz);
    const float tn = fmaxf(max3(fminf(ax, bx), fminf(ay, by), fminf(az, bz)), 0.0f);
    float tf = fminf(min3(fmaxf(ax, bx), fmaxf(ay, by), fmaxf(az, bz)), tmax);
    // (no slack on the comparison: the node boxes are padded by 1e-6 of the scene's reach, bvh.h: traversal_pad, eight times
    // the 2^-23 relative rounding of the FMA form for any hit within the scene's reach of the origin, and the best hit's
    // f32 bound is rounded up)
    tnear = tn;
    return tn <= tf;
}

// Node references on the traversal stack: primitive count in the top 3 bits, left_first below.
// (the count sits in the top 3 bits of a node's first word: api.cu folds it in after the upload, k_fold_node_refs - one word
// read per child instead of two combined; binary steps are 62 instructions, every one of them counts)
RT1W_DEV uint32_t node_ref(float4 n0, float4) { return __float_as_uint(n0.w); }

// Traversal state of one ray, resumable step by step (the wave kernel interleaves the steps of a warp's rays
// with refills of its idle lanes; the parity kernel just runs them to the end).
// The stack holds (node reference, entry distance) so that subtrees the best hit already beats are dropped
// on pop; its first kStackSmem entries live in the thread's column of a shared-memory array (stride =
// blockDim.x), deeper ones in a local-memory overflow.
constexpr uint32_t kTravDone = 0xffffffffu;
struct Trav {
    SlabRay s;
    double best;    // closest accepted root so far
    float bestf;    // its f32 upper bound, for the node tests
    int best_leaf;  // leaf | side << kLeafBits, or -1
    uint32_t ref;   // node to visit next: interior (count bits 0), leaf, or kTravDone
    int sp;
    uint32_t sbase; // shared-window address of the thread's stack column, held in a register (trav_bind_stack)
};

#ifdef RT1W_COUNT_TRAV // measurement build (build.py --variant trav -DRT1W_COUNT_TRAV): rays, interior steps, primitive tests, warp-level interior steps
static __device__ unsigned long long g_trav_counts[4];
#define RT1W_TRAV_COUNT(k) atomicAdd(&g_trav_counts[k], 1ull)
#else
#define RT1W_TRAV_COUNT(k)
#endif

// The stack column's shared-memory address as an opaque 32-bit value: left to itself the compiler re-derives it on EVERY node
// step (S2UR SR_CgaCtaId, UMOV, ULEA, S2R SR_TID, LEA: 5 of a step's 52 instructions) rather than keep one register alive.
RT1W_DEV void trav_bind_stack(Trav &T, const uint2 *stack) {
    T.sbase = uint32_t(__cvta_generic_to_shared(stack));
    asm volatile("" : "+r"(T.sbase));
}
RT1W_DEV void stack_store(uint32_t addr, uint2 e) { asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(e.x), "r"(e.y) : "memory"); }
RT1W_DEV uint2 stack_load(uint32_t addr) {
    uint2 e;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(e.x), "=r"(e.y) : "r"(addr) : "memory");
    return e;
}
RT1W_DEV void trav_begin(const SceneView &sc, const Ray &r, Trav &T) {
    RT1W_TRAV_COUNT(0);
    T.s.ix = rcp_capped(r.dx), T.s.iy = rcp_capped(r.dy), T.s.iz = rcp_capped(r.dz);
    T.s.ox = -__double2float_rn(r.ox) * T.s.ix, T.s.oy = -__double2float_rn(r.oy) * T.s.iy, T.s.oz = -__double2float_rn(r.oz) * T.s.iz;
    T.best = CUDART_INF, T.bestf = CUDART_INF_F, T.best_leaf = -1, T.sp = 0;
    const float4 n0 = __ldg(sc.nodes), n1 = __ldg(sc.nodes + 1);
    float tn;
    T.ref = slab(n0, n1, T.s, T.bestf, tn) ? node_ref(n0, n1) : kTravDone;
}

RT1W_DEV bool trav_interior(const Trav &T) { return (T.ref >> 29) == 0u; }
RT1W_DEV bool trav_done(const Trav &T) { return T.ref == kTravDone; }
RT1W_DEV bool trav_at_leaf(const Trav &T) { return !trav_interior(T) && !trav_done(T); }
RT1W_DEV void trav_reset(Trav &T) { T.ref = kTravDone, T.sp = 0; }

RT1W_DEV void trav_pop(Trav &T, const uint2 *stack, int stride, const uint2 *overflow) { // next stacked subtree that can still hold a closer hit
    // (taking one entry per step instead of looping here was measured slower: 479 vs 507 Mrays/s on the 1 M-sphere scene)
    while (T.sp > 0) {
        --T.sp;
        const uint2 e = T.sp < kStackSmem ? stack_load(T.sbase + uint32_t(T.sp * stride) * 8u) : overflow[T.sp - kStackSmem];
        if (__uint_as_float(e.y) <= T.bestf) {
            T.ref = e.x;
            return;
        }
    }
    T.ref = kTravDone;
}

// one interior node: both children (one 64-byte pair) tested, nearer one first
RT1W_DEV void trav_step_interior(const SceneView &sc, Trav &T, uint2 *stack, int stride, uint2 *overflow) {
    RT1W_TRAV_COUNT(1);
#ifdef RT1W_COUNT_TRAV
    if (int(threadIdx.x & 31) == __ffs(int(__activemask())) - 1) RT1W_TRAV_COUNT(3);
#endif
    const float4 *c = sc.nodes + 2 * size_t(T.ref); // (one IMAD.WIDE: ref * 32 bytes)
    const float4 l0 = __ldg(c), l1 = __ldg(c + 1), r0 = __ldg(c + 2), r1 = __ldg(c + 3);
    float tl, tr;
    const bool hl = slab(l0, l1, T.s, T.bestf, tl), hr = slab(r0, r1, T.s, T.bestf, tr);
    const uint32_t refl = node_ref(l0, l1), refr = node_ref(r0, r1);
    if (hl && hr) {
        const bool left_near = tl <= tr;
        const uint2 far_e = make_uint2(left_near ? refr : refl, __float_as_uint(left_near ? tr : tl));
        if (T.sp < kStackSmem) stack_store(T.sbase + uint32_t(T.sp * stride) * 8u, far_e);
        else overflow[T.sp - kStackSmem] = far_e;
        ++T.sp;
        T.ref = left_near ? refl : refr;
    } else if (hl || hr) {
        T.ref = hl ? refl : refr;
    } else {
        trav_pop(T, stack, stride, overflow);
    }
}

// one leaf: its primitives solved in f64, then the next subtree
template <bool EXACT, bool MEDIA>
RT1W_DEV void trav_step_leaf(const SceneView &sc, const Ray &r, const MediumRng &mr, Trav &T, const uint2 *stack, int stride, const uint2 *overflow) {
    const uint32_t first = T.ref & 0x1fffffffu, count = T.ref >> 29;
    for (uint32_t i = 0; i < count; ++i) {
        uint32_t box_sides = 0u;
        do {
            double t;
            int side = 0;
            RT1W_TRAV_COUNT(2);
            if (hit_prim<EXACT, MEDIA, true>(sc, sc.frames, sc.prims + (first + i), int(first + i), r, T.best, mr, t, box_sides, side)) {
                T.best = t, T.best_leaf = int(first + i) | (side << kLeafBits);
                T.bestf = __double2float_ru(t);
            }
        } while (box_sides != 0u);
    }
    trav_pop(T, stack, stride, overflow);
}

// The primitives that are in no tree (api.cu: spheres and sphere-bounded media whose box contains every other primitive's,
// e.g. a fog sphere around the whole scene): tested after the traversal, against the best hit it found - the whole warp
// at once, by a sphere-only copy of hit_prim (a full second copy cost final_scene 1.4 %: instruction fetch).
template <bool EXACT, bool MEDIA>
RT1W_DEV void hit_globals(const SceneView &sc, const Ray &r, const MediumRng &mr, double &best, int &best_leaf) {
    for (int g = sc.n_prims - sc.n_global; g < sc.n_prims; ++g) {
        uint32_t box_sides = 0u;
        do {
            double t;
            int side = 0;
            RT1W_TRAV_COUNT(2);
            if (hit_prim<EXACT, MEDIA, false, true>(sc, sc.frames, sc.prims + g, g, r, best, mr, t, box_sides, side)) best = t, best_leaf = g | (side << kLeafBits);
        } while (box_sides != 0u);
    }
}

// while-while traversal to the end: every lane descends to its next leaf before any lane runs the (f64)
// primitive tests, so those run with most of the warp converged.
template <bool EXACT, bool MEDIA>
RT1W_DEV bool closest_hit(const SceneView &sc, const Ray &r, const MediumRng &mr, uint2 *stack, int stride, double &t_best, int &leaf_best) {
    uint2 overflow[kStackLocal];
    Trav T;
    trav_bind_stack(T, stack);
    trav_begin(sc, r, T);
    while (!trav_done(T)) {
        while (trav_interior(T)) trav_step_interior(sc, T, stack, stride, overflow);
        if (!trav_done(T)) trav_step_leaf<EXACT, MEDIA>(sc, r, mr, T, stack, stride, overflow);
    }
    hit_globals<EXACT, MEDIA>(sc, r, mr, T.best, T.best_leaf);
    t_best = T.best, leaf_best = T.best_leaf;
    return T.best_leaf >= 0;
}

// ------------------------------------------------------------------------------------------
// extend: closest hit over the compressed 8-wide BVH (bvh8.h; replaces BVHNode::hit, bvh.rs:25-50, for big scenes)
// ------------------------------------------------------------------------------------------
// One step = ONE 80-byte node fetch and eight child tests.  Child boxes are bytes on the node's power-of-two grid, so a
// plane distance is t = q * (step / d) + (origin - o) / d: one int-to-float conversion and one FMA per plane, on the
// SlabRay terms of the binary traversal (same FMA form, same rounding, covered by the same box padding); the near and far
// byte of every axis is picked once per node from the sign of the direction instead of a min / max per child.
// The hit slots are kept as a bit mask in TRAVERSAL-PRIORITY order (bit slot ^ octant, bvh8.h): the highest set bit is the
// next child, and what is left of a node's mask is its single stack entry.  Leaf slots (one primitive each) are solved in
// f64 as soon as the node has been tested - before any of its interior children is entered - so the nearest hits shrink
// the ray early.  No entry distances are stored: a stacked child the best hit has meanwhile beaten is culled when its node
// is fetched (all of its children miss), as in Ylitie et al.
struct TravW {
    SlabRay s;
    double best;   // closest accepted root so far
    float bestf;   // its f32 upper bound (with the slack of `slab`), for the node tests
    int best_leaf; // leaf | side << kLeafBits, or -1
    uint2 ng;      // interior children still to visit: x = child_base, y = pending slots (bits 8..15) | imask (bits 0..7)
    uint2 lg;      // leaf slots the last node test hit: x = prim_base, y = pending slots (bits 8..15) | leaf_mask
    uint32_t oct;  // bit k set: direction component k >= 0
    int sp;
};
// The wide tree's stack lives in shared memory only (one entry per LEVEL: 16 entries reach deeper than any tree the
// collapse of a <= 62-level binary tree is used for; deeper wide trees fall back to the binary traversal, api.cu).
#ifndef RT1W_WIDE_STACK
#define RT1W_WIDE_STACK 12 // entries per thread: with 12 the persistent kernel's CTA fits the 132 KB shared-memory carveout four times (more L1 for the nodes)
#endif
constexpr int kWideStack = RT1W_WIDE_STACK;
constexpr int kWideMaxDepth = kWideStack - 2;

// 8-bit slot mask -> priority order: bit (s ^ oct) of the result = bit s of m
RT1W_DEV uint32_t octant_order(uint32_t m, uint32_t oct) {
    if (oct & 1u) m = ((m & 0xaau) >> 1) | ((m & 0x55u) << 1);
    if (oct & 2u) m = ((m & 0xccu) >> 2) | ((m & 0x33u) << 2);
    if (oct & 4u) m = ((m & 0xf0u) >> 4) | ((m & 0x0fu) << 4);
    return m;
}
// the pending slot (bits 8..15 of y) a ray of octant `oct` visits next: the one with the highest slot ^ oct
RT1W_DEV uint32_t next_slot(uint32_t y, uint32_t oct) { return (31u - uint32_t(__clz(int(octant_order(y >> 8, oct))))) ^ oct; }

RT1W_DEV void trav_bind_stack(TravW &, const uint2 *) {} // (measured on the wide tree too: nothing, 190 of a step's 230 instructions are the box tests)
RT1W_DEV void trav_reset(TravW &T) { T.ng = make_uint2(0u, 0u), T.lg = make_uint2(0u, 0u), T.sp = 0; }
RT1W_DEV bool trav_at_leaf(const TravW &T) { return (T.lg.y >> 8) != 0u; }
RT1W_DEV bool trav_interior(const TravW &T) { return (T.lg.y >> 8) == 0u && ((T.ng.y >> 8) != 0u || T.sp > 0); }
RT1W_DEV bool trav_done(const TravW &T) { return (T.lg.y >> 8) == 0u && (T.ng.y >> 8) == 0u && T.sp <= 0; }

constexpr float kBestSlack = 1.000001f; // the f32 node tests against the f64 solve's best hit: rcp.approx scales every plane distance by up to 2^-23
RT1W_DEV void trav_begin(const SceneView &sc, const Ray &r, TravW &T) {
    RT1W_TRAV_COUNT(0);
    T.s.ix = rcp_capped(r.dx), T.s.iy = rcp_capped(r.dy), T.s.iz = rcp_capped(r.dz);
    T.s.ox = -__double2float_rn(r.ox) * T.s.ix, T.s.oy = -__double2float_rn(r.oy) * T.s.iy, T.s.oz = -__double2float_rn(r.oz) * T.s.iz;
    T.best = CUDART_INF, T.bestf = CUDART_INF_F, T.best_leaf = -1, T.sp = 0;
    T.oct = (T.s.ix >= 0.0f ? 1u : 0u) | (T.s.iy >= 0.0f ? 2u : 0u) | (T.s.iz >= 0.0f ? 4u : 0u);
    T.ng = make_uint2(0u, 0x100u); // the root: "slot 0 of nothing" (imask 0: index = base + 0)
    T.lg = make_uint2(0u, 0u);
}

// byte k of `word` -> the float 1 + byte 2^-15 (the byte lands in the second mantissa byte of 1.0f): one PRMT with an
// immediate selector; `one` = 0x3f800000 held in a register the compiler cannot see through (else it puts the
// CONSTANT into the instruction's immediate slot and spends a second instruction on moving the selector into a register)
template <int K> RT1W_DEV float byte_to_float(uint32_t word, uint32_t one) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(word), "r"(one), "n"(0x7604 | (K << 4)));
    return __uint_as_float(r);
}

// one node: fetch, test the eight child boxes, split the hits into the interior group and the leaf group
RT1W_DEV void wide_visit(const SceneView &sc, uint32_t node, TravW &T) {
    const uint4 *n = sc.wide_nodes + 5u * size_t(node);
    const uint4 w0 = __ldg(n), w1 = __ldg(n + 1), w2 = __ldg(n + 2), w3 = __ldg(n + 3), w4 = __ldg(n + 4);
    const uint32_t em = w0.w; // step exponents x, y, z and imask, one byte each
    // A plane byte q becomes the float 1 + q 2^-15 with ONE byte permute (an int-to-float conversion would go through the
    // quarter-rate XU pipe, 48 times per node), and
    // t = (1 + q 2^-15) * (2^15 step / d) + ((origin - o) / d - 2^15 step / d) = q step / d + (origin - o) / d.
    // The subtraction rounds by at most 2^-9 of a grid step; the builder keeps 2^-7 of a step between every child box
    // and its quantised planes (bvh8.cpp), so the decoded box still contains the conservative box.
    const float ax = __uint_as_float(((em & 0xffu) + 15u) << 23) * T.s.ix, ay = __uint_as_float((((em >> 8) & 0xffu) + 15u) << 23) * T.s.iy,
                az = __uint_as_float((((em >> 16) & 0xffu) + 15u) << 23) * T.s.iz;
    const float bx = fmaf(__uint_as_float(w0.x), T.s.ix, T.s.ox) - ax, by = fmaf(__uint_as_float(w0.y), T.s.iy, T.s.oy) - ay,
                bz = fmaf(__uint_as_float(w0.z), T.s.iz, T.s.oz) - az;
    // words of four bytes (slots 0-3, 4-7): lo.x = w2.xy, lo.y = w2.zw, lo.z = w3.xy, hi.x = w3.zw, hi.y = w4.xy, hi.z = w4.zw;
    // the near and the far plane of every axis by the sign of the direction
    const bool px = (T.oct & 1u) != 0u, py = (T.oct & 2u) != 0u, pz = (T.oct & 4u) != 0u;
    const uint32_t nx[2] = {px ? w2.x : w3.z, px ? w2.y : w3.w}, fx[2] = {px ? w3.z : w2.x, px ? w3.w : w2.y};
    const uint32_t ny[2] = {py ? w2.z : w4.x, py ? w2.w : w4.y}, fy[2] = {py ? w4.x : w2.z, py ? w4.y : w2.w};
    const uint32_t nz[2] = {pz ? w3.x : w4.z, pz ? w3.y : w4.w}, fz[2] = {pz ? w4.z : w3.x, pz ? w4.w : w3.y};
    uint32_t one;
    asm("mov.b32 %0, 0x3f800000;" : "=r"(one));
    uint32_t hits = 0u;
#define RT1W_WIDE_SLOT(S)                                                                                                              \
    {                                                                                                                                  \
        constexpr int h = (S) >> 2, k = (S) & 3;                                                                                       \
        const float tnx = fmaf(byte_to_float<k>(nx[h], one), ax, bx), tfx = fmaf(byte_to_float<k>(fx[h], one), ax, bx);               \
        const float tny = fmaf(byte_to_float<k>(ny[h], one), ay, by), tfy = fmaf(byte_to_float<k>(fy[h], one), ay, by);               \
        const float tnz = fmaf(byte_to_float<k>(nz[h], one), az, bz), tfz = fmaf(byte_to_float<k>(fz[h], one), az, bz);               \
        const float tn = fmaxf(max3(tnx, tny, tnz), 0.0f);                                                                             \
        const float tf = fminf(min3(tfx, tfy, tfz), T.bestf);                                                                          \
        if (tn <= tf) hits |= 1u << (S);                                                                                               \
    }
    RT1W_WIDE_SLOT(0) RT1W_WIDE_SLOT(1) RT1W_WIDE_SLOT(2) RT1W_WIDE_SLOT(3) RT1W_WIDE_SLOT(4) RT1W_WIDE_SLOT(5) RT1W_WIDE_SLOT(6) RT1W_WIDE_SLOT(7)
#undef RT1W_WIDE_SLOT
    const uint32_t imask = em >> 24, lmask = w1.z & 0xffu; // empty slots are in neither
    T.ng = make_uint2(w1.x, ((hits & imask) << 8) | imask);
    T.lg = make_uint2(w1.y, ((hits & lmask) << 8) | lmask);
}

// the nearest pending interior child (of this node, else of the most recent node with children left)
RT1W_DEV void trav_step_interior(const SceneView &sc, TravW &T, uint2 *stack, int stride, uint2 *) {
    RT1W_TRAV_COUNT(1);
#ifdef RT1W_COUNT_TRAV
    if (int(threadIdx.x & 31) == __ffs(int(__activemask())) - 1) RT1W_TRAV_COUNT(3);
#endif
    if ((T.ng.y >> 8) == 0u) T.ng = stack[--T.sp * stride];
    const uint32_t slot = next_slot(T.ng.y, T.oct);
    const uint32_t node = T.ng.x + uint32_t(__popc(T.ng.y & ((1u << slot) - 1u))); // interior children below `slot` (imask: bits 0..7)
    T.ng.y &= ~(0x100u << slot);
    if ((T.ng.y >> 8) != 0u) stack[T.sp++ * stride] = T.ng; // its siblings wait on the stack
    wide_visit(sc, node, T);
}

// the leaf slots the last node test hit, nearest first: f64 solves
template <bool EXACT, bool MEDIA>
RT1W_DEV void trav_step_leaf(const SceneView &sc, const Ray &r, const MediumRng &mr, TravW &T, const uint2 *, int, const uint2 *) {
    const uint32_t lmask = T.lg.y & 0xffu;
    while ((T.lg.y >> 8) != 0u) {
        const uint32_t slot = next_slot(T.lg.y, T.oct);
        T.lg.y &= ~(0x100u << slot);
        const int leaf = int(T.lg.x + uint32_t(__popc(lmask & ((1u << slot) - 1u))));
        uint32_t box_sides = 0u;
        do {
            double t;
            int side = 0;
            RT1W_TRAV_COUNT(2);
            if (hit_prim<EXACT, MEDIA, true>(sc, sc.frames, sc.prims + leaf, leaf, r, T.best, mr, t, box_sides, side)) {
                T.best = t, T.best_leaf = leaf | (side << kLeafBits);
                T.bestf = __double2float_ru(t) * kBestSlack;
            }
        } while (box_sides != 0u);
    }
}

template <bool EXACT, bool MEDIA>
RT1W_DEV bool closest_hit_wide(const SceneView &sc, const Ray &r, const MediumRng &mr, uint2 *stack, int stride, double &t_best, int &leaf_best) {
    TravW T;
    trav_bind_stack(T, stack);
    trav_begin(sc, r, T);
    for (;;) {
        while (trav_interior(T)) trav_step_interior(sc, T, stack, stride, nullptr);
        if (!trav_at_leaf(T)) break;
        trav_step_leaf<EXACT, MEDIA>(sc, r, mr, T, stack, stride, nullptr);
    }
    hit_globals<EXACT, MEDIA>(sc, r, mr, T.best, T.best_leaf);
    t_best = T.best, leaf_best = T.best_leaf;
    return T.best_leaf >= 0;
}

// Small scenes (<= kFlatMax primitives and <= kFlatMaxFrames wrapper chains, e.g. the 13 + 1 of the Cornell
// box): a BVH over a handful of room-sized rectangles culls nothing, so the extend kernel scans the primitive
// list instead.  Records, boxes and frames sit in shared memory.
//   pass 1 (warp-uniform, f32): every lane slab-tests the same primitive at the same time (broadcast reads, no
//     divergence).  Boxes are the primitives' bounds in their OWN frame (tight around rotated box sides),
//     grouped by frame so the ray is re-expressed once per group; the entry distance of every box the ray
//     crosses beyond t_min is parked in shared memory and the nearest one is tracked.
//     Rectangles that are whole faces of one axis-aligned box in a frame (the five walls of the Cornell room, the
//     six sides of an AABox, aabox.rs:29-76) form a FACE GROUP (api.cu: find_face_groups): ONE slab computation on
//     the box names the face the ray enters through and the one it leaves through (the plane distances carry
//     their face number in the three lowest mantissa bits through the min / max network), and only those two
//     become candidates.  Rays that pass an edge of the box within the padding take a per-face path.
//   pass 2 (per lane, f64): solve the nearest candidate, then the nearest remaining one whose box is entered
//     before the best hit so far (the entry distance is a lower bound of the primitive's t), and so on:
//     ~1.2 solves per ray.
#ifndef RT1W_SCAN_UNROLL
#define RT1W_SCAN_UNROLL 1 // the wave kernel is bound by its instruction-cache footprint: unrolling by 4 was 5 % slower
#endif
constexpr int kScanUnroll = RT1W_SCAN_UNROLL;
#ifdef RT1W_COUNT_SOLVES // measurement build (build.py --variant count -DRT1W_COUNT_SOLVES): rays, pass-1 candidates, f64 solves, warp-level solve iterations
static __device__ unsigned long long g_scan_counts[4];
#endif
struct FlatScene {
    DPrim prims[kFlatMax];             // leaf order
    float4 lo[kFlatMax], hi[kFlatMax]; // scan order: padded f32 bounds in the frame of the group; lo.w = leaf (int bits)
    float4 sphere[kFlatMax];           // scan order, sphere groups: centre and radius in f32
    DFrame frames[kFlatMaxFrames];
    float4 frame_f[kFlatMaxFrames][2]; // f32 copy of the rigid part for pass 1: (sin, cos, b.x, b.y), (b.z, -, -, -)
    FlatGroups groups;                 // the scan-order groups (flat_plans.h), as the host built them
    uint32_t skip_bit[kFlatMax]; // leaf -> scan bit of a rectangle (a ray leaving a rectangle cannot hit it again), else 0
};

RT1W_DEV void flat_stage(const SceneView &sc, FlatScene &fs) { // call with the whole CTA, then __syncthreads()
    const int n = sc.n_prims;
    const uint32_t *src = reinterpret_cast<const uint32_t *>(sc.prims);
    uint32_t *dst = reinterpret_cast<uint32_t *>(fs.prims);
    for (int w = threadIdx.x; w < n * int(sizeof(DPrim) / 4); w += blockDim.x) dst[w] = src[w];
    src = reinterpret_cast<const uint32_t *>(sc.frames), dst = reinterpret_cast<uint32_t *>(fs.frames);
    for (int w = threadIdx.x; w < sc.n_frames * int(sizeof(DFrame) / 4); w += blockDim.x) dst[w] = src[w];
    for (int i = threadIdx.x; i < sc.n_frames; i += blockDim.x) {
        const DFrame &f = sc.frames[i];
        fs.frame_f[i][0] = make_float4(float(f.sin_t), float(f.cos_t), float(f.bx), float(f.by));
        fs.frame_f[i][1] = make_float4(float(f.bz), 0.0f, 0.0f, 0.0f);
    }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float4 lo = sc.prim_boxes[2 * i], hi = sc.prim_boxes[2 * i + 1];
        fs.lo[i] = lo, fs.hi[i] = hi;
        const DPrim &p = sc.prims[__float_as_int(lo.w)];
        fs.sphere[i] = make_float4(float(p.p[0]), float(p.p[1]), float(p.p[2]), float(p.p[3]));
        const int type = int(p.meta & 15u);
        fs.skip_bit[__float_as_int(lo.w)] = (type == P_XY_RECT || type == P_XZ_RECT || type == P_YZ_RECT) ? 1u << i : 0u;
    }
    static_assert(sizeof(FlatGroups) % 4 == 0, "group table copied in words");
    src = reinterpret_cast<const uint32_t *>(sc.flat_groups), dst = reinterpret_cast<uint32_t *>(&fs.groups);
    for (int w = threadIdx.x; w < int(sizeof(FlatGroups) / 4); w += blockDim.x) dst[w] = src[w];
}

// Slab test in the FMA form t = plane * (1/d) - o * (1/d).  |1/d| is capped at 1e18 so that no product
// overflows: an axis the ray is parallel to yields -+1e18-scale distances of the right sign instead of
// inf - inf.  The rounding of the form (cancellation 2^-23 |o / d|, rcp.approx 2^-23 |t|) is covered by the
// box padding (api.cu: scan_pad), so the comparison itself carries no slack.
struct SlabRayF {
    float ix, iy, iz, ox, oy, oz; // 1/d and -o/d
};
RT1W_DEV SlabRayF slab_ray(float ox, float oy, float oz, float dx, float dy, float dz) {
    SlabRayF s;
    s.ix = rcp_capped(dx), s.iy = rcp_capped(dy), s.iz = rcp_capped(dz);
    s.ox = -ox * s.ix, s.oy = -oy * s.iy, s.oz = -oz * s.iz;
    return s;
}
constexpr float kTMinSlab = 0.000999f; // just below t_min: a box the ray leaves before t_min cannot hold an accepted root
RT1W_DEV bool slab_fma(const float4 lo, const float4 hi, const SlabRayF &s, float &tnear) {
    const float ax = fmaf(lo.x, s.ix, s.ox), bx = fmaf(hi.x, s.ix, s.ox);
    const float ay = fmaf(lo.y, s.iy, s.oy), by = fmaf(hi.y, s.iy, s.oy);
    const float az = fmaf(lo.z, s.iz, s.oz), bz = fmaf(hi.z, s.iz, s.oz);
    tnear = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fmaxf(fminf(az, bz), kTMinSlab));
    const float tf = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fmaxf(az, bz));
    return tnear <= tf;
}

// a plane distance with its face number in the three lowest mantissa bits (face groups)
RT1W_DEV float face_tag(float t, uint32_t face) { return __uint_as_float((__float_as_uint(t) & ~7u) | face); }

// f32 screen of a plain sphere on top of its box: false only when the ray certainly misses it beyond t_min
// (discriminant below its rounding bound, or sphere behind an origin outside it).
RT1W_DEV bool sphere_maybe(const float4 sp, f3 o, f3 d) {
    const f3 oc = mk3(o.x - sp.x, o.y - sp.y, o.z - sp.z);
    const float a = dot(d, d), hb = dot(oc, d), oc2 = dot(oc, oc), r2 = sp.w * sp.w;
    const float cc = oc2 - r2, scale = oc2 + r2;
    const float disc = hb * hb - a * cc;
    if (disc < -4e-6f * (hb * hb + a * scale)) return false;
    return !(cc > 4e-6f * scale && hb > 0.0f);
}

// Pass 1 of the flat scan, one group at a time.  The generic scan (closest_hit_flat without a plan) reads the group table;
// a planned one (flat_plans.h) is unrolled over the plan's groups at compile time.  Both run these bodies, in scan order,
// so they find the same candidates, entry distances and nearest candidate (the first one in scan order on a tie).
struct ScanAcc {
    uint32_t cand; // scan bits of the candidates
    float t1;      // the nearest entry distance so far, and its slot
    int k1;
};

// the ray in frame `frame` (-1 = world) for the slab tests, f32
RT1W_DEV SlabRayF frame_slab_ray(const FlatScene &fs, int frame, const Ray &r, float ofx, float ofy, float ofz) {
    if (frame < 0) return slab_ray(ofx, ofy, ofz, r.dx, r.dy, r.dz);
    // hittable.rs:207,241-245 in f32: 1e-4 of error at Cornell coordinates, inside the box padding (api.cu)
    const float4 f0 = fs.frame_f[frame][0], f1 = fs.frame_f[frame][1]; // sin, cos, b.x, b.y | b.z
    return slab_ray(fmaf(f0.y, ofx, fmaf(-f0.x, ofz, f0.z)), ofy + f0.w, fmaf(f0.x, ofx, fmaf(f0.y, ofz, f1.x)),
                    fmaf(f0.y, r.dx, -f0.x * r.dz), r.dy, fmaf(f0.x, r.dx, f0.y * r.dz));
}

// the ray in frame `frame` for the sphere screen, f32
RT1W_DEV void sphere_group_ray(const FlatScene &fs, int frame, const Ray &r, f3 &o, f3 &d) {
    if (frame < 0) {
        o = mk3(float(r.ox), float(r.oy), float(r.oz)), d = mk3(r.dx, r.dy, r.dz);
    } else {
        const LocalRay l = to_local(frame_xf(fs.frames, frame), r);
        o = mk3(float(l.ox), float(l.oy), float(l.oz)), d = mk3(float(l.dx), float(l.dy), float(l.dz));
    }
}

// A face group whose slots start at k: face f's slot is slots(f), or -1.  group_delta: the group's delta (FlatGroups).
template <class Slots>
RT1W_DEV void scan_faces(const FlatScene &fs, const SlabRayF &s, int k, float group_delta, const Slots &slots, uint32_t keep, float *tn_col,
                         int stride, ScanAcc &acc) {
    // One slab computation for all faces of the group's box.  Plane distances are tagged with their face number
    // (lowest three mantissa bits), so the entry distance max(near) and the exit distance min(far) name their face.
    const float4 lo = fs.lo[k], hi = fs.hi[k];
    const float ax = face_tag(fmaf(lo.x, s.ix, s.ox), 0u), bx = face_tag(fmaf(hi.x, s.ix, s.ox), 1u);
    const float ay = face_tag(fmaf(lo.y, s.iy, s.oy), 2u), by = face_tag(fmaf(hi.y, s.iy, s.oy), 3u);
    const float az = face_tag(fmaf(lo.z, s.iz, s.oz), 4u), bz = face_tag(fmaf(hi.z, s.iz, s.oz), 5u);
    const float nx = fminf(ax, bx), ny = fminf(ay, by), nz = fminf(az, bz);
    const float fx = fmaxf(ax, bx), fy = fmaxf(ay, by), fz = fmaxf(az, bz);
    const float tn_raw = fmaxf(fmaxf(nx, ny), nz), tf = fminf(fminf(fx, fy), fz);
    const float tn = fmaxf(tn_raw, kTMinSlab);
    if (!(tn <= tf)) return;
    // A computed plane distance is within 2 * padding / |d_axis| of the true one (the padding covers the
    // rounding, see slab_fma): with delta = the sum over the axes, the face named by max / min is the true one
    // whenever the runner-up is further than delta away.
    const float delta = group_delta * (fabsf(s.ix) + fabsf(s.iy) + fabsf(s.iz));
    const float mid_n = fmaxf(fminf(nx, ny), fminf(fmaxf(nx, ny), nz));
    const float mid_f = fminf(fmaxf(fx, fy), fmaxf(fminf(fx, fy), fz));
    // the padded planes are crossed before the true ones: an entry up to delta before t_min may be a hit beyond it
    const bool enters = tn_raw + delta >= kTMinSlab;
    if (!((enters && mid_n >= tn_raw - delta) || mid_f <= tf + delta)) { // sure of the entry and of the exit face
        if (enters) { // the face the ray enters through (a ray leaving a face of the group names that face: skipped)
            const int sl = slots(__float_as_uint(tn_raw) & 7u);
            if (sl >= 0 && ((keep >> sl) & 1u)) {
                tn_col[sl * stride] = tn, acc.cand |= 1u << sl;
                if (tn < acc.t1) acc.t1 = tn, acc.k1 = sl;
            }
        }
        const int sl = slots(__float_as_uint(tf) & 7u); // the face it leaves through
        if (sl >= 0 && ((keep >> sl) & 1u)) {
            const float te = fmaxf(tf - delta, tn);
            tn_col[sl * stride] = te, acc.cand |= 1u << sl;
            if (te < acc.t1) acc.t1 = te, acc.k1 = sl;
        }
    } else { // the ray passes an edge of the box within the padding: every face whose plane it crosses inside the box
#pragma unroll 1
        for (int f = 0; f < 6; ++f) {
            const int sl = slots(uint32_t(f));
            if (sl < 0 || !((keep >> sl) & 1u)) continue;
            const int a = f >> 1;
            const float plane = reinterpret_cast<const float *>((f & 1) ? &fs.hi[k] : &fs.lo[k])[a];
            const float tp = fmaf(plane, a == 0 ? s.ix : (a == 1 ? s.iy : s.iz), a == 0 ? s.ox : (a == 1 ? s.oy : s.oz));
            if (tp + delta >= tn && tp - delta <= tf) {
                const float te = fmaxf(tp - delta, tn);
                tn_col[sl * stride] = te, acc.cand |= 1u << sl;
                if (te < acc.t1) acc.t1 = te, acc.k1 = sl;
            }
        }
    }
}

// slot k (scan bit `bit`) of a box group
RT1W_DEV void scan_box(const FlatScene &fs, const SlabRayF &s, int k, uint32_t bit, uint32_t keep, float *tn_col, int stride, ScanAcc &acc) {
    float tn;
    const bool in = slab_fma(fs.lo[k], fs.hi[k], s, tn) && (bit & keep) != 0u;
    tn_col[k * stride] = tn;
    if (in) acc.cand |= bit;
    if (in && tn < acc.t1) acc.t1 = tn, acc.k1 = k;
}

// slot k (scan bit `bit`) of a sphere group; (o, d): sphere_group_ray
RT1W_DEV void scan_sphere(const FlatScene &fs, const SlabRayF &s, f3 o, f3 d, int k, uint32_t bit, float *tn_col, int stride, ScanAcc &acc) {
    float tn;
    const bool in = slab_fma(fs.lo[k], fs.hi[k], s, tn) && sphere_maybe(fs.sphere[k], o, d);
    tn_col[k * stride] = tn;
    if (in) acc.cand |= bit;
    if (in && tn < acc.t1) acc.t1 = tn, acc.k1 = k;
}

struct TableSlots { // the generic scan's face map: a row of FlatGroups::face_slot
    const int8_t *slot;
    RT1W_DEV int operator()(uint32_t f) const { return slot[f]; }
};
template <int BEGIN, uint32_t FACES> struct PlanSlots { // a plan's face map, an immediate (FlatPlanGroup::faces)
    RT1W_DEV int operator()(uint32_t f) const {
        const uint32_t nib = (FACES >> (4u * f)) & 15u;
        return nib == 15u ? -1 : BEGIN + int(nib);
    }
};

template <bool MEDIA>
RT1W_DEV void scan_groups(const FlatScene &fs, const Ray &r, float ofx, float ofy, float ofz, uint32_t keep, float *tn_col, int stride, ScanAcc &acc) {
    const FlatGroups &gt = fs.groups;
    const int n_groups = gt.n_groups;
    uint32_t bit = 1;
    int k = 0, cur_frame = -2;
    SlabRayF s;
    for (int g = 0; g < n_groups; ++g) {
        const int frame = gt.frame[g], end = gt.end[g];
        if (frame != cur_frame) cur_frame = frame, s = frame_slab_ray(fs, frame, r, ofx, ofy, ofz);
        const int kind = gt.kind[g];
        if (kind == int(G_FACES)) {
            scan_faces(fs, s, k, gt.delta[g], TableSlots{gt.face_slot[g]}, keep, tn_col, stride, acc);
            k = end, bit = uint32_t(1ull << end);
        } else if (kind == int(G_SPHERES)) {
            f3 o, d;
            sphere_group_ray(fs, frame, r, o, d);
            // measured per kernel: with the loop rolled cornel_smoke gains 2.8 % (instruction fetch), the Cornell box loses 0.6 %
            if (MEDIA) {
#pragma unroll 1
                for (; k < end; ++k, bit <<= 1) scan_sphere(fs, s, o, d, k, bit, tn_col, stride, acc);
            } else {
                for (; k < end; ++k, bit <<= 1) scan_sphere(fs, s, o, d, k, bit, tn_col, stride, acc);
            }
        } else {
#pragma unroll(kScanUnroll)
            for (; k < end; ++k, bit <<= 1) scan_box(fs, s, k, bit, keep, tn_col, stride, acc);
        }
    }
}

// Group G of plan P onwards: frame switches, kinds, slots and scan bits are constants.
template <int P, int G>
RT1W_DEV void scan_plan(const FlatScene &fs, const Ray &r, float ofx, float ofy, float ofz, uint32_t keep, float *tn_col, int stride, SlabRayF &s,
                        ScanAcc &acc) {
    constexpr FlatPlanGroup q = kFlatPlans[P].g[G];
    if constexpr (G == 0 || kFlatPlans[P].g[G > 0 ? G - 1 : 0].frame != q.frame) s = frame_slab_ray(fs, q.frame, r, ofx, ofy, ofz);
    if constexpr (q.kind == G_FACES) {
        scan_faces(fs, s, q.begin, fs.groups.delta[G], PlanSlots<q.begin, q.faces>{}, keep, tn_col, stride, acc);
    } else if constexpr (q.kind == G_SPHERES) {
        f3 o, d;
        sphere_group_ray(fs, q.frame, r, o, d);
#pragma unroll
        for (int k = q.begin; k < q.end; ++k) scan_sphere(fs, s, o, d, k, 1u << k, tn_col, stride, acc);
    } else {
#pragma unroll
        for (int k = q.begin; k < q.end; ++k) scan_box(fs, s, k, 1u << k, keep, tn_col, stride, acc);
    }
    if constexpr (G + 1 < kFlatPlans[P].n_groups) scan_plan<P, G + 1>(fs, r, ofx, ofy, ofz, keep, tn_col, stride, s, acc);
}

// Pass 2 of a planned scan: candidate slot k (record Pr) solved by the class of its group - the hit_rect / hit_sphere /
// to_local calls of hit_prim, with the same arguments, without the type dispatch and with no code for the kinds a plan
// cannot hold (moving spheres, boxes, media).  ONE rectangle call site for walls, lights and box sides, the axis as data
// (DESIGN.md section 6).  The frame is read from the record as hit_prim reads it: the plan's slot-to-frame map instead
// cost the Cornell k_wave an 8-byte spill at its 80-register cap.
template <int P> RT1W_DEV bool hit_planned(const FlatScene &fs, int k, const DPrim *Pr, const Ray &r, double tmax, double &t) {
    const double2 *w = reinterpret_cast<const double2 *>(Pr);
    const int4 tail = *reinterpret_cast<const int4 *>(w + 3); // q2 | meta | frame
    const double2 p01 = w[0], p23 = w[1];
    const LocalRay l = to_local(tail.w < 0 ? nullptr : frame_xf(fs.frames, tail.w), r);
    constexpr uint32_t spheres = plan_slots(kFlatPlans[P], C_SPHERES);
    if ((spheres >> k) & 1u) return hit_sphere(l, p01.x, p01.y, p23.x, p23.y, kTMin, tmax, t);
    return hit_rect(l, P_YZ_RECT - int(uint32_t(tail.z) & 15u), p01.x, p01.y, p23.x, p23.y, w[2].x, kTMin, tmax, t);
}

// `tn_col`: this thread's column of the CTA's entry-distance table (stride = blockDim.x floats).
// `skip_leaf`: the rectangle the ray starts on (its only root is t ~ 0 < t_min), or -1.
// PLAN: the scene's plan (SceneView::flat_plan), or -1 for the generic scan of the group table and hit_prim.
template <bool EXACT, bool MEDIA, int PLAN = -1>
RT1W_DEV bool closest_hit_flat(const SceneView &sc, const FlatScene &fs, const Ray &r, const MediumRng &mr, float *tn_col, int stride,
                               int skip_leaf, double &t_best, int &leaf_best) {
    const uint32_t keep = ~(skip_leaf >= 0 ? fs.skip_bit[skip_leaf] : 0u);
    ScanAcc acc = {0u, CUDART_INF_F, -1};
    const float ofx = __double2float_rn(r.ox), ofy = __double2float_rn(r.oy), ofz = __double2float_rn(r.oz);
    if constexpr (PLAN >= 0) {
        SlabRayF s;
        scan_plan<PLAN, 0>(fs, r, ofx, ofy, ofz, keep, tn_col, stride, s, acc);
    } else {
        scan_groups<MEDIA>(fs, r, ofx, ofy, ofz, keep, tn_col, stride, acc);
    }
    uint32_t cand = acc.cand;
    double best = CUDART_INF;
    float bestf = CUDART_INF_F;
    int best_leaf = -1;
    int k = acc.k1;
#ifdef RT1W_COUNT_SOLVES
    atomicAdd(&g_scan_counts[0], 1ull), atomicAdd(&g_scan_counts[1], (unsigned long long)__popc(cand));
#endif
    while (k >= 0) {
#ifdef RT1W_COUNT_SOLVES
        atomicAdd(&g_scan_counts[2], 1ull);
        if (int(threadIdx.x & 31) == __ffs(int(__activemask())) - 1) atomicAdd(&g_scan_counts[3], 1ull);
#endif
        cand &= ~(1u << k);
        const int leaf = __float_as_int(fs.lo[k].w);
        double t;
        bool hit;
        if constexpr (PLAN >= 0) {
            hit = hit_planned<PLAN>(fs, k, fs.prims + leaf, r, best, t);
        } else {
            uint32_t box_sides = 0u;
            int side = 0;
            hit = hit_prim<EXACT, MEDIA, false>(sc, fs.frames, fs.prims + leaf, leaf, r, best, mr, t, box_sides, side);
        }
        if (hit) {
            best = t, best_leaf = leaf;
            bestf = __double2float_ru(t) * 1.000001f;
        }
        // next: the nearest remaining box that starts before the best hit; boxes beyond it are dropped for good
        k = -1;
        float tb = bestf;
        for (uint32_t m = cand; m != 0u; m &= m - 1u) {
            const int c = __ffs(int(m)) - 1;
            const float tc = tn_col[c * stride];
            if (tc <= tb) tb = tc, k = c;
            else if (tc > bestf) cand &= ~(1u << c);
        }
    }
    t_best = best, leaf_best = best_leaf;
    return best_leaf >= 0;
}

// ------------------------------------------------------------------------------------------
// HitRecord reconstruction (hittable.rs:10-47 + the wrapper rewrites)
// ------------------------------------------------------------------------------------------
struct HitInfo {
    double px, py, pz; // position
    f3 normal;         // oriented normal as the material sees it
    f3 n_out;          // outward unit normal in the leaf's own space (sphere_uv input)
    float u, v;
    bool front_face;
    int type; // PrimType
    uint32_t meta;
    // where the record came from, so that an image texture can ask for a rectangle's (u, v) after the fact (rect_uv)
    const DPrim *prim;
    const DFrame *frames;
    int side;
};

RT1W_DEV void sphere_uv(f3 p, float &u, float &v) { // math.rs:67-71
    // theta = acos(-y), written as atan2(|xz|, -y): identical for a unit vector but well conditioned
    // at the poles, where acos would amplify the f32 rounding of y to 1e-4
    const float theta = atan2f(sqrtf(fmaf(p.z, p.z, __fmul_rn(p.x, p.x))), -p.y);
    const float phi = atan2f(-p.z, p.x) + kPiF;
    u = phi * (0.5f / kPiF), v = theta * (1.0f / kPiF);
}

// (u, v) of a hit on a rectangle or a box side (aarect.rs:60-61,98-99,166-167): the hit point's in-plane coordinates
// normalised by the rectangle's intervals.  `type`: P_XY_RECT / P_XZ_RECT / P_YZ_RECT (for a P_BOX: the side's type),
// (lx, ly, lz): the hit point in the leaf's own space.
RT1W_DEV void rect_uv(const DPrim *P, int type, double lx, double ly, double lz, float &u, float &v) {
    const double2 *w = reinterpret_cast<const double2 *>(P);
    const double2 p01 = w[0], p23 = w[1];
    const double a = type == P_YZ_RECT ? ly : lx, b = type == P_XY_RECT ? ly : lz;
    double a0 = p01.x, a1 = p01.y, b0 = p23.x, b1 = p23.y;
    if (int(P->meta & 15u) == P_BOX) { // the side's in-plane intervals out of the box corners
        const int4 tail = *reinterpret_cast<const int4 *>(w + 3);
        const double2 q01 = w[2];
        const double x0 = p01.x, y0 = p01.y, z0 = p23.x, x1 = q01.x, y1 = q01.y, z1 = __hiloint2double(tail.y, tail.x);
        a0 = type == P_YZ_RECT ? y0 : x0, a1 = type == P_YZ_RECT ? y1 : x1;
        b0 = type == P_XY_RECT ? y0 : z0, b1 = type == P_XY_RECT ? y1 : z1;
    }
    u = float((a - a0) / (a1 - a0));
    v = float((b - b0) / (b1 - b0));
}

// P: the primitive's record, frames: the wrapper frames (global memory or the flat scan's shared-memory copies).
// `side`: which rectangle of a P_BOX was hit (see kLeafBits).
// PLAN: the scene's plan (flat_plans.h): the wrapper chains unrolled, no code for the kinds the plan cannot hold; or -1.
template <bool WANT_UV, int PLAN = -1> RT1W_DEV HitInfo finalize_hit(const DPrim *P, const DFrame *frames, int side, const Ray &r, double t) {
    HitInfo h;
    const double2 *w = reinterpret_cast<const double2 *>(P);
    const int4 tail = *reinterpret_cast<const int4 *>(w + 3);
    h.meta = uint32_t(tail.z);
    h.type = int(h.meta & 15u);
    h.prim = P, h.frames = frames, h.side = side;
    const bool box = PLAN < 0 && h.type == P_BOX;
    if (box) h.type = P_XY_RECT + (side >> 1); // the sides come in the order XY, XY, XZ, XZ, YZ, YZ (aabox.rs:29-76)
    const int frame = tail.w;
    // ray.at(t) is invariant under the rigid wrappers; evaluate it once in world space
    h.px = __fma_rn(t, double(r.dx), r.ox), h.py = __fma_rn(t, double(r.dy), r.oy), h.pz = __fma_rn(t, double(r.dz), r.oz);
    h.u = 0.0f, h.v = 0.0f;
    f3 n; // outward normal in the leaf's own space, then the record's normal on its way out through the wrappers
    bool ff;
    if (PLAN < 0 && (h.type == P_MEDIUM_SPHERE || h.type == P_MEDIUM_BOX)) { // constant_medium.rs:98-106: a literal record, not HitRecord::new;
        n = mk3(1.0f, 0.0f, 0.0f), ff = true;                  // the wrappers ABOVE the medium still rewrite it (the frame's ops)
        h.n_out = n;
    } else {
        f3 ld;             // ray direction in the leaf's own space
        double lx, ly, lz; // hit point in the leaf's own space
        if (frame < 0) {
            ld = mk3(r.dx, r.dy, r.dz);
            lx = h.px, ly = h.py, lz = h.pz;
        } else { // hittable.rs:207,241-245
            const FrameXf *f = frame_xf(frames, frame);
            const double s = f->sin_t, c = f->cos_t;
            ld = mk3(float(__fma_rn(c, double(r.dx), -__dmul_rn(s, double(r.dz)))), r.dy, float(__fma_rn(s, double(r.dx), __dmul_rn(c, double(r.dz)))));
            lx = __dadd_rn(__fma_rn(c, h.px, -__dmul_rn(s, h.pz)), f->bx), ly = __dadd_rn(h.py, f->by), lz = __dadd_rn(__fma_rn(s, h.px, __dmul_rn(c, h.pz)), f->bz);
        }
        if (h.type == P_SPHERE || (PLAN < 0 && h.type == P_MOVING_SPHERE)) {
            const double2 p01 = w[0], p23 = w[1];
            double cx = p01.x, cy = p01.y, cz = p23.x;
            if (PLAN < 0 && h.type == P_MOVING_SPHERE) {
                const float4 f = *reinterpret_cast<const float4 *>(w + 2);
                const double s = double((r.time - f.w) * __int_as_float(tail.x));
                cx = __fma_rn(s, double(f.x), cx), cy = __fma_rn(s, double(f.y), cy), cz = __fma_rn(s, double(f.z), cz);
            }
            const float inv_r = 1.0f / float(p23.y); // sphere.rs:51
            n = mk3(float(lx - cx) * inv_r, float(ly - cy) * inv_r, float(lz - cz) * inv_r);
            if (WANT_UV) sphere_uv(n, h.u, h.v);
            ff = dot(ld, n) < 0.0f; // HitRecord::new at the leaf, with the leaf-space ray (hittable.rs:30-35)
        } else {
            float dn;
            if (h.type == P_XY_RECT) n = mk3(0.0f, 0.0f, 1.0f), dn = ld.z;
            else if (h.type == P_XZ_RECT) n = mk3(0.0f, 1.0f, 0.0f), dn = ld.y;
            else n = mk3(1.0f, 0.0f, 0.0f), dn = ld.x;
            if (WANT_UV) rect_uv(P, h.type, lx, ly, lz, h.u, h.v); // aarect.rs:60-61
            ff = dn < 0.0f;
        }
        h.n_out = n;
        if (!ff) n = -n;
    }
    if (frame >= 0) {
        const DFrame *f = frames + frame;
        // a plan's chain: op count and kinds are constants (its one frame: plan_chain_kinds), the loop is unrolled
        constexpr uint32_t kPlanOps = PLAN >= 0 ? plan_chain_kinds(kFlatPlans[PLAN < 0 ? 0 : PLAN]) : 0u;
        const int n_ops = PLAN >= 0 ? int(kPlanOps & 15u) : f->n_ops;
        constexpr int kUnroll = PLAN >= 0 ? RT1W_MAX_CHAIN_OPS : 1;
#pragma unroll(kUnroll) // (unrolled by four otherwise: 1.7 KB more per copy of this function in kernels bound by instruction fetch; Cornell +1.9 %, cornel_smoke +3.7 %)
        for (int i = 0; i < n_ops; ++i) { // innermost wrapper first
            const DChainOp op = f->ops[i];
            const int kind = PLAN >= 0 ? int((kPlanOps >> (4 * i + 4)) & 15u) : op.kind;
            if (kind == OP_FLIP_FACE) { // hittable.rs:290-294
                ff = !ff;
                continue;
            }
            if (kind == OP_ROTATE_Y) { // hittable.rs:263-267
                const float nx = fmaf(op.cos_own, n.x, __fmul_rn(op.sin_own, n.z));
                const float nz = fmaf(-op.sin_own, n.x, __fmul_rn(op.cos_own, n.z));
                n.x = nx, n.z = nz;
            }
            // both wrappers re-run HitRecord::new with the ray INSIDE the wrapper (hittable.rs:221-229,269-277)
            const float dx = fmaf(op.cos_cum, r.dx, -__fmul_rn(op.sin_cum, r.dz));
            const float dz = fmaf(op.sin_cum, r.dx, __fmul_rn(op.cos_cum, r.dz));
            ff = dot(mk3(dx, r.dy, dz), n) < 0.0f;
            if (!ff) n = -n;
        }
    } else if ((h.meta >> 4) & PF_FLIP_FACE) {
        ff = !ff;
    }
    h.normal = n;
    h.front_face = ff;
    return h;
}

// front_face of a hit on a rectangle that sits under no wrapper chain (what finalize_hit computes for it), without the
// rest of the record: `dot(direction, +axis) < 0` (aarect.rs:62-70 with hittable.rs:30-35), toggled by FlipFace
// (hittable.rs:290-294).  Returns false for every other primitive.
RT1W_DEV bool plain_rect_front_face(const DPrim *P, const Ray &r, bool &front_face) {
    const int type = int(P->meta & 15u);
    if (P->frame >= 0 || (type != P_XY_RECT && type != P_XZ_RECT && type != P_YZ_RECT)) return false;
    const float dn = type == P_XY_RECT ? r.dz : (type == P_XZ_RECT ? r.dy : r.dx);
    front_face = (dn < 0.0f) != (((P->meta >> 4) & PF_FLIP_FACE) != 0u);
    return true;
}

// ------------------------------------------------------------------------------------------
// Textures (texture.rs, perlin.rs)
// ------------------------------------------------------------------------------------------
RT1W_DEV float perlin_noise(const DPerlin *tab, double px, double py, double pz) { // perlin.rs:46-72,88-106
    const double fx = floor(px), fy = floor(py), fz = floor(pz);
    const float u = float(px - fx), v = float(py - fy), w = float(pz - fz);
    const int i = int((long long)fx), j = int((long long)fy), k = int((long long)fz);
    const float uu = __fmul_rn(__fmul_rn(u, u), fmaf(-2.0f, u, 3.0f)), vv = __fmul_rn(__fmul_rn(v, v), fmaf(-2.0f, v, 3.0f));
    const float ww = __fmul_rn(__fmul_rn(w, w), fmaf(-2.0f, w, 3.0f));
    float accum = 0.0f;
#pragma unroll
    for (int di = 0; di < 2; ++di)
#pragma unroll
        for (int dj = 0; dj < 2; ++dj)
#pragma unroll
            for (int dk = 0; dk < 2; ++dk) {
                const int idx = tab->perm[0][(i + di) & 255] ^ tab->perm[1][(j + dj) & 255] ^ tab->perm[2][(k + dk) & 255];
                const float4 c = *reinterpret_cast<const float4 *>(tab->ranvec[idx]);
                const float wx = di ? uu : __fsub_rn(1.0f, uu), wy = dj ? vv : __fsub_rn(1.0f, vv), wz = dk ? ww : __fsub_rn(1.0f, ww);
                const float g = fmaf(c.z, __fsub_rn(w, float(dk)), fmaf(c.y, __fsub_rn(v, float(dj)), __fmul_rn(c.x, __fsub_rn(u, float(di)))));
                accum = fmaf(__fmul_rn(__fmul_rn(wx, wy), wz), g, accum);
            }
    return accum;
}

RT1W_DEV float perlin_turb(const DPerlin *tab, double px, double py, double pz, int depth) { // perlin.rs:74-86
    float accum = 0.0f, weight = 1.0f;
    for (int i = 0; i < depth; ++i) {
        accum = fmaf(weight, perlin_noise(tab, px, py, pz), accum);
        weight *= 0.5f;
        px *= 2.0, py *= 2.0, pz *= 2.0;
    }
    return fabsf(accum);
}

// sin of a f64 argument through f32 after an f64 range reduction (arguments reach 1e4 in the scenes).
// FAST: MUFU.SIN on the reduced argument in [-pi, pi] (2^-21 absolute) instead of sinf's 30 instructions + a slow path that
// is never taken: random_scene +3.3 %, final_scene +2.1 % in the lockstep kernels.  The persistent kernel keeps sinf: the
// stress scene, which never calls it, runs 4.7 % SLOWER with MUFU.SIN in the kernel (and 2 % slower with the texture code
// compiled out altogether) - the register allocation of its traversal loop at the 128-register cap is that sensitive.
template <bool FAST> RT1W_DEV float sin_reduced(double x) {
    const double two_pi = 6.283185307179586476925286766559;
    const double k = rint(x * (1.0 / two_pi));
    const float xr = float(__fma_rn(-k, two_pi, x));
    return FAST ? __sinf(xr) : sinf(xr);
}

// `perlins` may point at shared memory copies of the tables (render.cu stages them per CTA).
// RICH = false: the scene has only SolidColor textures (checker, Perlin and image code compiled out).
template <bool RICH, bool FAST_SIN = true> RT1W_DEV f3 texture_value(const SceneView &sc, const DPerlin *perlins, int tex, const HitInfo &h) {
    DTexture t = sc.textures[tex];
    if (!RICH) return mk3(t.color[0], t.color[1], t.color[2]);
    for (int guard = 0; guard < 9 && t.type == RT1W_TEX_CHECKER; ++guard) { // texture.rs:46-55
        const float sines = sin_reduced<FAST_SIN>(10.0 * h.px) * sin_reduced<FAST_SIN>(10.0 * h.py) * sin_reduced<FAST_SIN>(10.0 * h.pz);
        t = sc.textures[sines < 0.0f ? t.odd : t.even];
    }
    switch (t.type) {
    case RT1W_TEX_SOLID: return mk3(t.color[0], t.color[1], t.color[2]);
    case RT1W_TEX_NOISE: { // texture.rs:57-65
        const float turb = perlin_turb(perlins + t.table, h.px, h.py, h.pz, 7);
        const float s = 0.5f * (1.0f + sin_reduced<FAST_SIN>(__fma_rn(double(t.scale), h.pz, __dmul_rn(10.0, double(turb)))));
        return mk3(s, s, s);
    }
    case RT1W_TEX_PERLIN: { // perlin.rs:109-113 (a second copy of the lattice code: one shared, rolled copy cost two_perlin_spheres 11 %)
        const float s = perlin_noise(perlins + t.table, h.px, h.py, h.pz);
        return mk3(s, s, s);
    }
    case RT1W_TEX_IMAGE: { // texture.rs:67-89: nearest texel, (0,0) = top-left
        // the shading paths build their records without (u, v) (finalize_hit<false>): only this texture reads them
        float u = h.u, v = h.v;
        if (h.type == P_SPHERE || h.type == P_MOVING_SPHERE) {
            sphere_uv(h.n_out, u, v);
        } else if (h.prim != nullptr && (h.type == P_XY_RECT || h.type == P_XZ_RECT || h.type == P_YZ_RECT)) { // a rectangle or a box side (aarect.rs:60-61)
            double lx = h.px, ly = h.py, lz = h.pz;
            const int frame = h.prim->frame;
            if (frame >= 0) { // hittable.rs:207,241-245
                const FrameXf *f = frame_xf(h.frames, frame);
                lx = __dadd_rn(__fma_rn(f->cos_t, h.px, -__dmul_rn(f->sin_t, h.pz)), f->bx), ly = __dadd_rn(h.py, f->by);
                lz = __dadd_rn(__fma_rn(f->sin_t, h.px, __dmul_rn(f->cos_t, h.pz)), f->bz);
            }
            rect_uv(h.prim, h.type, lx, ly, lz, u, v);
        }
        u = fminf(fmaxf(u, 0.0f), 1.0f);
        v = 1.0f - fminf(fmaxf(v, 0.0f), 1.0f);
        const int2 dim = sc.image_dims[t.table];
        const int i = min(int(u * float(dim.x)), dim.x - 1), j = min(int(v * float(dim.y)), dim.y - 1);
        const float4 c = tex2D<float4>(sc.images[t.table], float(i) + 0.5f, float(j) + 0.5f);
        return mk3(c.x, c.y, c.z);
    }
    default: return mk3(0.0f, 0.0f, 0.0f);
    }
}

// ------------------------------------------------------------------------------------------
// Sampling (math.rs, onb.rs, pdf.rs) on a counter-based RNG
// ------------------------------------------------------------------------------------------
struct Rng { // Philox4x32-10 stream: key = (pixel, seed), counter = (sample, bounce, purpose, block)
    uint32_t k0, k1, c0, c1, c2, block;
    RT1W_DEV Philox4 next4() { return philox4x32_10(c0, c1, c2, block++, k0, k1); }
};

struct Onb {
    f3 u, v, w;
};
RT1W_DEV Onb onb_from_w(f3 n) { // onb.rs:13-24
    Onb o;
    o.w = normalize(n);
    const f3 a = fabsf(o.w.x) > 0.9f ? mk3(0.0f, 1.0f, 0.0f) : mk3(1.0f, 0.0f, 0.0f);
    o.v = normalize(cross(o.w, a));
    o.u = cross(o.w, o.v);
    return o;
}
RT1W_DEV f3 onb_local(const Onb &o, f3 a) { return fma3(a.z, o.w, fma3(a.y, o.v, a.x * o.u)); } // onb.rs:26-28

// math.rs:6-18 (three gen_range(-1..1) per try); `x`: the block the caller already drew, used by the first try
RT1W_DEV f3 random_in_unit_sphere(Philox4 x, Rng &rng) {
    for (;;) {
        const f3 p = mk3(2.0f * u01(x.x) - 1.0f, 2.0f * u01(x.y) - 1.0f, 2.0f * u01(x.z) - 1.0f);
        if (dot(p, p) < 1.0f) return p;
        x = rng.next4();
    }
}

// pdf_value of one light for the ray (o, v), hit range [0.001, inf) (aarect.rs:119-138, sphere.rs:72-90); kind: L.kind when
// the caller knows it (a plan), else -1.
// f32 on coordinates taken relative to the light in f64 first: the hit test only decides pdf = 0 at the light's
// silhouette, and the pdf value itself is an f32 quantity.
RT1W_DEV float light_pdf_value(const DLight &L, double ox, double oy, double oz, f3 v, int kind = -1) {
    if ((kind < 0 ? L.kind : kind) == L_XZ_RECT) {
        const float t = float(L.p[4] - oy) / v.y;
        if (t < float(kTMin) || t > CUDART_INF_F) return 0.0f; // NaN passes both comparisons, as in aarect.rs:85-88
        const float x = fmaf(t, v.x, float(ox - L.p[0])), z = fmaf(t, v.z, float(oz - L.p[2]));
        const float wx = float(L.p[1] - L.p[0]), wz = float(L.p[3] - L.p[2]);
        if (x < 0.0f || x > wx || z < 0.0f || z > wz) return 0.0f;
        const float len2 = dot(v, v);
        const float distance_squared = __fmul_rn(__fmul_rn(t, t), len2);
        const float cosine = fabsf(__fmul_rn(v.y, rsqrtf(len2))); // normal is +-y
        return distance_squared / __fmul_rn(cosine, __fmul_rn(wx, wz));
    }
    if ((kind < 0 ? L.kind : kind) == L_SPHERE) { // sphere.rs:24-48 with co = centre - origin
        const f3 co = mk3(float(L.p[0] - ox), float(L.p[1] - oy), float(L.p[2] - oz));
        const float r = float(L.p[3]);
        const float a = dot(v, v), cv = dot(co, v), d2 = dot(co, co);
        const float disc = fmaf(cv, cv, -__fmul_rn(a, fmaf(-r, r, d2)));
        if (disc < 0.0f) return 0.0f;
        const float sq = sqrtf(disc), inv_a = 1.0f / a;
        float root = __fmul_rn(__fsub_rn(cv, sq), inv_a);
        if (root < float(kTMin) || root > CUDART_INF_F) {
            root = __fmul_rn(__fadd_rn(cv, sq), inv_a);
            if (root < float(kTMin) || root > CUDART_INF_F) return 0.0f;
        }
        const float cos_theta_max = sqrtf(__fsub_rn(1.0f, __fmul_rn(r, r) / d2));
        const float solid_angle = __fmul_rn(2.0f * kPiF, __fsub_rn(1.0f, cos_theta_max));
        return 1.0f / solid_angle;
    }
    return 0.0f; // trait default, hittable.rs:66-68
}

// ------------------------------------------------------------------------------------------
// Materials (material.rs, constant_medium.rs:31-51).  Each returns the scattered direction and
// multiplies the throughput; `time_out` carries the reference's time quirk (main.rs:86).
// ------------------------------------------------------------------------------------------
RT1W_DEV f3 reflect(f3 v, f3 n) { return fma3(-2.0f * dot(v, n), n, v); } // material.rs:94-96

RT1W_DEV f3 refract(f3 uv, f3 n, float etai_over_etat) { // material.rs:114-119
    const float cos_theta = fminf(dot(-uv, n), 1.0f);
    const f3 r_out_perp = etai_over_etat * fma3(cos_theta, n, uv);
    return fma3(-sqrtf(fabsf(__fsub_rn(1.0f, dot(r_out_perp, r_out_perp)))), n, r_out_perp);
}

RT1W_DEV float reflectance(float cosine, float ref_idx) { // material.rs:121-125
    float r0 = (1.0f - ref_idx) / (1.0f + ref_idx);
    r0 = __fmul_rn(r0, r0);
    const float m = 1.0f - cosine;
    const float m2 = __fmul_rn(m, m);
    return fmaf(__fsub_rn(1.0f, r0), __fmul_rn(__fmul_rn(m2, m2), m), r0);
}

// Lambertian + MixturePdf(HittablePdf(lights), CosinePdf) — main.rs:75-104 / :142-160, material.rs:70-92, pdf.rs:36-69.
// A cosine sample (math.rs:39-49) and a sample towards a sphere light (math.rs:51-65, sphere.rs:92-99) are both
// `onb.local(cos(phi) q, sin(phi) q, z)` with q = sqrt(1 - z^2), about the normal resp. the direction to the
// sphere, so the two strategies share one code path; a rectangle light (aarect.rs:140-147) is the short branch.
// PLAN: the scene's plan (flat_plans.h): the light count and kinds are constants, the chosen light's branch follows from its
// index and the pdf sum runs over the list in order, i = 0 .. n - 1; or -1.
template <int PLAN = -1>
RT1W_DEV f3 scatter_lambertian(const SceneView &sc, const DLight *lights, const HitInfo &h, const Philox4 x, f3 &weight) {
    constexpr int kPlanLights = PLAN >= 0 ? kFlatPlans[PLAN < 0 ? 0 : PLAN].n_lights : 0;
    constexpr uint32_t kPlanKinds = PLAN >= 0 ? plan_light_kinds(kFlatPlans[PLAN < 0 ? 0 : PLAN]) : 0u;
    const f3 w = normalize(h.normal); // onb.rs:14
    const float r1 = u01(x.z), r2 = u01(x.w);
    f3 dir, axis = w;
    float z = sqrtf(1.0f - r2);
    bool local = true; // the direction comes out of an ONB
    const int n = PLAN >= 0 ? kPlanLights : (sc.has_lights ? sc.n_lights : 0);
    if (n > 0 && (x.x >> 31)) { // rng.gen::<bool>() -> HittablePdf (pdf.rs:63-64)
        const int li = min(int(u01(x.y) * float(n)), n - 1); // slice.choose (hittable.rs:153)
        const DLight &L = lights[li];
        const int kind = PLAN >= 0 ? int((kPlanKinds >> (2 * li)) & 3u) : L.kind;
        if (kind == L_XZ_RECT) { // un-normalised
            const double px = __fma_rn(L.p[1] - L.p[0], double(r1), L.p[0]), pz = __fma_rn(L.p[3] - L.p[2], double(r2), L.p[2]);
            dir = mk3(float(px - h.px), float(L.p[4] - h.py), float(pz - h.pz));
            local = false;
        } else if (kind == L_SPHERE) {
            axis = mk3(float(L.p[0] - h.px), float(L.p[1] - h.py), float(L.p[2] - h.pz));
            const float radius = float(L.p[3]);
            z = fmaf(r2, __fsub_rn(sqrtf(__fsub_rn(1.0f, __fmul_rn(radius, radius) / dot(axis, axis))), 1.0f), 1.0f);
        } else { // trait default, hittable.rs:69-71
            dir = mk3(1.0f, 0.0f, 0.0f);
            local = false;
        }
    }
    if (local) {
        const Onb uvw = onb_from_w(axis);
        float sn, cs;
        sn = __sinf(2.0f * kPiF * r1), cs = __cosf(2.0f * kPiF * r1); // MUFU.SIN / MUFU.COS on [0, 2 pi): 2^-21 absolute, 25 instructions fewer than sincospif (+0.6 %)
        const float q = sqrtf(fmaxf(fmaf(-z, z, 1.0f), 0.0f));
        dir = onb_local(uvw, mk3(__fmul_rn(cs, q), __fmul_rn(sn, q), z));
    }
    const float cosine = __fmul_rn(dot(normalize(dir), w), 1.0f / kPiF); // pdf.rs:37-40 and material.rs:82-91 (same expression)
    float pdf = fmaxf(cosine, 0.0f);
    if (n > 0) {
        float lsum = 0.0f;
        const float wl = 1.0f / float(PLAN >= 0 ? sc.n_lights : n); // (run time under a plan too: flat_plans.h)
        if constexpr (PLAN >= 0) { // (rolled: unrolled, the two pdf bodies cost the Cornell k_tail a 40-byte spill)
#pragma unroll 1
            for (int i = 0; i < kPlanLights; ++i) lsum = fmaf(wl, light_pdf_value(lights[i], h.px, h.py, h.pz, dir, int((kPlanKinds >> (2 * i)) & 3u)), lsum);
        } else {
            for (int i = 0; i < n; ++i) lsum = fmaf(wl, light_pdf_value(lights[i], h.px, h.py, h.pz, dir), lsum); // hittable.rs:144-150
        }
        pdf = fmaf(0.5f, lsum, __fmul_rn(0.5f, pdf)); // pdf.rs:58-60
    }
    const float s = fmaxf(cosine, 0.0f) / pdf; // unguarded, main.rs:102
    weight = mk3(s, s, s);
    return dir;
}

RT1W_DEV f3 scatter_metal(const DMaterial &m, const Ray &r, const HitInfo &h, const Philox4 x, Rng &rng) { // material.rs:98-112
    const f3 reflected = reflect(normalize(mk3(r.dx, r.dy, r.dz)), h.normal);
    if (m.fuzz == 0.0f) return reflected; // the reference still runs the sampler (material.rs:102) and multiplies it by zero
    return fma3(m.fuzz, random_in_unit_sphere(x, rng), reflected);
}

RT1W_DEV f3 scatter_dielectric(const DMaterial &m, const Ray &r, const HitInfo &h, const Philox4 x) { // material.rs:132-161
    const float ratio = h.front_face ? 1.0f / m.ir : m.ir;
    const f3 unit = normalize(mk3(r.dx, r.dy, r.dz));
    const float cos_theta = fminf(dot(-unit, h.normal), 1.0f);
    const float sin_theta = sqrtf(fmaf(-cos_theta, cos_theta, 1.0f));
    bool reflects = __fmul_rn(ratio, sin_theta) > 1.0f;
    if (!reflects) reflects = reflectance(cos_theta, ratio) > u01(x.x);
    return reflects ? reflect(unit, h.normal) : refract(unit, h.normal, ratio);
}

} // namespace rt1w
