// device_types.h — POD layouts shared by the host lowering code and the sm_100a kernels.
//
// HBM layout of a committed scene (all arrays read-only during a render, small enough to
// stay L1/L2 resident for every BASELINE config):
//   nodes   : 2 x float4 per BVH node (32 B).  n0 = (min.xyz, bits leftFirst), n1 = (max.xyz, bits count).
//             count == 0 -> interior, children at leftFirst and leftFirst+1 (a 64-B aligned pair);
//             count  > 0 -> leaf, primitives [leftFirst, leftFirst+count) in LEAF order.
//   prims   : 64 B per primitive in leaf order, see DPrim (f64 geometry parameters).
//   prim_id : leaf index -> primitive id (DFS order of the description).
//   frames, materials, textures, perlin tables, image texture objects, lights: small tables.
#pragma once

#include <stdint.h>

namespace rt1w {

enum PrimType : int {
    P_SPHERE = 0,
    P_MOVING_SPHERE = 1,
    P_XY_RECT = 2,
    P_XZ_RECT = 3,
    P_YZ_RECT = 4,
    P_MEDIUM_SPHERE = 5,
    P_MEDIUM_BOX = 6,
    P_BOX = 7, // AABox (aabox.rs): its six rectangles as one device primitive; the side travels with the leaf index
};

// A hit names its primitive as leaf index | side << 28 (side: 0 except for P_BOX, where it is the
// rectangle's position in aabox.rs:29-76: XY@z1, XY@z0, XZ@y1, XZ@y0, YZ@x1, YZ@x0).
constexpr int kLeafBits = 28;
constexpr int kLeafMask = (1 << kLeafBits) - 1;

enum PrimFlags : int { PF_FLIP_FACE = 1 };

// Shading queues of the wavefront: one per reference material family; the queue id of a hit is its
// rt1w_material_type (LAMBERTIAN..ISOTROPIC, DIFFUSE_LIGHT).  Misses and the null material `()`
// terminate inside the extend kernel.
enum QueueId : int { Q_COUNT = 5 }; // queue index == rt1w_material_type, RT1W_MAT_LAMBERTIAN (0) .. RT1W_MAT_ISOTROPIC (4)

// meta word: type[0:4) | flags[4:8) | material type[8:12) | material id[12:32)
static inline uint32_t pack_meta(int type, int flags, int mat_type, int mat_id) {
    return uint32_t(type) | (uint32_t(flags) << 4) | (uint32_t(mat_type) << 8) | (uint32_t(mat_id) << 12);
}

// One 64-byte device primitive (uploaded as 4 x 16-byte words, leaf order).  Geometry parameters are
// f64: the reference computes in f64 (main.rs:1) and B200 issues DFMA at half the FFMA rate, so the
// intersection solve keeps the reference's precision while node tests and shading stay f32.
//   sphere        : p0..2 = center, p3 = radius
//   rects         : p0,p1 = first in-plane interval, p2,p3 = second, q0 = k
//   moving sphere : p0..2 = center0, p3 = radius, f0..2 = center1-center0, f3 = time0, f4 = 1/(time1-time0)
//   medium sphere : p0..2 = center, p3 = radius, q0 = -1/density
//   medium box    : p0..2 = box min, p3 = -1/density, q0..2 = box max
//   box           : p0..2 = box min, q0..2 = box max
struct DPrim {
    double p[4];
    union {
        double q[3];
        float f[6];
    };
    uint32_t meta;
    int32_t frame; // -1: no wrapper chain
};
static_assert(sizeof(DPrim) == 64, "DPrim must be 4 x 16 bytes");

// One wrapper chain (Translate / RotateY / FlipFace stack above a leaf).
// local = Ry(p) + b with Ry: x' = c*x - s*z, z' = s*x + c*z (hittable.rs:241-245 composed with :207).
// ops replay the HitRecord::new calls of the wrappers, innermost first (hittable.rs:221-229, :269-277, :290).
#define RT1W_MAX_CHAIN_OPS 8
enum ChainOpKind : int { OP_TRANSLATE = 0, OP_ROTATE_Y = 1, OP_FLIP_FACE = 2 };
struct DChainOp {
    int32_t kind;
    float sin_own, cos_own; // this RotateY's own angle (normal back-rotation)
    float sin_cum, cos_cum; // cumulative angle of the ray direction INSIDE this wrapper
};
struct DFrame {
    double sin_t, cos_t;
    double bx, by, bz;
    int32_t n_ops;
    int32_t pad0;
    DChainOp ops[RT1W_MAX_CHAIN_OPS];
};

struct DMaterial { // 2 x float4
    float albedo[3];
    float fuzz;
    float ir;
    int32_t type;
    int32_t texture;
    int32_t pad;
};
static_assert(sizeof(DMaterial) == 32, "DMaterial must be 2 x float4");

struct DTexture { // 2 x float4
    float color[3];
    float scale;
    int32_t type;
    int32_t odd, even;
    int32_t table;
};
static_assert(sizeof(DTexture) == 32, "DTexture must be 2 x float4");

struct DPerlin {
    float ranvec[256][4]; // xyz + pad, 16-B aligned rows
    uint8_t perm[3][256];
};

enum LightKind : int { L_XZ_RECT = 0, L_SPHERE = 1, L_OTHER = 2 };
struct DLight { // pdf.rs / hittable.rs:144-154: only XZRect and Sphere implement pdf_value/random
    double p[5]; // XZ: x0,x1,z0,z1,k ; sphere: cx,cy,cz,r
    int32_t kind;
    int32_t pad;
};
#define RT1W_MAX_LIGHTS 32

struct DCamera { // the fields of `Camera` (camera.rs:8-19); kept f64, used once per path
    double origin[3];
    double llc_rel[3]; // lower_left_corner - origin
    double horizontal[3];
    double vertical[3];
    double u[3], v[3];
    double lens_radius;
    float time0, time1;
};

struct DRenderParams {
    int32_t width, height;
    int32_t sample_begin, n_samples;
    int32_t max_depth;
    uint32_t flags;
    uint32_t seed_lo, seed_hi;
    float background[3];
    float stat_clamp;
    unsigned long long total_paths;
    uint32_t n_pixels;
    int32_t pool;
    uint32_t tile_shift; // paths start tile by tile of 2^tile_shift pixels (render.cu: generate_ray)
    uint32_t tile_paths; // n_samples << tile_shift, at most 2^30
    // reciprocals prepared by the host: 1 / (width - 1), 1 / (height - 1) (main.rs:968-969) and, rounded UP so that
    // uint32(double(n) * r) == n / d for every n < 2^32 with n / d * d < 2^50, 1 / width and 1 / tile_paths
    double inv_w1, inv_h1, inv_width_up, inv_tile_paths_up;
};

// Batch renders (rt1w_render_batch): n_frames images of width x height pixels in one wavefront.  Batch pixel g =
// f * frame_pixels + (j * width + i) belongs to frame f, which renders with cams[f] and the Philox seed words
// seeds[2f] (lo), seeds[2f + 1] (hi).  One device allocation: this header, then the two tables it points to.
// f = g / frame_pixels through the rounded-up reciprocal 2^32 + magic of frame_pixels in fixed point (Granlund and
// Montgomery, PLDI 1994, figure 4.1): t = umulhi(g, magic), f = (t + ((g - t) >> shift1)) >> shift2, exact for every
// 32-bit g - integer registers only, where an f64 reciprocal read from memory costs the wave kernels spills.
struct DBatch {
    uint32_t frame_pixels, magic, shift1, shift2;
    const DCamera *cams;
    const uint32_t *seeds;
};

// Philox counter "stream" words (counter[2]); counter = {sample, bounce, stream, block}.
enum RngStream : uint32_t { RNG_CAMERA = 0, RNG_SCATTER = 1, RNG_MEDIUM = 2, RNG_TRACE_MEDIUM = 0x4d454449u };

} // namespace rt1w
