/*
 * rt1w.h — C ABI of the B200-native renderer for the per-pixel Monte Carlo
 * sample loop of hatoo/raytracing-1w (master, "The Rest of Your Life").
 *
 * This header is the drop-in boundary.  Everything a reference-side FFI layer
 * (Rust `extern "C"` block, see INTEGRATION.md) would bind for this path is
 * declared here with plain pointers and sizes.  All `file:line` citations are
 * relative to the reference tree (`src/...`).
 *
 * What crosses the boundary
 * -------------------------
 *  1. A *scene description*: the reference's object tree (`Box<dyn Hittable>`
 *     children, `Arc<Box<dyn Material>>` handles, `Texture` objects) lowered by
 *     the host into POD tables (rt1w_scene_desc).  One rt1w_node per reference
 *     constructor call; nothing is pre-flattened, so wrapper semantics
 *     (`Translate`, `RotateY`, `FlipFace`, hittable.rs:49-61) survive the trip.
 *  2. A camera (the private fields of `Camera`, camera.rs:8-19, as computed by
 *     `Camera::new`, camera.rs:22-59).
 *  3. Render parameters (the locals of `main`, main.rs:798-801,939).
 *  4. The result: per-pixel fp32 radiance SUMS (row 0 = top row, the order
 *     main.rs:957-1007 prints them), to which the host applies
 *     `Color::into_sampled` + `Display for SampledColor` (color.rs:14-21,56-65).
 *
 * The operator replaced is `ray_color` / `ray_color_without_light_objects`
 * (main.rs:51-190) together with the enclosing per-pixel loop (main.rs:957-1001):
 * one call renders a whole image (or one sample range of it), never one ray.
 *
 * Ownership: every input pointer is borrowed for the duration of the call and
 * copied; device memory lives behind the opaque handles; outputs are
 * caller-allocated.  Errors: integer status codes + rt1w_last_error(); nothing
 * unwinds across the ABI.  There is NO CPU fallback: without a usable CUDA
 * device rt1w_context_create fails with RT1W_ERR_NO_DEVICE.
 */
#ifndef RT1W_H
#define RT1W_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT1W_ABI_VERSION 2

typedef enum rt1w_status {
    RT1W_OK = 0,
    RT1W_ERR_INVALID = 1,     /* malformed description (mirrors the reference panics: bvh.rs:61,65-67; hittable.rs:153) */
    RT1W_ERR_UNSUPPORTED = 2, /* valid reference scene the device path does not lower (see DESIGN.md) */
    RT1W_ERR_CUDA = 3,        /* a CUDA runtime call failed */
    RT1W_ERR_NO_DEVICE = 4,   /* no usable sm_100 device; there is no CPU fallback */
    RT1W_ERR_STATE = 5
} rt1w_status;

/* ------------------------------------------------------------------------- */
/* Scene description (POD tables)                                              */
/* ------------------------------------------------------------------------- */

/* One node per reference `Hittable` value. */
typedef enum rt1w_node_type {
    RT1W_NODE_SPHERE = 0,          /* sphere.rs:16-20         p = {cx,cy,cz, radius} */
    RT1W_NODE_MOVING_SPHERE = 1,   /* moving_sphere.rs:13-20  p = {c0x,c0y,c0z, c1x,c1y,c1z, time0, time1, radius} */
    RT1W_NODE_XY_RECT = 2,         /* aarect.rs:15-22         p = {x0,x1,y0,y1,k} */
    RT1W_NODE_XZ_RECT = 3,         /* aarect.rs:25-32         p = {x0,x1,z0,z1,k} */
    RT1W_NODE_YZ_RECT = 4,         /* aarect.rs:35-42         p = {y0,y1,z0,z1,k} */
    RT1W_NODE_AABOX = 5,           /* aabox.rs:22-84          p = {p0x,p0y,p0z, p1x,p1y,p1z} */
    RT1W_NODE_TRANSLATE = 6,       /* hittable.rs:49-52       p = {ox,oy,oz}; 1 child */
    RT1W_NODE_ROTATE_Y = 7,        /* hittable.rs:158         p = {angle_deg, time0, time1}; 1 child */
    RT1W_NODE_FLIP_FACE = 8,       /* hittable.rs:61          1 child */
    RT1W_NODE_CONSTANT_MEDIUM = 9, /* constant_medium.rs:22   p = {density}; 1 child = boundary; material = its Isotropic phase function */
    RT1W_NODE_BVH = 10             /* bvh.rs:54-59            p = {time0,time1}; >=1 children (a grouping node; the device rebuilds one SAH BVH over all leaves) */
} rt1w_node_type;

typedef struct rt1w_node {
    int32_t type;        /* rt1w_node_type */
    int32_t material;    /* index into materials[] for leaves / CONSTANT_MEDIUM, else -1 */
    int32_t child_begin; /* first index into children[] (wrappers, BVH), else 0 */
    int32_t child_count;
    double p[10];
} rt1w_node;

typedef enum rt1w_material_type {
    RT1W_MAT_LAMBERTIAN = 0,    /* material.rs:52-55,70-92   texture = albedo */
    RT1W_MAT_METAL = 1,         /* material.rs:57-61,98-112  albedo[3], fuzz */
    RT1W_MAT_DIELECTRIC = 2,    /* material.rs:127-161       ir */
    RT1W_MAT_DIFFUSE_LIGHT = 3, /* material.rs:63-66,163-182 texture = emit */
    RT1W_MAT_ISOTROPIC = 4,     /* constant_medium.rs:31-51  texture = albedo */
    RT1W_MAT_NONE = 5           /* `impl Material for ()`, material.rs:68 */
} rt1w_material_type;

typedef struct rt1w_material {
    int32_t type;    /* rt1w_material_type */
    int32_t texture; /* index into textures[] or -1 */
    double albedo[3];
    double fuzz;
    double ir;
} rt1w_material;

typedef enum rt1w_texture_type {
    RT1W_TEX_SOLID = 0,   /* texture.rs:12-15,40-44  color */
    RT1W_TEX_CHECKER = 1, /* texture.rs:17-21,46-55  odd, even = texture ids */
    RT1W_TEX_NOISE = 2,   /* texture.rs:23-38,57-65  scale, table = perlin id */
    RT1W_TEX_IMAGE = 3,   /* texture.rs:67-89        table = image id */
    RT1W_TEX_PERLIN = 4   /* perlin.rs:109-113       table = perlin id (never instantiated by the reference scenes) */
} rt1w_texture_type;

typedef struct rt1w_texture {
    int32_t type; /* rt1w_texture_type */
    int32_t odd;
    int32_t even;
    int32_t table;
    double color[3];
    double scale;
} rt1w_texture;

/* The tables of one `Perlin<256>` (perlin.rs:7-12). */
typedef struct rt1w_perlin {
    double ranvec[256][3];
    int32_t perm_x[256];
    int32_t perm_y[256];
    int32_t perm_z[256];
} rt1w_perlin;

/* A decoded `image::DynamicImage` (texture.rs:67): tightly packed RGB8, row 0 = top. */
typedef struct rt1w_image {
    const uint8_t *rgb8;
    int32_t width;
    int32_t height;
} rt1w_image;

typedef struct rt1w_scene_desc {
    const rt1w_node *nodes;
    int32_t n_nodes;
    const int32_t *children; /* child node ids, referenced by child_begin/child_count */
    int32_t n_children;
    const rt1w_material *materials;
    int32_t n_materials;
    const rt1w_texture *textures;
    int32_t n_textures;
    const rt1w_perlin *perlins;
    int32_t n_perlins;
    const rt1w_image *images;
    int32_t n_images;
    int32_t world;         /* root node id (the `world` of main.rs:805) */
    int32_t has_lights;    /* `lights: Option<Vec<Box<dyn Hittable>>>` (main.rs:807-809): 0 = None */
    const int32_t *lights; /* node ids of the light hittables (separate null-material copies, main.rs:873-887) */
    int32_t n_lights;
} rt1w_scene_desc;

/* The fields of `Camera` after `Camera::new` (camera.rs:8-19,22-59). */
typedef struct rt1w_camera {
    double origin[3];
    double lower_left_corner[3];
    double horizontal[3];
    double vertical[3];
    double u[3], v[3], w[3];
    double lens_radius;
    double time0, time1;
} rt1w_camera;

#define RT1W_FLAG_STATS 1u   /* also accumulate per-pixel clamped sum and sum of squares (test statistic) */
#define RT1W_FLAG_PROFILE 2u /* bracket every kernel launch with CUDA events and fill rt1w_render_stats.kernel_ms (slower) */
/* BVH scenes: which wave kernel traverses (default: by BVH size).  Both return the same closest hits; parity tests force each. */
#define RT1W_FLAG_BVH_LOCKSTEP 4u   /* a warp runs its 32 rays to the end together (short, even traversals) */
#define RT1W_FLAG_BVH_PERSISTENT 8u /* lanes take a new ray as soon as theirs is done (long, uneven traversals) */
/* BVH scenes: which tree is walked (default: by BVH size).  Same leaves, same conservative boxes, same closest hits. */
#define RT1W_FLAG_BVH_BINARY 16u /* 32-byte nodes, two children per step */
#define RT1W_FLAG_BVH_WIDE 32u   /* compressed 8-wide nodes (80 bytes, eight quantised child boxes per step) */
/* Waves to the very end: without it, once about one hit per resident thread is left, one kernel follows every remaining path
 * to its end inside a thread (same scatter, same closest hit, same random numbers: same image). A/B measurements, tests. */
#define RT1W_FLAG_NO_TAIL 64u

/* kernel slots of rt1w_render_stats.kernel_ms / kernel_launches */
#define RT1W_KERNEL_WAVE 0  /* k_wave / k_wave_bvh: scatter queued hits / start camera paths, closest hit, regroup per material */
#define RT1W_KERNEL_COUNT 7 /* slots 1..6 reserved */

typedef struct rt1w_render_params {
    int32_t width;          /* image_width  (main.rs:799) */
    int32_t height;         /* image_height (main.rs:939) */
    int32_t sample_begin;   /* this call renders samples [sample_begin, sample_end) of every pixel; */
    int32_t sample_end;     /*   a full image is [0, samples_per_pixel) (main.rs:967)                 */
    int32_t max_depth;      /* MAX_DEPTH (main.rs:801) */
    uint32_t flags;
    uint64_t seed;          /* global Philox seed; the per-pixel stream id is j*width+i as in main.rs:964 */
    double background[3];   /* main.rs:806 */
    double stat_clamp;      /* per-sample, per-channel ceiling used only for the RT1W_FLAG_STATS buffers */
    int32_t pool_paths;     /* paths in flight per wave; 0 = library default */
    int32_t reserved;
} rt1w_render_params;

typedef struct rt1w_render_stats {
    uint64_t paths;       /* W*H*(sample_end-sample_begin) */
    uint64_t rays;        /* closest-hit queries (calls of `world.hit`, main.rs:62) */
    uint64_t waves;       /* wavefront iterations */
    uint64_t launches;    /* kernels launched inside the render */
    double render_ms;     /* device time generate -> accumulate, CUDA events on the render stream */
    double kernel_ms[RT1W_KERNEL_COUNT];         /* per kernel: device time summed over its launches (RT1W_FLAG_PROFILE only) */
    uint64_t kernel_launches[RT1W_KERNEL_COUNT]; /* per kernel: launches timed (RT1W_FLAG_PROFILE only) */
} rt1w_render_stats;

typedef struct rt1w_scene_info {
    int32_t n_prims;       /* leaf primitives after lowering */
    int32_t n_bvh_nodes;   /* 32-byte nodes of the device SAH BVH */
    int32_t n_frames;      /* distinct wrapper chains */
    int32_t n_lights;
    int32_t bvh_depth;
    int32_t material_mask; /* bit m set when some primitive uses rt1w_material_type m */
    double build_ms;       /* host lowering + BVH build (binary tree, then its collapse into the 8-wide tree) */
    double upload_ms;
    double sah_cost;
    int32_t n_wide_nodes;  /* 80-byte nodes of the compressed 8-wide BVH (0: flat-scan scene) */
    int32_t wide_depth;
    int32_t wide_default;  /* 1: render and trace calls walk the 8-wide tree unless a flag says otherwise */
    int32_t n_global_prims; /* spheres / sphere-bounded media kept out of the tree because their box contains every other primitive's (tested once per ray) */
    double wide_children;  /* occupied slots per wide node */
} rt1w_scene_info;

/* One lowered primitive, in PRIMITIVE-ID order (DFS order of the description,
 * an AABox expanding to its six rects in the order of aabox.rs:29-76). */
typedef struct rt1w_flat_prim {
    int32_t kind;     /* rt1w_node_type of the leaf (SPHERE..YZ_RECT) or CONSTANT_MEDIUM */
    int32_t node;     /* node id the primitive came from */
    int32_t material;
    int32_t frame;    /* wrapper-chain id or -1 */
    int32_t flags;    /* bit0: odd number of FlipFace wrappers */
    int32_t boundary; /* media: RT1W_NODE_SPHERE or RT1W_NODE_AABOX */
    double p[10];
    double bbox_min[3], bbox_max[3]; /* world-space bounds handed to the SAH builder */
    double time0, time1;             /* the bounding_box(time0,time1) arguments in scope (bvh.rs:54-59, hittable.rs:158) */
} rt1w_flat_prim;

typedef struct rt1w_ray {
    float origin[3];
    float direction[3];
    float time;
} rt1w_ray;

typedef struct rt1w_context rt1w_context;
typedef struct rt1w_scene rt1w_scene;

/* ------------------------------------------------------------------------- */
/* Entry points                                                                */
/* ------------------------------------------------------------------------- */

int32_t rt1w_abi_version(void);

/* Message of the most recent failure on this thread. */
const char *rt1w_last_error(void);

/* One context per process per GPU (`device_id` as in cudaSetDevice); several GPUs: see "Multi-GPU" below. */
rt1w_status rt1w_context_create(int32_t device_id, rt1w_context **out);
void rt1w_context_destroy(rt1w_context *ctx);

/* ---- Multi-GPU (SURVEY.md section 8e) -------------------------------------------------------------------------
 * The sample loop has no cross-pixel or cross-sample state (main.rs:957-993), so the path shards by SAMPLE RANGE: the
 * scene is replicated, rank r of n renders the r-th of n contiguous parts of [sample_begin, sample_end) of every pixel
 * (rt1w_shard_sample_range; the Philox counter carries the global sample index, so the image does not depend on n up to
 * fp32 summation order), and the partial radiance sums meet in ONE exchange step: ncclReduce(sum, fp32, 3*W*H) to rank
 * 0 on the render streams, over NVLink.  NCCL is bound at run time (libnccl.so.2; a copy the host process has already
 * loaded is shared); single-GPU use needs none.
 *
 * A context that belongs to a communicator makes EVERY render call (rt1w_render, rt1w_render_device, rt1w_render_rgb8)
 * collective: all ranks call with the same arguments, each renders its share, rank 0 receives the image (the other
 * ranks' output pointers may be NULL; after rt1w_render_device their buffers hold their own partial sums).
 * rt1w_render_stats then counts this rank's paths and rays (multi-process) or all devices' (multi-device context), and
 * render_ms includes the reduce.
 * Errors: a multi-device context checks the arguments and allocates every device's queues BEFORE any device starts, so a
 * call either fails on all devices or reaches the reduce on all of them.  Across processes (b) the usual rule of
 * collectives holds: a rank that returns an error before the reduce (bad arguments are rejected identically everywhere;
 * an allocation failure is not) leaves the other ranks waiting - destroy the contexts of a failed job.
 *
 *  (a) one process, n devices - what the reference's single `main` would use:
 *        rt1w_context_create_multi(ids, n, &ctx);  rt1w_scene_create(ctx, ...);  rt1w_render(scene, ...);
 *      The context owns one sub-context, render stream and host thread per device (rank i = device_ids[i]);
 *      rt1w_scene_create commits the scene on all of them in parallel; the handles are used exactly like single-GPU ones.
 *  (b) one process per device (MPI / torchrun style): rank 0 calls rt1w_comm_unique_id, the host side ships the id
 *      to the other ranks (any transport), and every rank calls rt1w_context_comm_init on its single-device context. */
#define RT1W_COMM_ID_BYTES 128 /* sizeof(ncclUniqueId) */
rt1w_status rt1w_context_create_multi(const int32_t *device_ids, int32_t n, rt1w_context **out);
rt1w_status rt1w_comm_unique_id(uint8_t *out_id, size_t capacity);
rt1w_status rt1w_context_comm_init(rt1w_context *ctx, const uint8_t *id, int32_t n_ranks, int32_t rank);
/* rank and size of the context's communicator (0 and 1 outside one) and the devices it drives itself. */
rt1w_status rt1w_context_get_comm(const rt1w_context *ctx, int32_t *rank, int32_t *n_ranks, int32_t *n_local_devices);
/* The split rule: contiguous parts whose sizes differ by at most one (host code, no device needed). */
void rt1w_shard_sample_range(int32_t rank, int32_t n_ranks, int32_t sample_begin, int32_t sample_end, int32_t *out_begin,
                             int32_t *out_end);

/* Lower + commit: walks the description, composes wrapper chains, expands
 * boxes, builds the SAH BVH (replaces `BVHNode::new`, bvh.rs:54-103) and
 * uploads everything.  The scene is immutable afterwards (`Send + Sync`,
 * hittable.rs:63). */
rt1w_status rt1w_scene_create(rt1w_context *ctx, const rt1w_scene_desc *desc, rt1w_scene **out);
void rt1w_scene_destroy(rt1w_scene *scene);
rt1w_status rt1w_scene_get_info(const rt1w_scene *scene, rt1w_scene_info *out);
/* Copies up to `capacity` lowered primitives; returns the total through *n_out. */
rt1w_status rt1w_scene_get_prims(const rt1w_scene *scene, rt1w_flat_prim *out, int32_t capacity, int32_t *n_out);
/* Test-only hook: the host copy of the primitive-id table the scene uploaded, in device leaf order - prim_id_of_leaf[leaf] is
 * the primitive id (rt1w_trace_closest numbering; a box: the id of its first rectangle) of leaf `leaf`.  The render keys the
 * free-flight draw of a ConstantMedium on its leaf index, which depends on the layout (flat scan or tree) and the builder;
 * a checker that replays the render's draws needs this table.  Copies up to `capacity` entries; returns the leaf count
 * through *n_out. */
rt1w_status rt1w_scene_get_leaf_prims(const rt1w_scene *scene, int32_t *prim_id_of_leaf, int32_t capacity, int32_t *n_out);

/* Host-side lowering only (no device needed): same primitive table as
 * rt1w_scene_get_prims would return after a create.  Used by tools and CPU tests. */
rt1w_status rt1w_lower_prims(const rt1w_scene_desc *desc, rt1w_flat_prim *out, int32_t capacity, int32_t *n_out);

/* Host-side only: the face groups the small-scene closest-hit scan forms over the lowered primitives - rectangles of
 * one wrapper frame that are whole faces of a common box (the walls of a room, the six sides of aabox.rs:29-76) are
 * tested with one slab computation.  Per primitive (rt1w_lower_prims order): group number or -1, and the face
 * 2 * axis + (upper plane ? 1 : 0) with axis 0 = x (YZRect), 1 = y (XZRect), 2 = z (XYRect).  Used by CPU tests. */
rt1w_status rt1w_lower_face_groups(const rt1w_scene_desc *desc, int32_t *group_of_prim, int32_t *face_of_prim, int32_t capacity,
                                   int32_t *n_groups);

/* Host-side only (no device needed): the two trees scene commit builds over the primitives' world-space boxes (n x 3
 * doubles each) - the binned-SAH binary tree of 32-byte nodes (replaces `BVHNode::new`, bvh.rs:54-103: min.xyz,
 * left_first, max.xyz, count; node 0 = root, node 1 = padding, the children of an interior node adjacent) and its
 * SAH-optimal collapse into the compressed 8-wide tree of 80-byte nodes (layout: csrc/bvh8.h).  Every output is optional;
 * capacities are in nodes.  prim_order[leaf] = input box of binary leaf `leaf`; wide_leaf_remap[slot primitive] = binary
 * leaf.  Used by CPU tests of the builders (tests/test_host_bvh.py). */
rt1w_status rt1w_build_bvh_host(const double *bbox_min3, const double *bbox_max3, int32_t n, void *nodes32, int32_t node_capacity,
                                int32_t *n_nodes, uint32_t *prim_order, void *wide_nodes80, int32_t wide_capacity, int32_t *n_wide,
                                uint32_t *wide_leaf_remap, int32_t *depth, int32_t *wide_depth);

/* Replaces the pixel loop + ray_color (main.rs:957-1001, 51-190).
 * out_rgb_sum: HOST buffer, width*height*3 floats, row 0 = top, per-pixel SUM
 *   over the rendered sample range (not yet divided by spp).
 * out_stat (nullable, needs RT1W_FLAG_STATS): HOST buffer width*height*6 floats:
 *   sum of min(x,stat_clamp) and sum of min(x,stat_clamp)^2 per channel
 *   (NaN samples counted as 0). */
rt1w_status rt1w_render(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params,
                        float *out_rgb_sum, float *out_stat, rt1w_render_stats *stats);

/* Same, but the result stays on the device (d_rgb_sum: width*height*3 floats,
 * zeroed by the call) and work is enqueued on `cuda_stream` (a cudaStream_t, 0 =
 * default stream); returns after the stream has drained.  Lets the caller
 * combine partial sums across GPUs (ncclReduce) without a host round trip. */
rt1w_status rt1w_render_device(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params,
                               float *d_rgb_sum, void *cuda_stream, rt1w_render_stats *stats);

/* Render + the output path of main.rs:992,1003-1007 on the device: the per-pixel sums are resolved to 8-bit
 * channels (`Color::into_sampled`, `Display for SampledColor`, color.rs:14-21,56-65) before they leave the GPU.
 * out_rgb8: HOST buffer, width*height*3 bytes, row 0 = top - what the reference prints as its P3 body.
 * The mean divides by sample_end - sample_begin. */
rt1w_status rt1w_render_rgb8(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params,
                             uint8_t *out_rgb8, rt1w_render_stats *stats);

/* Adaptive sampling: every pixel is rendered until its 8-bit output has converged.
 * Schedule: round 0 renders samples [0, min_spp) of every pixel; round k+1 renders [n, min(2n, sample_end)) of every
 * pixel still active after n samples.  Sample s of pixel p is the same path whichever round renders it (Philox key =
 * pixel seed, counter = global sample index), so a pixel that ends with n samples holds what rt1w_render of [0, n) gives
 * it, up to the order of the fp32 additions.
 * Convergence rule, after each round, in f64 from the fp32 sums of the pixels still active (n samples each).  Per
 * channel, with S1, S2 the sum and sum of squares of min(x, stat_clamp) (the RT1W_FLAG_STATS buffers):
 *     m = S1 / n,  v = max(S2 / n - m*m, 0) * n / (n - 1),  se = sqrt(v / n),
 *     e = 128 * (sqrt(clamp(m + se, 0, 1)) - sqrt(clamp(m - se, 0, 1)))
 * i.e. the half-width of the +-1 standard-error interval of the mean in 8-bit output levels, through the gamma 2 and
 * x 256 of color.rs:56-65 (a saturated channel has e = 0).  A channel whose radiance SUM is NaN counts as converged: it
 * resolves to 0 whatever follows (color.rs:16-18).  A pixel stops when n >= sample_end or when e <= max_error on all
 * three channels.  max_error = 0 turns the rule off: every pixel gets sample_end samples.
 * params: as for rt1w_render, except that sample_begin must be 0 and sample_end is the per-pixel cap; the statistics
 * buffers are always kept (RT1W_FLAG_STATS need not be set).  2 <= min_spp <= sample_end; max_error >= 0.
 * Outputs: HOST buffers, row 0 = top, each may be NULL - out_rgb_sum width*height*3 sums, out_spp width*height sample
 * counts, out_rgb8 width*height*3 bytes (into_sampled + Display with each pixel's own count, resolved on the device),
 * out_stat width*height*6 (as rt1w_render's).  stats: paths = the sum of out_spp; rays, waves, launches summed over the
 * rounds; render_ms the whole call.
 * One device only: a context that belongs to a communicator or drives several devices returns RT1W_ERR_UNSUPPORTED. */
rt1w_status rt1w_render_adaptive(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params,
                                 int32_t min_spp, double max_error, float *out_rgb_sum, int32_t *out_spp,
                                 uint8_t *out_rgb8, float *out_stat, rt1w_render_stats *stats);

/* Batch rendering: n_frames images of one scene in ONE wavefront (an animation through shutter windows, a turntable, a set
 * of views).  Frame f is rendered with cameras[f] and the seed seeds[f] (every frame params->seed when seeds is NULL);
 * size, sample range, depth, background, flags and pool come from params and are the same for all frames.  Frame f equals
 * rt1w_render(scene, &cameras[f], params with seed = seeds[f]) up to the order of the fp32 additions: its sample s of pixel
 * p keys Philox exactly as that render does.  The waves stay full until the last frame's paths have started, and the call
 * drains once instead of once per frame.
 * Outputs: HOST buffers, frame-major, row 0 = top within each frame; either may be NULL, but rank 0 must pass one -
 * out_rgb_sum n_frames*width*height*3 sums, out_rgb8 the same layout in bytes (resolved on the device, divided by
 * sample_end - sample_begin).  stats: paths = n_frames*width*height*(sample_end - sample_begin); rays, waves, launches and
 * render_ms cover the whole call.  Contexts: as rt1w_render (the sample range is sharded across devices or ranks, and
 * one ncclReduce of n_frames*width*height*3 floats collects the sums).
 * RT1W_ERR_INVALID: n_frames < 1, NULL cameras, n_frames*width*height >= 2^32 (checked before anything is allocated),
 * RT1W_FLAG_STATS, both outputs NULL on rank 0, and the argument checks of rt1w_render. */
rt1w_status rt1w_render_batch(rt1w_scene *scene, const rt1w_camera *cameras, int32_t n_frames, const uint64_t *seeds,
                              const rt1w_render_params *params, float *out_rgb_sum, uint8_t *out_rgb8,
                              rt1w_render_stats *stats);

/* First-hit feature buffers (AOVs) for denoisers and compositing: per pixel, sums over the sample range of what the first
 * segment of every path sees.
 * Definition.  For pixel p and global sample index s in [sample_begin, sample_end), take the render's own first ray of
 * path (p, s) - direction, origin, lens offset and time from the Philox key, counter and purpose words of the render's
 * camera ray - and its depth-0 closest hit, media included (the free-flight draw of the wave kernels at bounce 0: key
 * (pixel seed, seed lo), counter (s, 0, RNG_MEDIUM purpose)).  The buffers describe exactly the first segment of the paths
 * rt1w_render traces with the same camera and params.  Per sample the call adds
 *     albedo (3)    hit: Lambertian / Isotropic the texture value at the hit (the attenuation scatter uses), Metal its
 *                   albedo, Dielectric (1,1,1), DiffuseLight its emission on the front face (else 0) clamped to [0,1],
 *                   the null material 0;  miss: background clamped to [0,1]
 *     normal (3)    hit: the hit record's normal (what rt1w_trace_closest reports in normal3), 0 for a medium hit
 *                   (constant_medium.rs:98-106 writes an arbitrary (1,0,0), not a surface);  miss: 0
 *     distance (1)  hit: t * |d| (f64 hit parameter times the length of the un-normalised direction) rounded to f32,
 *                   the distance from the ray's origin on the lens;  miss: 0
 *     hits (1)      hit: 1;  miss: 0
 * The outputs are SUMS over the sample range, like rgb_sum: they add across sample ranges and reduce across ranks; hit
 * counts are exact (fewer than 2^24 samples per call).  Mean albedo and normal = sum / n (the normal mean is not
 * renormalised); mean distance = distance_sum / hits, 0 where hits == 0.
 * Outputs: HOST buffers, row 0 = top - out_albedo_sum and out_normal_sum width*height*3, out_distance_sum and out_hits
 * width*height.  Any may be NULL, but rank 0 must pass one.
 * params: size, sample range, seed and background as for rt1w_render; RT1W_FLAG_BVH_BINARY / _WIDE choose the tree as for
 * the render; max_depth, pool_paths, RT1W_FLAG_BVH_LOCKSTEP / _PERSISTENT and RT1W_FLAG_NO_TAIL are not used.  The call
 * allocates no path pool: one buffer of 8*width*height floats per device, kept by the context.  Contexts: as rt1w_render
 * (the sample range is sharded across devices or ranks, one ncclReduce of the 8*width*height sums to rank 0).
 * Deterministic: no float atomics, two calls with the same arguments on the same kind of context give identical bits.
 * stats: paths = rays = width*height*(sample_end - sample_begin) (one closest hit per sample), waves = 0, launches, render_ms.
 * RT1W_ERR_INVALID: RT1W_FLAG_STATS, all outputs NULL on rank 0, and the size and sample-range checks of rt1w_render. */
rt1w_status rt1w_render_aov(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params,
                            float *out_albedo_sum, float *out_normal_sum, float *out_distance_sum, float *out_hits,
                            rt1w_render_stats *stats);

/* Parity hook (test-only, like rt1w_eval_*): the render's first ray of path (pixel seed pixel_seed[i] = j*width+i, global
 * sample index sample[i]) for the camera and params (size and seed are used), i.e. what the wave kernels and
 * rt1w_render_aov trace.  The f64 origin is rounded to f32: exact for pinhole cameras (lens_radius == 0) whose origin is
 * representable in f32.  All buffers are HOST buffers. */
rt1w_status rt1w_eval_camera_rays(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params,
                                  const uint32_t *pixel_seed, const int32_t *sample, size_t n, rt1w_ray *out);

/* Parity hook: closest hit (`world.hit(ray, 0.001, inf)`, main.rs:62) for n
 * host rays.  prim_id = -1 on a miss.  Media draw their free-flight number from
 * Philox keyed by (seed, ray index, primitive id) so a CPU checker can replay it.
 * Any output pointer may be NULL. */
rt1w_status rt1w_trace_closest(rt1w_scene *scene, const rt1w_ray *rays, size_t n, uint64_t seed,
                               int32_t *prim_id, float *t, float *normal3, uint8_t *front_face, float *uv2);

/* Pointwise parity hooks for the shading functions (test-only entry points, like rt1w_trace_closest): the device
 * functions the wave kernels call, evaluated for n host inputs, so that a checker can hold them against the reference
 * formulas value by value.  All buffers are HOST buffers.
 *   rt1w_eval_light_pdf   light >= 0: `pdf_value(o, v)` of that entry of the light list (XZRect aarect.rs:119-138,
 *                         Sphere sphere.rs:72-90, others 0 by the trait default hittable.rs:66-68); light < 0: the
 *                         list's own `sum (1/n) pdf_value_i` (hittable.rs:144-150), i.e. HittablePdf::value (pdf.rs:47-49)
 *   rt1w_eval_texture     `Texture::value(u, v, p)` (texture.rs:40-89); uv2 may be NULL (u = v = 0)
 *   rt1w_eval_perlin      `Perlin::noise(p)` (turb_depth = 0, perlin.rs:46-72) or `turb(p, turb_depth)` (perlin.rs:74-86)
 *   rt1w_eval_dielectric  `reflect`, `refract`, `reflectance(min(dot(-uv, n), 1), ratio)` (material.rs:94-96,114-125)
 *   rt1w_eval_scatter     closest hit of ray i, then `Material::scatter` there as the render runs it for the path
 *                         (pixel seed i, sample i & 0xffff, bounce 0): Philox key (i, seed lo), counter (i & 0xffff, 0,
 *                         1 ^ (seed hi << 4), block).  material_type: rt1w_material_type of the hit or -1 (miss);
 *                         dir3: the scattered direction (zero when the path ends); weight3: attenuation * scattering_pdf
 *                         / pdf for scattering materials (main.rs:100-103), the emitted radiance for a DiffuseLight
 *                         (material.rs:168-181); time: the scattered ray's time (main.rs:86: the hit's t after a
 *                         Lambertian bounce).  Any output pointer may be NULL. */
rt1w_status rt1w_eval_light_pdf(rt1w_scene *scene, int32_t light, const double *origin3, const float *dir3, size_t n, float *pdf);
rt1w_status rt1w_eval_texture(rt1w_scene *scene, int32_t texture, const double *p3, const float *uv2, size_t n, float *rgb3);
rt1w_status rt1w_eval_perlin(rt1w_scene *scene, int32_t table, int32_t turb_depth, const double *p3, size_t n, float *out);
rt1w_status rt1w_eval_dielectric(rt1w_context *ctx, const float *unit_dir3, const float *normal3, const float *ratio, size_t n,
                                 float *reflect3, float *refract3, float *reflectance);
rt1w_status rt1w_eval_scatter(rt1w_scene *scene, const rt1w_ray *rays, size_t n, uint64_t seed, int32_t *prim_id,
                              int32_t *material_type, float *dir3, float *weight3, float *time);

/* `Color::into_sampled` + `Display for SampledColor` (color.rs:14-21,56-65):
 * NaN sum -> 0, mean, sqrt, clamp to [0,0.999], *256, truncate.  Host code. */
void rt1w_resolve_rgb8(const float *rgb_sum, int32_t width, int32_t height, int32_t samples_per_pixel, uint8_t *out_rgb8);

/* Philox4x32-10 block, exported so checkers can replay device draws. */
void rt1w_philox4x32(const uint32_t counter[4], const uint32_t key[2], uint32_t out[4]);

#ifdef __cplusplus
}
#endif
#endif /* RT1W_H */
