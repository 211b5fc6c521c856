/* oracle.h — C interface of the CPU oracle (TEST INFRASTRUCTURE, never shipped).
 *
 * The oracle is a C++17 / f64 restatement of the reference's per-pixel sample loop
 * (src/main.rs:51-190,957-1001 and every module it calls).  Only tests/, the smoke
 * check in __graft_entry__.py and bench.py's cpu_baseline / --impl reference legs may
 * load it.  It consumes the same POD scene description as the product
 * (include/rt1w.h) but shares no code with it.
 */
#ifndef RT1W_ORACLE_H
#define RT1W_ORACLE_H
#include "../include/rt1w.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct oracle_scene oracle_scene;

typedef struct oracle_render_stats {
    uint64_t paths;
    uint64_t rays; /* closest-hit queries: calls of world.hit from ray_color (main.rs:62) */
    double seconds;
    int32_t threads;
    int32_t reserved;
} oracle_render_stats;

const char *oracle_last_error(void);

/* Builds the reference object tree: nested BVHNode::new with random axis + median split
 * (bvh.rs:54-103, axis RNG = StdRng::seed_from_u64(bvh_seed)), AABox with its inner BVH
 * (aabox.rs:22-84), wrappers as wrappers. */
oracle_scene *oracle_scene_load(const rt1w_scene_desc *desc, uint64_t bvh_seed);
void oracle_scene_free(oracle_scene *s);
int32_t oracle_scene_num_prims(const oracle_scene *s);
/* BVHNode count and depth of the world tree (bvh.rs:60-101), AABox inner trees excluded. */
void oracle_scene_bvh_shape(const oracle_scene *s, int32_t *n_nodes, int32_t *depth);

/* world.hit(ray, 0.001, inf) for n rays (f32 inputs widened to f64).  Media replay the
 * device's keyed Philox free-flight draw.  ambiguous[i] != 0 on genuine (near-)ties only: two
 * leaves within 1e-9 relative of the winning t (e.g. the Cornell box bottom on the floor — the
 * reference's winner depends on its random BVH order there, bvh.rs:39-46,84), a candidate within
 * 1e-9 of t_min / t_max, or a winner that changes under a 1e-9-relative perturbation of the ray. */
int32_t oracle_trace_closest(const oracle_scene *s, const rt1w_ray *rays, size_t n, uint64_t seed, int32_t *prim_id,
                             double *t, double *normal3, uint8_t *front_face, double *uv2, uint8_t *ambiguous,
                             int32_t threads);

/* The pixel loop (main.rs:957-1001) for samples [sample_begin, sample_end).
 * rgb_sum: width*height*3 doubles, row 0 = top.  stat (nullable): width*height*6 doubles
 * (sum and sum of squares of min(sample, stat_clamp), NaN -> 0).  The per-pixel RNG is
 * StdRng::seed_from_u64(j*width+i) advanced past the first sample_begin samples' worth of
 * draws only when sample_begin == 0 (otherwise seeded with a mixed key). threads<=0: all cores. */
int32_t oracle_render(const oracle_scene *s, const rt1w_camera *camera, const rt1w_render_params *params,
                      int32_t threads, double *rgb_sum, double *stat, oracle_render_stats *stats);

/* Path replay: for each (pixel seed pixel_seed[i] = j*width+i, global sample index sample[i]) the path rt1w_render traces,
 * computed by ray_color / ray_color_without_light_objects above (f64 hits, virtual dispatch, the reference's formulas) with
 * every random number taken from the product's Philox stream.  At one sample per pixel, rt1w_render's rgb_sum of the pixel
 * is this path's radiance.
 *
 * The draw map (render.cu: camera_ray, scatter; kernels.cuh: medium_sample, scatter_*, random_in_unit_sphere):
 *   key     = (pixel seed j*w+i, seed lo)
 *   counter = (s, d, purpose ^ (seed hi << 4), block), d = the depth of the ray (0 = the camera ray)
 *   u01(x)  = (x >> 8) * 2^-24 in f32;  purposes RNG_CAMERA = 0, RNG_SCATTER = 1, RNG_MEDIUM = 2
 *   camera        (s, 0, CAMERA, 0): u01(x.x) s-jitter, u01(x.y) t-jitter, u01(x.z) shutter time.  The ray is the
 *                 product's: f32 direction and time, f64 origin.
 *   lens          (lens_radius != 0 only) blocks 1, 2, ...: try (y.x, y.y), then (y.z, y.w) as 2 u01 - 1; accept on the
 *                 f32 test px^2 + py^2 < 1
 *   free flight   of a medium hit by the ray of depth d: (s, d, MEDIUM, device LEAF index of the medium); xi = u01(x.x),
 *                 distance -1/density log(xi) (the device takes __logf, the replay the f64 log)
 *   Lambertian    at depth d: (s, d, SCATTER, 0): x.x >> 31 = sample towards the lights (only when the scene has a light
 *                 list); light = min(int(u01(x.y) n), n - 1) in f32; r1 = u01(x.z), r2 = u01(x.w) for the cosine or the
 *                 light sample; a light kind with no pdf gives the direction (1, 0, 0)
 *   Metal fuzz>0  random_in_unit_sphere: block 0, then 1, 2, ...: (2 u01 - 1) of x.x, x.y, x.z, f32 test |p|^2 < 1
 *   Dielectric    block 0: u01(x.x) against reflectance
 *   Isotropic     random_in_unit_sphere, as Metal
 * leaf_of_prim[prim id] (oracle_scene_num_prims entries; NULL when the scene has no media): the device leaf index of each
 * primitive, the inverse of rt1w_scene_get_leaf_prims.
 * Outputs: out_rgb[3n] radiance (f64), out_rays[n] calls of world.hit (nullable), out_flags[n] (nullable):
 *   bit 0  a closest hit that is not robust: the oracle_trace_closest tie bookkeeping, a winner that changes when the
 *          direction moves by 1e-5 relative, or a moving sphere met at a time outside [time0, time1] no later than the
 *          winner (it has left its bounding box, so whether a tree finds it depends on the tree)
 *   bit 1  a draw decision within 1e-4 of its threshold: Schlick vs xi, ratio sin(theta) vs 1, the rejection tests, the
 *          free-flight distance vs the distance inside the medium
 *   bit 2  a Lambertian pdf or weight outside the normal f32 range (0 included), or a textured attenuation that moves by
 *          more than 1e-3 relative within the device ray's position uncertainty (PathTracer::fragile_texture)
 * mutation (test-only): 0 = the product's scheme; each other value replays one plausible kernel bug, so that a test can show
 * that its bars catch it: 1 the scatter counter uses d+1; 2 the seed hi word is left out of the purpose words; 3 the light
 * index comes from x.x; 4 the Metal / Isotropic retry reuses block 0 (given up after 64 tries); 5 the medium block is the
 * primitive id instead of the leaf; 6 lights emit on the back face too; 7 the Lambertian bounce keeps the ray's time;
 * 8 the depth limit is one bounce later; 9 the camera's s and t jitters are swapped.
 * Returns 0, or non-zero with oracle_last_error set. */
int32_t oracle_replay_paths(const oracle_scene *s, const rt1w_camera *camera, const rt1w_render_params *params, const int32_t *leaf_of_prim,
                            size_t n, const uint32_t *pixel_seed, const int32_t *sample, int32_t mutation, int32_t threads, double *out_rgb,
                            uint32_t *out_rays, uint8_t *out_flags);
/* One replayed path as text (radiance, rays, flags, then per bounce: primitive, rt1w_material_type, t, weight, flags so far),
 * so that a failing pixel can explain itself. */
int32_t oracle_replay_path_log(const oracle_scene *s, const rt1w_camera *camera, const rt1w_render_params *params, const int32_t *leaf_of_prim,
                               uint32_t pixel_seed, int32_t sample, int32_t mutation, char *buf, size_t capacity);
/* The replay's camera rays (origin f64, direction and time f32 values widened). */
void oracle_replay_camera_rays(const oracle_scene *s, const rt1w_camera *camera, const rt1w_render_params *params, size_t n,
                               const uint32_t *pixel_seed, const int32_t *sample, int32_t mutation, double *origin3, double *dir3, double *time);

/* ---- known-answer probes (SURVEY.md §4 table) ---- */
double oracle_xz_rect_pdf_value(const double rect[5], const double o[3], const double v[3]);
double oracle_sphere_pdf_value(const double center[3], double radius, const double o[3], const double v[3]);
double oracle_sphere_hit_t(const double center[3], double radius, const double o[3], const double d[3], double t_min, double t_max);
double oracle_reflectance(double cosine, double ref_idx);
void oracle_refract(const double uv[3], const double n[3], double etai_over_etat, double out[3]);
void oracle_sphere_uv(const double p[3], double out_uv[2]);
void oracle_onb_from_w(const double n[3], double out_uvw[9]);
void oracle_quantise(const double rgb_sum[3], int32_t spp, int32_t out[3]);
void oracle_camera_ray(const rt1w_camera *cam, double s, double t, double out_origin[3], double out_dir[3]); /* lens_radius 0 */
void oracle_rotate_y_bbox(const double bmin[3], const double bmax[3], double deg, double out_min[3], double out_max[3]);
/* Closest hit of one f64 ray against a described scene: returns prim id (or -1). */
int32_t oracle_hit_one(const oracle_scene *s, const double o[3], const double d[3], double time, double *t, double p[3],
                       double n[3], int32_t *front_face);
double oracle_perlin_noise(const rt1w_perlin *tab, const double p[3]);
double oracle_perlin_turb(const rt1w_perlin *tab, const double p[3], int32_t depth);
void oracle_texture_value(const oracle_scene *s, int32_t texture, double u, double v, const double p[3], double out[3]);
void oracle_bvh_count(int32_t n_objects, uint64_t seed, int32_t *n_nodes, int32_t *depth);
/* RNG probes */
void oracle_chacha_block(const uint32_t state[16], int32_t rounds, uint32_t out[16]);
void oracle_stdrng_u32(uint64_t seed, int32_t n, uint32_t *out);
void oracle_stdrng_from_seed_u32(const uint8_t seed[32], int32_t n, uint32_t *out);
void oracle_stdrng_f64(uint64_t seed, int32_t n, double *out);
void oracle_philox(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

#ifdef __cplusplus
}
#endif
#endif
