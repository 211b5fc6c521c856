// render.h — host-side interface of the wavefront renderer (render.cu) used by the C ABI (api.cu).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rt1w.h"
#include "device_types.h"
#include "kernels.cuh"

namespace rt1w {

// Device-side counters of the wavefront queues (one struct per context, zeroed per render).  Three copies
// rotate: wave w reads slot w % 3, appends to slot (w + 1) % 3 and clears slot (w + 2) % 3 for wave w + 1.
struct Counters {
    uint32_t n_mat[3][Q_COUNT];      // hits queued per material family (rt1w_material_type) for the wave that reads the slot
    unsigned long long next_path[3]; // next (pixel, sample) pair to start, as seen by the wave that reads the slot
    unsigned long long rays;         // closest-hit queries so far
    uint32_t tail_ticket;            // k_tail: CTAs that have finished (the last one closes the queues)
};

// One queue = SoA payload arrays; entry i of every array belongs to the same ray, so a warp reading
// entries [i, i+32) issues fully coalesced 16-byte-per-lane loads (DESIGN.md "Data layout").
struct RayQueue {
    double2 *a = nullptr; // origin.x, origin.y
    RayB *b = nullptr;    // origin.z, direction.x, direction.y
    RayC *c = nullptr;    // direction.z, time, state, pixel
    float4 *t = nullptr;  // throughput rgb (+ unused lane)
    HitRec *h = nullptr;  // t, leaf, meta of the hit the ray ended on
};

// The queues of a render: one hit queue per scattering material family, double-buffered between waves.
// No path owns a slot: rays move from queue to queue, compacted at every stage.
struct Pool {
    RayQueue mat[2][Q_COUNT];
    Counters *ctr = nullptr;
    uint32_t capacity = 0;  // rays in flight per wave (<= allocated)
    uint32_t allocated = 0; // entries every queue was allocated with
    int material_mask = 0; // material queues allocated
};

cudaError_t pool_alloc(Pool &pool, uint32_t capacity, int material_mask);
void pool_free(Pool &pool);

struct RenderArgs {
    SceneView sc;
    Pool pool;
    DRenderParams rp;
    DCamera cam;
    float *accum; // width*height*3 radiance sums
    float *stat;  // width*height*6 clamped sum / sum of squares, or nullptr
};

enum KernelSlot : int { K_WAVE = 0, K_COUNT = RT1W_KERNEL_COUNT };

struct WaveStats {
    uint64_t waves = 0, launches = 0, rays = 0;
    bool profile = false;        // RT1W_FLAG_PROFILE: bracket every launch with CUDA events
    double kernel_ms[K_COUNT] = {0};
    uint64_t kernel_launches[K_COUNT] = {0};
};

// Runs the wave loop to completion on `stream`, adding to accum/stat (zeroed by the caller before the first range).
// list: nullptr (pixel seeds 0 .. rp.n_pixels - 1) or rp.n_pixels pixel seeds j*w+i, ascending, on the device.
// batch: nullptr, or (with list == nullptr) the device tables of a batch render (device_types.h: DBatch): rp.n_pixels is
// then n_frames * width * height, and accum holds the frames' sums one after the other.
// groups: nullptr, or (with list == batch == nullptr) the light-group table of a light-group render on the device: entry 0
// the background group, entry 1 + leaf the group of device leaf `leaf` (rt1w.h: rt1w_render_light_groups); accum then holds
// the groups' images one after the other, rp.n_pixels each.
// material_mask: bit m set when some primitive uses rt1w_material_type m.
// h_ctr: TWO pinned host snapshots of the counters (the termination poll runs one chunk of waves behind).
cudaError_t render_waves(const RenderArgs &args, const uint32_t *list, const DBatch *batch, const int32_t *groups, int material_mask, Counters *h_ctr,
                         cudaStream_t stream, int sm_count, WaveStats &ws);

// Adaptive sampling, after a round of n samples over n_active pixels (d_list, or every pixel when null): the convergence
// rule (rt1w.h: rt1w_render_adaptive); d_spp[pixel] = n for the pixels that stop; the others, in list order, to d_next.
// d_keep: n_active bytes; d_counts: converge_blocks(n_active) + 1 entries, the last one receives the count of d_next.
uint32_t converge_blocks(uint32_t n_active);
cudaError_t converge_launch(const float *d_accum, const float *d_stat, const uint32_t *d_list, uint32_t n_active, int width, int height, int n, int max_spp,
                            double max_error, int32_t *d_spp, uint8_t *d_keep, uint32_t *d_counts, uint32_t *d_next, cudaStream_t stream);

// Closest-hit parity kernel (rt1w_trace_closest).  All pointers are device pointers; outputs may be null.
// leaf / t64 (nullable): the hit as the kernels carry it (leaf | side << 28, f64 distance), input of eval_scatter_launch.
cudaError_t trace_closest_launch(const SceneView &sc, const rt1w_ray *rays, size_t n, uint64_t seed, int32_t *prim_id, float *t,
                                 float *normal3, uint8_t *front_face, float *uv2, cudaStream_t stream, int32_t *leaf = nullptr,
                                 double *t64 = nullptr);

// Pointwise parity hooks (rt1w.h: rt1w_eval_*); all pointers are device pointers.
cudaError_t eval_light_pdf_launch(const SceneView &sc, int light, const double *o3, const float *v3, size_t n, float *pdf, cudaStream_t stream);
cudaError_t eval_texture_launch(const SceneView &sc, int texture, int perlin_table, int turb_depth, const double *p3, const float *uv2, size_t n,
                                float *out, cudaStream_t stream);
cudaError_t eval_dielectric_launch(const float *uv3, const float *n3, const float *ratio, size_t n, float *reflect3, float *refract3,
                                   float *reflectance, cudaStream_t stream);
cudaError_t eval_scatter_launch(const SceneView &sc, const rt1w_ray *rays, const int32_t *leaf, const double *t64, size_t n, uint64_t seed,
                                int32_t *material, float *dir3, float *weight3, float *time_out, cudaStream_t stream);

// First-hit feature buffers (rt1w.h: rt1w_render_aov) of the sample range [rp.sample_begin, + rp.n_samples) of every pixel of
// args' image: d_out receives 8 * width * height floats [albedo 3P | normal 3P | distance P | hits P], every one written.
// One launch; args.pool and args.accum are not used.
cudaError_t aov_launch(const RenderArgs &args, int material_mask, float *d_out, int sm_count, cudaStream_t stream);
// The render's first ray of path (pixel_seed[i], global sample index sample[i]) (rt1w_eval_camera_rays); device pointers.
cudaError_t eval_camera_rays_launch(const RenderArgs &args, const uint32_t *pixel_seed, const int32_t *sample, size_t n, rt1w_ray *out, cudaStream_t stream);

// The denoiser (denoise.cu; rt1w.h: rt1w_denoise): the sums of n_samples samples - d_rgb_sum 3P, d_stat 6P (RT1W_FLAG_STATS
// layout), d_aov 8P (aov_launch's layout) - filtered into *d_out_rgb (3P mean radiance, inside d_scratch) and, when d_rgb8 is
// not null, resolved into it.  d_scratch: denoise_scratch_bytes(P).  dp has been checked.  *launches: kernels enqueued.
size_t denoise_scratch_bytes(size_t pixels);
cudaError_t denoise_launch(const float *d_rgb_sum, const float *d_stat, const float *d_aov, int width, int height, int n_samples, const rt1w_denoise_params &dp,
                           void *d_scratch, float **d_out_rgb, uint8_t *d_rgb8, uint64_t *launches, cudaStream_t stream);

// Device-side image resolve (color.rs:14-21,56-65): width*height*3 radiance sums -> 8-bit channels.
cudaError_t resolve_launch(const float *d_rgb_sum, size_t n_values, int samples_per_pixel, uint8_t *d_rgb8, cudaStream_t stream);
// The same with each pixel's own sample count (d_spp: width*height counts).
cudaError_t resolve_counts_launch(const float *d_rgb_sum, const int32_t *d_spp, size_t n_values, uint8_t *d_rgb8, cudaStream_t stream);

} // namespace rt1w
