// render.cu — the wavefront kernel and the wave loop (sm_100a).
//
// The reference's pixel loop + recursive ray_color (main.rs:51-190, 957-1001) become a sequence of waves.
// One wave = ONE launch of k_wave, in which every thread
//
//   1. takes one unit of work: a hit queued by the previous wave for one of the scattering material
//      families (its material decides the scatter code: material.rs, pdf.rs, constant_medium.rs:31-51), or,
//      past the queued hits, a new camera path (main.rs:968-971, camera.rs:61-73);
//   2. extends the resulting ray: closest hit over the scene (bvh.rs:25-50 and every `hit()` below it);
//   3. ends the path there (miss -> background, null material, DiffuseLight -> emission; main.rs:110-115) or
//      appends ray + path state + hit to the queue of the material it landed on, for the next wave.
//
// Ray and path state live in SoA queues in HBM (render.h: RayQueue), one per material family and double
// buffered between waves.  Rays do not own a slot: a wave reads its input queues front to back (fully
// coalesced 16-byte-per-lane loads; the queues are laid end to end in the thread index space, each padded
// to a multiple of 32, so a warp only ever shades one material) and appends the survivors to the output
// queues, regrouped per material with __ballot_sync + __popc + __shfl_sync and one atomic instruction per
// warp.  The recursion `emitted + attenuation * f * L / pdf` is unrolled into a running throughput: only
// terminal events carry radiance, so a path adds to its pixel once.
//
// Per ray segment the wave moves 80 B in and 80 B out of HBM (SURVEY.md section 8d counts 148 B for a
// minimal fp32 wavefront); an earlier split pipeline (generate / extend / one shade kernel per material,
// 288 B per segment, 7 launches per wave) ran 1.3x slower.
#include "render.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <utility>
#include <vector>

namespace rt1w {

// tunables (overridable at build time for sweeps: build.py --variant NAME -DRT1W_...=N)
#ifndef RT1W_WAVE_THREADS
#define RT1W_WAVE_THREADS 128
#endif
#ifndef RT1W_FLAT_MIN_BLOCKS
#define RT1W_FLAT_MIN_BLOCKS 5 // CTAs per SM of the flat-scan wave kernel with media (128 threads, 96 registers)
#endif
#ifndef RT1W_BVH_MIN_BLOCKS
#define RT1W_BVH_MIN_BLOCKS 5 // lockstep BVH wave kernel with media; one more without
#endif
#ifndef RT1W_PERSISTENT_MIN_BLOCKS
#define RT1W_PERSISTENT_MIN_BLOCKS 4 // persistent BVH wave kernel: more resident rays only thrash L1 on the big trees it is used for
#endif
constexpr int kWaveThreads = RT1W_WAVE_THREADS;
#ifndef RT1W_FLAT_THREADS
#define RT1W_FLAT_THREADS 256 // medium-free flat-scan wave kernel: 3 CTAs of 256 threads per SM (80 registers) beat 6 of 128 by 1.4 %
#endif
// CTA size and CTAs per SM of the wave kernel variants (the launch uses the same functions)
__host__ __device__ constexpr int wave_threads(bool flat, bool media) { return flat && !media ? RT1W_FLAT_THREADS : kWaveThreads; }
#ifndef RT1W_FLAT_PLAIN_MIN_BLOCKS
#define RT1W_FLAT_PLAIN_MIN_BLOCKS (6 * 128 / RT1W_FLAT_THREADS)
#endif
__host__ __device__ constexpr int wave_min_blocks(bool flat, bool media) {
    return flat ? (media ? RT1W_FLAT_MIN_BLOCKS : RT1W_FLAT_PLAIN_MIN_BLOCKS) : RT1W_BVH_MIN_BLOCKS + (media ? 0 : 1);
}
constexpr int kExtendThreads = kWaveThreads; // k_trace shares the traversal-stack geometry

// Scattering material families, in the order their queues are laid out in a wave's thread index space.
__host__ __device__ constexpr int scatter_mat(int s) { return s < 3 ? s : int(RT1W_MAT_ISOTROPIC); } // LAMBERTIAN, METAL, DIELECTRIC, ISOTROPIC
static_assert(RT1W_MAT_LAMBERTIAN == 0 && RT1W_MAT_METAL == 1 && RT1W_MAT_DIELECTRIC == 2, "segment order");

// Sorts the lanes of a warp into the per-material hit queues with ONE atomic instruction: lane q
// reserves queue q's entries for the whole warp (Q_COUNT lanes, Q_COUNT addresses, one round trip),
// then every lane fetches the base of its own destination with a shuffle.  dest < 0: nothing to append.
// Two halves, so that the caller can put independent work (the splat of the paths that end) between the atomic
// and the first use of its result: the round trip to L2 was 40 % of the wave kernel's long-scoreboard stalls.
struct QueueReservation {
    uint32_t base; // lane q: start of the warp's entries in queue q
    uint32_t mine; // lanes with the same destination as this one
};
RT1W_DEV QueueReservation warp_sort_begin(uint32_t *n_mat, int dest) {
    const int lane = threadIdx.x & 31;
    QueueReservation res;
    res.base = 0, res.mine = 0;
    uint32_t count_for_lane = 0;
#pragma unroll
    for (int q = 0; q < Q_COUNT; ++q) {
        if (q == RT1W_MAT_DIFFUSE_LIGHT) continue; // lights end the path inside the wave
        const unsigned m = __ballot_sync(0xffffffffu, dest == q);
        if (dest == q) res.mine = m;
        if (lane == q) count_for_lane = uint32_t(__popc(m));
    }
    if (count_for_lane) res.base = atomicAdd(&n_mat[lane], count_for_lane);
    return res;
}
RT1W_DEV uint32_t warp_sort_end(const QueueReservation &res, int dest) {
    const int lane = threadIdx.x & 31;
    const uint32_t base = __shfl_sync(0xffffffffu, res.base, dest < 0 ? 0 : dest);
    return base + __popc(res.mine & ((1u << lane) - 1u));
}

// Programmatic dependent launch (sm_90+): a wave kernel is launched while its predecessor still runs; everything
// before this call must not touch what the predecessor writes.  Once the predecessor is complete the next wave may
// start its own prologue.
RT1W_DEV void grid_dependency_wait() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// A path ends: pixel += throughput * radiance.  A NaN product must reach the sum even when the
// radiance is zero: the reference turns a NaN pixel SUM into black (color.rs:14-21), and
// `li / pdf` with pdf == 0 is NaN there whatever li is (main.rs:102).
// `seed`: the path's pixel as the reference numbers it (j * width + i, row j counted from the bottom, main.rs:964).
// n / d through the host-prepared reciprocal of d rounded up (device_types.h: DRenderParams): three instructions instead of the ~20 of a 32-bit division
RT1W_DEV uint32_t div_by(uint32_t n, double inv_up) { return __double2uint_rz(double(n) * inv_up); }

// `first`: the image's first pixel in the sums (a frame of a batch render).
RT1W_DEV void splat(const RenderArgs &a, uint32_t seed, f3 thr, f3 radiance, uint32_t first = 0u) {
    const float c[3] = {thr.x * radiance.x, thr.y * radiance.y, thr.z * radiance.z};
    const uint32_t j = div_by(seed, a.rp.inv_width_up), col = seed - j * uint32_t(a.rp.width);
    const uint32_t pixel = first + (uint32_t(a.rp.height) - 1u - j) * uint32_t(a.rp.width) + col; // main.rs:959: rows are emitted top first
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (c[k] != 0.0f) atomicAdd(a.accum + 3 * size_t(pixel) + k, c[k]);
    }
    if (a.stat) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            float x = c[k];
            if (x != x) x = 0.0f;
            x = fminf(x, a.rp.stat_clamp);
            if (x != 0.0f) {
                atomicAdd(a.stat + 6 * size_t(pixel) + k, x);
                atomicAdd(a.stat + 6 * size_t(pixel) + 3 + k, x * x);
            }
        }
    }
}
RT1W_DEV bool finite3(f3 v) { return (fabsf(v.x) + fabsf(v.y) + fabsf(v.z)) < CUDART_INF_F; } // false for NaN and inf

// Queue entries are read once and written once per wave: streaming (evict-first) accesses keep them from
// pushing the radiance sums and the scene out of L2.
template <class T> RT1W_DEV T stream_load(const T *p) {
    static_assert(sizeof(T) == 16, "queue arrays hold 16-byte elements");
    const float4 v = __ldcs(reinterpret_cast<const float4 *>(p));
    return *reinterpret_cast<const T *>(&v);
}
template <class T> RT1W_DEV void stream_store(T *p, const T &x) {
    static_assert(sizeof(T) == 16, "queue arrays hold 16-byte elements");
    __stcs(reinterpret_cast<float4 *>(p), *reinterpret_cast<const float4 *>(&x));
}

// Philox key/counter of a path: key = (reference pixel seed j*w+i (main.rs:964), seed), counter = (sample, bounce, purpose, block)
RT1W_DEV void path_rng_key(const DRenderParams &rp, uint32_t seed, uint32_t &k0, uint32_t &k1) { k0 = seed, k1 = rp.seed_lo; }
RT1W_DEV uint32_t purpose_word(const DRenderParams &rp, uint32_t stream) { return stream ^ (rp.seed_hi << 4); }

// ------------------------------------------------------------------------------------------
// path numbering: what the pixel word of a path (RayC::pixel) names, a compile-time choice of the wave kernels, so that
// the instantiations of one mode carry no code of the others (these kernels move by percents on code they never run,
// DESIGN.md section 7)
// ------------------------------------------------------------------------------------------
enum Numbering : int {
    NUM_IMAGE = 0, // paths number the pixels of one image: the pixel word is the reference seed j*w+i
    NUM_LIST = 1,  // adaptive rounds: new paths go to the pixels of a list (generate_ray); the pixel word is as NUM_IMAGE's
    NUM_BATCH = 2, // batch renders: the pixel word is the batch pixel g = f * frame_pixels + (j*w+i) of frame f (DBatch)
    NUM_GROUP = 3, // light groups: NUM_IMAGE's numbering; a path's sum goes to the image of the group of whatever ended it (group_first)
};

RT1W_DEV uint32_t batch_frame(const DBatch *batch, uint32_t g) { // g / frame_pixels (device_types.h: DBatch)
    const uint32_t t = __umulhi(g, __ldg(&batch->magic));
    return (t + ((g - t) >> __ldg(&batch->shift1))) >> __ldg(&batch->shift2);
}
RT1W_DEV uint2 batch_seed(const DBatch *batch, uint32_t f) { return __ldg(reinterpret_cast<const uint2 *>(batch->seeds) + f); } // (lo, hi)

// The Philox key, purpose words and pixel of a path in mode NUM: frame f of a batch keys exactly as a render of its own
// (its pixel seed, its seed words), so that every frame equals that render.
template <int NUM> RT1W_DEV void path_rng_key(const DRenderParams &rp, const DBatch *batch, uint32_t pixel, uint32_t &k0, uint32_t &k1) {
    if (NUM == NUM_BATCH) {
        const uint32_t f = batch_frame(batch, pixel);
        k0 = pixel - f * __ldg(&batch->frame_pixels), k1 = batch_seed(batch, f).x;
    } else {
        path_rng_key(rp, pixel, k0, k1);
    }
}
template <int NUM> RT1W_DEV uint32_t purpose_word(const DRenderParams &rp, const DBatch *batch, uint32_t pixel, uint32_t stream) {
    if (NUM == NUM_BATCH) return stream ^ (batch_seed(batch, batch_frame(batch, pixel)).y << 4);
    return purpose_word(rp, stream);
}
// NUM_GROUP: the kernels' trailing table pointer carries the light-group table instead of batch tables (render_waves):
// int32 entry 0 = the background group, entry 1 + leaf = the group of device leaf `leaf` (read for DiffuseLight leaves only).
// The first of the sums of the group a path ends in: its light's group when it ends on a DiffuseLight hit, else the
// background group (a miss, the null material, the depth limit - where h is no hit and is not read).
RT1W_DEV uint32_t group_first(const RenderArgs &a, const DBatch *batch, int mat_type, const HitRec &h) {
    const int32_t *table = reinterpret_cast<const int32_t *>(batch);
    return uint32_t(__ldg(table + (mat_type == RT1W_MAT_DIFFUSE_LIGHT ? 1 + (h.leaf & kLeafMask) : 0))) * a.rp.n_pixels;
}

template <int NUM> RT1W_DEV void splat(const RenderArgs &a, const DBatch *batch, uint32_t pixel, f3 thr, f3 radiance, int mat_type, const HitRec &h) {
    if (NUM == NUM_BATCH) { // frame f's sums follow frames 0 .. f-1's
        const uint32_t first = batch_frame(batch, pixel) * __ldg(&batch->frame_pixels);
        splat(a, pixel - first, thr, radiance, first);
    } else if (NUM == NUM_GROUP) { // group g's image follows groups 0 .. g-1's
        splat(a, pixel, thr, radiance, group_first(a, batch, mat_type, h));
    } else {
        splat(a, pixel, thr, radiance);
    }
}

// ------------------------------------------------------------------------------------------
// a new camera path (main.rs:968-971, camera.rs:61-73, math.rs:30-37)
// ------------------------------------------------------------------------------------------
// The first ray of path (pixel, global sample index rp.sample_begin + sample_rel): `pix` is the pixel's reference seed j*w+i
// in its image, (key1, camera_word) the Philox key word and RNG_CAMERA purpose word of the render (or of its frame).  One copy for the
// wave kernels (generate_ray), the feature buffers (k_aov) and their parity hook, so that they cannot drift apart.
RT1W_DEV Ray camera_ray(const DCamera &cam, const DRenderParams &rp, uint32_t pix, uint32_t key1, uint32_t camera_word, uint32_t sample_rel) {
    const uint32_t j = div_by(pix, rp.inv_width_up), col = pix - j * uint32_t(rp.width);
    Rng rng;
    rng.k0 = pix, rng.k1 = key1;
    rng.c0 = uint32_t(rp.sample_begin) + sample_rel, rng.c1 = 0;
    rng.c2 = camera_word, rng.block = 0;
    const Philox4 x = rng.next4();
    const double s = (double(col) + double(u01(x.x))) * rp.inv_w1; // main.rs:968
    const double t = (double(j) + double(u01(x.y))) * rp.inv_h1;   // main.rs:969
    double offx = 0.0, offy = 0.0, offz = 0.0;
    if (cam.lens_radius != 0.0) { // camera.rs:62-63; the rejection loop of math.rs:30-37
        float px, py;
        for (;;) {
            const Philox4 y = rng.next4();
            px = 2.0f * u01(y.x) - 1.0f, py = 2.0f * u01(y.y) - 1.0f;
            if (px * px + py * py < 1.0f) break;
            px = 2.0f * u01(y.z) - 1.0f, py = 2.0f * u01(y.w) - 1.0f;
            if (px * px + py * py < 1.0f) break;
        }
        const double rx = cam.lens_radius * double(px), ry = cam.lens_radius * double(py);
        offx = cam.u[0] * rx + cam.v[0] * ry;
        offy = cam.u[1] * rx + cam.v[1] * ry;
        offz = cam.u[2] * rx + cam.v[2] * ry;
    }
    Ray r;
    // camera.rs:67-70: direction = lower_left_corner + s*horizontal + t*vertical - origin - offset (never normalised)
    r.dx = float(cam.llc_rel[0] + s * cam.horizontal[0] + t * cam.vertical[0] - offx);
    r.dy = float(cam.llc_rel[1] + s * cam.horizontal[1] + t * cam.vertical[1] - offy);
    r.dz = float(cam.llc_rel[2] + s * cam.horizontal[2] + t * cam.vertical[2] - offz);
    r.ox = cam.origin[0] + offx, r.oy = cam.origin[1] + offy, r.oz = cam.origin[2] + offz;
    r.time = cam.time0 + (cam.time1 - cam.time0) * u01(x.z); // camera.rs:71
    return r;
}

// Path numbering.  Paths are started tile by tile: all samples of a tile of 2^tile_shift consecutive pixels (sample
// by sample, pixel by pixel inside it) before the next tile, so that the pixels the paths in flight add to - a wave
// holds millions of paths - stay a small, L2-resident part of a big image (3840x2160: 100 MB of sums).  A small
// image is one tile, i.e. sample-major order.  Path number path0 + i = tile t0 + (w0 + i) / tile_paths, position
// (w0 + i) % tile_paths inside it, with t0 = path0 / tile_paths and w0 = path0 % tile_paths split once per CTA.
// NUM_LIST (adaptive rounds): the same numbering runs over slots of a pixel list - n_pixels is its length, and slot k
// renders the pixel whose reference seed is list[k].  The list is ascending, so a tile still adds to a compact range of sums.
// NUM_BATCH: it runs over the n_frames * width * height batch pixels (tiles may straddle frames); batch pixel g renders
// pixel g - f * frame_pixels of frame f with the frame's camera (lens, shutter) and seed words.
template <int NUM = NUM_IMAGE>
RT1W_DEV Ray generate_ray(const RenderArgs &a, const uint32_t *list, const DBatch *batch, uint32_t t0, uint32_t w0, uint32_t i, uint32_t &state,
                          uint32_t &seed_out) {
    const uint32_t w = w0 + i, dt = div_by(w, a.rp.inv_tile_paths_up);
    const uint32_t within = w - dt * a.rp.tile_paths, first = (t0 + dt) << a.rp.tile_shift;
    uint32_t sample_rel, seed;
    if (a.rp.n_pixels - first >= (1u << a.rp.tile_shift)) { // a whole tile
        sample_rel = within >> a.rp.tile_shift, seed = first + (within & ((1u << a.rp.tile_shift) - 1u));
    } else { // the last, partial tile
        const uint32_t tp = a.rp.n_pixels - first;
        sample_rel = within / tp, seed = first + (within - sample_rel * tp);
    }
    if (NUM == NUM_LIST) seed = __ldg(list + seed);
    uint32_t frame = 0, frame_first = 0;
    uint2 frame_seed = make_uint2(0u, 0u);
    if (NUM == NUM_BATCH) frame = batch_frame(batch, seed), frame_first = frame * __ldg(&batch->frame_pixels), frame_seed = batch_seed(batch, frame);
    const DCamera &cam = NUM == NUM_BATCH ? batch->cams[frame] : a.cam;
    const uint32_t pix = seed - frame_first; // the pixel's reference seed in its image
    const Ray r = camera_ray(cam, a.rp, pix, NUM == NUM_BATCH ? frame_seed.x : a.rp.seed_lo,
                             NUM == NUM_BATCH ? RNG_CAMERA ^ (frame_seed.y << 4) : purpose_word(a.rp, RNG_CAMERA), sample_rel);
    state = sample_rel << 8;
    seed_out = seed;
    return r;
}

// ------------------------------------------------------------------------------------------
// scatter at a queued hit of material family `mat` (warp-uniform in the wave kernels).  Rewrites `r` into the
// scattered ray, advances the depth in c.state and folds the attenuation into `thr`.  Returns false when
// the path ends here (depth limit, main.rs:59-61).  One copy of the hit reconstruction, the Philox setup and the
// epilogue serves all families: instruction-cache footprint is what the wave kernel is most sensitive to.
// ------------------------------------------------------------------------------------------
// `prims`, `frames`: the scene tables (global memory, or the flat scan's shared-memory copies).
// MEDIA = false: no Isotropic hits can be queued (ConstantMedium::new is the only source, constant_medium.rs:22-28).
// NUM, batch: the path numbering (Numbering) and its tables.
// PLAN: the flat scene's plan (flat_plans.h: the wrapper chains and the light list compiled in), or -1.
template <bool MEDIA, bool RICH, bool FAST_SIN = true, int NUM = NUM_IMAGE, int PLAN = -1>
RT1W_DEV bool scatter(const int mat, const RenderArgs &a, const DPrim *prims, const DFrame *frames, const DPerlin *perlins, const DLight *lights,
                      Ray &r, const HitRec &hr, RayC &c, f3 &thr, const DBatch *batch) {
    const DMaterial m = a.sc.materials[hr.meta >> 12];
    const HitInfo h = finalize_hit<false, PLAN>(prims + (hr.leaf & kLeafMask), frames, hr.leaf >> kLeafBits, r, hr.t);
    const uint32_t depth = c.state & 255u;
    Rng rng;
    path_rng_key<NUM>(a.rp, batch, c.pixel, rng.k0, rng.k1);
    rng.c0 = uint32_t(a.rp.sample_begin) + (c.state >> 8), rng.c1 = depth, rng.c2 = purpose_word<NUM>(a.rp, batch, c.pixel, RNG_SCATTER), rng.block = 0;
    const Philox4 x0 = rng.next4(); // every family starts from this block (one Philox body for the four of them; the Dielectric ignores it on total reflection)
    f3 dir;
    float time = r.time; // specular scatters keep ray.time (material.rs:104,157; constant_medium.rs:46)
    if (mat == RT1W_MAT_LAMBERTIAN) {
        const f3 att = texture_value<RICH, FAST_SIN>(a.sc, perlins, m.texture, h);
        f3 weight;
        dir = scatter_lambertian<PLAN>(a.sc, lights, h, x0, weight);
        thr = thr * att * weight;
        time = float(hr.t); // main.rs:86,145: the scattered ray's time is the hit parameter t
    } else if (mat == RT1W_MAT_METAL) {
        dir = scatter_metal(m, r, h, x0, rng);
        thr = thr * mk3(m.albedo[0], m.albedo[1], m.albedo[2]);
    } else if (mat == RT1W_MAT_DIELECTRIC || !MEDIA) {
        dir = scatter_dielectric(m, r, h, x0); // attenuation (1,1,1)
    } else {                                    // Isotropic, constant_medium.rs:36-51
        thr = thr * texture_value<RICH, FAST_SIN>(a.sc, perlins, m.texture, h);
        dir = random_in_unit_sphere(x0, rng);
    }
    if (depth + 1u >= uint32_t(a.rp.max_depth)) return false; // main.rs:59-61: the next ray_color call returns black (the caller keeps a NaN throughput alive in the pixel)
    r.ox = h.px, r.oy = h.py, r.oz = h.pz;
    r.dx = dir.x, r.dy = dir.y, r.dz = dir.z;
    r.time = time;
    c.state += 1u;
    return true;
}

// ------------------------------------------------------------------------------------------
// the steps of a bounce, one copy for the three kernels that advance paths (k_wave, k_tail, k_wave_bvh): they must
// give every path the same bits whichever of them runs its bounce (DESIGN.md section 13)
// ------------------------------------------------------------------------------------------
// Scene tables into shared memory (call with the whole CTA; visible after the next barrier): the flat scan's primitive
// list (FLAT), the light list, and the Perlin tables when the host made room for them (perlin_in_smem: render_waves).
// Returns where the Perlin tables are read from.
template <bool FLAT, bool RICH>
RT1W_DEV const DPerlin *stage_scene(const SceneView &sc, int perlin_in_smem, unsigned char *s_dyn, FlatScene *s_flat, DLight *s_lights) {
    if (FLAT) flat_stage(sc, s_flat[0]);
    const DPerlin *perlins = sc.perlins;
    if (RICH && perlin_in_smem) {
        const uint32_t words = uint32_t(sc.n_perlins) * uint32_t(sizeof(DPerlin) / 4);
        const uint32_t *src = reinterpret_cast<const uint32_t *>(sc.perlins);
        uint32_t *dst = reinterpret_cast<uint32_t *>(s_dyn);
        for (uint32_t w = threadIdx.x; w < words; w += blockDim.x) dst[w] = src[w];
        perlins = reinterpret_cast<const DPerlin *>(s_dyn);
    }
    for (int l = threadIdx.x; l < sc.n_lights; l += blockDim.x) s_lights[l] = sc.lights[l];
    return perlins;
}

// The thread index space of a wave: [lambertian hits | metal | dielectric | isotropic | new paths], each hit segment
// padded to whole warps; the new paths start at path gen_t0 * tile_paths + gen_w0 (generate_ray).
struct WaveLayout {
    uint32_t off1, off2, off3, off4, cnt0, cnt1, cnt2, cnt3, total, gen_t0, gen_w0;
};

// The layout of the wave that reads counter slot `slot`.  NEW = false (k_tail): the queued hits only.  NEW: then as
// many new paths as the pool has room for; thread 0 of CTA 0 hands the counters over to the next wave (nobody else
// writes those slots during this wave), and gen_t0 / gen_w0 are set in thread 0 only, the one that publishes the layout.
template <bool NEW> RT1W_DEV WaveLayout wave_layout(const RenderArgs &a, int slot) {
    Counters *ctr = a.pool.ctr;
    WaveLayout l;
    l.cnt0 = ctr->n_mat[slot][scatter_mat(0)], l.cnt1 = ctr->n_mat[slot][scatter_mat(1)];
    l.cnt2 = ctr->n_mat[slot][scatter_mat(2)], l.cnt3 = ctr->n_mat[slot][scatter_mat(3)];
    l.off1 = (l.cnt0 + 31u) & ~31u, l.off2 = l.off1 + ((l.cnt1 + 31u) & ~31u), l.off3 = l.off2 + ((l.cnt2 + 31u) & ~31u);
    l.off4 = l.off3 + ((l.cnt3 + 31u) & ~31u);
    l.total = l.off4, l.gen_t0 = 0u, l.gen_w0 = 0u;
    if (NEW) {
        const int nxt = slot == 2 ? 0 : slot + 1, clr = nxt == 2 ? 0 : nxt + 1;
        const uint32_t queued = l.cnt0 + l.cnt1 + l.cnt2 + l.cnt3;
        const unsigned long long path0 = ctr->next_path[slot];
        const unsigned long long left = a.rp.total_paths - min(a.rp.total_paths, path0);
        const uint32_t n_new = uint32_t(min((unsigned long long)(a.pool.capacity - min(a.pool.capacity, queued)), left));
        l.total = l.off4 + n_new;
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            ctr->next_path[nxt] = path0 + n_new;
#pragma unroll
            for (int q = 0; q < Q_COUNT; ++q) ctr->n_mat[clr][q] = 0;
        }
        if (threadIdx.x == 0) l.gen_t0 = uint32_t(path0 / a.rp.tile_paths), l.gen_w0 = uint32_t(path0 - (unsigned long long)l.gen_t0 * a.rp.tile_paths);
    }
    return l;
}

// Work item i < lay.off4 of a wave: the hit it was queued with, its material family (warp-uniform), ray, path state and
// throughput.  False for the padding past a segment's count.  `lay`: a WaveLayout, or a volatile one in shared memory.
template <class L>
RT1W_DEV bool load_queued(const RenderArgs &a, int parity, const L &lay, uint32_t i, int &mat, Ray &r, RayC &c, HitRec &hr, f3 &thr) {
    const uint32_t off1 = lay.off1, off2 = lay.off2, off3 = lay.off3;
    const int seg = i < off1 ? 0 : (i < off2 ? 1 : (i < off3 ? 2 : 3));
    const uint32_t j = i - (seg == 0 ? 0u : (seg == 1 ? off1 : (seg == 2 ? off2 : off3)));
    if (j >= (seg == 0 ? lay.cnt0 : (seg == 1 ? lay.cnt1 : (seg == 2 ? lay.cnt2 : lay.cnt3)))) return false;
    mat = scatter_mat(seg);
    const RayQueue &in = a.pool.mat[parity][mat];
    const double2 o = stream_load(in.a + j);
    const RayB b = stream_load(in.b + j);
    c = stream_load(in.c + j);
    r.ox = o.x, r.oy = o.y, r.oz = b.oz;
    r.dx = b.dx, r.dy = b.dy, r.dz = c.dz;
    r.time = c.time;
    hr = stream_load(in.h + j);
    const float4 th4 = stream_load(in.t + j);
    thr = mk3(th4.x, th4.y, th4.z);
    return true;
}

// The Philox key and counter of the free-flight draws of ConstantMedium candidates (constant_medium.rs:85), the only
// draws inside a traversal; zero without MEDIA.
template <bool MEDIA, int NUM> RT1W_DEV MediumRng medium_rng(const DRenderParams &rp, const DBatch *batch, const RayC &c) {
    MediumRng mr = {0, 0, 0, 0, 0};
    if (MEDIA) {
        path_rng_key<NUM>(rp, batch, c.pixel, mr.k0, mr.k1);
        mr.c0 = uint32_t(rp.sample_begin) + (c.state >> 8), mr.c1 = c.state & 255u, mr.c2 = purpose_word<NUM>(rp, batch, c.pixel, RNG_MEDIUM);
    }
    return mr;
}

// Closest hit of `r`: the flat scan over the staged list (tn_col: this thread's column of entry distances; skip_leaf: the
// primitive the ray starts on; PLAN: the scan's plan or -1, see closest_hit_flat), the 8-wide tree (WIDE) or the binary one
// (stack: this thread's column); `stride`: the CTA size.
template <bool FLAT, bool MEDIA, bool WIDE, int PLAN = -1>
RT1W_DEV bool closest_hit_of(const SceneView &sc, const FlatScene &fs, const Ray &r, const MediumRng &mr, float *tn_col, uint2 *stack, int stride,
                             int skip_leaf, double &t, int &leaf) {
    return FLAT   ? closest_hit_flat<false, MEDIA, PLAN>(sc, fs, r, mr, tn_col, stride, skip_leaf, t, leaf)
           : WIDE ? closest_hit_wide<false, MEDIA>(sc, r, mr, stack, stride, t, leaf)
                  : closest_hit<false, MEDIA>(sc, r, mr, stack, stride, t, leaf);
}

// The material of the closest hit (h.meta is filled in), RT1W_MAT_NONE on a miss.  `prims`: the flat scan's staged list
// (FLAT) or the scene's.  DiffuseLight and NONE end the path (main.rs:110-115); the others queue it for their scatter.
template <bool FLAT> RT1W_DEV int hit_material(const SceneView &sc, const DPrim *prims, bool hit, HitRec &h) {
    if (!hit) return RT1W_MAT_NONE;
    h.meta = FLAT ? prims[h.leaf & kLeafMask].meta : __ldg(&sc.prims[h.leaf & kLeafMask].meta);
    return int((h.meta >> 8) & 15u);
}

// The radiance a path ends on: a light's emission, on its front face only (material.rs:168-181); the background when its
// last extend missed (main.rs:113-115); zero at a hit of `impl Material for ()` (material.rs:68) or on the depth limit.
// FAST_SIN: the sine of the kernel's build of the shading code (see sin_reduced).  SIDE_ONLY: a solid-colour rectangle light
// outside any wrapper needs only the side the ray comes from, not the hit record (the wave kernel's shorter code; k_tail
// keeps the full record).  PLAN: as scatter's.
template <bool RICH, bool FAST_SIN, bool SIDE_ONLY, int PLAN = -1>
RT1W_DEV f3 end_radiance(const RenderArgs &a, const DPrim *prims, const DFrame *frames, const DPerlin *perlins, const Ray &r, const HitRec &h, bool miss,
                         int mat_type) {
    f3 rad = mk3(0.0f, 0.0f, 0.0f);
    if (mat_type == RT1W_MAT_DIFFUSE_LIGHT) {
        const DPrim *P = prims + (h.leaf & kLeafMask);
        bool front;
        if (SIDE_ONLY && !RICH && plain_rect_front_face(P, r, front)) {
            if (front) rad = texture_value<false>(a.sc, perlins, a.sc.materials[h.meta >> 12].texture, HitInfo());
        } else {
            const HitInfo hi = finalize_hit<false, PLAN>(P, frames, h.leaf >> kLeafBits, r, h.t);
            if (hi.front_face) rad = texture_value<RICH, FAST_SIN>(a.sc, perlins, a.sc.materials[h.meta >> 12].texture, hi);
        }
    } else if (miss) {
        rad = mk3(a.rp.background[0], a.rp.background[1], a.rp.background[2]);
    }
    return rad;
}

// A path ends: its pixel gets throughput * radiance.  Zero radiance still has to deliver a NaN / inf throughput (splat).
// mat_type, h: what ended it (RT1W_MAT_NONE on the depth limit), for the light groups (NUM_GROUP) alone.
template <int NUM> RT1W_DEV void end_path(const RenderArgs &a, const DBatch *batch, uint32_t pixel, f3 thr, f3 rad, int mat_type, const HitRec &h) {
    if (rad.x != 0.0f || rad.y != 0.0f || rad.z != 0.0f || !finite3(thr)) splat<NUM>(a, batch, pixel, thr, rad, mat_type, h);
}

// Ray + path state + hit go to entry e of `out`, the queue of the material the ray landed on.
RT1W_DEV void append_queued(const RayQueue &out, uint32_t e, const Ray &r, RayC c, f3 thr, const HitRec &h) {
    stream_store(out.a + e, make_double2(r.ox, r.oy));
    RayB b;
    b.oz = r.oz, b.dx = r.dx, b.dy = r.dy;
    stream_store(out.b + e, b);
    c.dz = r.dz, c.time = r.time;
    stream_store(out.c + e, c);
    stream_store(out.t + e, make_float4(thr.x, thr.y, thr.z, 0.0f));
    stream_store(out.h + e, h);
}

// This thread's closest-hit queries -> the render's ray count (s_traced: zeroed before the CTA's barrier).  Call with the whole CTA.
RT1W_DEV void count_rays(uint32_t traced, unsigned int &s_traced, Counters *ctr) {
    traced = __reduce_add_sync(0xffffffffu, traced);
    if ((threadIdx.x & 31) == 0 && traced) atomicAdd(&s_traced, traced);
    __syncthreads();
    if (threadIdx.x == 0 && s_traced) atomicAdd(&ctr->rays, (unsigned long long)s_traced);
}

// ------------------------------------------------------------------------------------------
// the wave kernel
// ------------------------------------------------------------------------------------------
// FLAT: scan the primitive list staged in shared memory (small scenes) instead of walking the BVH.
// MEDIA: the scene has ConstantMedium primitives (their candidates draw random numbers inside the traversal).
// RICH: some texture is not a SolidColor (else checker / Perlin / image code is compiled out: a third of the kernel).
// WIDE (BVH scenes): walk the compressed 8-wide tree (bvh8.h) instead of the binary one.
// NUM: the path numbering (Numbering) - new camera paths go to the pixels of `list` (NUM_LIST) or to the frames of `batch`
// (NUM_BATCH); NUM_GROUP: `batch` is the light-group table (group_first).
// PLAN (FLAT): the scene's plan (flat_plans.h) compiled into the scan, the wrapper chains and the light list, or -1.
template <bool FLAT, bool MEDIA, bool RICH, bool WIDE, int NUM = NUM_IMAGE, int PLAN = -1>
__global__ void __launch_bounds__(wave_threads(FLAT, MEDIA), wave_min_blocks(FLAT, MEDIA))
    k_wave(const __grid_constant__ RenderArgs a, const int slot, const int parity, const int perlin_in_smem, const uint32_t *list, const DBatch *batch) {
    extern __shared__ __align__(16) unsigned char s_dyn[]; // Perlin tables (perlin.rs:7-12), when the scene has any
    // one static buffer: the staged primitive list + entry-distance table (FLAT) or the per-thread traversal stacks (BVH)
    constexpr int kThreads = wave_threads(FLAT, MEDIA);
    constexpr size_t kFlatBytes = sizeof(FlatScene) + sizeof(float) * kFlatMax * kThreads;
    __shared__ __align__(16) unsigned char s_raw[FLAT ? kFlatBytes : sizeof(uint2) * kStackSmem * kWaveThreads];
    __shared__ DLight s_lights[RT1W_MAX_LIGHTS];
    __shared__ unsigned int s_traced;
    __shared__ WaveLayout s_layout; // read back from shared memory inside the loop instead of pinning a dozen registers
    uint2 *s_stack = reinterpret_cast<uint2 *>(s_raw);
    FlatScene *s_flat = reinterpret_cast<FlatScene *>(s_raw);
    float *s_tn = reinterpret_cast<float *>(s_raw + sizeof(FlatScene)); // entry distances, [primitive][thread]

    // Scene tables into shared memory first: they do not depend on the previous wave, so with programmatic dependent
    // launch (render_waves) this part runs while the previous wave drains.
    const DPerlin *perlins = stage_scene<FLAT, RICH>(a.sc, perlin_in_smem, s_dyn, s_flat, s_lights);
    grid_dependency_wait(); // the previous wave's queues and counters are complete and visible from here on

    Counters *ctr = a.pool.ctr;
    const int nxt = slot == 2 ? 0 : slot + 1;
    const WaveLayout l = wave_layout<true>(a, slot);
    if (blockIdx.x * blockDim.x >= l.total) return;
    if (threadIdx.x == 0) s_traced = 0, s_layout = l;
    __syncthreads();

    const DPrim *prims = FLAT ? s_flat[0].prims : a.sc.prims;
    const DFrame *frames = FLAT ? s_flat[0].frames : a.sc.frames;
    const volatile WaveLayout &lay = s_layout;
    uint32_t traced = 0;
    for (uint32_t i0 = blockIdx.x * blockDim.x; i0 < lay.total; i0 += gridDim.x * blockDim.x) {
        const uint32_t i = i0 + threadIdx.x;
        Ray r;
        RayC c;
        f3 thr;
        bool alive = false, ends = false; // ends: the path is over and its pixel gets throughput * rad
        int skip_leaf = -1;               // the primitive the ray starts on
        const uint32_t off4 = lay.off4;
        if (i < off4) { // a hit queued by the previous wave: scatter
            int mat;
            HitRec hr;
            if (load_queued(a, parity, lay, i, mat, r, c, hr, thr)) {
                skip_leaf = hr.leaf;
                alive = scatter<MEDIA, RICH, true, NUM, PLAN>(mat, a, prims, frames, perlins, s_lights, r, hr, c, thr, batch);
                ends = !alive; // depth limit: zero radiance
            }
        } else if (i < lay.total) { // a new camera path
            r = generate_ray<NUM>(a, list, batch, lay.gen_t0, lay.gen_w0, i - off4, c.state, c.pixel);
            thr = mk3(1.0f, 1.0f, 1.0f);
            alive = true;
        }

        int dest = -1;
        HitRec h;
        int mat_type = RT1W_MAT_NONE;
        bool hit = false;
        if (alive) { // extend: closest hit, then end the path or hand it to the material it landed on
            ++traced;
            hit = closest_hit_of<FLAT, MEDIA, WIDE, PLAN>(a.sc, s_flat[0], r, medium_rng<MEDIA, NUM>(a.rp, batch, c), s_tn + threadIdx.x,
                                                          s_stack + threadIdx.x, kThreads, skip_leaf, h.t, h.leaf);
            mat_type = hit_material<FLAT>(a.sc, prims, hit, h);
            if (mat_type == RT1W_MAT_DIFFUSE_LIGHT || mat_type == RT1W_MAT_NONE) ends = true;
            else dest = mat_type;
        }
        __syncwarp();
        // the queue entries are reserved while the paths that end here reach their pixels (the atomic's round trip is hidden)
        const QueueReservation res = warp_sort_begin(ctr->n_mat[nxt], dest);
        if (ends) end_path<NUM>(a, batch, c.pixel, thr, end_radiance<RICH, true, true, PLAN>(a, prims, frames, perlins, r, h, alive && !hit, mat_type), mat_type, h);
        __syncwarp();
        const uint32_t e = warp_sort_end(res, dest);
        if (dest >= 0) append_queued(a.pool.mat[parity ^ 1][dest], e, r, c, thr, h);
    }
    count_rays(traced, s_traced, ctr);
}

// ------------------------------------------------------------------------------------------
// the end of a render: the last paths run to completion, one thread each
// ------------------------------------------------------------------------------------------
// Depth 50 and no Russian roulette (main.rs:59-61): after the last path has started, the rays in flight shrink by a
// fifth per bounce, and the last ~45 of a Cornell render's ~72 waves hold less than one ray per resident thread - each of
// them still costs the latency of one trip through scatter + closest hit (~10 us), a barrier per bounce.  Once the
// queues hold few enough hits (max_items: about a ray per resident thread), this kernel - launched after every chunk of
// waves, a no-op until then - takes every queued hit and follows its path bounce after bounce inside ONE thread until it
// ends: no barrier between bounces, the warp diverges over materials and depths instead.  Same scatter, same closest hit,
// same Philox counters as the waves: the image does not depend on when (or whether) it takes over.
// The last CTA to finish zeroes the queue counters it consumed, so the waves launched after it find nothing to do.
// WIDE / FAST_SIN: the scenes of the persistent kernel (k_wave_bvh below) end the same way, on the tree and with the sine
// that kernel uses, so that the image does not depend on when the tail takes over.
// NUM: the waves' path numbering (NUM_IMAGE also serves NUM_LIST: the pixel words are the same), and NUM_GROUP's table in `batch`.
// PLAN: the waves' plan (k_wave), so that the tail takes their paths over bit for bit.
template <bool FLAT, bool MEDIA, bool RICH, bool WIDE = false, bool FAST_SIN = true, int NUM = NUM_IMAGE, int PLAN = -1>
__global__ void __launch_bounds__(wave_threads(FLAT, MEDIA), wave_min_blocks(FLAT, MEDIA))
    k_tail(const __grid_constant__ RenderArgs a, const int slot, const int parity, const int perlin_in_smem, const uint32_t max_items, const DBatch *batch) {
    extern __shared__ __align__(16) unsigned char s_dyn[];
    constexpr int kThreads = wave_threads(FLAT, MEDIA);
    constexpr size_t kFlatBytes = sizeof(FlatScene) + sizeof(float) * kFlatMax * kThreads;
    __shared__ __align__(16) unsigned char s_raw[FLAT ? kFlatBytes : sizeof(uint2) * kStackSmem * kWaveThreads];
    __shared__ DLight s_lights[RT1W_MAX_LIGHTS];
    __shared__ unsigned int s_traced;
    uint2 *s_stack = reinterpret_cast<uint2 *>(s_raw);
    FlatScene *s_flat = reinterpret_cast<FlatScene *>(s_raw);
    float *s_tn = reinterpret_cast<float *>(s_raw + sizeof(FlatScene));

    Counters *ctr = a.pool.ctr;
    const WaveLayout l = wave_layout<false>(a, slot);
    const uint32_t queued = l.cnt0 + l.cnt1 + l.cnt2 + l.cnt3;
    if (queued == 0u || queued > max_items || ctr->next_path[slot] < a.rp.total_paths) return; // not yet (or nothing left): every CTA decides alike

    const DPerlin *perlins = stage_scene<FLAT, RICH>(a.sc, perlin_in_smem, s_dyn, s_flat, s_lights);
    if (threadIdx.x == 0) s_traced = 0;
    __syncthreads();
    const DPrim *prims = FLAT ? s_flat[0].prims : a.sc.prims;
    const DFrame *frames = FLAT ? s_flat[0].frames : a.sc.frames;

    uint32_t traced = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < l.off4; i += gridDim.x * blockDim.x) {
        int mat;
        Ray r;
        RayC c;
        HitRec hr;
        f3 thr;
        if (!load_queued(a, parity, l, i, mat, r, c, hr, thr)) continue;
        for (;;) { // one bounce per trip: scatter at the hit, closest hit of the scattered ray
            if (!scatter<MEDIA, RICH, FAST_SIN, NUM, PLAN>(mat, a, prims, frames, perlins, s_lights, r, hr, c, thr, batch)) { // depth limit: zero radiance
                end_path<NUM>(a, batch, c.pixel, thr, mk3(0.0f, 0.0f, 0.0f), RT1W_MAT_NONE, hr);
                break;
            }
            ++traced;
            HitRec h;
            const bool hit = closest_hit_of<FLAT, MEDIA, WIDE, PLAN>(a.sc, s_flat[0], r, medium_rng<MEDIA, NUM>(a.rp, batch, c), s_tn + threadIdx.x,
                                                                     s_stack + threadIdx.x, kThreads, hr.leaf, h.t, h.leaf);
            const int mat_type = hit_material<FLAT>(a.sc, prims, hit, h);
            if (mat_type == RT1W_MAT_DIFFUSE_LIGHT || mat_type == RT1W_MAT_NONE) {
                end_path<NUM>(a, batch, c.pixel, thr, end_radiance<RICH, FAST_SIN, false, PLAN>(a, prims, frames, perlins, r, h, !hit, mat_type), mat_type, h);
                break;
            }
            hr = h, mat = mat_type;
        }
    }
    count_rays(traced, s_traced, ctr);
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&ctr->tail_ticket, 1u) == gridDim.x - 1u) { // the last CTA: every CTA has read the counters it is about to close
#pragma unroll
            for (int q = 0; q < Q_COUNT; ++q) ctr->n_mat[slot][q] = 0;
        }
    }
}

// ------------------------------------------------------------------------------------------
// the wave kernel of BVH scenes: persistent warps, rays replaced lane by lane
// ------------------------------------------------------------------------------------------
// BVH traversal lengths vary wildly from ray to ray (a 1 M-sphere scene: 5 of 32 lanes busy when a warp
// runs 32 rays to the end together), while scattering wants a whole warp on one material.  So a warp
// alternates between two jobs:
//   produce   takes the next 32-item block of its CTA's share of the wave (one material, or new camera
//             paths), scatters / generates with all 32 lanes, and parks the surviving rays + path state in
//             the warp's private ring buffer in shared memory;
//   traverse  bounded while-while rounds (interior steps until the next leaf, then the f64 primitive
//             tests); a lane whose ray is done hands the path over (queue of the material it landed on,
//             or the pixel) and takes the next ray out of the ring at once.
// The traversals in flight simply wait in registers while the warp produces.
#ifndef RT1W_INNER_STEPS
#define RT1W_INNER_STEPS 32 // at most this many interior steps per round
#endif
#ifndef RT1W_LEAF_LANES
#define RT1W_LEAF_LANES 24 // a round's interior steps stop once this many lanes wait at a leaf
#endif
// the 8-wide tree: a third of the steps per ray, each four times the work - rays end (and lanes idle) after fewer steps, so
// the rounds are shorter (measured on the 1 M-sphere scene: 32 steps 547 Mrays/s, 8 steps 794, 4 steps 694), and a lane takes
// two steps per vote (4 votes of 2 steps: 910 against 888 Mrays/s for 8 votes of 1)
#ifndef RT1W_INNER_STEPS_WIDE
#define RT1W_INNER_STEPS_WIDE 4
#endif
#ifndef RT1W_LEAF_LANES_WIDE
#define RT1W_LEAF_LANES_WIDE 24
#endif
constexpr int kPersistentFromNodes = 32768;
constexpr int kRing = 64; // rays per warp ring; a block is produced whenever 32 entries are free

struct __align__(16) RingRay { // 64 bytes: a ray and the state of its path, between scatter and traversal
    double ox, oy, oz;
    float dx, dy, dz, time;
    float tr, tg, tb;
    uint32_t state, pixel;
    uint32_t pad;
};
static_assert(sizeof(RingRay) == 64, "RingRay must be 4 x 16 bytes");

template <bool WIDE> struct TravOf {
    using type = Trav;
};
template <> struct TravOf<true> {
    using type = TravW;
};

template <bool MEDIA, bool WIDE, int NUM = NUM_IMAGE> // NUM: as k_wave's
__global__ void __launch_bounds__(kWaveThreads, RT1W_PERSISTENT_MIN_BLOCKS)
    k_wave_bvh(const __grid_constant__ RenderArgs a, const int slot, const int parity, const int perlin_in_smem, const uint32_t *list, const DBatch *batch) {
    extern __shared__ __align__(16) unsigned char s_dyn[]; // Perlin tables (perlin.rs:7-12), when the scene has any
    __shared__ uint2 s_stack[(WIDE ? kWideStack : kStackSmem) * kWaveThreads];
    __shared__ RingRay s_ring[(kWaveThreads / 32) * kRing];
    __shared__ DLight s_lights[RT1W_MAX_LIGHTS];
    __shared__ unsigned int s_traced, s_next;
    __shared__ WaveLayout s_layout;

    // scene tables first (independent of the previous wave: overlaps its tail under programmatic dependent launch)
    const DPerlin *perlins = stage_scene<false, true>(a.sc, perlin_in_smem, s_dyn, nullptr, s_lights);
    grid_dependency_wait(); // the previous wave's queues and counters are complete and visible from here on

    Counters *ctr = a.pool.ctr;
    const int nxt = slot == 2 ? 0 : slot + 1;
    const WaveLayout l = wave_layout<true>(a, slot);
    if (threadIdx.x == 0) s_traced = 0, s_next = 0, s_layout = l;
    // this CTA's share of the wave: the 32-item blocks blockIdx.x, blockIdx.x + gridDim.x, ...
    const uint32_t n_blocks = (l.total + 31u) >> 5;
    const uint32_t my_blocks = blockIdx.x < n_blocks ? (n_blocks - blockIdx.x + gridDim.x - 1u) / gridDim.x : 0u;
    if (my_blocks == 0u) return;

    __syncthreads();

    const volatile WaveLayout &lay = s_layout;
    const int lane = threadIdx.x & 31;
    uint2 *stack = s_stack + threadIdx.x;
    RingRay *ring = s_ring + (threadIdx.x >> 5) * kRing;
    uint2 overflow[WIDE ? 1 : kStackLocal]; // (the wide tree's stack is shared memory only)
    uint32_t traced = 0;
    uint32_t ring_rd = 0, ring_cnt = 0; // warp-uniform
    bool more = true;                   // warp-uniform: the CTA's share still has blocks
    bool has_ray = false;
    Ray r;
    RayC c;
    f3 thr;
    typename TravOf<WIDE>::type T;
    trav_reset(T);
    trav_bind_stack(T, stack);
    for (;;) {
        // ---- produce: one 32-item block -> scatter / generate with the whole warp -> surviving rays into the ring
        if (more && ring_cnt <= uint32_t(kRing - 32)) {
            uint32_t qb = 0;
            if (lane == 0) qb = atomicAdd(&s_next, 1u);
            qb = __shfl_sync(0xffffffffu, qb, 0);
            more = qb + 1u < my_blocks;
            if (qb < my_blocks) {
                const uint32_t i = ((qb * gridDim.x + blockIdx.x) << 5) + uint32_t(lane);
                Ray nr;
                RayC nc;
                f3 nthr;
                bool alive = false;
                const uint32_t off4 = lay.off4;
                if (i < off4) { // a hit queued by the previous wave: scatter (one material per block)
                    int mat;
                    HitRec hr;
                    if (load_queued(a, parity, lay, i, mat, nr, nc, hr, nthr)) {
                        alive = scatter<MEDIA, true, false, NUM>(mat, a, a.sc.prims, a.sc.frames, perlins, s_lights, nr, hr, nc, nthr, batch); // (sinf: see sin_reduced)
                        if (!alive) end_path<NUM>(a, batch, nc.pixel, nthr, mk3(0.0f, 0.0f, 0.0f), RT1W_MAT_NONE, hr); // depth limit: zero radiance
                    }
                } else if (i < lay.total) { // a new camera path
                    nr = generate_ray<NUM>(a, list, batch, lay.gen_t0, lay.gen_w0, i - off4, nc.state, nc.pixel);
                    nthr = mk3(1.0f, 1.0f, 1.0f);
                    alive = true;
                }
                const unsigned alive_mask = __ballot_sync(0xffffffffu, alive);
                if (alive) {
                    RingRay e;
                    e.ox = nr.ox, e.oy = nr.oy, e.oz = nr.oz, e.dx = nr.dx, e.dy = nr.dy, e.dz = nr.dz, e.time = nr.time;
                    e.tr = nthr.x, e.tg = nthr.y, e.tb = nthr.z, e.state = nc.state, e.pixel = nc.pixel, e.pad = 0;
                    ring[(ring_rd + ring_cnt + __popc(alive_mask & ((1u << lane) - 1u))) & (kRing - 1)] = e;
                }
                ring_cnt += __popc(alive_mask);
                __syncwarp();
            }
        }
        // ---- idle lanes take rays out of the ring
        const unsigned idle = __ballot_sync(0xffffffffu, !has_ray);
        if (idle != 0u && ring_cnt != 0u) {
            const uint32_t rank = __popc(idle & ((1u << lane) - 1u));
            if (!has_ray && rank < ring_cnt) {
                const RingRay e = ring[(ring_rd + rank) & (kRing - 1)];
                r.ox = e.ox, r.oy = e.oy, r.oz = e.oz, r.dx = e.dx, r.dy = e.dy, r.dz = e.dz, r.time = e.time;
                thr = mk3(e.tr, e.tg, e.tb);
                c.state = e.state, c.pixel = e.pixel;
                ++traced;
                trav_begin(a.sc, r, T);
                has_ray = true;
            }
            const uint32_t taken = min(uint32_t(__popc(idle)), ring_cnt);
            ring_rd = (ring_rd + taken) & (kRing - 1), ring_cnt -= taken;
            __syncwarp();
        } else if (idle == 0xffffffffu && !more) {
            break; // nothing in flight, nothing parked, nothing left to produce
        }
        // ---- one while-while round: interior steps until enough lanes wait at a leaf (or finished), then the leaves
        constexpr int kInnerSteps = WIDE ? RT1W_INNER_STEPS_WIDE : RT1W_INNER_STEPS, kLeafLanes = WIDE ? RT1W_LEAF_LANES_WIDE : RT1W_LEAF_LANES;
        for (int step = 0; step < kInnerSteps; ++step) {
            const bool interior = has_ray && trav_interior(T);
            const unsigned walking = __ballot_sync(0xffffffffu, interior);
            const unsigned at_leaf = __ballot_sync(0xffffffffu, has_ray && trav_at_leaf(T));
            if (walking == 0u || __popc(at_leaf) >= kLeafLanes) break; // every round steps or solves: it always makes progress
            if (interior) trav_step_interior(a.sc, T, stack, kWaveThreads, overflow);
            if (WIDE && interior && trav_interior(T)) trav_step_interior(a.sc, T, stack, kWaveThreads, overflow); // a second step on the same vote
        }
        if (has_ray && trav_at_leaf(T)) trav_step_leaf<false, MEDIA>(a.sc, r, medium_rng<MEDIA, NUM>(a.rp, batch, c), T, stack, kWaveThreads, overflow);
        // ---- rays that reached the end: finish the path or hand it to the material it landed on
        const bool fin = has_ray && trav_done(T);
        if (__any_sync(0xffffffffu, fin)) {
            int dest = -1;
            HitRec h;
            if (fin) {
                has_ray = false;
                if (a.sc.n_global > 0) hit_globals<false, MEDIA>(a.sc, r, medium_rng<MEDIA, NUM>(a.rp, batch, c), T.best, T.best_leaf); // the primitives that are in no tree
                const bool hit = T.best_leaf >= 0;
                h.t = T.best, h.leaf = T.best_leaf;
                const int mat_type = hit_material<false>(a.sc, a.sc.prims, hit, h);
                if (mat_type == RT1W_MAT_DIFFUSE_LIGHT || mat_type == RT1W_MAT_NONE)
                    end_path<NUM>(a, batch, c.pixel, thr, end_radiance<true, false, false>(a, a.sc.prims, a.sc.frames, perlins, r, h, !hit, mat_type), mat_type, h);
                else dest = mat_type;
            }
            __syncwarp();
            const uint32_t e = warp_sort_end(warp_sort_begin(ctr->n_mat[nxt], dest), dest);
            if (dest >= 0) append_queued(a.pool.mat[parity ^ 1][dest], e, r, c, thr, h);
        }
    }
    count_rays(traced, s_traced, ctr);
}

// ------------------------------------------------------------------------------------------
// closest-hit parity kernel
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kExtendThreads) k_trace(const __grid_constant__ SceneView sc, const rt1w_ray *__restrict__ rays, const size_t n,
                                                          const uint32_t seed_lo, const uint32_t seed_hi, int32_t *prim_id, float *t_out,
                                                          float *normal3, uint8_t *front_face, float *uv2, int32_t *leaf_out, double *t64_out) {
    __shared__ uint2 s_stack[kStackSmem * kExtendThreads];
    __shared__ FlatScene s_flat;
    float *s_tn = reinterpret_cast<float *>(s_stack); // the flat scan's entry-distance table shares the stack space
    static_assert(sizeof(float) * kFlatMax <= sizeof(uint2) * kStackSmem, "entry-distance table must fit the stack buffer");
    const bool flat = sc.flat != 0; // same choice as the render path, so parity covers both traversals
    if (flat) {
        flat_stage(sc, s_flat);
        __syncthreads();
    }
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) {
        const rt1w_ray in = rays[i];
        Ray r;
        r.ox = in.origin[0], r.oy = in.origin[1], r.oz = in.origin[2];
        r.dx = in.direction[0], r.dy = in.direction[1], r.dz = in.direction[2];
        r.time = in.time;
        MediumRng mr;
        mr.c0 = uint32_t(i), mr.c1 = uint32_t(uint64_t(i) >> 32), mr.c2 = RNG_TRACE_MEDIUM, mr.k0 = seed_lo, mr.k1 = seed_hi;
        double t;
        int leaf;
        const bool hit = flat      ? closest_hit_flat<true, true>(sc, s_flat, r, mr, s_tn + threadIdx.x, kExtendThreads, -1, t, leaf)
                         : sc.wide ? closest_hit_wide<true, true>(sc, r, mr, s_stack + threadIdx.x, kExtendThreads, t, leaf)
                                   : closest_hit<true, true>(sc, r, mr, s_stack + threadIdx.x, kExtendThreads, t, leaf);
        HitInfo h;
        if (hit) h = finalize_hit<true>(sc.prims + (leaf & kLeafMask), sc.frames, leaf >> kLeafBits, r, t);
        if (prim_id) prim_id[i] = hit ? sc.prim_id[leaf & kLeafMask] + (leaf >> kLeafBits) : -1; // a box: its first rectangle + the side
        if (t_out) t_out[i] = hit ? float(t) : CUDART_INF_F;
        if (normal3) {
            normal3[3 * i] = hit ? h.normal.x : 0.0f, normal3[3 * i + 1] = hit ? h.normal.y : 0.0f, normal3[3 * i + 2] = hit ? h.normal.z : 0.0f;
        }
        if (front_face) front_face[i] = hit ? uint8_t(h.front_face) : uint8_t(0);
        if (uv2) uv2[2 * i] = hit ? h.u : 0.0f, uv2[2 * i + 1] = hit ? h.v : 0.0f;
        if (leaf_out) leaf_out[i] = hit ? leaf : -1; // (the shading hooks below continue from here)
        if (t64_out) t64_out[i] = hit ? t : CUDART_INF;
    }
}

// ------------------------------------------------------------------------------------------
// pointwise parity hooks for the shading functions (rt1w.h: rt1w_eval_*): the device functions the wave kernels
// call, one thread per input, so that tests can hold them against the reference's formulas value by value
// ------------------------------------------------------------------------------------------
// `[T]: Hittable::pdf_value` over the light list (hittable.rs:144-150) or one light's own (aarect.rs:119-138, sphere.rs:72-90)
__global__ void __launch_bounds__(256) k_eval_light_pdf(const __grid_constant__ SceneView sc, const int light, const double *__restrict__ o3,
                                                        const float *__restrict__ v3, const size_t n, float *__restrict__ out) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) {
        const f3 v = mk3(v3[3 * i], v3[3 * i + 1], v3[3 * i + 2]);
        float pdf = 0.0f;
        if (light >= 0) {
            pdf = light_pdf_value(sc.lights[light], o3[3 * i], o3[3 * i + 1], o3[3 * i + 2], v);
        } else {
            const float wl = 1.0f / float(sc.n_lights);
            for (int l = 0; l < sc.n_lights; ++l) pdf += wl * light_pdf_value(sc.lights[l], o3[3 * i], o3[3 * i + 1], o3[3 * i + 2], v);
        }
        out[i] = pdf;
    }
}

// Texture::value(u, v, p) (texture.rs:40-89) / Perlin::noise, turb (perlin.rs:46-106; depth 0 = noise)
__global__ void __launch_bounds__(256) k_eval_texture(const __grid_constant__ SceneView sc, const int texture, const int perlin_table, const int turb_depth,
                                                      const double *__restrict__ p3, const float *__restrict__ uv2, const size_t n,
                                                      float *__restrict__ out) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) {
        if (texture < 0) {
            const DPerlin *tab = sc.perlins + perlin_table;
            out[i] = turb_depth > 0 ? perlin_turb(tab, p3[3 * i], p3[3 * i + 1], p3[3 * i + 2], turb_depth) : perlin_noise(tab, p3[3 * i], p3[3 * i + 1], p3[3 * i + 2]);
            continue;
        }
        HitInfo h;
        h.px = p3[3 * i], h.py = p3[3 * i + 1], h.pz = p3[3 * i + 2];
        h.u = uv2 ? uv2[2 * i] : 0.0f, h.v = uv2 ? uv2[2 * i + 1] : 0.0f;
        h.type = P_XY_RECT, h.prim = nullptr, h.frames = nullptr, h.side = 0; // prim == nullptr: (u, v) are given
        h.normal = h.n_out = mk3(0.0f, 0.0f, 1.0f), h.front_face = true, h.meta = 0u;
        const f3 c = texture_value<true>(sc, sc.perlins, texture, h);
        out[3 * i] = c.x, out[3 * i + 1] = c.y, out[3 * i + 2] = c.z;
    }
}

// reflect, refract, reflectance (material.rs:94-96,114-125) on unit directions
__global__ void __launch_bounds__(256) k_eval_dielectric(const float *__restrict__ uv3, const float *__restrict__ n3, const float *__restrict__ ratio,
                                                         const size_t n, float *__restrict__ reflect3, float *__restrict__ refract3,
                                                         float *__restrict__ reflectance_out) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) {
        const f3 uv = mk3(uv3[3 * i], uv3[3 * i + 1], uv3[3 * i + 2]), nn = mk3(n3[3 * i], n3[3 * i + 1], n3[3 * i + 2]);
        const f3 a = reflect(uv, nn), b = refract(uv, nn, ratio[i]);
        reflect3[3 * i] = a.x, reflect3[3 * i + 1] = a.y, reflect3[3 * i + 2] = a.z;
        refract3[3 * i] = b.x, refract3[3 * i + 1] = b.y, refract3[3 * i + 2] = b.z;
        reflectance_out[i] = reflectance(fminf(dot(-uv, nn), 1.0f), ratio[i]);
    }
}

// Material::scatter at the closest hit of ray i (found by k_trace: leaf, t) - the same `scatter` the wave kernels run, for
// path (pixel seed i, sample i & 0xffff, bounce 0).  A hit that ends the path reports what it emits instead.
__global__ void __launch_bounds__(kExtendThreads) k_eval_scatter(const __grid_constant__ RenderArgs a, const rt1w_ray *__restrict__ rays,
                                                                 const int32_t *__restrict__ leaf_in, const double *__restrict__ t_in, const size_t n,
                                                                 int32_t *__restrict__ material_out, float *__restrict__ dir3,
                                                                 float *__restrict__ weight3, float *__restrict__ time_out) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) {
        const rt1w_ray in = rays[i];
        Ray r;
        r.ox = in.origin[0], r.oy = in.origin[1], r.oz = in.origin[2];
        r.dx = in.direction[0], r.dy = in.direction[1], r.dz = in.direction[2];
        r.time = in.time;
        const int leaf = leaf_in[i];
        int mat_type = -1;
        f3 w = mk3(0.0f, 0.0f, 0.0f), d = mk3(0.0f, 0.0f, 0.0f);
        if (leaf >= 0) {
            HitRec hr;
            hr.t = t_in[i], hr.leaf = leaf, hr.meta = a.sc.prims[leaf & kLeafMask].meta;
            mat_type = int((hr.meta >> 8) & 15u);
            if (mat_type == RT1W_MAT_LAMBERTIAN || mat_type == RT1W_MAT_METAL || mat_type == RT1W_MAT_DIELECTRIC || mat_type == RT1W_MAT_ISOTROPIC) {
                RayC c;
                c.dz = r.dz, c.time = r.time, c.state = (uint32_t(i) & 0xffffu) << 8, c.pixel = uint32_t(i);
                w = mk3(1.0f, 1.0f, 1.0f);
                scatter<true, true>(mat_type, a, a.sc.prims, a.sc.frames, a.sc.perlins, a.sc.lights, r, hr, c, w, nullptr);
                d = mk3(r.dx, r.dy, r.dz);
            } else if (mat_type == RT1W_MAT_DIFFUSE_LIGHT) { // material.rs:168-181
                const HitInfo hi = finalize_hit<false>(a.sc.prims + (leaf & kLeafMask), a.sc.frames, leaf >> kLeafBits, r, hr.t);
                if (hi.front_face) w = texture_value<true>(a.sc, a.sc.perlins, a.sc.materials[hr.meta >> 12].texture, hi);
            }
        }
        material_out[i] = mat_type;
        dir3[3 * i] = d.x, dir3[3 * i + 1] = d.y, dir3[3 * i + 2] = d.z;
        weight3[3 * i] = w.x, weight3[3 * i + 1] = w.y, weight3[3 * i + 2] = w.z;
        time_out[i] = r.time;
    }
}

// ------------------------------------------------------------------------------------------
// first-hit feature buffers (rt1w.h: rt1w_render_aov)
// ------------------------------------------------------------------------------------------
// The render's first ray of path (pixel seed, global sample index) - the camera-ray parity hook (rt1w_eval_camera_rays);
// a.rp.sample_begin = 0
__global__ void __launch_bounds__(256) k_eval_camera_rays(const __grid_constant__ RenderArgs a, const uint32_t *__restrict__ pixel_seed,
                                                          const int32_t *__restrict__ sample, const size_t n, rt1w_ray *__restrict__ out) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) {
        const Ray r = camera_ray(a.cam, a.rp, pixel_seed[i], a.rp.seed_lo, purpose_word(a.rp, RNG_CAMERA), uint32_t(sample[i]));
        rt1w_ray o;
        o.origin[0] = float(r.ox), o.origin[1] = float(r.oy), o.origin[2] = float(r.oz);
        o.direction[0] = r.dx, o.direction[1] = r.dy, o.direction[2] = r.dz;
        o.time = r.time;
        out[i] = o;
    }
}

constexpr int kAovThreads = 128;
RT1W_DEV f3 clamp01(f3 c) { return mk3(fminf(fmaxf(c.x, 0.0f), 1.0f), fminf(fmaxf(c.y, 0.0f), 1.0f), fminf(fmaxf(c.z, 0.0f), 1.0f)); }

// Per pixel, the sums over the render's sample range of what the first segment of every path sees (rt1w.h: albedo, normal,
// distance, hit).  Work mapping: 2^group_log2 consecutive lanes share one pixel, lane g of the group takes the samples g,
// g + G, ... in order, then a fixed __shfl_xor tree adds the group's sums - a warp covers 32 / G neighbouring pixels of one
// row, whose camera rays are coherent, and no float atomics: the sums do not depend on scheduling.  The host widens the
// groups until small images at high sample counts fill the GPU (aov_launch).  The same closest hit, with the same template
// arguments and the same medium draws, as the depth-0 extend of the wave kernels; the flat scan stages its tables in
// shared memory as k_trace does.  out: [albedo 3P | normal 3P | distance P | hits P] for P = width * height, row 0 = top.
template <bool FLAT, bool MEDIA, bool RICH, bool WIDE>
__global__ void __launch_bounds__(kAovThreads) k_aov(const __grid_constant__ RenderArgs a, const int group_log2, float *__restrict__ out) {
    __shared__ __align__(16) uint2 s_stack[kStackSmem * kAovThreads]; // traversal stacks, or the flat scan's entry distances
    __shared__ __align__(16) unsigned char s_raw[FLAT ? sizeof(FlatScene) : 16];
    FlatScene *s_flat = reinterpret_cast<FlatScene *>(s_raw);
    float *s_tn = reinterpret_cast<float *>(s_stack);
    static_assert(sizeof(float) * kFlatMax <= sizeof(uint2) * kStackSmem, "entry-distance table must fit the stack buffer");
    if (FLAT) {
        flat_stage(a.sc, s_flat[0]);
        __syncthreads();
    }
    const DPrim *prims = FLAT ? s_flat[0].prims : a.sc.prims;
    const DFrame *frames = FLAT ? s_flat[0].frames : a.sc.frames;
    const uint32_t n_pixels = uint32_t(a.rp.width) * uint32_t(a.rp.height), group = 1u << group_log2;
    const uint32_t total = n_pixels << group_log2;
    const uint32_t camera_word = purpose_word(a.rp, RNG_CAMERA), medium_word = purpose_word(a.rp, RNG_MEDIUM);
    // whole CTAs run the loop (the shuffles below need every lane of a warp)
    for (uint32_t k0 = blockIdx.x * kAovThreads; k0 < total; k0 += gridDim.x * kAovThreads) {
        const uint32_t k = k0 + threadIdx.x, pix = k >> group_log2, lane_in_group = k & (group - 1u);
        float acc[8] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f}; // albedo, normal, distance, hits
        for (uint32_t s = lane_in_group; k < total && s < uint32_t(a.rp.n_samples); s += group) {
            const uint32_t sample = uint32_t(a.rp.sample_begin) + s;
            const Ray r = camera_ray(a.cam, a.rp, pix, a.rp.seed_lo, camera_word, s);
            MediumRng mr = {0, 0, 0, 0, 0};
            if (MEDIA) mr.c0 = sample, mr.c1 = 0u, mr.c2 = medium_word, mr.k0 = pix, mr.k1 = a.rp.seed_lo; // the wave kernels' draw at bounce 0
            double t;
            int leaf;
            const bool hit = closest_hit_of<FLAT, MEDIA, WIDE>(a.sc, s_flat[0], r, mr, s_tn + threadIdx.x, s_stack + threadIdx.x, kAovThreads, -1, t, leaf);
            f3 albedo = clamp01(mk3(a.rp.background[0], a.rp.background[1], a.rp.background[2])), normal = mk3(0.0f, 0.0f, 0.0f);
            float dist = 0.0f;
            if (hit) {
                const HitInfo h = finalize_hit<false>(prims + (leaf & kLeafMask), frames, leaf >> kLeafBits, r, t);
                const DMaterial m = a.sc.materials[h.meta >> 12];
                const int mat = int((h.meta >> 8) & 15u);
                if (mat == RT1W_MAT_LAMBERTIAN || mat == RT1W_MAT_ISOTROPIC) albedo = texture_value<RICH>(a.sc, a.sc.perlins, m.texture, h); // scatter's attenuation
                else if (mat == RT1W_MAT_METAL) albedo = mk3(m.albedo[0], m.albedo[1], m.albedo[2]);
                else if (mat == RT1W_MAT_DIELECTRIC) albedo = mk3(1.0f, 1.0f, 1.0f);
                else if (mat == RT1W_MAT_DIFFUSE_LIGHT && h.front_face) albedo = clamp01(texture_value<RICH>(a.sc, a.sc.perlins, m.texture, h));
                else albedo = mk3(0.0f, 0.0f, 0.0f);
                if (h.type != P_MEDIUM_SPHERE && h.type != P_MEDIUM_BOX) normal = h.normal; // a medium's record carries no surface normal
                const double dx = r.dx, dy = r.dy, dz = r.dz;
                dist = float(__dmul_rn(t, __dsqrt_rn(__fma_rn(dz, dz, __fma_rn(dy, dy, __dmul_rn(dx, dx))))));
            }
            acc[0] += albedo.x, acc[1] += albedo.y, acc[2] += albedo.z;
            acc[3] += normal.x, acc[4] += normal.y, acc[5] += normal.z;
            acc[6] += dist, acc[7] += hit ? 1.0f : 0.0f;
        }
        for (uint32_t o = group >> 1; o > 0u; o >>= 1)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[c] += __shfl_xor_sync(0xffffffffu, acc[c], int(o));
        if (k < total && lane_in_group == 0u) {
            const uint32_t j = div_by(pix, a.rp.inv_width_up), q = (uint32_t(a.rp.height) - 1u - j) * uint32_t(a.rp.width) + (pix - j * uint32_t(a.rp.width));
#pragma unroll
            for (int c = 0; c < 3; ++c) out[3 * size_t(q) + c] = acc[c], out[3 * size_t(n_pixels) + 3 * size_t(q) + c] = acc[3 + c];
            out[6 * size_t(n_pixels) + q] = acc[6], out[7 * size_t(n_pixels) + q] = acc[7];
        }
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static cudaError_t queue_alloc(RayQueue &q, uint32_t capacity) {
    cudaError_t e;
    if ((e = cudaMalloc(&q.a, sizeof(double2) * size_t(capacity))) != cudaSuccess) return e;
    if ((e = cudaMalloc(&q.b, sizeof(RayB) * size_t(capacity))) != cudaSuccess) return e;
    if ((e = cudaMalloc(&q.c, sizeof(RayC) * size_t(capacity))) != cudaSuccess) return e;
    if ((e = cudaMalloc(&q.t, sizeof(float4) * size_t(capacity))) != cudaSuccess) return e;
    if ((e = cudaMalloc(&q.h, sizeof(HitRec) * size_t(capacity))) != cudaSuccess) return e;
    return cudaSuccess;
}

static void queue_free(RayQueue &q) {
    cudaFree(q.a), cudaFree(q.b), cudaFree(q.c), cudaFree(q.t), cudaFree(q.h);
    q = RayQueue();
}

// material_mask: only the hit queues of the scattering material families the scene uses are allocated.
cudaError_t pool_alloc(Pool &pool, uint32_t capacity, int material_mask) {
    pool_free(pool);
    cudaError_t e = cudaSuccess;
    for (int k = 0; k < 2; ++k)
        for (int q = 0; q < Q_COUNT && e == cudaSuccess; ++q)
            if ((material_mask & (1 << q)) && q != RT1W_MAT_DIFFUSE_LIGHT) e = queue_alloc(pool.mat[k][q], capacity);
    if (e == cudaSuccess) e = cudaMalloc(&pool.ctr, sizeof(Counters));
    if (e != cudaSuccess) {
        pool_free(pool);
        return e;
    }
    pool.capacity = pool.allocated = capacity;
    pool.material_mask = material_mask;
    return cudaSuccess;
}

void pool_free(Pool &pool) {
    for (int k = 0; k < 2; ++k)
        for (int q = 0; q < Q_COUNT; ++q) queue_free(pool.mat[k][q]);
    cudaFree(pool.ctr);
    pool = Pool();
}

// grid: every CTA resident at once (SM count x occupancy); the kernel grid-strides over a device-side count
using WaveKernel = void (*)(const RenderArgs, const int, const int, const int, const uint32_t *, const DBatch *);
// The kernels of the plans (flat_plans.h): image renders of solid-colour flat scenes without media.
template <int... P> static WaveKernel planned_wave(int plan, std::integer_sequence<int, P...>) {
    const WaveKernel k[] = {k_wave<true, false, false, false, NUM_IMAGE, P>...};
    return k[plan];
}
template <int NUM> static WaveKernel wave_kernel(bool flat, bool persistent, bool wide, bool media, bool rich, int plan = -1) {
    if (flat && plan >= 0 && !media && !rich && NUM == NUM_IMAGE) return planned_wave(plan, std::make_integer_sequence<int, kNumFlatPlans>());
    if (flat)
        return media ? (rich ? k_wave<true, true, true, false, NUM> : k_wave<true, true, false, false, NUM>)
                     : (rich ? k_wave<true, false, true, false, NUM> : k_wave<true, false, false, false, NUM>);
    if (persistent)
        return wide ? (media ? k_wave_bvh<true, true, NUM> : k_wave_bvh<false, true, NUM>) : (media ? k_wave_bvh<true, false, NUM> : k_wave_bvh<false, false, NUM>);
    return wide ? (media ? (rich ? k_wave<false, true, true, true, NUM> : k_wave<false, true, false, true, NUM>)
                         : (rich ? k_wave<false, false, true, true, NUM> : k_wave<false, false, false, true, NUM>))
                : (media ? (rich ? k_wave<false, true, true, false, NUM> : k_wave<false, true, false, false, NUM>)
                         : (rich ? k_wave<false, false, true, false, NUM> : k_wave<false, false, false, false, NUM>));
}

// the kernel that runs the last paths to completion (k_tail), or none: WIDE scenes only end that way on the persistent kernel
using TailKernel = void (*)(const RenderArgs, const int, const int, const int, const uint32_t, const DBatch *);
template <int... P> static TailKernel planned_tail(int plan, std::integer_sequence<int, P...>) {
    const TailKernel k[] = {k_tail<true, false, false, false, true, NUM_IMAGE, P>...};
    return k[plan];
}
template <int NUM> static TailKernel tail_kernel_of(bool flat, bool persistent, bool wide, bool media, bool rich, int plan = -1) {
    if (flat && plan >= 0 && !media && !rich && NUM == NUM_IMAGE) return planned_tail(plan, std::make_integer_sequence<int, kNumFlatPlans>());
    if (!flat && persistent) // the persistent kernel's build of the shading code: every texture kind, sinf
        return wide ? (media ? k_tail<false, true, true, true, false, NUM> : k_tail<false, false, true, true, false, NUM>)
                    : (media ? k_tail<false, true, true, false, false, NUM> : k_tail<false, false, true, false, false, NUM>);
    if (wide) return nullptr;
    return flat ? (media ? (rich ? k_tail<true, true, true, false, true, NUM> : k_tail<true, true, false, false, true, NUM>)
                         : (rich ? k_tail<true, false, true, false, true, NUM> : k_tail<true, false, false, false, true, NUM>))
                : (media ? (rich ? k_tail<false, true, true, false, true, NUM> : k_tail<false, true, false, false, true, NUM>)
                         : (rich ? k_tail<false, false, true, false, true, NUM> : k_tail<false, false, false, false, true, NUM>));
}

// The Perlin tables ride on top of a wave kernel's static shared memory: beyond 48 KB in total the kernel has to opt in.
// False (the error cleared) when `kernel` cannot take `bytes` more.
template <class K> static bool perlin_opt_in(K kernel, size_t bytes) {
    cudaFuncAttributes fa;
    int optin = 0, dev = 0;
    if (cudaFuncGetAttributes(&fa, kernel) != cudaSuccess || cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    const size_t need = fa.sharedSizeBytes + bytes;
    if (need > size_t(optin)) return false;
    if (need > 48 * 1024 && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes)) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return true;
}

// BVH scenes: the 8-wide tree (the scene's default by size) unless a flag picks a tree
static bool walk_wide(const SceneView &sc, uint32_t flags) {
    if ((flags & RT1W_FLAG_BVH_BINARY) || sc.wide_nodes == nullptr) return false;
    return (flags & RT1W_FLAG_BVH_WIDE) || sc.wide != 0;
}

cudaError_t render_waves(const RenderArgs &args, const uint32_t *list, const DBatch *batch, const int32_t *groups, int material_mask, Counters *h_ctr,
                         cudaStream_t stream, int sm_count, WaveStats &ws) {
    cudaError_t e = cudaMemsetAsync(args.pool.ctr, 0, sizeof(Counters), stream);
    if (e != cudaSuccess) return e;
    const bool flat = args.sc.flat != 0;
    const bool media = (material_mask & (1 << RT1W_MAT_ISOTROPIC)) != 0;
    size_t perlin_bytes = size_t(args.sc.n_perlins) * sizeof(DPerlin);
    int perlin_in_smem = perlin_bytes > 0 && perlin_bytes <= 40 * 1024;
    const int poll_every = 8;
    // BVH scenes: traversals of a big tree vary too much in length to run a warp's rays in lockstep (1 M spheres:
    // 5 of 32 lanes busy); small trees are walked faster by the leaner lockstep kernel (measured crossover)
    bool persistent = args.sc.n_nodes > kPersistentFromNodes;
    if (args.rp.flags & RT1W_FLAG_BVH_LOCKSTEP) persistent = false;
    if (args.rp.flags & RT1W_FLAG_BVH_PERSISTENT) persistent = true;
    const bool rich = args.sc.rich_textures != 0;
    const bool wide = walk_wide(args.sc, args.rp.flags);
    // the planned scan (flat_plans.h) for image renders; the waves and the tail of a render scan alike
    const int plan = flat && !batch && !list && !groups ? args.sc.flat_plan : -1;
    const WaveKernel kernel = batch    ? wave_kernel<NUM_BATCH>(flat, persistent, wide, media, rich)
                              : list   ? wave_kernel<NUM_LIST>(flat, persistent, wide, media, rich)
                              : groups ? wave_kernel<NUM_GROUP>(flat, persistent, wide, media, rich)
                                       : wave_kernel<NUM_IMAGE>(flat, persistent, wide, media, rich, plan);
    if (groups) batch = reinterpret_cast<const DBatch *>(groups); // the trailing table argument of NUM_GROUP's kernels
    if (flat) cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared); // scene + scan tables live in shared memory
    // A scene with more Perlin tables than fit reads them from global memory instead (perlin.rs:7-12 keeps them on the heap).
    if (!perlin_in_smem || !perlin_opt_in(kernel, perlin_bytes)) perlin_in_smem = 0, perlin_bytes = 0;
    // the kernel that runs the last paths to completion (k_tail); RT1W_FLAG_NO_TAIL keeps waves to the end (A/B, tests)
    TailKernel tail_kernel = nullptr;
    if (!(args.rp.flags & RT1W_FLAG_NO_TAIL))
        tail_kernel = groups  ? tail_kernel_of<NUM_GROUP>(flat, persistent, wide, media, rich)
                      : batch ? tail_kernel_of<NUM_BATCH>(flat, persistent, wide, media, rich)
                              : tail_kernel_of<NUM_IMAGE>(flat, persistent, wide, media, rich, plan);
    if (tail_kernel && perlin_bytes > 0 && !perlin_opt_in(tail_kernel, perlin_bytes)) tail_kernel = nullptr; // it reads the tables where the waves do
    if (tail_kernel && flat) cudaFuncSetAttribute(tail_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    const int threads = wave_threads(flat, media);
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, perlin_bytes)) != cudaSuccess) return e;
    const int blocks = sm_count * (per_sm > 0 ? per_sm : 1);
    uint32_t tail_items = uint32_t(blocks) * uint32_t(threads); // one queued hit per resident thread
    if (const char *env = std::getenv("RT1W_TAIL_FACTOR")) // (A/B: take over earlier / later; a thread then follows several paths, one after the other)
        tail_items = uint32_t(std::min(double(args.pool.capacity), std::max(1.0, std::atof(env) * double(tail_items))));
    // every wave may start (scene tables -> shared memory) while the wave before it drains: programmatic dependent launch
    cudaLaunchAttribute launch_attr[1];
    launch_attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    launch_attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t launch = {};
    launch.gridDim = dim3(unsigned(blocks)), launch.blockDim = dim3(unsigned(threads)), launch.dynamicSmemBytes = perlin_bytes, launch.stream = stream;
    launch.attrs = launch_attr, launch.numAttrs = 1;

    // profiling mode: one event before every launch and one at the end of the chunk
    struct Mark {
        cudaEvent_t ev;
        int slot;
    };
    std::vector<Mark> marks;
    std::vector<cudaEvent_t> spare;
    auto mark = [&](int slot) {
        if (!ws.profile) return;
        cudaEvent_t ev;
        if (!spare.empty()) ev = spare.back(), spare.pop_back();
        else cudaEventCreate(&ev);
        cudaEventRecord(ev, stream);
        marks.push_back(Mark{ev, slot});
    };
    auto drain_marks = [&]() {
        for (size_t i = 0; i + 1 < marks.size(); ++i) {
            if (marks[i].slot < 0) continue;
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, marks[i].ev, marks[i + 1].ev);
            ws.kernel_ms[marks[i].slot] += ms, ws.kernel_launches[marks[i].slot] += 1;
        }
        for (auto &m : marks) spare.push_back(m.ev);
        marks.clear();
    };

    // Termination poll, one chunk behind: the counters after chunk c are copied to a pinned snapshot while chunk
    // c + 1 is already queued, so the GPU never idles waiting for the host.  The price is one chunk of empty waves
    // (a few microseconds each) after the last useful one.
    auto finished = [&](const Counters &c, uint64_t next_wave) { // what wave `next_wave` would see: no path left to start, no hit queued
        const int slot = int(next_wave % 3);
        uint32_t queued = 0;
        for (int q = 0; q < Q_COUNT; ++q) queued += c.n_mat[slot][q];
        return c.next_path[slot] >= args.rp.total_paths && queued == 0;
    };
    cudaEvent_t snap_ev[2] = {nullptr, nullptr};
    for (int k = 0; k < 2 && e == cudaSuccess; ++k) e = cudaEventCreateWithFlags(&snap_ev[k], cudaEventDisableTiming);
    uint64_t wave = 0, chunk = 0;
    const Counters *last = h_ctr;
    while (e == cudaSuccess) {
        for (int k = 0; k < poll_every; ++k, ++wave) {
            const int slot = int(wave % 3), parity = int(wave & 1);
            mark(K_WAVE);
            if ((e = cudaLaunchKernelEx(&launch, kernel, args, slot, parity, perlin_in_smem, list, batch)) != cudaSuccess) break;
            ++ws.launches;
        }
        if (tail_kernel && e == cudaSuccess) { // a no-op until few enough hits are queued, then the rest of the render (k_tail)
            cudaLaunchConfig_t cfg = launch;
            cfg.attrs = nullptr, cfg.numAttrs = 0;
            mark(K_WAVE);
            if ((e = cudaLaunchKernelEx(&cfg, tail_kernel, args, int(wave % 3), int(wave & 1), perlin_in_smem, tail_items, batch)) != cudaSuccess) break;
            ++ws.launches;
        }
        mark(-1);
        Counters *snap = h_ctr + (chunk & 1);
        if ((e = cudaGetLastError()) != cudaSuccess) break;
        if ((e = cudaMemcpyAsync(snap, args.pool.ctr, sizeof(Counters), cudaMemcpyDeviceToHost, stream)) != cudaSuccess) break;
        if ((e = cudaEventRecord(snap_ev[chunk & 1], stream)) != cudaSuccess) break;
        if (ws.profile) { // per-launch event times are read chunk by chunk
            if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) break;
            drain_marks();
            last = snap;
            if (finished(*snap, wave)) break;
        } else if (chunk >= 1) {
            const Counters *prev = h_ctr + ((chunk - 1) & 1);
            if ((e = cudaEventSynchronize(snap_ev[(chunk - 1) & 1])) != cudaSuccess) break;
            if (finished(*prev, wave - poll_every)) {
                e = cudaStreamSynchronize(stream); // the chunk queued meanwhile ran on empty queues
                last = snap;
                break;
            }
        }
        ++chunk;
    }
    for (int k = 0; k < 2; ++k)
        if (snap_ev[k]) cudaEventDestroy(snap_ev[k]);
    for (auto &m : marks) cudaEventDestroy(m.ev);
    for (auto ev : spare) cudaEventDestroy(ev);
    if (e != cudaSuccess) return e;
    ws.waves = wave;
    ws.rays = last->rays;
#ifdef RT1W_COUNT_SOLVES
    if (flat) {
        unsigned long long d[4] = {0, 0, 0, 0}, zero[4] = {0, 0, 0, 0};
        cudaMemcpyFromSymbol(d, g_scan_counts, sizeof(d));
        cudaMemcpyToSymbol(g_scan_counts, zero, sizeof(zero));
        std::fprintf(stderr, "[flat scan] rays %llu, candidates per ray %.3f, f64 solves per ray %.3f, solve iterations per warp of 32 rays %.3f\n", d[0],
                     double(d[1]) / double(d[0]), double(d[2]) / double(d[0]), 32.0 * double(d[3]) / double(d[0]));
    }
#endif
#ifdef RT1W_COUNT_TRAV
    if (!flat) {
        unsigned long long d[4] = {0, 0, 0, 0}, zero[4] = {0, 0, 0, 0};
        cudaMemcpyFromSymbol(d, g_trav_counts, sizeof(d));
        cudaMemcpyToSymbol(g_trav_counts, zero, sizeof(zero));
        std::fprintf(stderr, "[bvh] rays %llu, interior steps per ray %.2f, primitive tests per ray %.3f, lanes per warp-level interior step %.2f\n", d[0],
                     double(d[1]) / double(d[0]), double(d[2]) / double(d[0]), double(d[1]) / double(d[3] ? d[3] : 1));
    }
#endif
    return cudaSuccess;
}

// `Color::into_sampled` + `Display for SampledColor` (color.rs:14-21,56-65) on the device: NaN sum -> 0, mean, sqrt,
// clamp to [0, 0.999], * 256, truncate; same f64 arithmetic as the host rt1w_resolve_rgb8 (bit-identical output).
RT1W_DEV uint8_t resolve_value(float sum, double scale) {
    double x = double(sum);
    if (x != x) x = 0.0;
    x *= scale;
    double g = sqrt(x);
    g = g < 0.0 ? 0.0 : (g > 0.999 ? 0.999 : g);
    const double q = 256.0 * g;
    return q != q ? uint8_t(0) : uint8_t(int(q));
}

__global__ void __launch_bounds__(256) k_resolve(const float *__restrict__ rgb_sum, const size_t n, const double scale, uint8_t *__restrict__ out) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) out[i] = resolve_value(rgb_sum[i], scale);
}

// the same with each pixel's own sample count (adaptive renders): scale 1 / spp[pixel], as the host computes it
__global__ void __launch_bounds__(256) k_resolve_counts(const float *__restrict__ rgb_sum, const int32_t *__restrict__ spp, const size_t n,
                                                        uint8_t *__restrict__ out) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x)
        out[i] = resolve_value(rgb_sum[i], 1.0 / double(spp[i / 3]));
}

cudaError_t resolve_launch(const float *d_rgb_sum, size_t n_values, int samples_per_pixel, uint8_t *d_rgb8, cudaStream_t stream) {
    if (n_values == 0) return cudaSuccess;
    const size_t want = (n_values + 255) / 256;
    k_resolve<<<int(want < 148 * 8 ? want : 148 * 8), 256, 0, stream>>>(d_rgb_sum, n_values, 1.0 / double(samples_per_pixel), d_rgb8);
    return cudaGetLastError();
}

cudaError_t resolve_counts_launch(const float *d_rgb_sum, const int32_t *d_spp, size_t n_values, uint8_t *d_rgb8, cudaStream_t stream) {
    if (n_values == 0) return cudaSuccess;
    const size_t want = (n_values + 255) / 256;
    k_resolve_counts<<<int(want < 148 * 8 ? want : 148 * 8), 256, 0, stream>>>(d_rgb_sum, d_spp, n_values, d_rgb8);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// adaptive sampling (rt1w.h: rt1w_render_adaptive): after every round, the convergence rule over the pixels still active
// and their ordered compaction into the next round's list - per-CTA counts, one scan of them, a scatter.  Once per round,
// not on the hot path; the list keeps ascending seed order and no result depends on the order of atomics.
// ------------------------------------------------------------------------------------------
constexpr int kConvergeThreads = 256;

// The rule of rt1w.h after n samples, per channel in f64 from the fp32 sums: the half-width of the +-1 standard-error
// interval of the mean (clamped statistics), through the gamma 2 and x 256 of color.rs:56-65, is at most max_error 8-bit
// levels - or the channel's radiance sum is NaN (it resolves to 0 whatever follows, color.rs:16-18).  m * m unfused: the
// same value the rule gives in numpy.
RT1W_DEV bool pixel_converged(const float *sum3, const float *stat6, int n, double max_error) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        if (sum3[c] != sum3[c]) continue;
        const double m = double(stat6[c]) / n;
        const double v = fmax(double(stat6[3 + c]) / n - __dmul_rn(m, m), 0.0) * n / (n - 1);
        const double se = sqrt(v / n);
        const double hi = fmin(fmax(m + se, 0.0), 1.0), lo = fmin(fmax(m - se, 0.0), 1.0);
        if (!(128.0 * (sqrt(hi) - sqrt(lo)) <= max_error)) return false;
    }
    return true;
}

// warp counts of `flag` into s_warp, then this thread's rank among the flagged threads of the CTA before it
RT1W_DEV uint32_t cta_rank(bool flag, uint32_t *s_warp, uint32_t &cta_total) {
    const unsigned m = __ballot_sync(0xffffffffu, flag);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = uint32_t(__popc(m));
    __syncthreads();
    uint32_t before = 0, total = 0;
    for (int w = 0; w < kConvergeThreads / 32; ++w) {
        if (w < int(threadIdx.x >> 5)) before += s_warp[w];
        total += s_warp[w];
    }
    cta_total = total;
    return before + uint32_t(__popc(m & ((1u << (threadIdx.x & 31)) - 1u)));
}

// One thread per active pixel: list slot k (list == nullptr: every pixel, seed k).  A pixel that stops gets its count n;
// keep[k] = 1 for one that goes on; counts[b] = how many of CTA b's go on.  max_error = 0 turns the rule off.
__global__ void __launch_bounds__(kConvergeThreads) k_converge(const float *__restrict__ accum, const float *__restrict__ stat, const uint32_t *__restrict__ list,
                                                               const uint32_t n_active, const int width, const int height, const int n, const int max_spp,
                                                               const double max_error, int32_t *__restrict__ spp, uint8_t *__restrict__ keep,
                                                               uint32_t *__restrict__ counts) {
    __shared__ uint32_t s_warp[kConvergeThreads / 32];
    const uint32_t k = blockIdx.x * kConvergeThreads + threadIdx.x;
    bool go_on = false;
    if (k < n_active) {
        const uint32_t seed = list ? list[k] : k, j = seed / uint32_t(width);
        const uint32_t pixel = (uint32_t(height) - 1u - j) * uint32_t(width) + (seed - j * uint32_t(width)); // row 0 = top (splat)
        go_on = n < max_spp && !(max_error > 0.0 && pixel_converged(accum + 3 * size_t(pixel), stat + 6 * size_t(pixel), n, max_error));
        if (!go_on) spp[pixel] = n;
        keep[k] = go_on ? 1 : 0;
    }
    uint32_t total;
    cta_rank(go_on, s_warp, total);
    if (threadIdx.x == 0) counts[blockIdx.x] = total;
}

// Exclusive scan of the per-CTA counts in place (one CTA); counts[n] = the sum: the next round's pixel count.
__global__ void __launch_bounds__(1024) k_scan_counts(uint32_t *counts, const uint32_t n) {
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t i = base + threadIdx.x, x = i < n ? counts[i] : 0u;
        uint32_t v = x; // inclusive scan inside the warp, then over the warps' totals
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += y;
        }
        if (lane == 31) s_warp[warp] = v;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        const uint32_t inclusive = s_carry + (warp > 0 ? s_warp[warp - 1] : 0u) + v;
        if (i < n) counts[i] = inclusive - x;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = inclusive;
        __syncthreads();
    }
    if (threadIdx.x == 0) counts[n] = s_carry;
}

// The pixels that go on, in list order, to next[offsets[b] + rank inside CTA b].
__global__ void __launch_bounds__(kConvergeThreads) k_compact(const uint32_t *__restrict__ list, const uint8_t *__restrict__ keep, const uint32_t n_active,
                                                              const uint32_t *__restrict__ offsets, uint32_t *__restrict__ next) {
    __shared__ uint32_t s_warp[kConvergeThreads / 32];
    const uint32_t k = blockIdx.x * kConvergeThreads + threadIdx.x;
    const bool go_on = k < n_active && keep[k] != 0;
    uint32_t total;
    const uint32_t rank = cta_rank(go_on, s_warp, total);
    if (go_on) next[offsets[blockIdx.x] + rank] = list ? list[k] : k;
}

uint32_t converge_blocks(uint32_t n_active) { return (n_active + kConvergeThreads - 1) / kConvergeThreads; }

cudaError_t converge_launch(const float *d_accum, const float *d_stat, const uint32_t *d_list, uint32_t n_active, int width, int height, int n, int max_spp,
                            double max_error, int32_t *d_spp, uint8_t *d_keep, uint32_t *d_counts, uint32_t *d_next, cudaStream_t stream) {
    const uint32_t blocks = converge_blocks(n_active);
    if (blocks == 0) return cudaMemsetAsync(d_counts, 0, sizeof(uint32_t), stream);
    k_converge<<<blocks, kConvergeThreads, 0, stream>>>(d_accum, d_stat, d_list, n_active, width, height, n, max_spp, max_error, d_spp, d_keep, d_counts);
    k_scan_counts<<<1, 1024, 0, stream>>>(d_counts, blocks);
    k_compact<<<blocks, kConvergeThreads, 0, stream>>>(d_list, d_keep, n_active, d_counts, d_next);
    return cudaGetLastError();
}

cudaError_t trace_closest_launch(const SceneView &sc, const rt1w_ray *rays, size_t n, uint64_t seed, int32_t *prim_id, float *t,
                                 float *normal3, uint8_t *front_face, float *uv2, cudaStream_t stream, int32_t *leaf, double *t64) {
    if (n == 0) return cudaSuccess;
    const size_t want = (n + kExtendThreads - 1) / kExtendThreads;
    const int blocks = int(want < 148 * 16 ? want : 148 * 16);
    k_trace<<<blocks, kExtendThreads, 0, stream>>>(sc, rays, n, uint32_t(seed), uint32_t(seed >> 32), prim_id, t, normal3, front_face, uv2, leaf, t64);
    return cudaGetLastError();
}

static int eval_blocks(size_t n, int threads) {
    const size_t want = (n + threads - 1) / threads;
    return int(want < 148 * 8 ? want : 148 * 8);
}

cudaError_t eval_light_pdf_launch(const SceneView &sc, int light, const double *o3, const float *v3, size_t n, float *pdf, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    k_eval_light_pdf<<<eval_blocks(n, 256), 256, 0, stream>>>(sc, light, o3, v3, n, pdf);
    return cudaGetLastError();
}

cudaError_t eval_texture_launch(const SceneView &sc, int texture, int perlin_table, int turb_depth, const double *p3, const float *uv2, size_t n,
                                float *out, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    k_eval_texture<<<eval_blocks(n, 256), 256, 0, stream>>>(sc, texture, perlin_table, turb_depth, p3, uv2, n, out);
    return cudaGetLastError();
}

cudaError_t eval_dielectric_launch(const float *uv3, const float *n3, const float *ratio, size_t n, float *reflect3, float *refract3,
                                   float *reflectance, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    k_eval_dielectric<<<eval_blocks(n, 256), 256, 0, stream>>>(uv3, n3, ratio, n, reflect3, refract3, reflectance);
    return cudaGetLastError();
}

cudaError_t eval_scatter_launch(const SceneView &sc, const rt1w_ray *rays, const int32_t *leaf, const double *t64, size_t n, uint64_t seed,
                                int32_t *material, float *dir3, float *weight3, float *time_out, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    RenderArgs a = {};
    a.sc = sc;
    a.rp.sample_begin = 0, a.rp.n_samples = 1 << 16, a.rp.max_depth = 50, a.rp.seed_lo = uint32_t(seed), a.rp.seed_hi = uint32_t(seed >> 32);
    k_eval_scatter<<<eval_blocks(n, kExtendThreads), kExtendThreads, 0, stream>>>(a, rays, leaf, t64, n, material, dir3, weight3, time_out);
    return cudaGetLastError();
}

cudaError_t eval_camera_rays_launch(const RenderArgs &args, const uint32_t *pixel_seed, const int32_t *sample, size_t n, rt1w_ray *out, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    k_eval_camera_rays<<<eval_blocks(n, 256), 256, 0, stream>>>(args, pixel_seed, sample, n, out);
    return cudaGetLastError();
}

using AovKernel = void (*)(const RenderArgs, const int, float *);
static AovKernel aov_kernel(bool flat, bool wide, bool media, bool rich) {
    if (flat) return media ? (rich ? k_aov<true, true, true, false> : k_aov<true, true, false, false>) : (rich ? k_aov<true, false, true, false> : k_aov<true, false, false, false>);
    if (wide) return media ? (rich ? k_aov<false, true, true, true> : k_aov<false, true, false, true>) : (rich ? k_aov<false, false, true, true> : k_aov<false, false, false, true>);
    return media ? (rich ? k_aov<false, true, true, false> : k_aov<false, true, false, false>) : (rich ? k_aov<false, false, true, false> : k_aov<false, false, false, false>);
}

cudaError_t aov_launch(const RenderArgs &args, int material_mask, float *d_out, int sm_count, cudaStream_t stream) {
    const bool flat = args.sc.flat != 0, media = (material_mask & (1 << RT1W_MAT_ISOTROPIC)) != 0;
    const AovKernel kernel = aov_kernel(flat, !flat && walk_wide(args.sc, args.rp.flags), media, args.sc.rich_textures != 0);
    cudaError_t e;
    if (flat && (e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)) != cudaSuccess) return e;
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kAovThreads, 0)) != cudaSuccess) return e;
    const uint64_t resident = uint64_t(sm_count) * uint64_t(per_sm > 0 ? per_sm : 1) * kAovThreads;
    // Lanes per pixel: one while the pixels alone give every resident thread four of them (large images, or few samples:
    // 3840x2160 at 1 spp is a pixel per lane), doubled up to a warp per pixel while they do not (256^2 at 1024 spp: 8 lanes
    // of 128 samples each), and never more lanes than samples.
    const uint64_t pixels = uint64_t(args.rp.width) * uint64_t(args.rp.height);
    int group_log2 = 0;
    while (group_log2 < 5 && (1 << group_log2) < args.rp.n_samples && (pixels << group_log2) < 4 * resident) ++group_log2;
    const uint64_t blocks = std::min(resident / kAovThreads, ((pixels << group_log2) + kAovThreads - 1) / kAovThreads);
    kernel<<<unsigned(blocks), kAovThreads, 0, stream>>>(args, group_log2, d_out);
    return cudaGetLastError();
}

} // namespace rt1w
