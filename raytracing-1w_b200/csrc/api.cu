// api.cu — the C ABI of include/rt1w.h: handles, scene commit (lowering + SAH build + upload),
// render entry points, the closest-hit parity hook and the host-side output quantisation.
#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <cstring>
#include <limits>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/rt1w.h"
#include "bvh.h"
#include "bvh8.h"
#include "lbvh.h"
#include "lower.h"
#include "nccl_dl.h"
#include "render.h"

using namespace rt1w;

namespace {

thread_local std::string g_error;

rt1w_status fail(rt1w_status s, const std::string &msg) {
    g_error = msg;
    return s;
}
rt1w_status fail_cuda(const char *what, cudaError_t e) {
    g_error = std::string(what) + ": " + cudaGetErrorString(e);
    return RT1W_ERR_CUDA;
}

#define RT1W_CUDA(call)                                                                                                                               \
    do {                                                                                                                                              \
        cudaError_t e__ = (call);                                                                                                                     \
        if (e__ != cudaSuccess) return fail_cuda(#call, e__);                                                                                         \
    } while (0)

constexpr uint32_t kDefaultPool = 1u << 23; // rays in flight per wave: the queues stream through HBM, so bigger waves amortise launches and the tail
constexpr int kLbvhFromPrims = 1 << 17;      // scenes from this many primitives on get their BVH built on the device
// The traversal's node reference (primitive count << 29 | left_first) folded into the first word of every node once, so that
// a node step reads it instead of combining two words per child (kernels.cuh: node_ref)
__global__ void k_fold_node_refs(uint4 *nodes, size_t n) {
    const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) nodes[2 * i].w |= nodes[2 * i + 1].w << 29;
}
static void fold_node_refs(float4 *nodes, size_t n, cudaStream_t stream) {
    k_fold_node_refs<<<unsigned((n + 255) / 256), 256, 0, stream>>>(reinterpret_cast<uint4 *>(nodes), n);
}
constexpr int kWideFromNodes = 32768;        // BVHs from this many binary nodes on are walked through the compressed 8-wide tree by default
constexpr int kMaxLeaf = 1; // single-primitive leaves: the f32 leaf-box test screens the f64 primitive solve

// Bounds of a lowered primitive in its own frame (the box its wrapper chain rotates and translates).
void local_bounds(const rt1w_flat_prim &fp, double lo[3], double hi[3]) {
    const double *p = fp.p;
    switch (fp.kind) {
    case RT1W_NODE_XY_RECT:
    case RT1W_NODE_XZ_RECT:
    case RT1W_NODE_YZ_RECT: { // in-plane intervals + the reference's +-0.0001 slab (aarect.rs:74-79,112-117,180-185)
        const int ax = fp.kind == RT1W_NODE_XY_RECT ? 2 : (fp.kind == RT1W_NODE_XZ_RECT ? 1 : 0);
        const int a = ax == 0 ? 1 : 0, b = ax == 2 ? 1 : 2;
        lo[a] = p[0], hi[a] = p[1], lo[b] = p[2], hi[b] = p[3], lo[ax] = p[4] - 0.0001, hi[ax] = p[4] + 0.0001;
        break;
    }
    case RT1W_NODE_AABOX: // merged box: p = min xyz, max xyz
        for (int c = 0; c < 3; ++c) lo[c] = p[c], hi[c] = p[3 + c];
        break;
    case RT1W_NODE_CONSTANT_MEDIUM:
        if (fp.boundary != RT1W_NODE_SPHERE) { // p = min xyz, -1/density, max xyz
            for (int c = 0; c < 3; ++c) lo[c] = p[c], hi[c] = p[4 + c];
            break;
        }
        // fall through: p = center, radius, ...
    case RT1W_NODE_SPHERE:
        for (int c = 0; c < 3; ++c) lo[c] = p[c] - p[3], hi[c] = p[c] + p[3];
        break;
    default: // not expected (moving spheres keep their world box)
        for (int c = 0; c < 3; ++c) lo[c] = fp.bbox_min[c], hi[c] = fp.bbox_max[c];
        break;
    }
}

// Face groups of the flat scan.  A rectangle is a face of the box B when its plane is one of B's bounds on its axis and
// its in-plane intervals are exactly B's on the two other axes.  Two rectangles of different axes in one frame fix a
// box; every unassigned rectangle of the frame that is a face of it joins, one per face.  Groups of fewer than three
// faces are not worth the shared slab computation.  `order`: leaf -> index into dev.  Output per leaf: group number
// and face = 2 * axis + (upper plane ? 1 : 0), or -1; per group: the box (min xyz, max xyz).
void find_face_groups(const std::vector<rt1w_flat_prim> &dev, const std::vector<uint32_t> &order, std::vector<int> &face_group,
                      std::vector<int> &face_of, std::vector<std::array<double, 6>> &group_box) {
    const int n = int(order.size());
    auto prim = [&](int leaf) -> const rt1w_flat_prim & { return dev[order[leaf]]; };
    auto axis_of = [&](int leaf) {
        const int kind = prim(leaf).kind;
        return kind == RT1W_NODE_YZ_RECT ? 0 : (kind == RT1W_NODE_XZ_RECT ? 1 : (kind == RT1W_NODE_XY_RECT ? 2 : -1));
    };
    // extents of a rectangle: lo / hi on its two in-plane axes, plane on its own
    auto rect_extents = [&](int leaf, double lo[3], double hi[3]) {
        const int ax = axis_of(leaf), a = ax == 0 ? 1 : 0, b = ax == 2 ? 1 : 2;
        const double *p = prim(leaf).p;
        lo[a] = p[0], hi[a] = p[1], lo[b] = p[2], hi[b] = p[3], lo[ax] = hi[ax] = p[4];
    };
    auto face_in = [&](int leaf, const std::array<double, 6> &box) { // face number of the rectangle in the box, or -1
        const int ax = axis_of(leaf);
        double lo[3], hi[3];
        rect_extents(leaf, lo, hi);
        for (int c = 0; c < 3; ++c)
            if (c != ax && (lo[c] != box[c] || hi[c] != box[3 + c])) return -1;
        if (lo[ax] == box[ax]) return 2 * ax;
        if (lo[ax] == box[3 + ax]) return 2 * ax + 1;
        return -1;
    };
    for (int r1 = 0; r1 < n; ++r1) {
        if (axis_of(r1) < 0 || face_group[r1] >= 0) continue;
        for (int r2 = 0; r2 < n; ++r2) {
            if (r2 == r1 || axis_of(r2) < 0 || axis_of(r2) == axis_of(r1) || face_group[r2] >= 0 || prim(r2).frame != prim(r1).frame) continue;
            std::array<double, 6> box;
            double lo[3], hi[3], lo2[3], hi2[3];
            rect_extents(r1, lo, hi), rect_extents(r2, lo2, hi2);
            const int ax = axis_of(r1);
            for (int c = 0; c < 3; ++c) box[c] = c == ax ? lo2[c] : lo[c], box[3 + c] = c == ax ? hi2[c] : hi[c];
            if (!(box[0] < box[3] && box[1] < box[4] && box[2] < box[5])) continue;
            if (face_in(r1, box) < 0 || face_in(r2, box) < 0) continue;
            int members[6] = {-1, -1, -1, -1, -1, -1}, count = 0;
            for (int r = 0; r < n; ++r) {
                if (axis_of(r) < 0 || face_group[r] >= 0 || prim(r).frame != prim(r1).frame) continue;
                const int f = face_in(r, box);
                if (f >= 0 && members[f] < 0) members[f] = r, ++count;
            }
            if (count < 3) continue;
            for (int f = 0; f < 6; ++f)
                if (members[f] >= 0) face_group[members[f]] = int(group_box.size()), face_of[members[f]] = f;
            group_box.push_back(box);
            break;
        }
    }
}

template <class T> cudaError_t upload(const std::vector<T> &v, T **out) {
    *out = nullptr;
    const size_t bytes = sizeof(T) * (v.empty() ? 1 : v.size());
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(out), bytes);
    if (e != cudaSuccess) return e;
    if (!v.empty()) e = cudaMemcpy(*out, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice);
    return e;
}

struct DeviceArena { // device copies of host arrays for one hook call; freed on scope exit
    std::vector<void *> ptrs;
    cudaError_t err = cudaSuccess;
    template <class T> T *alloc(size_t count) {
        void *p = nullptr;
        if (err == cudaSuccess) err = cudaMalloc(&p, sizeof(T) * (count ? count : 1));
        if (p) ptrs.push_back(p);
        return static_cast<T *>(p);
    }
    template <class T> T *upload(const T *host, size_t count, cudaStream_t stream) {
        T *d = alloc<T>(count);
        if (err == cudaSuccess && host && count) err = cudaMemcpyAsync(d, host, sizeof(T) * count, cudaMemcpyHostToDevice, stream);
        return d;
    }
    template <class T> void download(T *host, const T *dev, size_t count, cudaStream_t stream) {
        if (err == cudaSuccess && host && count) err = cudaMemcpyAsync(host, dev, sizeof(T) * count, cudaMemcpyDeviceToHost, stream);
    }
    ~DeviceArena() {
        for (void *p : ptrs) cudaFree(p);
    }
};

} // namespace

struct rt1w_context {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    Pool pool;
    Counters *h_ctr = nullptr; // pinned
    float *d_accum = nullptr, *d_stat = nullptr;
    uint8_t *d_rgb8 = nullptr;
    size_t accum_pixels = 0, stat_pixels = 0, rgb8_pixels = 0;
    // adaptive renders: per-pixel sample counts, the pixel lists of two consecutive rounds, the compaction's flags and
    // per-CTA counts, and the pinned copy of the next round's pixel count
    int32_t *d_spp = nullptr;
    uint32_t *d_list[2] = {nullptr, nullptr};
    uint8_t *d_keep = nullptr;
    uint32_t *d_counts = nullptr, *h_active = nullptr;
    size_t adaptive_pixels = 0;
    // batch renders: the frame tables of the last call (DBatch header, cameras, seed words), one allocation grown on demand
    unsigned char *d_batch = nullptr;
    size_t batch_bytes = 0;
    // feature buffers (rt1w_render_aov): the packed sums of the last call, 8 floats per pixel
    float *d_aov = nullptr;
    size_t aov_pixels = 0;
    std::mutex lock; // calls on one context are serialised (rt1w.h "Threading")
    // Multi-GPU (SURVEY.md 8e): a context that belongs to a communicator renders ITS share of the sample range of every
    // render call and adds its radiance sums to rank 0's with one ncclReduce on the render stream.
    ncclComm_t comm = nullptr;
    int comm_rank = 0, comm_size = 1;
    std::vector<rt1w_context *> members; // rt1w_context_create_multi: the other devices' contexts (ranks 1..n-1), owned by this one
};

struct rt1w_scene {
    rt1w_context *ctx = nullptr;
    int device = 0; // where the allocations below live (kept here: a scene may be released after its context)
    std::vector<rt1w_flat_prim> prims; // primitive-id order
    std::vector<int32_t> leaf_prim_id; // host copy of d_prim_id (device leaf order)
    rt1w_scene_info info{};
    SceneView view{};
    int material_mask = 0;
    int n_textures = 0;
    // device allocations
    float4 *d_nodes = nullptr;
    uint4 *d_wide_nodes = nullptr;
    DPrim *d_prims = nullptr;
    float4 *d_prim_boxes = nullptr;
    int32_t *d_prim_id = nullptr;
    DFrame *d_frames = nullptr;
    DMaterial *d_materials = nullptr;
    DTexture *d_textures = nullptr;
    DPerlin *d_perlins = nullptr;
    cudaTextureObject_t *d_images = nullptr;
    int2 *d_image_dims = nullptr;
    DLight *d_lights = nullptr;
    std::vector<cudaArray_t> arrays;
    std::vector<cudaTextureObject_t> tex_objects;
    std::vector<rt1w_scene *> replicas; // multi-device context: the same scene committed on ranks 1..n-1
};

static void scene_release(rt1w_scene *s) {
    if (!s) return;
    for (rt1w_scene *r : s->replicas) scene_release(r);
    cudaSetDevice(s->device);
    for (auto t : s->tex_objects) cudaDestroyTextureObject(t);
    for (auto a : s->arrays) cudaFreeArray(a);
    cudaFree(s->d_nodes), cudaFree(s->d_wide_nodes), cudaFree(s->d_prims), cudaFree(s->d_prim_boxes), cudaFree(s->d_prim_id), cudaFree(s->d_frames), cudaFree(s->d_materials);
    cudaFree(s->d_textures), cudaFree(s->d_perlins), cudaFree(s->d_images), cudaFree(s->d_image_dims), cudaFree(s->d_lights);
    delete s;
}

extern "C" {

int32_t rt1w_abi_version(void) { return RT1W_ABI_VERSION; }

const char *rt1w_last_error(void) { return g_error.c_str(); }

static rt1w_status context_create_impl(int32_t device_id, rt1w_context **out) {
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(RT1W_ERR_NO_DEVICE, "no CUDA device (this library has no CPU fallback)");
    }
    if (device_id < 0 || device_id >= count) return fail(RT1W_ERR_INVALID, "device id out of range");
    cudaDeviceProp prop;
    RT1W_CUDA(cudaGetDeviceProperties(&prop, device_id));
    if (prop.major != 10) return fail(RT1W_ERR_NO_DEVICE, "device is not sm_100 (kernels are built for sm_100a only)");
    RT1W_CUDA(cudaSetDevice(device_id));
    auto ctx = std::make_unique<rt1w_context>();
    ctx->device = device_id;
    ctx->sm_count = prop.multiProcessorCount;
    RT1W_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    RT1W_CUDA(cudaEventCreate(&ctx->ev0));
    RT1W_CUDA(cudaEventCreate(&ctx->ev1));
    RT1W_CUDA(cudaMallocHost(reinterpret_cast<void **>(&ctx->h_ctr), 2 * sizeof(Counters))); // two snapshots: the poll runs one chunk behind
    *out = ctx.release();
    return RT1W_OK;
}

rt1w_status rt1w_context_create(int32_t device_id, rt1w_context **out) {
    if (!out) return fail(RT1W_ERR_INVALID, "null output pointer");
    return context_create_impl(device_id, out);
}

static rt1w_status fail_nccl(const char *what, ncclResult_t r) {
    const NcclApi &nccl = nccl_api();
    g_error = std::string(what) + ": " + (nccl.GetErrorString ? nccl.GetErrorString(r) : "NCCL error");
    return RT1W_ERR_CUDA;
}

rt1w_status rt1w_context_create_multi(const int32_t *device_ids, int32_t n, rt1w_context **out) {
    if (!out || !device_ids || n <= 0) return fail(RT1W_ERR_INVALID, "null output pointer or empty device list");
    *out = nullptr;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < i; ++j)
            if (device_ids[i] == device_ids[j]) return fail(RT1W_ERR_INVALID, "a device may appear only once in the device list");
    std::vector<rt1w_context *> all(size_t(n), nullptr);
    auto destroy_all = [&] {
        for (rt1w_context *c : all)
            if (c) c->members.clear(), rt1w_context_destroy(c);
    };
    for (int i = 0; i < n; ++i) {
        rt1w_status st = context_create_impl(device_ids[i], &all[i]);
        if (st != RT1W_OK) {
            destroy_all();
            return st;
        }
    }
    if (n > 1) {
        const NcclApi &nccl = nccl_api();
        if (!nccl.error.empty()) {
            destroy_all();
            return fail(RT1W_ERR_UNSUPPORTED, nccl.error);
        }
        std::vector<ncclComm_t> comms(size_t(n), nullptr);
        std::vector<int> devs(device_ids, device_ids + n);
        ncclResult_t r = nccl.CommInitAll(comms.data(), n, devs.data());
        if (r != ncclSuccess) {
            destroy_all();
            return fail_nccl("ncclCommInitAll", r);
        }
        for (int i = 0; i < n; ++i) all[i]->comm = comms[i], all[i]->comm_rank = i, all[i]->comm_size = n;
    }
    all[0]->members.assign(all.begin() + 1, all.end());
    *out = all[0];
    return RT1W_OK;
}

rt1w_status rt1w_comm_unique_id(uint8_t *out_id, size_t capacity) {
    if (!out_id || capacity < RT1W_COMM_ID_BYTES) return fail(RT1W_ERR_INVALID, "the id buffer must hold RT1W_COMM_ID_BYTES bytes");
    static_assert(RT1W_COMM_ID_BYTES == sizeof(ncclUniqueId), "rt1w.h must reserve an ncclUniqueId");
    const NcclApi &nccl = nccl_api();
    if (!nccl.error.empty()) return fail(RT1W_ERR_UNSUPPORTED, nccl.error);
    ncclUniqueId id;
    ncclResult_t r = nccl.GetUniqueId(&id);
    if (r != ncclSuccess) return fail_nccl("ncclGetUniqueId", r);
    std::memcpy(out_id, &id, sizeof(id));
    return RT1W_OK;
}

rt1w_status rt1w_context_comm_init(rt1w_context *ctx, const uint8_t *id, int32_t n_ranks, int32_t rank) {
    if (!ctx || !id || n_ranks <= 0 || rank < 0 || rank >= n_ranks) return fail(RT1W_ERR_INVALID, "bad communicator arguments");
    std::lock_guard<std::mutex> guard(ctx->lock);
    if (ctx->comm || !ctx->members.empty()) return fail(RT1W_ERR_STATE, "the context already belongs to a communicator");
    if (n_ranks == 1) return RT1W_OK;
    const NcclApi &nccl = nccl_api();
    if (!nccl.error.empty()) return fail(RT1W_ERR_UNSUPPORTED, nccl.error);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    ncclUniqueId uid;
    std::memcpy(&uid, id, sizeof(uid));
    ncclComm_t comm = nullptr;
    ncclResult_t r = nccl.CommInitRank(&comm, n_ranks, uid, rank);
    if (r != ncclSuccess) return fail_nccl("ncclCommInitRank", r);
    ctx->comm = comm, ctx->comm_rank = rank, ctx->comm_size = n_ranks;
    return RT1W_OK;
}

rt1w_status rt1w_context_get_comm(const rt1w_context *ctx, int32_t *rank, int32_t *n_ranks, int32_t *n_local_devices) {
    if (!ctx) return fail(RT1W_ERR_INVALID, "null context");
    if (rank) *rank = ctx->comm_rank;
    if (n_ranks) *n_ranks = ctx->comm_size;
    if (n_local_devices) *n_local_devices = int32_t(1 + ctx->members.size());
    return RT1W_OK;
}

void rt1w_shard_sample_range(int32_t rank, int32_t n_ranks, int32_t sample_begin, int32_t sample_end, int32_t *out_begin, int32_t *out_end) {
    // contiguous ranges whose sizes differ by at most one; the Philox counter carries the GLOBAL sample index, so the image
    // does not depend on the split (up to the order of the fp32 additions)
    const int64_t total = sample_end > sample_begin ? int64_t(sample_end) - sample_begin : 0;
    const int64_t base = n_ranks > 0 ? total / n_ranks : total, extra = n_ranks > 0 ? total % n_ranks : 0;
    const int64_t b = int64_t(rank) * base + std::min<int64_t>(rank, extra);
    if (out_begin) *out_begin = int32_t(sample_begin + b);
    if (out_end) *out_end = int32_t(sample_begin + b + base + (rank < extra ? 1 : 0));
}

void rt1w_context_destroy(rt1w_context *ctx) {
    if (!ctx) return;
    for (rt1w_context *m : ctx->members) rt1w_context_destroy(m);
    ctx->members.clear();
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->comm && nccl_api().CommDestroy) nccl_api().CommDestroy(ctx->comm);
    pool_free(ctx->pool);
    cudaFree(ctx->d_accum), cudaFree(ctx->d_stat), cudaFree(ctx->d_rgb8);
    cudaFree(ctx->d_spp), cudaFree(ctx->d_list[0]), cudaFree(ctx->d_list[1]), cudaFree(ctx->d_keep), cudaFree(ctx->d_counts);
    cudaFree(ctx->d_batch), cudaFree(ctx->d_aov);
    cudaFreeHost(ctx->h_active);
    cudaFreeHost(ctx->h_ctr);
    cudaEventDestroy(ctx->ev0), cudaEventDestroy(ctx->ev1);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

rt1w_status rt1w_lower_prims(const rt1w_scene_desc *desc, rt1w_flat_prim *out, int32_t capacity, int32_t *n_out) {
    LoweredScene low;
    std::string err;
    rt1w_status st = lower_scene(desc, low, err);
    if (st != RT1W_OK) return fail(st, err);
    if (n_out) *n_out = int32_t(low.prims.size());
    if (out)
        for (int32_t i = 0; i < capacity && i < int32_t(low.prims.size()); ++i) out[i] = low.prims[i];
    return RT1W_OK;
}

rt1w_status rt1w_lower_face_groups(const rt1w_scene_desc *desc, int32_t *group_of_prim, int32_t *face_of_prim, int32_t capacity, int32_t *n_groups) {
    LoweredScene low;
    std::string err;
    rt1w_status st = lower_scene(desc, low, err);
    if (st != RT1W_OK) return fail(st, err);
    std::vector<uint32_t> order(low.prims.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = uint32_t(i);
    std::vector<int> group(low.prims.size(), -1), face(low.prims.size(), -1);
    std::vector<std::array<double, 6>> boxes;
    find_face_groups(low.prims, order, group, face, boxes);
    for (int32_t i = 0; i < capacity && i < int32_t(low.prims.size()); ++i) {
        if (group_of_prim) group_of_prim[i] = group[i];
        if (face_of_prim) face_of_prim[i] = face[i];
    }
    if (n_groups) *n_groups = int32_t(boxes.size());
    return RT1W_OK;
}

rt1w_status rt1w_build_bvh_host(const double *bbox_min3, const double *bbox_max3, int32_t n, void *nodes32, int32_t node_capacity, int32_t *n_nodes,
                                uint32_t *prim_order, void *wide_nodes80, int32_t wide_capacity, int32_t *n_wide, uint32_t *wide_leaf_remap,
                                int32_t *depth, int32_t *wide_depth) {
    if (!bbox_min3 || !bbox_max3 || n <= 0) return fail(RT1W_ERR_INVALID, "No objects in bvh_node constructor. (bvh.rs:61)");
    for (size_t i = 0; i < 3 * size_t(n); ++i)
        if (!std::isfinite(bbox_min3[i]) || !std::isfinite(bbox_max3[i]))
            return fail(RT1W_ERR_INVALID, "No bounding box in bvh_node constructor. (bvh.rs:65-67): non-finite primitive bounds");
    BvhBuildResult bvh;
    build_sah_bvh(bbox_min3, bbox_max3, size_t(n), kMaxLeaf, bvh);
    Bvh8BuildResult wide;
    collapse_to_bvh8(bvh.nodes.data(), bvh.nodes.size(), wide);
    if (wide.leaf_remap.size() != size_t(n)) return fail(RT1W_ERR_STATE, "wide BVH collapse lost primitives");
    if (n_nodes) *n_nodes = int32_t(bvh.nodes.size());
    if (n_wide) *n_wide = int32_t(wide.nodes.size());
    if (depth) *depth = bvh.depth;
    if (wide_depth) *wide_depth = wide.depth;
    if (nodes32) std::memcpy(nodes32, bvh.nodes.data(), sizeof(BvhNode32) * std::min(bvh.nodes.size(), size_t(std::max(node_capacity, 0))));
    if (wide_nodes80) std::memcpy(wide_nodes80, wide.nodes.data(), sizeof(Bvh8Node) * std::min(wide.nodes.size(), size_t(std::max(wide_capacity, 0))));
    if (prim_order) std::memcpy(prim_order, bvh.prim_order.data(), sizeof(uint32_t) * size_t(n));
    if (wide_leaf_remap) std::memcpy(wide_leaf_remap, wide.leaf_remap.data(), sizeof(uint32_t) * size_t(n));
    return RT1W_OK;
}

static rt1w_status scene_create_impl(rt1w_context *ctx, const rt1w_scene_desc *desc, rt1w_scene **out) {
    *out = nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    LoweredScene low;
    std::string err;
    rt1w_status st = lower_scene(desc, low, err);
    if (st != RT1W_OK) return fail(st, err);

    // Device primitives: the lowered primitives, except that the six rectangles of an AABox (aabox.rs:29-76) travel
    // as ONE box primitive (kernels.cuh: hit_box); hits still name the rectangle (first id + side).
    std::vector<rt1w_flat_prim> dev;
    std::vector<int32_t> dev_first_id;
    // scenes small enough for the flat scan keep their rectangles: the scan's frame-local boxes already cull five of a
    // box's six sides, and one code path for walls and box sides beats the shorter list (measured, Cornell box)
    // ONE decision for both: a scene is either scanned with its rectangles kept (flat) or traversed with its boxes merged.
    // (Deciding `flat` on the merged count would send P_BOX primitives into the scan, which compiles them out.)
    const bool flat = low.prims.size() <= size_t(kFlatMax) && low.frames.size() <= size_t(kFlatMaxFrames);
    const bool merge_boxes = !flat;
    for (size_t i = 0; i < low.prims.size();) {
        const rt1w_flat_prim &f0 = low.prims[i];
        bool is_box = merge_boxes && f0.kind == RT1W_NODE_XY_RECT && f0.node >= 0 && f0.node < desc->n_nodes && desc->nodes[f0.node].type == RT1W_NODE_AABOX &&
                      i + 6 <= low.prims.size();
        for (size_t k = 1; is_box && k < 6; ++k) is_box = low.prims[i + k].node == f0.node && low.prims[i + k].frame == f0.frame;
        if (!is_box) {
            dev.push_back(f0), dev_first_id.push_back(int32_t(i));
            ++i;
            continue;
        }
        rt1w_flat_prim b = f0; // sides: XY@z1, XY@z0, XZ@y1, ... with p = a0, a1, b0, b1, k
        b.kind = RT1W_NODE_AABOX;
        b.p[0] = f0.p[0], b.p[1] = f0.p[2], b.p[2] = low.prims[i + 1].p[4]; // x0, y0, z0
        b.p[3] = f0.p[1], b.p[4] = f0.p[3], b.p[5] = f0.p[4];               // x1, y1, z1
        for (size_t k = 1; k < 6; ++k)
            for (int c = 0; c < 3; ++c) {
                b.bbox_min[c] = std::min(b.bbox_min[c], low.prims[i + k].bbox_min[c]);
                b.bbox_max[c] = std::max(b.bbox_max[c], low.prims[i + k].bbox_max[c]);
            }
        dev.push_back(b), dev_first_id.push_back(int32_t(i));
        i += 6;
    }
    const size_t n = dev.size();
    if (n >= size_t(1) << kLeafBits) return fail(RT1W_ERR_UNSUPPORTED, "more than 2^28 primitives");
    for (size_t i = 0; i < n; ++i)
        for (int k = 0; k < 3; ++k)
            if (!std::isfinite(dev[i].bbox_min[k]) || !std::isfinite(dev[i].bbox_max[k]))
                return fail(RT1W_ERR_INVALID, "No bounding box in bvh_node constructor. (bvh.rs:65-67): non-finite primitive bounds");
    // Primitives whose box contains every other primitive's box - final_scene's 5000-unit fog sphere (main.rs:734-745) -
    // stay OUT of the tree: no box test ever culls them, in the tree they are one more level and one divergent leaf visit
    // for every ray.  They go to the end of the primitive array and are tested once per ray after the traversal, by all
    // lanes of the warp together (kernels.cuh: hit_globals).  RT1W_GLOBAL_PRIMS=0 keeps them in the tree (A/B, tests).
    size_t n_global = 0;
    const char *glob_env = std::getenv("RT1W_GLOBAL_PRIMS");
    if (!flat && n >= 8 && !(glob_env && std::strcmp(glob_env, "0") == 0)) {
        constexpr size_t kMaxGlobal = 4;
        std::vector<char> is_global(n, 0);
        for (size_t round = 0; round < kMaxGlobal; ++round) { // the box of all the OTHER primitives still in the tree, per candidate, from the two extremes of each bound
            double lo1[3], lo2[3], hi1[3], hi2[3];
            size_t lo_at[3], hi_at[3];
            for (int k = 0; k < 3; ++k) lo1[k] = lo2[k] = INFINITY, hi1[k] = hi2[k] = -INFINITY, lo_at[k] = hi_at[k] = n;
            for (size_t i = 0; i < n; ++i) {
                if (is_global[i]) continue;
                for (int k = 0; k < 3; ++k) {
                    const double a = dev[i].bbox_min[k], b = dev[i].bbox_max[k];
                    if (a < lo1[k]) lo2[k] = lo1[k], lo1[k] = a, lo_at[k] = i;
                    else if (a < lo2[k]) lo2[k] = a;
                    if (b > hi1[k]) hi2[k] = hi1[k], hi1[k] = b, hi_at[k] = i;
                    else if (b > hi2[k]) hi2[k] = b;
                }
            }
            size_t found = n;
            for (size_t i = 0; i < n && found == n; ++i) {
                if (is_global[i]) continue;
                // (spheres and sphere-bounded media only: hit_globals carries the sphere tests alone)
                if (!(dev[i].kind == RT1W_NODE_SPHERE || (dev[i].kind == RT1W_NODE_CONSTANT_MEDIUM && dev[i].boundary == RT1W_NODE_SPHERE))) continue;
                bool contains = true;
                for (int k = 0; k < 3 && contains; ++k) {
                    const double olo = lo_at[k] == i ? lo2[k] : lo1[k], ohi = hi_at[k] == i ? hi2[k] : hi1[k];
                    contains = dev[i].bbox_min[k] <= olo && dev[i].bbox_max[k] >= ohi;
                }
                if (contains) found = i;
            }
            if (found == n) break;
            is_global[found] = 1, ++n_global;
        }
        if (n_global > 0) { // stable: tree primitives first, globals last (primitive ids travel with them)
            std::vector<rt1w_flat_prim> d2;
            std::vector<int32_t> id2;
            for (int pass = 0; pass < 2; ++pass)
                for (size_t i = 0; i < n; ++i)
                    if (int(is_global[i]) == pass) d2.push_back(dev[i]), id2.push_back(dev_first_id[i]);
            dev.swap(d2), dev_first_id.swap(id2);
        }
    }
    const size_t nb = n - n_global; // primitives in the tree
    std::vector<double> bmin(3 * nb), bmax(3 * nb);
    for (size_t i = 0; i < nb; ++i)
        for (int k = 0; k < 3; ++k) bmin[3 * i + k] = dev[i].bbox_min[k], bmax[3 * i + k] = dev[i].bbox_max[k];
    // Builder: binned SAH on the host (best trees; seconds for a million primitives) or, for big scenes, a linear BVH
    // on the device (lbvh.cu; milliseconds).  RT1W_BVH_BUILDER=sah|lbvh overrides the size rule (tuning, tests).
    BvhBuildResult bvh;
    BvhNode32 *d_lbvh_nodes = nullptr;
    size_t n_bvh_nodes = 0;
    bool use_lbvh = nb >= size_t(kLbvhFromPrims);
    if (const char *env = std::getenv("RT1W_BVH_BUILDER")) use_lbvh = std::strcmp(env, "lbvh") == 0 ? nb >= 2 : (std::strcmp(env, "sah") == 0 ? false : use_lbvh);
    if (use_lbvh) {
        RT1W_CUDA(cudaSetDevice(ctx->device));
        std::vector<float> boxes(6 * nb);
        const double pad = traversal_pad(bmin.data(), bmax.data(), nb);
        for (size_t i = 0; i < nb; ++i) conservative_box(dev[i].bbox_min, dev[i].bbox_max, &boxes[6 * i], &boxes[6 * i + 3], pad);
        int depth = 0;
        cudaError_t e = build_lbvh(boxes.data(), nb, ctx->stream, &d_lbvh_nodes, &n_bvh_nodes, bvh.prim_order, &depth);
        if (e != cudaSuccess) return fail_cuda("device BVH build", e);
        bvh.depth = depth;
        if (depth > kStackSmem + kStackLocal - 2) { // many coincident centroids: let the SAH builder split by index instead
            cudaFree(d_lbvh_nodes), d_lbvh_nodes = nullptr;
            use_lbvh = false;
        }
    }
    if (!use_lbvh) {
        build_sah_bvh(bmin.data(), bmax.data(), nb, kMaxLeaf, bvh);
        n_bvh_nodes = bvh.nodes.size();
    }
    struct NodeGuard { // the device nodes belong to the scene once it exists
        BvhNode32 *&p;
        ~NodeGuard() { cudaFree(p); }
    } node_guard{d_lbvh_nodes};
    if (bvh.depth > kStackSmem + kStackLocal - 2) return fail(RT1W_ERR_UNSUPPORTED, "BVH deeper than the traversal stack");
    // BVH scenes also get the compressed 8-wide tree (bvh8.h), collapsed from the binary one whichever builder made it.
    // The leaves take the wide tree's order (a node's leaf slots are adjacent), the binary tree's leaf nodes are re-pointed:
    // both trees index ONE primitive array and find the same closest hits.
    Bvh8BuildResult wide;
    if (!flat) {
        if (d_lbvh_nodes) { // device-built: bring the nodes back (64 MB for a million primitives)
            bvh.nodes.resize(n_bvh_nodes);
            RT1W_CUDA(cudaMemcpy(bvh.nodes.data(), d_lbvh_nodes, sizeof(BvhNode32) * n_bvh_nodes, cudaMemcpyDeviceToHost));
            cudaFree(d_lbvh_nodes), d_lbvh_nodes = nullptr;
        }
        collapse_to_bvh8(bvh.nodes.data(), bvh.nodes.size(), wide);
        if (wide.leaf_remap.size() != nb) return fail(RT1W_ERR_STATE, "wide BVH collapse lost primitives");
        std::vector<uint32_t> new_of_old(nb), order(nb);
        for (size_t i = 0; i < nb; ++i) new_of_old[wide.leaf_remap[i]] = uint32_t(i), order[i] = bvh.prim_order[wide.leaf_remap[i]];
        for (BvhNode32 &nd : bvh.nodes)
            if (nd.count != 0) nd.left_first = new_of_old[nd.left_first];
        bvh.prim_order.swap(order);
    }
    for (size_t g = nb; g < n; ++g) bvh.prim_order.push_back(uint32_t(g)); // the global primitives: leaf indices nb .. n - 1
    std::vector<DPrim> dprims(n);
    std::vector<int32_t> prim_id(n);
    for (size_t i = 0; i < n; ++i) {
        const rt1w_flat_prim &fp = dev[bvh.prim_order[i]];
        dprims[i] = make_device_prim(fp, low.materials);
        prim_id[i] = dev_first_id[bvh.prim_order[i]];
    }
    // Small scenes are scanned, not traversed (kernels.cuh: closest_hit_flat): one padded f32 box per primitive in
    // the primitive's own frame, listed frame by frame; lo.w = leaf index, hi.w = frame of the BOX (-1 = world).
    std::vector<float4> prim_boxes;
    if (flat) {
        // the scan's FMA-form slab test cancels o/d against plane/d (2^-23 |o| of absolute error per plane) and uses
        // rcp.approx (2^-23 of the distance travelled): covered for ray origins up to twice the scene's largest
        // coordinate away from the world origin
        double reach = 0.0;
        for (size_t i = 0; i < n; ++i) {
            double llo[3], lhi[3];
            local_bounds(dev[i], llo, lhi);
            for (int c = 0; c < 3; ++c) {
                reach = std::max(reach, std::max(std::fabs(dev[i].bbox_min[c]), std::fabs(dev[i].bbox_max[c])));
                reach = std::max(reach, std::max(std::fabs(llo[c]), std::fabs(lhi[c])));
            }
        }
        const double scan_pad = 1e-6 * reach;
        // Face groups (kernels.cuh: closest_hit_flat): rectangles of one frame that are whole faces of a common box -
        // the walls of a room, the sides of an AABox (aabox.rs:29-76) - are tested with ONE slab computation on that box.
        std::vector<int> face_group(n, -1), face_of(n, -1); // by leaf
        std::vector<std::array<double, 6>> group_box;
        const char *fg_env = std::getenv("RT1W_FACE_GROUPS"); // =0: one box per rectangle (A/B measurements, tests)
        if (!fg_env || std::strcmp(fg_env, "0") != 0) find_face_groups(dev, bvh.prim_order, face_group, face_of, group_box);
        std::vector<int> scan(n);
        for (size_t i = 0; i < n; ++i) scan[i] = int(i);
        auto box_frame = [&](int leaf) { // a moving sphere keeps its world box: the reference tests that box (bvh.rs:31) before
                                         // evaluating the sphere at a time that may lie outside [time0, time1] (main.rs:86)
            const rt1w_flat_prim &fp = dev[bvh.prim_order[leaf]];
            return fp.kind == RT1W_NODE_MOVING_SPHERE ? -1 : fp.frame;
        };
        auto is_sphere = [&](int leaf) { // plain spheres get an f32 discriminant screen (kernels.cuh: flat_is_sphere)
            const rt1w_flat_prim &fp = dev[bvh.prim_order[leaf]];
            return fp.kind == RT1W_NODE_SPHERE ? 1 : 0;
        };
        auto scan_class = [&](int leaf) { return face_group[leaf] >= 0 ? 0 : 1 + is_sphere(leaf); }; // face groups, other boxes, plain spheres
        std::stable_sort(scan.begin(), scan.end(), [&](int a, int b) {
            if (box_frame(a) != box_frame(b)) return box_frame(a) < box_frame(b);
            if (scan_class(a) != scan_class(b)) return scan_class(a) < scan_class(b);
            if (face_group[a] != face_group[b]) return face_group[a] < face_group[b];
            return face_of[a] < face_of[b];
        });
        for (size_t k = 0; k < n; ++k) { // three float4 per scan slot: (lo.xyz, leaf), (hi.xyz, frame), (face group + 1, face, delta, -)
            const rt1w_flat_prim &fp = dev[bvh.prim_order[scan[k]]];
            const int bf = box_frame(scan[k]);
            double dlo[3], dhi[3];
            float lo[3], hi[3];
            float4 extra = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            const int fg = face_group[scan[k]];
            if (fg >= 0) { // every face slot carries the group's box, its planes moved outward by the f32 error of a tagged plane
                           // distance: 2^-23 |o| + (2^-22 + 2^-21) |plane - o| in space units, below 2e-6 reach for origins
                           // within 2 x reach (see scan_pad), + the f32 frame transform of pass 1 (3 roundings of reach-sized terms).
                           // A rectangle is hit ON its plane: its +-0.0001 slab is not needed.
                const double face_pad = 4e-6 * reach;
                double pad = 0.0; // distance of the padded planes from the true faces after rounding outward
                for (int c = 0; c < 3; ++c) {
                    lo[c] = std::nextafter(float(group_box[fg][c] - face_pad), -std::numeric_limits<float>::infinity());
                    hi[c] = std::nextafter(float(group_box[fg][3 + c] + face_pad), std::numeric_limits<float>::infinity());
                    pad = std::max(pad, std::max(group_box[fg][c] - double(lo[c]), double(hi[c]) - group_box[fg][3 + c]));
                }
                const int32_t g1 = fg + 1, face = face_of[scan[k]];
                std::memcpy(&extra.x, &g1, 4), std::memcpy(&extra.y, &face, 4);
                extra.z = float(2.02 * pad);
            } else {
                if (bf < 0) {
                    for (int c = 0; c < 3; ++c) dlo[c] = fp.bbox_min[c], dhi[c] = fp.bbox_max[c];
                } else {
                    local_bounds(fp, dlo, dhi);
                }
                conservative_box(dlo, dhi, lo, hi, scan_pad);
            }
            float4 l = make_float4(lo[0], lo[1], lo[2], 0.0f), h = make_float4(hi[0], hi[1], hi[2], 0.0f);
            const int32_t leaf = scan[k], frame = bf;
            std::memcpy(&l.w, &leaf, 4), std::memcpy(&h.w, &frame, 4);
            prim_boxes.push_back(l), prim_boxes.push_back(h), prim_boxes.push_back(extra);
        }
    }
    const auto t1 = std::chrono::steady_clock::now();

    RT1W_CUDA(cudaSetDevice(ctx->device));
    std::unique_ptr<rt1w_scene, void (*)(rt1w_scene *)> s(new rt1w_scene(), scene_release);
    s->ctx = ctx, s->device = ctx->device;
    static_assert(sizeof(BvhNode32) == 2 * sizeof(float4), "node layout");
    if (d_lbvh_nodes) {
        s->d_nodes = reinterpret_cast<float4 *>(d_lbvh_nodes), d_lbvh_nodes = nullptr;
    } else {
        RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&s->d_nodes), sizeof(BvhNode32) * bvh.nodes.size()));
        RT1W_CUDA(cudaMemcpy(s->d_nodes, bvh.nodes.data(), sizeof(BvhNode32) * bvh.nodes.size(), cudaMemcpyHostToDevice));
    }
    if (n_bvh_nodes > 0) fold_node_refs(s->d_nodes, n_bvh_nodes, ctx->stream);
    if (!wide.nodes.empty() && wide.depth <= kWideMaxDepth) {
        static_assert(sizeof(Bvh8Node) == 5 * sizeof(uint4), "wide node layout");
        RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&s->d_wide_nodes), sizeof(Bvh8Node) * wide.nodes.size()));
        RT1W_CUDA(cudaMemcpy(s->d_wide_nodes, wide.nodes.data(), sizeof(Bvh8Node) * wide.nodes.size(), cudaMemcpyHostToDevice));
    }
    RT1W_CUDA(upload(dprims, &s->d_prims));
    RT1W_CUDA(upload(prim_boxes, &s->d_prim_boxes));
    RT1W_CUDA(upload(prim_id, &s->d_prim_id));
    RT1W_CUDA(upload(low.frames, &s->d_frames));
    RT1W_CUDA(upload(low.materials, &s->d_materials));
    RT1W_CUDA(upload(low.textures, &s->d_textures));
    RT1W_CUDA(upload(low.perlins, &s->d_perlins));
    RT1W_CUDA(upload(low.lights, &s->d_lights));
    // images -> CUDA texture objects (point sampled, normalised-float reads give texel/255 as texture.rs:81-87)
    std::vector<int2> dims;
    for (const LoweredImage &im : low.images) {
        std::vector<uchar4> rgba(size_t(im.width) * im.height);
        for (size_t p = 0; p < rgba.size(); ++p) rgba[p] = make_uchar4(im.rgb8[3 * p], im.rgb8[3 * p + 1], im.rgb8[3 * p + 2], 255);
        cudaChannelFormatDesc fmt = cudaCreateChannelDesc<uchar4>();
        cudaArray_t arr = nullptr;
        RT1W_CUDA(cudaMallocArray(&arr, &fmt, size_t(im.width), size_t(im.height)));
        s->arrays.push_back(arr);
        RT1W_CUDA(cudaMemcpy2DToArray(arr, 0, 0, rgba.data(), size_t(im.width) * 4, size_t(im.width) * 4, size_t(im.height), cudaMemcpyHostToDevice));
        cudaResourceDesc res;
        std::memset(&res, 0, sizeof(res));
        res.resType = cudaResourceTypeArray;
        res.res.array.array = arr;
        cudaTextureDesc td;
        std::memset(&td, 0, sizeof(td));
        td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModePoint;
        td.readMode = cudaReadModeNormalizedFloat;
        td.normalizedCoords = 0;
        cudaTextureObject_t tex = 0;
        RT1W_CUDA(cudaCreateTextureObject(&tex, &res, &td, nullptr));
        s->tex_objects.push_back(tex);
        dims.push_back(make_int2(im.width, im.height));
    }
    RT1W_CUDA(upload(s->tex_objects, &s->d_images));
    RT1W_CUDA(upload(dims, &s->d_image_dims));
    const auto t2 = std::chrono::steady_clock::now();

    SceneView &v = s->view;
    v.nodes = s->d_nodes, v.prims = s->d_prims, v.prim_boxes = s->d_prim_boxes, v.prim_id = s->d_prim_id, v.frames = s->d_frames;
    v.materials = s->d_materials, v.textures = s->d_textures, v.perlins = s->d_perlins;
    v.images = s->d_images, v.image_dims = s->d_image_dims, v.lights = s->d_lights;
    v.n_lights = int32_t(low.lights.size()), v.has_lights = low.has_lights ? 1 : 0;
    v.n_global = int32_t(n_global);
    v.n_prims = int32_t(n), v.n_nodes = int32_t(n_bvh_nodes), v.n_perlins = int32_t(low.perlins.size()), v.n_frames = int32_t(low.frames.size());
    v.flat = flat ? 1 : 0;
    v.wide_nodes = s->d_wide_nodes, v.n_wide = s->d_wide_nodes ? int32_t(wide.nodes.size()) : 0;
    v.wide = !flat && n_bvh_nodes >= size_t(kWideFromNodes) ? 1 : 0;
    if (const char *env = std::getenv("RT1W_BVH_LAYOUT")) // binary | wide: overrides the size rule (tuning, tests)
        v.wide = !flat && std::strcmp(env, "wide") == 0 ? 1 : (std::strcmp(env, "binary") == 0 ? 0 : v.wide);
    if (!s->d_wide_nodes) v.wide = 0; // (a degenerate tree deeper than the wide traversal's stack keeps the binary walk)
    v.rich_textures = 0;
    for (const DTexture &t : low.textures)
        if (t.type != RT1W_TEX_SOLID) v.rich_textures = 1;
    s->material_mask = low.material_mask;
    s->n_textures = int(low.textures.size());
    s->prims = low.prims;
    s->leaf_prim_id = prim_id;
    s->info.n_prims = int32_t(low.prims.size()), s->info.n_bvh_nodes = int32_t(n_bvh_nodes), s->info.n_frames = int32_t(low.frames.size());
    s->info.n_lights = int32_t(low.lights.size()), s->info.bvh_depth = bvh.depth, s->info.material_mask = low.material_mask;
    s->info.build_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    s->info.upload_ms = std::chrono::duration<double, std::milli>(t2 - t1).count();
    s->info.sah_cost = bvh.sah_cost;
    s->info.n_wide_nodes = int32_t(wide.nodes.size()), s->info.wide_depth = wide.depth, s->info.wide_default = v.wide;
    s->info.wide_children = wide.avg_children, s->info.n_global_prims = int32_t(n_global);
    *out = s.release();
    return RT1W_OK;
}

rt1w_status rt1w_scene_create(rt1w_context *ctx, const rt1w_scene_desc *desc, rt1w_scene **out) {
    if (!ctx || !out) return fail(RT1W_ERR_INVALID, "null context or output pointer");
    *out = nullptr;
    std::lock_guard<std::mutex> guard(ctx->lock);
    if (ctx->members.empty()) return scene_create_impl(ctx, desc, out);
    // a multi-device context: the scene is replicated (SURVEY.md 8e), every device commits its own copy, all at once
    const size_t n = 1 + ctx->members.size();
    std::vector<rt1w_scene *> made(n, nullptr);
    std::vector<rt1w_status> status(n, RT1W_OK);
    std::vector<std::string> message(n);
    std::vector<std::thread> workers;
    for (size_t i = 1; i < n; ++i)
        workers.emplace_back([&, i] {
            status[i] = scene_create_impl(ctx->members[i - 1], desc, &made[i]);
            if (status[i] != RT1W_OK) message[i] = g_error;
        });
    status[0] = scene_create_impl(ctx, desc, &made[0]);
    if (status[0] != RT1W_OK) message[0] = g_error;
    for (auto &w : workers) w.join();
    for (size_t i = 0; i < n; ++i)
        if (status[i] != RT1W_OK) {
            for (rt1w_scene *m : made) scene_release(m);
            return fail(status[i], message[i]);
        }
    made[0]->replicas.assign(made.begin() + 1, made.end());
    *out = made[0];
    return RT1W_OK;
}

void rt1w_scene_destroy(rt1w_scene *scene) { scene_release(scene); }

rt1w_status rt1w_scene_get_info(const rt1w_scene *scene, rt1w_scene_info *out) {
    if (!scene || !out) return fail(RT1W_ERR_INVALID, "null scene or output pointer");
    *out = scene->info;
    return RT1W_OK;
}

rt1w_status rt1w_scene_get_prims(const rt1w_scene *scene, rt1w_flat_prim *out, int32_t capacity, int32_t *n_out) {
    if (!scene) return fail(RT1W_ERR_INVALID, "null scene");
    if (n_out) *n_out = int32_t(scene->prims.size());
    if (out)
        for (int32_t i = 0; i < capacity && i < int32_t(scene->prims.size()); ++i) out[i] = scene->prims[i];
    return RT1W_OK;
}

rt1w_status rt1w_scene_get_leaf_prims(const rt1w_scene *scene, int32_t *prim_id_of_leaf, int32_t capacity, int32_t *n_out) {
    if (!scene) return fail(RT1W_ERR_INVALID, "null scene");
    if (n_out) *n_out = int32_t(scene->leaf_prim_id.size());
    if (prim_id_of_leaf)
        for (int32_t i = 0; i < capacity && i < int32_t(scene->leaf_prim_id.size()); ++i) prim_id_of_leaf[i] = scene->leaf_prim_id[i];
    return RT1W_OK;
}

static rt1w_status ensure_buffers(rt1w_context *ctx, size_t pixels, bool stat, bool rgb8) {
    if (ctx->accum_pixels < pixels) {
        cudaFree(ctx->d_accum), ctx->d_accum = nullptr, ctx->accum_pixels = 0;
        RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&ctx->d_accum), sizeof(float) * 3 * pixels));
        ctx->accum_pixels = pixels;
    }
    if (stat && ctx->stat_pixels < pixels) {
        cudaFree(ctx->d_stat), ctx->d_stat = nullptr, ctx->stat_pixels = 0;
        RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&ctx->d_stat), sizeof(float) * 6 * pixels));
        ctx->stat_pixels = pixels;
    }
    if (rgb8 && ctx->rgb8_pixels < pixels) {
        cudaFree(ctx->d_rgb8), ctx->d_rgb8 = nullptr, ctx->rgb8_pixels = 0;
        RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&ctx->d_rgb8), 3 * pixels));
        ctx->rgb8_pixels = pixels;
    }
    return RT1W_OK;
}

static rt1w_status ensure_adaptive_buffers(rt1w_context *ctx, size_t pixels) {
    if (ctx->adaptive_pixels >= pixels) return RT1W_OK;
    cudaFree(ctx->d_spp), cudaFree(ctx->d_list[0]), cudaFree(ctx->d_list[1]), cudaFree(ctx->d_keep), cudaFree(ctx->d_counts);
    ctx->d_spp = nullptr, ctx->d_list[0] = ctx->d_list[1] = nullptr, ctx->d_keep = nullptr, ctx->d_counts = nullptr, ctx->adaptive_pixels = 0;
    if (!ctx->h_active) RT1W_CUDA(cudaMallocHost(reinterpret_cast<void **>(&ctx->h_active), sizeof(uint32_t)));
    RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&ctx->d_spp), sizeof(int32_t) * pixels));
    for (int k = 0; k < 2; ++k) RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&ctx->d_list[k]), sizeof(uint32_t) * pixels));
    RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&ctx->d_keep), pixels));
    RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&ctx->d_counts), sizeof(uint32_t) * (converge_blocks(uint32_t(pixels)) + 1)));
    ctx->adaptive_pixels = pixels;
    return RT1W_OK;
}

// One device's part of a render call: its share of the sample range (all of it outside a communicator), then - inside a
// communicator - the one exchange step of the path, ncclReduce(sum, fp32) of the radiance sums to rank 0 on the render
// stream (SURVEY.md 8e).  d_accum / d_stat: this device's buffers; after the call rank 0's hold the whole image.
// Everything of a render call that can fail before the first launch: argument checks, this rank's share of the sample range,
// the wave capacity and the queue allocation.  render_dispatch runs it for EVERY device of a multi-device context before any
// of them starts: a device that failed here alone would leave the others waiting in the reduce.
// The frames of a batch render (rt1w_render_batch): frame f renders with cameras[f] and seed seeds[f] (params->seed when seeds is null).
struct BatchFrames {
    const rt1w_camera *cameras;
    const uint64_t *seeds;
    int32_t n_frames;
};

// Byte offsets of the tables in the device allocation of a batch render (device_types.h: DBatch).
static size_t batch_cams_offset() { return (sizeof(DBatch) + 15) & ~size_t(15); }
static size_t batch_seeds_offset(size_t n_frames) { return batch_cams_offset() + sizeof(DCamera) * n_frames; }

static rt1w_status ensure_batch_tables(rt1w_context *ctx, size_t n_frames) {
    const size_t bytes = batch_seeds_offset(n_frames) + 2 * sizeof(uint32_t) * n_frames;
    if (ctx->batch_bytes >= bytes) return RT1W_OK;
    cudaFree(ctx->d_batch), ctx->d_batch = nullptr, ctx->batch_bytes = 0;
    RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&ctx->d_batch), bytes));
    ctx->batch_bytes = bytes;
    return RT1W_OK;
}

// The image size and sample range of a call (every render entry point and rt1w_render_aov).
static rt1w_status check_size_and_range(const rt1w_render_params &p) {
    if (p.width <= 0 || p.height <= 0) return fail(RT1W_ERR_INVALID, "image size must be positive");
    if (p.sample_end <= p.sample_begin || p.sample_begin < 0) return fail(RT1W_ERR_INVALID, "empty sample range");
    if (p.sample_end - p.sample_begin >= (1 << 24)) return fail(RT1W_ERR_UNSUPPORTED, "more than 2^24-1 samples per pixel in one call");
    if (uint64_t(p.width) * uint64_t(p.height) >= (1ull << 31)) return fail(RT1W_ERR_UNSUPPORTED, "image too large");
    return RT1W_OK;
}

static rt1w_status render_prepare(rt1w_scene *scene, const rt1w_render_params *params, rt1w_render_params &p, uint32_t &want_pool, int32_t &my_samples,
                                  const BatchFrames *frames = nullptr) {
    rt1w_context *ctx = scene->ctx;
    p = *params;
    const rt1w_status checked = check_size_and_range(p);
    if (checked != RT1W_OK) return checked;
    if (p.max_depth < 0 || p.max_depth > 255) return fail(RT1W_ERR_UNSUPPORTED, "max_depth must be in [0, 255]");
    if (p.pool_paths > (1 << 30)) return fail(RT1W_ERR_UNSUPPORTED, "pool_paths must not exceed 2^30");
    const bool sharded = ctx->comm != nullptr && ctx->comm_size > 1;
    if (sharded) rt1w_shard_sample_range(ctx->comm_rank, ctx->comm_size, params->sample_begin, params->sample_end, &p.sample_begin, &p.sample_end);
    my_samples = p.sample_end - p.sample_begin; // 0: more ranks than samples - this one only joins the reduce
    const uint64_t n_frames = frames ? uint64_t(frames->n_frames) : 1u;
    const uint64_t all_paths = n_frames * uint64_t(p.width) * uint64_t(p.height) * uint64_t(my_samples);
    want_pool = p.pool_paths > 0 ? uint32_t(p.pool_paths) : kDefaultPool;
    if (p.pool_paths <= 0 && all_paths < want_pool) want_pool = uint32_t((all_paths + 1023u) & ~uint64_t(1023u)); // small renders: one wave holds every path
    if (want_pool == 0) want_pool = 1024;
    if (frames) {
        const rt1w_status st = ensure_batch_tables(ctx, size_t(n_frames));
        if (st != RT1W_OK) return st;
    }
    if (ctx->pool.allocated < want_pool || (ctx->pool.material_mask & scene->material_mask) != scene->material_mask) {
        const uint32_t grow = ctx->pool.allocated > want_pool ? ctx->pool.allocated : want_pool;
        cudaError_t e = pool_alloc(ctx->pool, grow, scene->material_mask | ctx->pool.material_mask);
        if (e != cudaSuccess) return fail_cuda("path pool allocation", e);
    }
    return RT1W_OK;
}

static DCamera device_camera(const rt1w_camera *camera) {
    DCamera c;
    for (int k = 0; k < 3; ++k) {
        c.origin[k] = camera->origin[k];
        c.llc_rel[k] = camera->lower_left_corner[k] - camera->origin[k];
        c.horizontal[k] = camera->horizontal[k], c.vertical[k] = camera->vertical[k];
        c.u[k] = camera->u[k], c.v[k] = camera->v[k];
    }
    c.lens_radius = camera->lens_radius;
    c.time0 = float(camera->time0), c.time1 = float(camera->time1);
    return c;
}

// The wave loop's arguments for the sample range [p.sample_begin, p.sample_begin + n_samples) of n_pixels pixels: every
// pixel of the image, the pixels of a list, or every pixel of every frame of a batch (render_waves).  The sums of
// d_accum / d_stat are added to, not zeroed.
static RenderArgs render_args(const rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params &p, uint32_t want_pool, int32_t n_samples,
                              uint32_t n_pixels, float *d_accum, float *d_stat) {
    RenderArgs args;
    args.sc = scene->view;
    args.pool = scene->ctx->pool;
    args.pool.capacity = want_pool;
    DRenderParams &rp = args.rp;
    rp.width = p.width, rp.height = p.height, rp.sample_begin = p.sample_begin, rp.n_samples = n_samples;
    rp.max_depth = p.max_depth, rp.flags = p.flags, rp.seed_lo = uint32_t(p.seed), rp.seed_hi = uint32_t(p.seed >> 32);
    for (int k = 0; k < 3; ++k) rp.background[k] = float(p.background[k]);
    rp.stat_clamp = p.stat_clamp > 0.0 ? float(p.stat_clamp) : INFINITY;
    rp.n_pixels = n_pixels;
    rp.total_paths = p.max_depth == 0 ? 0ull : (unsigned long long)rp.n_pixels * (unsigned long long)rp.n_samples; // depth 0: ray_color returns black at once
    rp.pool = int32_t(want_pool);
    rp.tile_shift = 16; // 65536 pixels = 768 KB of sums per tile; fewer when the sample count is huge (tile_paths <= 2^30)
    while (rp.tile_shift > 5 && (uint64_t(rp.n_samples) << rp.tile_shift) > (1ull << 30)) --rp.tile_shift;
    rp.tile_paths = uint32_t(std::max(rp.n_samples, 1)) << rp.tile_shift;
    rp.inv_w1 = 1.0 / double(p.width - 1), rp.inv_h1 = 1.0 / double(p.height - 1); // a 1-pixel axis: inf, as the reference's division by zero
    rp.inv_width_up = (1.0 / double(p.width)) * (1.0 + 0x1p-50), rp.inv_tile_paths_up = (1.0 / double(rp.tile_paths)) * (1.0 + 0x1p-50);
    args.cam = device_camera(camera);
    args.accum = d_accum;
    args.stat = d_stat;
    return args;
}

// The frame tables of a batch render to ctx->d_batch (allocated by render_prepare), on `stream` ahead of the waves.
static rt1w_status upload_batch(rt1w_context *ctx, const BatchFrames &frames, const rt1w_render_params &p, cudaStream_t stream) {
    const size_t n = size_t(frames.n_frames), cams = batch_cams_offset(), seeds = batch_seeds_offset(n);
    std::vector<unsigned char> host(seeds + 2 * sizeof(uint32_t) * n);
    DBatch h;
    const uint32_t d = uint32_t(p.width) * uint32_t(p.height);
    uint32_t l = 0; // ceil(log2(d))
    while (l < 32 && (uint64_t(1) << l) < d) ++l;
    h.frame_pixels = d;
    h.magic = uint32_t(((uint64_t(1) << 32) * ((uint64_t(1) << l) - d)) / d + 1); // (2^l - d < d, so the product fits 64 bits)
    h.shift1 = l < 1 ? l : 1, h.shift2 = l < 1 ? 0 : l - 1;
    h.cams = reinterpret_cast<const DCamera *>(ctx->d_batch + cams), h.seeds = reinterpret_cast<const uint32_t *>(ctx->d_batch + seeds);
    std::memcpy(host.data(), &h, sizeof(h));
    for (size_t f = 0; f < n; ++f) {
        const DCamera c = device_camera(&frames.cameras[f]);
        const uint64_t seed = frames.seeds ? frames.seeds[f] : p.seed;
        const uint32_t words[2] = {uint32_t(seed), uint32_t(seed >> 32)};
        std::memcpy(host.data() + cams + sizeof(DCamera) * f, &c, sizeof(c));
        std::memcpy(host.data() + seeds + sizeof(words) * f, words, sizeof(words));
    }
    // (from pageable memory: the call returns once `host` has been staged)
    RT1W_CUDA(cudaMemcpyAsync(ctx->d_batch, host.data(), host.size(), cudaMemcpyHostToDevice, stream));
    return RT1W_OK;
}

// frames: nullptr, or the frames of a batch render - every frame's sums, one after the other, in d_accum.
static rt1w_status render_common(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params, float *d_accum, float *d_stat,
                                 cudaStream_t stream, rt1w_render_stats *stats, const BatchFrames *frames = nullptr) {
    rt1w_context *ctx = scene->ctx;
    rt1w_render_params p;
    uint32_t want_pool = 0;
    int32_t my_samples = 0;
    const rt1w_status prepared = render_prepare(scene, params, p, want_pool, my_samples, frames);
    if (prepared != RT1W_OK) return prepared;
    const bool sharded = ctx->comm != nullptr && ctx->comm_size > 1;
    const uint32_t n_frames = frames ? uint32_t(frames->n_frames) : 1u;
    const RenderArgs args = render_args(scene, frames ? frames->cameras : camera, p, want_pool, my_samples, n_frames * uint32_t(p.width) * uint32_t(p.height),
                                        d_accum, d_stat);
    const DRenderParams &rp = args.rp;

    RT1W_CUDA(cudaEventRecord(ctx->ev0, stream));
    if (frames) {
        const rt1w_status st = upload_batch(ctx, *frames, p, stream);
        if (st != RT1W_OK) return st;
    }
    RT1W_CUDA(cudaMemsetAsync(d_accum, 0, sizeof(float) * 3 * size_t(rp.n_pixels), stream));
    if (d_stat) RT1W_CUDA(cudaMemsetAsync(d_stat, 0, sizeof(float) * 6 * size_t(rp.n_pixels), stream));
    WaveStats ws;
    ws.profile = (p.flags & RT1W_FLAG_PROFILE) != 0;
    if (rp.total_paths > 0) {
        const DBatch *batch = frames ? reinterpret_cast<const DBatch *>(ctx->d_batch) : nullptr;
        cudaError_t e = render_waves(args, nullptr, batch, scene->material_mask, ctx->h_ctr, stream, ctx->sm_count, ws);
        if (e != cudaSuccess) return fail_cuda("wavefront render", e);
    }
    if (sharded) { // in place: rank 0 receives where it sent
        const NcclApi &nccl = nccl_api();
        ncclResult_t r = nccl.Reduce(d_accum, d_accum, 3 * size_t(rp.n_pixels), ncclFloat, ncclSum, 0, ctx->comm, stream);
        if (r == ncclSuccess && d_stat) r = nccl.Reduce(d_stat, d_stat, 6 * size_t(rp.n_pixels), ncclFloat, ncclSum, 0, ctx->comm, stream);
        if (r != ncclSuccess) return fail_nccl("ncclReduce of the radiance sums", r);
    }
    RT1W_CUDA(cudaEventRecord(ctx->ev1, stream));
    RT1W_CUDA(cudaStreamSynchronize(stream));
    if (stats) {
        float ms = 0.0f;
        RT1W_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        std::memset(stats, 0, sizeof(*stats));
        stats->paths = uint64_t(rp.n_pixels) * uint64_t(rp.n_samples);
        stats->rays = ws.rays, stats->waves = ws.waves, stats->launches = ws.launches;
        stats->render_ms = ms;
        static_assert(RT1W_KERNEL_COUNT == K_COUNT, "kernel slot tables must agree");
        for (int k = 0; k < K_COUNT; ++k) stats->kernel_ms[k] = ws.kernel_ms[k], stats->kernel_launches[k] = ws.kernel_launches[k];
    }
    return RT1W_OK;
}

// A call on a multi-device context (rt1w_context_create_multi): one host thread per device, each running `run` on its
// replica of the scene, after `prepare` has run for EVERY device: whatever can fail before the first launch fails there, for
// every device, before any of them enters the collective part (a device that failed alone would leave the others waiting in
// the reduce).  stats: paths, rays and launches summed, waves and time the maximum.
// prepare(i, context, scene) and run(i, context, scene, stats) for device i (0: the context's own).
extern "C++" {
template <class Prepare, class Run>
static rt1w_status for_each_device(rt1w_scene *scene, Prepare prepare, Run run, rt1w_render_stats *stats) {
    rt1w_context *ctx = scene->ctx;
    const size_t n = 1 + ctx->members.size();
    if (scene->replicas.size() + 1 != n) return fail(RT1W_ERR_STATE, "the scene was not committed on this multi-device context");
    std::vector<rt1w_status> status(n, RT1W_OK);
    std::vector<std::string> message(n);
    std::vector<rt1w_render_stats> st(n);
    for (size_t i = 0; i < n; ++i) {
        rt1w_context *c = i == 0 ? ctx : ctx->members[i - 1];
        rt1w_status s0 = cudaSetDevice(c->device) == cudaSuccess ? RT1W_OK : fail(RT1W_ERR_CUDA, "cudaSetDevice failed");
        if (s0 == RT1W_OK) s0 = prepare(i, c, i == 0 ? scene : scene->replicas[i - 1]);
        if (s0 != RT1W_OK) {
            const std::string why = g_error;
            cudaSetDevice(ctx->device);
            return fail(s0, "device " + std::to_string(i) + ": " + why);
        }
    }
    auto run_one = [&](size_t i) {
        rt1w_context *c = i == 0 ? ctx : ctx->members[i - 1];
        if (cudaSetDevice(c->device) != cudaSuccess) {
            status[i] = RT1W_ERR_CUDA, message[i] = "cudaSetDevice failed";
            return;
        }
        status[i] = run(i, c, i == 0 ? scene : scene->replicas[i - 1], &st[i]);
        if (status[i] != RT1W_OK) message[i] = g_error;
    };
    std::vector<std::thread> workers;
    for (size_t i = 1; i < n; ++i) workers.emplace_back(run_one, i);
    run_one(0);
    for (auto &w : workers) w.join();
    cudaSetDevice(ctx->device);
    for (size_t i = 0; i < n; ++i)
        if (status[i] != RT1W_OK) return fail(status[i], "device " + std::to_string(i) + ": " + message[i]);
    if (stats) {
        *stats = st[0];
        for (size_t i = 1; i < n; ++i) {
            stats->paths += st[i].paths, stats->rays += st[i].rays, stats->launches += st[i].launches;
            stats->waves = std::max(stats->waves, st[i].waves), stats->render_ms = std::max(stats->render_ms, st[i].render_ms);
            for (int k = 0; k < K_COUNT; ++k) stats->kernel_ms[k] += st[i].kernel_ms[k], stats->kernel_launches[k] += st[i].kernel_launches[k];
        }
    }
    return RT1W_OK;
}
} // extern "C++"

// A render call on a multi-device context: render_common on every device's replica of the scene; the reduce inside leaves
// the image in rank 0's buffers (d_accum / d_stat on the first device, stream = its render stream).
static rt1w_status render_dispatch(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params, float *d_accum, float *d_stat,
                                   cudaStream_t stream, rt1w_render_stats *stats, const BatchFrames *frames = nullptr) {
    rt1w_context *ctx = scene->ctx;
    if (ctx->members.empty()) return render_common(scene, camera, params, d_accum, d_stat, stream, stats, frames);
    const size_t pixels = params->width > 0 && params->height > 0 ? size_t(frames ? frames->n_frames : 1) * size_t(params->width) * size_t(params->height) : 0;
    auto prepare = [&](size_t i, rt1w_context *c, rt1w_scene *sc) {
        rt1w_render_params p;
        uint32_t want_pool = 0;
        int32_t my_samples = 0;
        const rt1w_status s0 = i > 0 ? ensure_buffers(c, pixels, d_stat != nullptr, false) : RT1W_OK;
        return s0 != RT1W_OK ? s0 : render_prepare(sc, params, p, want_pool, my_samples, frames);
    };
    auto run = [&](size_t i, rt1w_context *c, rt1w_scene *sc, rt1w_render_stats *st) {
        if (i == 0) return render_common(sc, camera, params, d_accum, d_stat, stream, st, frames);
        return render_common(sc, camera, params, c->d_accum, d_stat ? c->d_stat : nullptr, c->stream, st, frames);
    };
    return for_each_device(scene, prepare, run, stats);
}

rt1w_status rt1w_render(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params, float *out_rgb_sum, float *out_stat,
                        rt1w_render_stats *stats) {
    if (!scene || !camera || !params) return fail(RT1W_ERR_INVALID, "null argument");
    rt1w_context *ctx = scene->ctx;
    const bool root = ctx->comm_rank == 0; // only rank 0 of a communicator receives the image
    if (root && !out_rgb_sum) return fail(RT1W_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> guard(ctx->lock);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    if (params->width <= 0 || params->height <= 0) return fail(RT1W_ERR_INVALID, "image size must be positive");
    const size_t pixels = size_t(params->width) * size_t(params->height);
    // (the flag alone decides whether the statistics buffers exist: in a communicator every rank must join the same reduces)
    const bool want_stat = (params->flags & RT1W_FLAG_STATS) != 0;
    if (out_stat && !want_stat) return fail(RT1W_ERR_INVALID, "out_stat needs RT1W_FLAG_STATS");
    rt1w_status st = ensure_buffers(ctx, pixels, want_stat, false);
    if (st != RT1W_OK) return st;
    st = render_dispatch(scene, camera, params, ctx->d_accum, want_stat ? ctx->d_stat : nullptr, ctx->stream, stats);
    if (st != RT1W_OK) return st;
    if (root) {
        RT1W_CUDA(cudaMemcpyAsync(out_rgb_sum, ctx->d_accum, sizeof(float) * 3 * pixels, cudaMemcpyDeviceToHost, ctx->stream));
        if (want_stat && out_stat) RT1W_CUDA(cudaMemcpyAsync(out_stat, ctx->d_stat, sizeof(float) * 6 * pixels, cudaMemcpyDeviceToHost, ctx->stream));
        RT1W_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return RT1W_OK;
}

rt1w_status rt1w_render_rgb8(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params, uint8_t *out_rgb8,
                             rt1w_render_stats *stats) {
    if (!scene || !camera || !params) return fail(RT1W_ERR_INVALID, "null argument");
    rt1w_context *ctx = scene->ctx;
    const bool root = ctx->comm_rank == 0;
    if (root && !out_rgb8) return fail(RT1W_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> guard(ctx->lock);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    if (params->width <= 0 || params->height <= 0) return fail(RT1W_ERR_INVALID, "image size must be positive");
    if (params->flags & RT1W_FLAG_STATS) return fail(RT1W_ERR_INVALID, "RT1W_FLAG_STATS is only available through rt1w_render");
    const size_t pixels = size_t(params->width) * size_t(params->height);
    rt1w_status st = ensure_buffers(ctx, pixels, false, root);
    if (st != RT1W_OK) return st;
    st = render_dispatch(scene, camera, params, ctx->d_accum, nullptr, ctx->stream, stats);
    if (st != RT1W_OK) return st;
    if (root) { // the mean divides by the WHOLE sample range: the reduce has added every rank's share
        RT1W_CUDA(resolve_launch(ctx->d_accum, 3 * pixels, params->sample_end - params->sample_begin, ctx->d_rgb8, ctx->stream));
        RT1W_CUDA(cudaMemcpyAsync(out_rgb8, ctx->d_rgb8, 3 * pixels, cudaMemcpyDeviceToHost, ctx->stream));
        RT1W_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return RT1W_OK;
}

rt1w_status rt1w_render_device(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params, float *d_rgb_sum,
                               void *cuda_stream, rt1w_render_stats *stats) {
    if (!scene || !camera || !params || !d_rgb_sum) return fail(RT1W_ERR_INVALID, "null argument");
    rt1w_context *ctx = scene->ctx;
    std::lock_guard<std::mutex> guard(ctx->lock);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    if (params->flags & RT1W_FLAG_STATS) return fail(RT1W_ERR_INVALID, "RT1W_FLAG_STATS is only available through rt1w_render");
    return render_dispatch(scene, camera, params, d_rgb_sum, nullptr, static_cast<cudaStream_t>(cuda_stream), stats);
}

// All frames in ONE wavefront: paths are numbered over n_frames * width * height batch pixels (render.cu: Numbering), so the
// waves stay full until the last frame's paths have started and the render drains once.
rt1w_status rt1w_render_batch(rt1w_scene *scene, const rt1w_camera *cameras, int32_t n_frames, const uint64_t *seeds, const rt1w_render_params *params,
                              float *out_rgb_sum, uint8_t *out_rgb8, rt1w_render_stats *stats) {
    if (!scene || !cameras || !params) return fail(RT1W_ERR_INVALID, "null argument");
    if (n_frames < 1) return fail(RT1W_ERR_INVALID, "n_frames must be at least 1");
    rt1w_context *ctx = scene->ctx;
    const bool root = ctx->comm_rank == 0;
    if (root && !out_rgb_sum && !out_rgb8) return fail(RT1W_ERR_INVALID, "rank 0 needs out_rgb_sum or out_rgb8");
    std::lock_guard<std::mutex> guard(ctx->lock);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    if (params->width <= 0 || params->height <= 0) return fail(RT1W_ERR_INVALID, "image size must be positive");
    if (params->flags & RT1W_FLAG_STATS) return fail(RT1W_ERR_INVALID, "RT1W_FLAG_STATS is only available through rt1w_render");
    const uint64_t pixels = uint64_t(n_frames) * uint64_t(params->width) * uint64_t(params->height);
    if (pixels >= (1ull << 32)) return fail(RT1W_ERR_INVALID, "n_frames * width * height must be below 2^32 (a path's pixel word is 32 bits)");
    rt1w_status st = ensure_buffers(ctx, size_t(pixels), false, root && out_rgb8);
    if (st != RT1W_OK) return st;
    const BatchFrames frames{cameras, seeds, n_frames};
    st = render_dispatch(scene, cameras, params, ctx->d_accum, nullptr, ctx->stream, stats, &frames);
    if (st != RT1W_OK) return st;
    if (root) { // the mean divides by the WHOLE sample range: the reduce has added every rank's share
        if (out_rgb8) {
            RT1W_CUDA(resolve_launch(ctx->d_accum, 3 * size_t(pixels), params->sample_end - params->sample_begin, ctx->d_rgb8, ctx->stream));
            RT1W_CUDA(cudaMemcpyAsync(out_rgb8, ctx->d_rgb8, 3 * size_t(pixels), cudaMemcpyDeviceToHost, ctx->stream));
        }
        if (out_rgb_sum) RT1W_CUDA(cudaMemcpyAsync(out_rgb_sum, ctx->d_accum, sizeof(float) * 3 * size_t(pixels), cudaMemcpyDeviceToHost, ctx->stream));
        RT1W_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return RT1W_OK;
}

// Rounds of ordinary sample ranges: [0, min_spp) over the whole image, then [n, min(2n, max_spp)) over the list of the
// pixels the convergence pass kept, in ascending seed order, adding to the same sums and statistics.
rt1w_status rt1w_render_adaptive(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params, int32_t min_spp, double max_error,
                                 float *out_rgb_sum, int32_t *out_spp, uint8_t *out_rgb8, float *out_stat, rt1w_render_stats *stats) {
    if (!scene || !camera || !params) return fail(RT1W_ERR_INVALID, "null argument");
    rt1w_context *ctx = scene->ctx;
    std::lock_guard<std::mutex> guard(ctx->lock);
    if (ctx->comm != nullptr || !ctx->members.empty())
        return fail(RT1W_ERR_UNSUPPORTED, "adaptive rendering runs on one device: this context belongs to a communicator or drives several devices");
    RT1W_CUDA(cudaSetDevice(ctx->device));
    if (params->sample_begin != 0) return fail(RT1W_ERR_INVALID, "adaptive rendering starts at sample 0: sample_begin must be 0 (sample_end is the cap)");
    if (min_spp < 2 || min_spp > params->sample_end) return fail(RT1W_ERR_INVALID, "min_spp must be in [2, sample_end]");
    if (!(max_error >= 0.0)) return fail(RT1W_ERR_INVALID, "max_error must be a number >= 0");
    rt1w_render_params p;
    uint32_t want_pool = 0;
    int32_t max_spp = 0;
    rt1w_status st = render_prepare(scene, params, p, want_pool, max_spp);
    if (st != RT1W_OK) return st;
    const uint32_t pixels = uint32_t(p.width) * uint32_t(p.height);
    if ((st = ensure_buffers(ctx, pixels, true, out_rgb8 != nullptr)) != RT1W_OK) return st;
    if ((st = ensure_adaptive_buffers(ctx, pixels)) != RT1W_OK) return st;
    const cudaStream_t stream = ctx->stream;

    RT1W_CUDA(cudaEventRecord(ctx->ev0, stream));
    RT1W_CUDA(cudaMemsetAsync(ctx->d_accum, 0, sizeof(float) * 3 * size_t(pixels), stream));
    RT1W_CUDA(cudaMemsetAsync(ctx->d_stat, 0, sizeof(float) * 6 * size_t(pixels), stream));
    WaveStats all;
    uint64_t paths = 0;
    const uint32_t *list = nullptr; // round 0: every pixel
    uint32_t active = pixels;
    int32_t n = 0, next = min_spp;
    for (int round = 0; active > 0; ++round) {
        p.sample_begin = n;
        const RenderArgs args = render_args(scene, camera, p, want_pool, next - n, active, ctx->d_accum, ctx->d_stat);
        if (args.rp.total_paths > 0) {
            WaveStats ws;
            ws.profile = (p.flags & RT1W_FLAG_PROFILE) != 0;
            const cudaError_t e = render_waves(args, list, nullptr, scene->material_mask, ctx->h_ctr, stream, ctx->sm_count, ws);
            if (e != cudaSuccess) return fail_cuda("wavefront render", e);
            all.rays += ws.rays, all.waves += ws.waves, all.launches += ws.launches;
            for (int k = 0; k < K_COUNT; ++k) all.kernel_ms[k] += ws.kernel_ms[k], all.kernel_launches[k] += ws.kernel_launches[k];
        }
        paths += uint64_t(active) * uint64_t(next - n);
        n = next;
        uint32_t *out_list = ctx->d_list[round & 1];
        RT1W_CUDA(converge_launch(ctx->d_accum, ctx->d_stat, list, active, p.width, p.height, n, max_spp, max_error, ctx->d_spp, ctx->d_keep, ctx->d_counts,
                                  out_list, stream));
        RT1W_CUDA(cudaMemcpyAsync(ctx->h_active, ctx->d_counts + converge_blocks(active), sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
        RT1W_CUDA(cudaStreamSynchronize(stream));
        active = *ctx->h_active;
        list = out_list;
        next = int32_t(std::min<int64_t>(2 * int64_t(n), max_spp));
    }
    if (out_rgb8) RT1W_CUDA(resolve_counts_launch(ctx->d_accum, ctx->d_spp, 3 * size_t(pixels), ctx->d_rgb8, stream));
    RT1W_CUDA(cudaEventRecord(ctx->ev1, stream));
    if (out_rgb_sum) RT1W_CUDA(cudaMemcpyAsync(out_rgb_sum, ctx->d_accum, sizeof(float) * 3 * size_t(pixels), cudaMemcpyDeviceToHost, stream));
    if (out_spp) RT1W_CUDA(cudaMemcpyAsync(out_spp, ctx->d_spp, sizeof(int32_t) * size_t(pixels), cudaMemcpyDeviceToHost, stream));
    if (out_rgb8) RT1W_CUDA(cudaMemcpyAsync(out_rgb8, ctx->d_rgb8, 3 * size_t(pixels), cudaMemcpyDeviceToHost, stream));
    if (out_stat) RT1W_CUDA(cudaMemcpyAsync(out_stat, ctx->d_stat, sizeof(float) * 6 * size_t(pixels), cudaMemcpyDeviceToHost, stream));
    RT1W_CUDA(cudaStreamSynchronize(stream));
    if (stats) {
        float ms = 0.0f;
        RT1W_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        std::memset(stats, 0, sizeof(*stats));
        stats->paths = paths;
        stats->rays = all.rays, stats->waves = all.waves, stats->launches = all.launches;
        stats->render_ms = ms;
        for (int k = 0; k < K_COUNT; ++k) stats->kernel_ms[k] = all.kernel_ms[k], stats->kernel_launches[k] = all.kernel_launches[k];
    }
    return RT1W_OK;
}

// ---- first-hit feature buffers (rt1w.h: rt1w_render_aov) ----
// Everything of an AOV call that can fail before its launch, on one device: the argument checks, this rank's share of the
// sample range and the output buffer.  No path pool: the call traces one closest hit per sample and keeps no path state.
static rt1w_status aov_prepare(rt1w_scene *scene, const rt1w_render_params *params, rt1w_render_params &p, int32_t &my_samples) {
    rt1w_context *ctx = scene->ctx;
    p = *params;
    const rt1w_status checked = check_size_and_range(p);
    if (checked != RT1W_OK) return checked;
    if (p.flags & RT1W_FLAG_STATS) return fail(RT1W_ERR_INVALID, "RT1W_FLAG_STATS is only available through rt1w_render");
    if (ctx->comm != nullptr && ctx->comm_size > 1)
        rt1w_shard_sample_range(ctx->comm_rank, ctx->comm_size, params->sample_begin, params->sample_end, &p.sample_begin, &p.sample_end);
    my_samples = p.sample_end - p.sample_begin; // 0: more ranks than samples - this one only joins the reduce
    const size_t pixels = size_t(p.width) * size_t(p.height);
    if (ctx->aov_pixels < pixels) {
        cudaFree(ctx->d_aov), ctx->d_aov = nullptr, ctx->aov_pixels = 0;
        RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&ctx->d_aov), sizeof(float) * 8 * pixels));
        ctx->aov_pixels = pixels;
    }
    return RT1W_OK;
}

// One device's part of an AOV call: its share of the sample range into ctx->d_aov, then - inside a communicator - ONE
// ncclReduce of the packed 8 * width * height sums to rank 0.
static rt1w_status aov_common(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params, rt1w_render_stats *stats) {
    rt1w_context *ctx = scene->ctx;
    rt1w_render_params p;
    int32_t my_samples = 0;
    const rt1w_status prepared = aov_prepare(scene, params, p, my_samples);
    if (prepared != RT1W_OK) return prepared;
    const uint32_t pixels = uint32_t(p.width) * uint32_t(p.height);
    const RenderArgs args = render_args(scene, camera, p, 0, my_samples, pixels, nullptr, nullptr);
    const cudaStream_t stream = ctx->stream;
    RT1W_CUDA(cudaEventRecord(ctx->ev0, stream));
    if (my_samples > 0) RT1W_CUDA(aov_launch(args, scene->material_mask, ctx->d_aov, ctx->sm_count, stream));
    else RT1W_CUDA(cudaMemsetAsync(ctx->d_aov, 0, sizeof(float) * 8 * size_t(pixels), stream));
    if (ctx->comm != nullptr && ctx->comm_size > 1) {
        const ncclResult_t r = nccl_api().Reduce(ctx->d_aov, ctx->d_aov, 8 * size_t(pixels), ncclFloat, ncclSum, 0, ctx->comm, stream);
        if (r != ncclSuccess) return fail_nccl("ncclReduce of the feature buffers", r);
    }
    RT1W_CUDA(cudaEventRecord(ctx->ev1, stream));
    RT1W_CUDA(cudaStreamSynchronize(stream));
    if (stats) {
        float ms = 0.0f;
        RT1W_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        std::memset(stats, 0, sizeof(*stats));
        stats->paths = stats->rays = uint64_t(pixels) * uint64_t(my_samples); // one closest hit per sample
        stats->launches = my_samples > 0 ? 1 : 0;
        stats->render_ms = ms;
    }
    return RT1W_OK;
}

rt1w_status rt1w_render_aov(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params, float *out_albedo_sum, float *out_normal_sum,
                            float *out_distance_sum, float *out_hits, rt1w_render_stats *stats) {
    if (!scene || !camera || !params) return fail(RT1W_ERR_INVALID, "null argument");
    rt1w_context *ctx = scene->ctx;
    const bool root = ctx->comm_rank == 0;
    if (root && !out_albedo_sum && !out_normal_sum && !out_distance_sum && !out_hits) return fail(RT1W_ERR_INVALID, "rank 0 needs at least one output");
    std::lock_guard<std::mutex> guard(ctx->lock);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    rt1w_status st;
    if (ctx->members.empty()) {
        st = aov_common(scene, camera, params, stats);
    } else {
        auto prepare = [&](size_t, rt1w_context *, rt1w_scene *sc) {
            rt1w_render_params p;
            int32_t my_samples = 0;
            return aov_prepare(sc, params, p, my_samples);
        };
        auto run = [&](size_t, rt1w_context *, rt1w_scene *sc, rt1w_render_stats *s) { return aov_common(sc, camera, params, s); };
        st = for_each_device(scene, prepare, run, stats);
    }
    if (st != RT1W_OK || !root) return st;
    const size_t pixels = size_t(params->width) * size_t(params->height);
    float *outs[4] = {out_albedo_sum, out_normal_sum, out_distance_sum, out_hits};
    const size_t offset[4] = {0, 3 * pixels, 6 * pixels, 7 * pixels}, count[4] = {3 * pixels, 3 * pixels, pixels, pixels};
    for (int k = 0; k < 4; ++k)
        if (outs[k]) RT1W_CUDA(cudaMemcpyAsync(outs[k], ctx->d_aov + offset[k], sizeof(float) * count[k], cudaMemcpyDeviceToHost, ctx->stream));
    RT1W_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT1W_OK;
}

rt1w_status rt1w_eval_camera_rays(rt1w_scene *scene, const rt1w_camera *camera, const rt1w_render_params *params, const uint32_t *pixel_seed,
                                  const int32_t *sample, size_t n, rt1w_ray *out) {
    if (!scene || !camera || !params || ((!pixel_seed || !sample || !out) && n)) return fail(RT1W_ERR_INVALID, "null argument");
    if (params->width <= 0 || params->height <= 0 || uint64_t(params->width) * uint64_t(params->height) >= (1ull << 31))
        return fail(RT1W_ERR_INVALID, "image size must be positive and below 2^31 pixels");
    const uint64_t pixels = uint64_t(params->width) * uint64_t(params->height);
    for (size_t i = 0; i < n; ++i)
        if (pixel_seed[i] >= pixels || sample[i] < 0) return fail(RT1W_ERR_INVALID, "pixel seed outside the image or negative sample index");
    rt1w_context *ctx = scene->ctx;
    std::lock_guard<std::mutex> guard(ctx->lock);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    rt1w_render_params p = *params;
    p.sample_begin = 0; // the samples are global indices
    const RenderArgs args = render_args(scene, camera, p, 0, 1, uint32_t(pixels), nullptr, nullptr);
    DeviceArena a;
    const uint32_t *d_seed = a.upload(pixel_seed, n, ctx->stream);
    const int32_t *d_sample = a.upload(sample, n, ctx->stream);
    rt1w_ray *d_out = a.alloc<rt1w_ray>(n);
    RT1W_CUDA(a.err);
    RT1W_CUDA(eval_camera_rays_launch(args, d_seed, d_sample, n, d_out, ctx->stream));
    a.download(out, d_out, n, ctx->stream);
    RT1W_CUDA(a.err);
    RT1W_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT1W_OK;
}

rt1w_status rt1w_trace_closest(rt1w_scene *scene, const rt1w_ray *rays, size_t n, uint64_t seed, int32_t *prim_id, float *t, float *normal3,
                               uint8_t *front_face, float *uv2) {
    if (!scene || (!rays && n)) return fail(RT1W_ERR_INVALID, "null argument");
    if (n == 0) return RT1W_OK;
    rt1w_context *ctx = scene->ctx;
    std::lock_guard<std::mutex> guard(ctx->lock);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    struct Buffers {
        rt1w_ray *rays = nullptr;
        int32_t *prim = nullptr;
        float *t = nullptr, *normal = nullptr, *uv = nullptr;
        uint8_t *ff = nullptr;
        ~Buffers() { cudaFree(rays), cudaFree(prim), cudaFree(t), cudaFree(normal), cudaFree(uv), cudaFree(ff); }
    } b;
    RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&b.rays), sizeof(rt1w_ray) * n));
    RT1W_CUDA(cudaMemcpyAsync(b.rays, rays, sizeof(rt1w_ray) * n, cudaMemcpyHostToDevice, ctx->stream));
    if (prim_id) RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&b.prim), sizeof(int32_t) * n));
    if (t) RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&b.t), sizeof(float) * n));
    if (normal3) RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&b.normal), sizeof(float) * 3 * n));
    if (uv2) RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&b.uv), sizeof(float) * 2 * n));
    if (front_face) RT1W_CUDA(cudaMalloc(reinterpret_cast<void **>(&b.ff), n));
    RT1W_CUDA(trace_closest_launch(scene->view, b.rays, n, seed, b.prim, b.t, b.normal, b.ff, b.uv, ctx->stream));
    if (prim_id) RT1W_CUDA(cudaMemcpyAsync(prim_id, b.prim, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (t) RT1W_CUDA(cudaMemcpyAsync(t, b.t, sizeof(float) * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (normal3) RT1W_CUDA(cudaMemcpyAsync(normal3, b.normal, sizeof(float) * 3 * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (uv2) RT1W_CUDA(cudaMemcpyAsync(uv2, b.uv, sizeof(float) * 2 * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (front_face) RT1W_CUDA(cudaMemcpyAsync(front_face, b.ff, n, cudaMemcpyDeviceToHost, ctx->stream));
    RT1W_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT1W_OK;
}

// ---- pointwise parity hooks (tests only) ----
rt1w_status rt1w_eval_light_pdf(rt1w_scene *scene, int32_t light, const double *origin3, const float *dir3, size_t n, float *pdf) {
    if (!scene || ((!origin3 || !dir3 || !pdf) && n)) return fail(RT1W_ERR_INVALID, "null argument");
    if (light >= scene->view.n_lights || (light < 0 && scene->view.n_lights == 0)) return fail(RT1W_ERR_INVALID, "light index out of range");
    rt1w_context *ctx = scene->ctx;
    std::lock_guard<std::mutex> guard(ctx->lock);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    DeviceArena a;
    const double *d_o = a.upload(origin3, 3 * n, ctx->stream);
    const float *d_v = a.upload(dir3, 3 * n, ctx->stream);
    float *d_out = a.alloc<float>(n);
    RT1W_CUDA(a.err);
    RT1W_CUDA(eval_light_pdf_launch(scene->view, light, d_o, d_v, n, d_out, ctx->stream));
    a.download(pdf, d_out, n, ctx->stream);
    RT1W_CUDA(a.err);
    RT1W_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT1W_OK;
}

rt1w_status rt1w_eval_texture(rt1w_scene *scene, int32_t texture, const double *p3, const float *uv2, size_t n, float *rgb3) {
    if (!scene || ((!p3 || !rgb3) && n)) return fail(RT1W_ERR_INVALID, "null argument");
    if (texture < 0 || texture >= scene->n_textures) return fail(RT1W_ERR_INVALID, "texture id out of range");
    rt1w_context *ctx = scene->ctx;
    std::lock_guard<std::mutex> guard(ctx->lock);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    DeviceArena a;
    const double *d_p = a.upload(p3, 3 * n, ctx->stream);
    const float *d_uv = uv2 ? a.upload(uv2, 2 * n, ctx->stream) : nullptr;
    float *d_out = a.alloc<float>(3 * n);
    RT1W_CUDA(a.err);
    RT1W_CUDA(eval_texture_launch(scene->view, texture, 0, 0, d_p, d_uv, n, d_out, ctx->stream));
    a.download(rgb3, d_out, 3 * n, ctx->stream);
    RT1W_CUDA(a.err);
    RT1W_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT1W_OK;
}

rt1w_status rt1w_eval_perlin(rt1w_scene *scene, int32_t table, int32_t turb_depth, const double *p3, size_t n, float *out) {
    if (!scene || ((!p3 || !out) && n)) return fail(RT1W_ERR_INVALID, "null argument");
    if (table < 0 || table >= scene->view.n_perlins || turb_depth < 0) return fail(RT1W_ERR_INVALID, "perlin table id out of range");
    rt1w_context *ctx = scene->ctx;
    std::lock_guard<std::mutex> guard(ctx->lock);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    DeviceArena a;
    const double *d_p = a.upload(p3, 3 * n, ctx->stream);
    float *d_out = a.alloc<float>(n);
    RT1W_CUDA(a.err);
    RT1W_CUDA(eval_texture_launch(scene->view, -1, table, turb_depth, d_p, nullptr, n, d_out, ctx->stream));
    a.download(out, d_out, n, ctx->stream);
    RT1W_CUDA(a.err);
    RT1W_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT1W_OK;
}

rt1w_status rt1w_eval_dielectric(rt1w_context *ctx, const float *unit_dir3, const float *normal3, const float *ratio, size_t n, float *reflect3,
                                 float *refract3, float *reflectance) {
    if (!ctx || ((!unit_dir3 || !normal3 || !ratio) && n)) return fail(RT1W_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> guard(ctx->lock);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    DeviceArena a;
    const float *d_uv = a.upload(unit_dir3, 3 * n, ctx->stream), *d_n = a.upload(normal3, 3 * n, ctx->stream), *d_r = a.upload(ratio, n, ctx->stream);
    float *d_refl = a.alloc<float>(3 * n), *d_refr = a.alloc<float>(3 * n), *d_f = a.alloc<float>(n);
    RT1W_CUDA(a.err);
    RT1W_CUDA(eval_dielectric_launch(d_uv, d_n, d_r, n, d_refl, d_refr, d_f, ctx->stream));
    a.download(reflect3, d_refl, 3 * n, ctx->stream), a.download(refract3, d_refr, 3 * n, ctx->stream), a.download(reflectance, d_f, n, ctx->stream);
    RT1W_CUDA(a.err);
    RT1W_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT1W_OK;
}

rt1w_status rt1w_eval_scatter(rt1w_scene *scene, const rt1w_ray *rays, size_t n, uint64_t seed, int32_t *prim_id, int32_t *material_type, float *dir3,
                              float *weight3, float *time) {
    if (!scene || (!rays && n)) return fail(RT1W_ERR_INVALID, "null argument");
    if (n >= (size_t(1) << 32)) return fail(RT1W_ERR_UNSUPPORTED, "more than 2^32-1 rays in one call");
    rt1w_context *ctx = scene->ctx;
    std::lock_guard<std::mutex> guard(ctx->lock);
    RT1W_CUDA(cudaSetDevice(ctx->device));
    DeviceArena a;
    const rt1w_ray *d_rays = a.upload(rays, n, ctx->stream);
    int32_t *d_prim = a.alloc<int32_t>(n), *d_leaf = a.alloc<int32_t>(n), *d_mat = a.alloc<int32_t>(n);
    double *d_t = a.alloc<double>(n);
    float *d_dir = a.alloc<float>(3 * n), *d_w = a.alloc<float>(3 * n), *d_time = a.alloc<float>(n);
    RT1W_CUDA(a.err);
    RT1W_CUDA(trace_closest_launch(scene->view, d_rays, n, seed, d_prim, nullptr, nullptr, nullptr, nullptr, ctx->stream, d_leaf, d_t));
    RT1W_CUDA(eval_scatter_launch(scene->view, d_rays, d_leaf, d_t, n, seed, d_mat, d_dir, d_w, d_time, ctx->stream));
    a.download(prim_id, d_prim, n, ctx->stream), a.download(material_type, d_mat, n, ctx->stream);
    a.download(dir3, d_dir, 3 * n, ctx->stream), a.download(weight3, d_w, 3 * n, ctx->stream), a.download(time, d_time, n, ctx->stream);
    RT1W_CUDA(a.err);
    RT1W_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT1W_OK;
}

void rt1w_resolve_rgb8(const float *rgb_sum, int32_t width, int32_t height, int32_t samples_per_pixel, uint8_t *out_rgb8) {
    // color.rs:14-21 (NaN sum -> 0, then * 1/spp) and color.rs:56-65 (gamma 2, clamp to [0, 0.999], * 256, truncate)
    const double scale = 1.0 / double(samples_per_pixel);
    const size_t n = size_t(width) * size_t(height) * 3;
    for (size_t i = 0; i < n; ++i) {
        double x = double(rgb_sum[i]);
        if (std::isnan(x)) x = 0.0;
        x *= scale;
        double g = std::sqrt(x);
        g = g < 0.0 ? 0.0 : (g > 0.999 ? 0.999 : g);
        const double q = 256.0 * g;
        out_rgb8[i] = std::isnan(q) ? uint8_t(0) : uint8_t(int(q));
    }
}

void rt1w_philox4x32(const uint32_t counter[4], const uint32_t key[2], uint32_t out[4]) {
    const Philox4 r = philox4x32_10(counter[0], counter[1], counter[2], counter[3], key[0], key[1]);
    out[0] = r.x, out[1] = r.y, out[2] = r.z, out[3] = r.w;
}

} // extern "C"
