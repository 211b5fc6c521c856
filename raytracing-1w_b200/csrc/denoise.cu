// denoise.cu — the edge-avoiding à-trous filter of rt1w_denoise / rt1w_render_denoised (include/rt1w.h: the definition):
// the radiance mean is divided by the first-hit albedo, the irradiance is filtered with weights from the normals, the
// distances and the luminance variance of the statistics buffers, and the result is multiplied by the albedo again.
// Three kernels: prepare (sums -> packed per-pixel images), K passes (one thread per pixel, ping-pong between two float4
// images), finish (remodulate).  Every output is a fixed-order sum: no atomics, repeated calls give identical bits.
#include "render.h"

namespace rt1w {
namespace {

constexpr int kTileX = 32, kTileY = 8; // 2-D blocks over a 1-D grid of tiles (the grid's y extent would cap the height)
constexpr float kAlbedoFloor = 1e-3f;
constexpr float kLumR = 0.2126f, kLumG = 0.7152f, kLumB = 0.0722f;
constexpr float kLog2e = 1.4426950408889634f;

struct Tile {
    int x, y;
    bool inside;
};
__device__ __forceinline__ Tile tile_pixel(int width, int height) {
    const int tiles_x = (width + kTileX - 1) / kTileX;
    const int tx = int(blockIdx.x) % tiles_x, ty = int(blockIdx.x) / tiles_x;
    Tile t;
    t.x = tx * kTileX + int(threadIdx.x), t.y = ty * kTileY + int(threadIdx.y);
    t.inside = t.x < width && t.y < height;
    return t;
}

__device__ __forceinline__ float depth_of(const float *__restrict__ aov, size_t pixels, size_t q) {
    const float hits = aov[7 * pixels + q];
    return hits > 0.0f ? aov[6 * pixels + q] / hits : 0.0f;
}

__device__ __forceinline__ float albedo_floored(const float *__restrict__ aov, size_t q, int c, float inv_n) {
    return fmaxf(aov[3 * q + c] * inv_n, kAlbedoFloor);
}

__device__ __forceinline__ float luminance(float4 v) { return kLumR * v.x + kLumG * v.y + kLumB * v.z; }

__device__ __forceinline__ bool normal_zero(float4 g) { return g.x == 0.0f && g.y == 0.0f && g.z == 0.0f; }

// The taps the normal test does not stop: w_n(p, q) > 0.  Both normals zero, or both non-zero and (sigma_n == 0 or N_p.N_q > 0).
__device__ __forceinline__ bool same_surface(float4 gp, bool p_zero, float4 gq, bool sigma_n_zero, float &dot) {
    const bool q_zero = normal_zero(gq);
    dot = gp.x * gq.x + gp.y * gq.y + gp.z * gq.z;
    if (p_zero || q_zero) return p_zero == q_zero;
    return sigma_n_zero || dot > 0.0f;
}

// sums [rgb 3P] [S1 rgb | S2 rgb per pixel: 6P] [albedo 3P | normal 3P | distance P | hits P] -> (I, Var), (N, z), grad z
__global__ void __launch_bounds__(kTileX *kTileY) k_denoise_prepare(const float *__restrict__ rgb_sum, const float *__restrict__ stat, const float *__restrict__ aov,
                                                                    int width, int height, float inv_n, float inv_n1, float4 *__restrict__ img,
                                                                    float4 *__restrict__ guide, float2 *__restrict__ grad) {
    const Tile t = tile_pixel(width, height);
    if (!t.inside) return;
    const size_t pixels = size_t(width) * size_t(height), p = size_t(t.y) * width + t.x;
    const float lum[3] = {kLumR, kLumG, kLumB};
    float irr[3], var = 0.0f;
    for (int c = 0; c < 3; ++c) {
        const float s = rgb_sum[3 * p + c];
        const float color = isfinite(s) ? s * inv_n : 0.0f; // color.rs:16-18 makes a NaN sum black; an infinite one too here
        const float a = albedo_floored(aov, p, c, inv_n);
        irr[c] = color / a;
        const float m = stat[6 * p + c] * inv_n;
        float v = fmaxf(stat[6 * p + 3 + c] * inv_n - m * m, 0.0f) * inv_n1;
        if (!isfinite(v)) v = 0.0f; // an infinite sample (stat_clamp 0) leaves no variance estimate
        const float k = lum[c] / a;
        var += k * k * v;
    }
    const float nx = aov[3 * pixels + 3 * p], ny = aov[3 * pixels + 3 * p + 1], nz = aov[3 * pixels + 3 * p + 2];
    const float nn = nx * nx + ny * ny + nz * nz;
    const float r = nn > 0.0f ? rsqrtf(nn) : 0.0f;
    img[p] = make_float4(irr[0], irr[1], irr[2], var);
    guide[p] = make_float4(nx * r, ny * r, nz * r, depth_of(aov, pixels, p));
    const size_t row = size_t(t.y) * width;
    const int xl = t.x > 0 ? t.x - 1 : 0, xr = t.x + 1 < width ? t.x + 1 : t.x;
    const int yu = t.y > 0 ? t.y - 1 : 0, yd = t.y + 1 < height ? t.y + 1 : t.y;
    grad[p] = make_float2(0.5f * (depth_of(aov, pixels, row + xr) - depth_of(aov, pixels, row + xl)),
                          0.5f * (depth_of(aov, pixels, size_t(yd) * width + t.x) - depth_of(aov, pixels, size_t(yu) * width + t.x)));
}

// One pass at step s: 5x5 taps p + s (i, j), B3 spline h, weight w_n w_z w_l (one exp2 for the three), centre tap w = 1.
__global__ void __launch_bounds__(kTileX *kTileY) k_denoise_pass(const float4 *__restrict__ in, float4 *__restrict__ out, const float4 *__restrict__ guide,
                                                                 const float2 *__restrict__ grad, int width, int height, int step, float sigma_l,
                                                                 float sigma_n, float sigma_z) {
    const Tile t = tile_pixel(width, height);
    if (!t.inside) return;
    const size_t p = size_t(t.y) * width + t.x;
    const float4 gp = guide[p], cp = in[p];
    const float2 dz = grad[p];
    const bool p_zero = normal_zero(gp), sigma_n_zero = sigma_n == 0.0f;
    // g3: the 3x3 binomial blur of the variance over the taps the normal test does not stop, renormalised
    float vsum = 0.0f, vw = 0.0f;
#pragma unroll
    for (int j = -1; j <= 1; ++j) {
        const int qy = t.y + j;
        if (qy < 0 || qy >= height) continue;
#pragma unroll
        for (int i = -1; i <= 1; ++i) {
            const int qx = t.x + i;
            if (qx < 0 || qx >= width) continue;
            const size_t q = size_t(qy) * width + qx;
            float dot;
            if ((i | j) != 0 && !same_surface(gp, p_zero, guide[q], sigma_n_zero, dot)) continue;
            const float k = float((2 - abs(i)) * (2 - abs(j)));
            vsum += k * in[q].w, vw += k;
        }
    }
    const float inv_l = 1.0f / (sigma_l * sqrtf(vsum / vw) + 1e-6f);
    const float lp = luminance(cp), zp = gp.w, z_floor = 1e-3f * zp + 1e-6f;
    const bool pow_normals = !p_zero && !sigma_n_zero;
    const float h1[5] = {1.0f / 16.0f, 4.0f / 16.0f, 6.0f / 16.0f, 4.0f / 16.0f, 1.0f / 16.0f};
    float sr = 0.0f, sg = 0.0f, sb = 0.0f, sw = 0.0f, sv = 0.0f;
#pragma unroll
    for (int j = -2; j <= 2; ++j) {
        const int qy = t.y + step * j;
        if (qy < 0 || qy >= height) continue;
#pragma unroll
        for (int i = -2; i <= 2; ++i) {
            const int qx = t.x + step * i;
            if (qx < 0 || qx >= width) continue;
            const size_t q = size_t(qy) * width + qx;
            const float4 cq = in[q];
            float w = 1.0f;
            if ((i | j) != 0) {
                const float4 gq = guide[q];
                float dot;
                if (!same_surface(gp, p_zero, gq, sigma_n_zero, dot)) continue;
                const float zd = fabsf(zp - gq.w) / (sigma_z * fabsf(dz.x * float(step * i) + dz.y * float(step * j)) + z_floor);
                const float ld = fabsf(lp - luminance(cq)) * inv_l;
                float e = -(zd + ld) * kLog2e;
                if (pow_normals) e += sigma_n * __log2f(dot); // max(0, N_p.N_q)^sigma_n (dot > 0 here)
                w = exp2f(e);
            }
            const float hw = h1[i + 2] * h1[j + 2] * w;
            sr += hw * cq.x, sg += hw * cq.y, sb += hw * cq.z, sw += hw, sv += hw * hw * cq.w;
        }
    }
    const float inv = 1.0f / sw;
    out[p] = make_float4(sr * inv, sg * inv, sb * inv, sv * (inv * inv));
}

// out_rgb = a * I_K (the floored albedo, as prepare computed it)
__global__ void __launch_bounds__(256) k_denoise_finish(const float4 *__restrict__ img, const float *__restrict__ aov, size_t pixels, float inv_n,
                                                         float *__restrict__ out) {
    for (size_t p = size_t(blockIdx.x) * blockDim.x + threadIdx.x; p < pixels; p += size_t(gridDim.x) * blockDim.x) {
        const float4 v = img[p];
        out[3 * p] = albedo_floored(aov, p, 0, inv_n) * v.x;
        out[3 * p + 1] = albedo_floored(aov, p, 1, inv_n) * v.y;
        out[3 * p + 2] = albedo_floored(aov, p, 2, inv_n) * v.z;
    }
}

} // namespace

size_t denoise_scratch_bytes(size_t pixels) { return pixels * (3 * sizeof(float4) + sizeof(float2) + 3 * sizeof(float)); }

cudaError_t denoise_launch(const float *d_rgb_sum, const float *d_stat, const float *d_aov, int width, int height, int n_samples, const rt1w_denoise_params &dp,
                           void *d_scratch, float **d_out_rgb, uint8_t *d_rgb8, uint64_t *launches, cudaStream_t stream) {
    const size_t pixels = size_t(width) * size_t(height);
    float4 *img[2] = {static_cast<float4 *>(d_scratch), static_cast<float4 *>(d_scratch) + pixels};
    float4 *guide = img[1] + pixels;
    float2 *grad = reinterpret_cast<float2 *>(guide + pixels);
    float *out = reinterpret_cast<float *>(grad + pixels);
    const float inv_n = float(1.0 / double(n_samples)), inv_n1 = float(1.0 / double(n_samples - 1));
    const unsigned tiles = unsigned(((width + kTileX - 1) / kTileX) * size_t((height + kTileY - 1) / kTileY));
    const dim3 block(kTileX, kTileY);
    k_denoise_prepare<<<tiles, block, 0, stream>>>(d_rgb_sum, d_stat, d_aov, width, height, inv_n, inv_n1, img[0], guide, grad);
    for (int k = 0; k < dp.iterations; ++k)
        k_denoise_pass<<<tiles, block, 0, stream>>>(img[k & 1], img[(k + 1) & 1], guide, grad, width, height, 1 << k, float(dp.sigma_luminance),
                                                    float(dp.sigma_normal), float(dp.sigma_depth));
    const size_t want = (pixels + 255) / 256;
    k_denoise_finish<<<unsigned(want < 148 * 8 ? want : 148 * 8), 256, 0, stream>>>(img[dp.iterations & 1], d_aov, pixels, inv_n, out);
    *launches = 2 + uint64_t(dp.iterations);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && d_rgb8) { // the arithmetic of rt1w_render_rgb8's resolve, with one sample: out_rgb is already a mean
        e = resolve_launch(out, 3 * pixels, 1, d_rgb8, stream);
        *launches += 1;
    }
    *d_out_rgb = out;
    return e;
}

} // namespace rt1w
