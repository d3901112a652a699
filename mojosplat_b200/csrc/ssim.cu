// Photometric training loss: SSIM (3DGS's `ssim`: 11x11 Gaussian window, sigma 1.5, zero padding 5, per-channel,
// C1 = 0.01^2, C2 = 0.03^2) and L1, forward and backward, on (H, W, C) fp32 images.
//
// Forward (ssim_fwd_kernel + ssim_finish_kernel): one CTA per 32x32 pixel tile, the channels one after another.  Per
// channel the tile and its 5-pixel halo (42x42) are staged in shared memory as five planes x, y, x^2, y^2, xy (the
// products computed once per element); a horizontal 11-tap pass writes the five planes of 42x32 row sums to shared
// memory, and a vertical pass gives mu_x, mu_y, E[x^2], E[y^2], E[xy] for the 32x32 outputs.  From them every pixel
// gets S and, when a gradient is wanted, the three maps the backward convolves (A = dS/dmu_x - 2 mu_x dS/dsigma_x^2 -
// mu_y dS/dsigma_xy, B = dS/dsigma_x^2, Cxy = dS/dsigma_xy).  The sums of S and |x - y| go to one fp32 pair per CTA in
// the workspace; ssim_finish_kernel adds them in a fixed order (no floating-point atomics: bit-identical results).
//
// Backward (ssim_bwd_kernel): the same tiling over the three maps, then
//   v_img = g_s / (HWC) (w*A + 2 x (w*B) + y (w*Cxy)) + g_l / (HWC) sign(x - y)
// (the window is symmetric, so the transposed convolution is the same zero-padded convolution).
//
// Register blocking keeps both passes off the shared-memory port: a horizontal item is 8 outputs of one row of one
// plane (18 loads, 88 FMA), a vertical item is 4 outputs of one column of every plane (14 loads per plane, 44 FMA).
#include "common.cuh"

namespace bsplat {

constexpr int kSsimTile = 32;                        // output pixels per CTA side
constexpr int kSsimHalo = 5;
constexpr int kSsimIn = kSsimTile + 2 * kSsimHalo;   // 42 staged rows / columns
constexpr int kSsimStride = 45;                      // staged row stride: odd, so the 8 rows x 4 runs of a
                                                     // horizontal warp fall into 32 different banks
constexpr int kSsimThreads = 256;
constexpr int kSsimHRun = 8;                         // horizontal outputs per item
constexpr int kSsimVRun = 4;                         // vertical outputs per thread (32 columns x 8 runs = 256 threads)
constexpr int kSsimPlane = kSsimIn * kSsimStride;    // staged plane (floats)
constexpr int kSsimHPlane = kSsimIn * kSsimTile;     // horizontal-pass plane (floats)
static_assert(kSsimTile == 32 && kSsimThreads == kSsimTile * (kSsimTile / kSsimVRun), "one vertical item per thread");

constexpr float kSsimC1 = 0.01f * 0.01f;
constexpr float kSsimC2 = 0.03f * 0.03f;

// exp(-(i - 5)^2 / (2 * 1.5^2)) normalised to sum 1 (computed in double, rounded to fp32)
__device__ __forceinline__ float ssim_w(const int t) {
    constexpr float w[11] = {0.001028380123898387f, 0.0075987582094967365f, 0.036000773310661316f,
                             0.10936068743467331f,  0.21300554275512695f,   0.26601171493530273f,
                             0.21300554275512695f,  0.10936068743467331f,   0.036000773310661316f,
                             0.0075987582094967365f, 0.001028380123898387f};
    return w[t];
}

// Stages NQ planes of the 42x42 window around tile (tile_x, tile_y) of channel c; load(e, v) fills v[0..NQ) for the
// in-image element offset e, everything outside the image is zero (the convolution's zero padding).
template <int NQ, typename Load>
__device__ __forceinline__ void ssim_stage(float* __restrict__ s_in, const int H, const int W, const int C, const int c,
                                           const int gx0, const int gy0, Load load) {
    for (int i = threadIdx.x; i < kSsimIn * kSsimIn; i += kSsimThreads) {
        const int r = i / kSsimIn, col = i - r * kSsimIn;
        const int gy = gy0 - kSsimHalo + r, gx = gx0 - kSsimHalo + col;
        float v[NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q) v[q] = 0.0f;
        if (gy >= 0 && gy < H && gx >= 0 && gx < W) load(((int64_t)gy * W + gx) * C + c, v);
        const int s = r * kSsimStride + col;
        BSPLAT_DASSERT(r < kSsimIn && col < kSsimIn && (NQ - 1) * kSsimPlane + s < NQ * kSsimPlane);
#pragma unroll
        for (int q = 0; q < NQ; ++q) s_in[q * kSsimPlane + s] = v[q];
    }
}

// Horizontal 11-tap pass: s_h[q][row][col] = sum_t w[t] s_in[q][row][col + t] for the 42 rows x 32 output columns.
template <int NQ>
__device__ __forceinline__ void ssim_hpass(const float* __restrict__ s_in, float* __restrict__ s_h) {
    constexpr int runs = kSsimTile / kSsimHRun;
    for (int it = threadIdx.x; it < NQ * kSsimIn * runs; it += kSsimThreads) {
        const int run = it % runs, row = (it / runs) % kSsimIn, q = it / (runs * kSsimIn);
        const float* src = s_in + q * kSsimPlane + row * kSsimStride + run * kSsimHRun;
        BSPLAT_DASSERT(run * kSsimHRun + kSsimHRun + 9 < kSsimIn);
        float v[kSsimHRun + 10];
#pragma unroll
        for (int k = 0; k < kSsimHRun + 10; ++k) v[k] = src[k];
        float o[kSsimHRun];
#pragma unroll
        for (int i = 0; i < kSsimHRun; ++i) {
            float a = 0.0f;
#pragma unroll
            for (int t = 0; t < 11; ++t) a = fmaf(ssim_w(t), v[i + t], a);
            o[i] = a;
        }
        float4* dst = reinterpret_cast<float4*>(s_h + q * kSsimHPlane + row * kSsimTile + run * kSsimHRun);
#pragma unroll
        for (int i = 0; i < kSsimHRun / 4; ++i) dst[i] = make_float4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
    }
}

// Vertical 11-tap pass for this thread's column and kSsimVRun rows: out[q][i] at tile row r0 + i.
template <int NQ>
__device__ __forceinline__ void ssim_vpass(const float* __restrict__ s_h, const int col, const int r0,
                                           float (&out)[NQ][kSsimVRun]) {
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        float v[kSsimVRun + 10];
#pragma unroll
        for (int k = 0; k < kSsimVRun + 10; ++k) v[k] = s_h[q * kSsimHPlane + (r0 + k) * kSsimTile + col];
#pragma unroll
        for (int i = 0; i < kSsimVRun; ++i) {
            float a = 0.0f;
#pragma unroll
            for (int t = 0; t < 11; ++t) a = fmaf(ssim_w(t), v[i + t], a);
            out[q][i] = a;
        }
    }
}

__global__ void __launch_bounds__(kSsimThreads)
ssim_fwd_kernel(const int H, const int W, const int C, const int tiles_x, const float* __restrict__ img,
                const float* __restrict__ target, float* __restrict__ maps, float2* __restrict__ partials) {
    extern __shared__ __align__(16) float s_ssim[];
    float* s_h = s_ssim;                      // [5][42][32]
    float* s_in = s_ssim + 5 * kSsimHPlane;   // [5][42][45]: x, y, x^2, y^2, xy
    const int tile = blockIdx.x;
    const int gx0 = (tile % tiles_x) * kSsimTile, gy0 = (tile / tiles_x) * kSsimTile;
    const int col = threadIdx.x & (kSsimTile - 1), r0 = (threadIdx.x / kSsimTile) * kSsimVRun;
    const int64_t HWC = (int64_t)H * W * C;
    float sum_s = 0.0f, sum_l1 = 0.0f;
    for (int c = 0; c < C; ++c) {
        ssim_stage<5>(s_in, H, W, C, c, gx0, gy0, [&](const int64_t e, float (&v)[5]) {
            const float x = __ldg(img + e), y = __ldg(target + e);
            v[0] = x; v[1] = y; v[2] = x * x; v[3] = y * y; v[4] = x * y;
        });
        __syncthreads();
        ssim_hpass<5>(s_in, s_h);
        __syncthreads();
        float m[5][kSsimVRun];
        ssim_vpass<5>(s_h, col, r0, m);
#pragma unroll
        for (int i = 0; i < kSsimVRun; ++i) {
            const int gy = gy0 + r0 + i, gx = gx0 + col;
            if (gy >= H || gx >= W) continue;
            const float mx = m[0][i], my = m[1][i];
            const float sxx = m[2][i] - mx * mx, syy = m[3][i] - my * my, sxy = m[4][i] - mx * my;
            const float a1 = 2.0f * mx * my + kSsimC1, a2 = 2.0f * sxy + kSsimC2;
            const float rb1 = 1.0f / (mx * mx + my * my + kSsimC1), rb2 = 1.0f / (sxx + syy + kSsimC2);
            const float s = a1 * a2 * rb1 * rb2;
            sum_s += s;
            const int si = (r0 + i + kSsimHalo) * kSsimStride + col + kSsimHalo;
            sum_l1 += fabsf(s_in[si] - s_in[kSsimPlane + si]);
            if (maps != nullptr) {
                const float d_mx = 2.0f * my * a2 * rb1 * rb2 - 2.0f * mx * s * rb1;
                const float d_sxx = -s * rb2;
                const float d_sxy = 2.0f * a1 * rb1 * rb2;
                const int64_t e = ((int64_t)gy * W + gx) * C + c;
                maps[e] = d_mx - 2.0f * mx * d_sxx - my * d_sxy;
                maps[HWC + e] = d_sxx;
                maps[2 * HWC + e] = d_sxy;
            }
        }
        __syncthreads();  // the next channel overwrites s_in / s_h
    }
    // fixed-order block reduction (shuffle tree, then the 8 warp sums in order)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sum_s += __shfl_xor_sync(0xffffffffu, sum_s, o);
        sum_l1 += __shfl_xor_sync(0xffffffffu, sum_l1, o);
    }
    __shared__ float2 s_red[kSsimThreads / kWarp];
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = make_float2(sum_s, sum_l1);
    __syncthreads();
    if (threadIdx.x == 0) {
        float2 t = s_red[0];
#pragma unroll
        for (int w = 1; w < kSsimThreads / kWarp; ++w) { t.x += s_red[w].x; t.y += s_red[w].y; }
        partials[tile] = t;
    }
}

// out2 = (sum of the per-CTA pairs) / HWC, added in a fixed order in double precision.
__global__ void __launch_bounds__(kSsimThreads)
ssim_finish_kernel(const float2* __restrict__ partials, const int n, const double inv_n, float* __restrict__ out2) {
    __shared__ double s_a[kSsimThreads], s_b[kSsimThreads];
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < n; i += kSsimThreads) {
        const float2 p = partials[i];
        a += (double)p.x;
        b += (double)p.y;
    }
    s_a[threadIdx.x] = a;
    s_b[threadIdx.x] = b;
    __syncthreads();
    for (int o = kSsimThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            s_a[threadIdx.x] += s_a[threadIdx.x + o];
            s_b[threadIdx.x] += s_b[threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out2[0] = (float)(s_a[0] * inv_n);
        out2[1] = (float)(s_b[0] * inv_n);
    }
}

__global__ void __launch_bounds__(kSsimThreads)
ssim_bwd_kernel(const int H, const int W, const int C, const int tiles_x, const float* __restrict__ img,
                const float* __restrict__ target, const float* __restrict__ maps, const float* __restrict__ v_out2,
                float* __restrict__ v_img) {
    extern __shared__ __align__(16) float s_ssim[];
    float* s_h = s_ssim;                      // [3][42][32]
    float* s_in = s_ssim + 3 * kSsimHPlane;   // [3][42][45]: A, B, Cxy
    const int tile = blockIdx.x;
    const int gx0 = (tile % tiles_x) * kSsimTile, gy0 = (tile / tiles_x) * kSsimTile;
    const int col = threadIdx.x & (kSsimTile - 1), r0 = (threadIdx.x / kSsimTile) * kSsimVRun;
    const int64_t HWC = (int64_t)H * W * C;
    const float g_s = (float)((double)__ldg(v_out2) / (double)HWC);
    const float g_l = (float)((double)__ldg(v_out2 + 1) / (double)HWC);
    for (int c = 0; c < C; ++c) {
        ssim_stage<3>(s_in, H, W, C, c, gx0, gy0, [&](const int64_t e, float (&v)[3]) {
            v[0] = __ldg(maps + e); v[1] = __ldg(maps + HWC + e); v[2] = __ldg(maps + 2 * HWC + e);
        });
        __syncthreads();
        ssim_hpass<3>(s_in, s_h);
        __syncthreads();
        float m[3][kSsimVRun];
        ssim_vpass<3>(s_h, col, r0, m);
#pragma unroll
        for (int i = 0; i < kSsimVRun; ++i) {
            const int gy = gy0 + r0 + i, gx = gx0 + col;
            if (gy >= H || gx >= W) continue;
            const int64_t e = ((int64_t)gy * W + gx) * C + c;
            const float x = __ldg(img + e), y = __ldg(target + e);
            const float d = x - y;
            const float sgn = (float)(d > 0.0f) - (float)(d < 0.0f);
            v_img[e] = g_s * (m[0][i] + 2.0f * x * m[1][i] + y * m[2][i]) + g_l * sgn;
        }
        __syncthreads();
    }
}

constexpr size_t kSsimFwdSmem = (size_t)5 * (kSsimHPlane + kSsimPlane) * sizeof(float);
constexpr size_t kSsimBwdSmem = (size_t)3 * (kSsimHPlane + kSsimPlane) * sizeof(float);

inline bool ssim_dims_ok(const int32_t H, const int32_t W, const int32_t C) {
    return H >= 1 && W >= 1 && C >= 1 && C <= 4;
}

inline int64_t ssim_tiles(const int32_t H, const int32_t W) { return ceil_div(W, kSsimTile) * ceil_div(H, kSsimTile); }

}  // namespace bsplat

using namespace bsplat;

extern "C" size_t bsplat_ssim_workspace_bytes(int32_t H, int32_t W, int32_t C) {
    if (!ssim_dims_ok(H, W, C)) return 0;
    return (size_t)ssim_tiles(H, W) * sizeof(float2);
}

extern "C" int bsplat_ssim_fwd(int32_t H, int32_t W, int32_t C, const float* img, const float* target, float* out2,
                               float* maps, void* workspace, size_t workspace_bytes, size_t* needed_bytes,
                               void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!ssim_dims_ok(H, W, C) || !img || !target || !out2) return BSPLAT_E_ARG;
    const int64_t tiles = ssim_tiles(H, W);
    if (tiles > 0x7fffffff) return BSPLAT_E_ARG;
    const size_t need = bsplat_ssim_workspace_bytes(H, W, C);
    if (needed_bytes) *needed_bytes = need;
    if (!workspace || workspace_bytes < need) return BSPLAT_E_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(workspace) & 7u) return BSPLAT_E_ARG;
    float2* partials = static_cast<float2*>(workspace);
    BSPLAT_CUDA_TRY(cudaFuncSetAttribute(ssim_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)kSsimFwdSmem));
    ssim_fwd_kernel<<<(unsigned)tiles, kSsimThreads, kSsimFwdSmem, stream>>>(
        H, W, C, (int)ceil_div(W, kSsimTile), img, target, maps, partials);
    BSPLAT_LAUNCH_CHECK();
    ssim_finish_kernel<<<1, kSsimThreads, 0, stream>>>(partials, (int)tiles, 1.0 / ((double)H * W * C), out2);
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}

extern "C" int bsplat_ssim_bwd(int32_t H, int32_t W, int32_t C, const float* img, const float* target,
                               const float* maps, const float* v_out2, float* v_img, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!ssim_dims_ok(H, W, C) || !img || !target || !maps || !v_out2 || !v_img) return BSPLAT_E_ARG;
    const int64_t tiles = ssim_tiles(H, W);
    if (tiles > 0x7fffffff) return BSPLAT_E_ARG;
    ssim_bwd_kernel<<<(unsigned)tiles, kSsimThreads, kSsimBwdSmem, stream>>>(
        H, W, C, (int)ceil_div(W, kSsimTile), img, target, maps, v_out2, v_img);
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}
