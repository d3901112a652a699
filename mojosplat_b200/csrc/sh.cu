// Colour stage -- real spherical harmonics (degree 0..3) evaluated along the view direction
// (SURVEY.md 8f rank 4).
//
// The reference only has a placeholder here (mojosplat/render.py:82-87: "SH evaluation not implemented",
// the first three feature channels are used as RGB), so there is no reference arithmetic to restate; this is
// the standard 3D-Gaussian-splatting convention: dir = normalize(mean - camera position),
// colour = max(sum_k Y_k(dir) c_k + 0.5, 0), Y_k the real SH basis with the usual constants, coefficients
// laid out [N, K, 3] with K = (degree_used + 1)^2 <= coefficients stored per Gaussian.  Checked against a float64
// numpy restatement kept with the tests (sh_eval_np).
//
// HBM-bound: 12 B (mean) + 12 K B (coefficients) read + 12 B written per Gaussian.  The [N, K, 3] rows of a
// CTA are one contiguous block: they are copied into shared memory with fully coalesced 128-bit loads and each
// thread then reads its own row (stride 3K words -- odd multiples of 3 are conflict-free, K = 4 / 16 are 2-way).
#include "common.cuh"

namespace bsplat {

constexpr int kShThreads = 128;

__device__ __forceinline__ float3 sh_row(const float* c, int k) { return make_float3(c[3 * k], c[3 * k + 1], c[3 * k + 2]); }

template <int DEG>
__global__ void __launch_bounds__(kShThreads)
sh_eval_kernel(const int64_t N, const int K_stored, const float* __restrict__ coeffs,
               const float* __restrict__ means3d, const float cx, const float cy, const float cz,
               float* __restrict__ colors) {
    extern __shared__ float s_c[];  // [kShThreads][K_stored * 3]
    const int tid = threadIdx.x;
    const int64_t base = (int64_t)blockIdx.x * kShThreads;
    const int n_here = (int)min((int64_t)kShThreads, N - base);
    const int row = K_stored * 3;
    const int64_t words = (int64_t)n_here * row;
    const float* src = coeffs + base * row;
    if ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) {
        const int64_t n4 = words >> 2;
        for (int64_t i = tid; i < n4; i += kShThreads)
            reinterpret_cast<float4*>(s_c)[i] = __ldg(reinterpret_cast<const float4*>(src) + i);
        for (int64_t i = (n4 << 2) + tid; i < words; i += kShThreads) s_c[i] = __ldg(src + i);
    } else {
        for (int64_t i = tid; i < words; i += kShThreads) s_c[i] = __ldg(src + i);
    }
    __syncthreads();
    if (tid >= n_here) return;
    const int64_t g = base + tid;
    const float* c = s_c + tid * row;
    float3 r = sh_row(c, 0);
    const float C0 = 0.28209479177387814f;
    r.x *= C0; r.y *= C0; r.z *= C0;
    if (DEG >= 1) {
        float x = __ldg(means3d + 3 * g) - cx, y = __ldg(means3d + 3 * g + 1) - cy, z = __ldg(means3d + 3 * g + 2) - cz;
        const float inv = rsqrtf(fmaxf(x * x + y * y + z * z, 1e-30f));
        x *= inv; y *= inv; z *= inv;
        const float C1 = 0.4886025119029199f;
        float3 a = sh_row(c, 1), b = sh_row(c, 2), d = sh_row(c, 3);
        r.x += C1 * (-y * a.x + z * b.x - x * d.x);
        r.y += C1 * (-y * a.y + z * b.y - x * d.y);
        r.z += C1 * (-y * a.z + z * b.z - x * d.z);
        if (DEG >= 2) {
            const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
            const float w4 = 1.0925484305920792f * xy, w5 = -1.0925484305920792f * yz,
                        w6 = 0.31539156525252005f * (2.0f * zz - xx - yy), w7 = -1.0925484305920792f * xz,
                        w8 = 0.5462742152960396f * (xx - yy);
            const float wv[5] = {w4, w5, w6, w7, w8};
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const float3 q = sh_row(c, 4 + k);
                r.x += wv[k] * q.x; r.y += wv[k] * q.y; r.z += wv[k] * q.z;
            }
            if (DEG >= 3) {
                const float u[7] = {-0.5900435899266435f * y * (3.0f * xx - yy),
                                    2.890611442640554f * xy * z,
                                    -0.4570457994644658f * y * (4.0f * zz - xx - yy),
                                    0.3731763325901154f * z * (2.0f * zz - 3.0f * xx - 3.0f * yy),
                                    -0.4570457994644658f * x * (4.0f * zz - xx - yy),
                                    1.445305721320277f * z * (xx - yy),
                                    -0.5900435899266435f * x * (xx - 3.0f * yy)};
#pragma unroll
                for (int k = 0; k < 7; ++k) {
                    const float3 q = sh_row(c, 9 + k);
                    r.x += u[k] * q.x; r.y += u[k] * q.y; r.z += u[k] * q.z;
                }
            }
        }
    }
    colors[3 * g] = fmaxf(r.x + 0.5f, 0.0f);
    colors[3 * g + 1] = fmaxf(r.y + 0.5f, 0.0f);
    colors[3 * g + 2] = fmaxf(r.z + 0.5f, 0.0f);
}

// Backward of sh_eval_kernel: v_coeffs [N, K_stored, 3] (bands above DEG written as zeros) and, when v_means3d is not
// null, d loss / d means3d through dir = normalize(mean - campos).  The clamp max(r + 0.5, 0) passes the gradient
// where r + 0.5 >= 0 (torch.clamp(min=0)).  The coefficient rows of a CTA are staged in shared memory as in the
// forward; each thread overwrites its own row with its gradient, and the block is stored with 128-bit stores.
template <int DEG>
__global__ void __launch_bounds__(kShThreads, 8)
sh_bwd_kernel(const int64_t N, const int K_stored, const float* __restrict__ coeffs,
              const float* __restrict__ means3d, const float cx, const float cy, const float cz,
              const float* __restrict__ v_colors, float* __restrict__ v_coeffs, float* __restrict__ v_means3d) {
    extern __shared__ float s_c[];  // [kShThreads][K_stored * 3]
    const int tid = threadIdx.x;
    const int64_t base = (int64_t)blockIdx.x * kShThreads;
    const int n_here = (int)min((int64_t)kShThreads, N - base);
    const int row = K_stored * 3;
    const int64_t words = (int64_t)n_here * row;
    const float* src = coeffs + base * row;
    float* dst = v_coeffs + base * row;
    const bool vec = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0;
    const int64_t n4 = vec ? words >> 2 : 0;
    for (int64_t i = tid; i < n4; i += kShThreads)
        reinterpret_cast<float4*>(s_c)[i] = __ldg(reinterpret_cast<const float4*>(src) + i);
    for (int64_t i = (n4 << 2) + tid; i < words; i += kShThreads) s_c[i] = __ldg(src + i);
    __syncthreads();
    if (tid < n_here) {
        const int64_t g = base + tid;
        float* c = s_c + tid * row;
        constexpr int K = (DEG + 1) * (DEG + 1);
        float Y[K];
        Y[0] = 0.28209479177387814f;
        float x = 0.0f, y = 0.0f, z = 0.0f, inv = 0.0f;
        if (DEG >= 1) {
            x = __ldg(means3d + 3 * g) - cx; y = __ldg(means3d + 3 * g + 1) - cy; z = __ldg(means3d + 3 * g + 2) - cz;
            inv = rsqrtf(fmaxf(x * x + y * y + z * z, 1e-30f));
            x *= inv; y *= inv; z *= inv;
            const float C1 = 0.4886025119029199f;
            Y[1] = -C1 * y; Y[2] = C1 * z; Y[3] = -C1 * x;
        }
        const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
        if (DEG >= 2) {
            Y[4] = 1.0925484305920792f * xy; Y[5] = -1.0925484305920792f * yz;
            Y[6] = 0.31539156525252005f * (2.0f * zz - xx - yy); Y[7] = -1.0925484305920792f * xz;
            Y[8] = 0.5462742152960396f * (xx - yy);
        }
        if (DEG >= 3) {
            Y[9] = -0.5900435899266435f * y * (3.0f * xx - yy);
            Y[10] = 2.890611442640554f * xy * z;
            Y[11] = -0.4570457994644658f * y * (4.0f * zz - xx - yy);
            Y[12] = 0.3731763325901154f * z * (2.0f * zz - 3.0f * xx - 3.0f * yy);
            Y[13] = -0.4570457994644658f * x * (4.0f * zz - xx - yy);
            Y[14] = 1.445305721320277f * z * (xx - yy);
            Y[15] = -0.5900435899266435f * x * (xx - 3.0f * yy);
        }
        float3 r = make_float3(0.0f, 0.0f, 0.0f);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float3 q = sh_row(c, k);
            r.x += Y[k] * q.x; r.y += Y[k] * q.y; r.z += Y[k] * q.z;
        }
        float3 vr = make_float3(__ldg(v_colors + 3 * g), __ldg(v_colors + 3 * g + 1), __ldg(v_colors + 3 * g + 2));
        vr.x = (r.x + 0.5f >= 0.0f) ? vr.x : 0.0f;
        vr.y = (r.y + 0.5f >= 0.0f) ? vr.y : 0.0f;
        vr.z = (r.z + 0.5f >= 0.0f) ? vr.z : 0.0f;
        // g_k = c_k . v_r (for the direction), then the row is overwritten with v_c_k = Y_k v_r
        float gk[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float3 q = sh_row(c, k);
            gk[k] = q.x * vr.x + q.y * vr.y + q.z * vr.z;
            c[3 * k] = Y[k] * vr.x; c[3 * k + 1] = Y[k] * vr.y; c[3 * k + 2] = Y[k] * vr.z;
        }
        for (int k = 3 * K; k < row; ++k) c[k] = 0.0f;
        if (v_means3d != nullptr) {
            float vx = 0.0f, vy = 0.0f, vz = 0.0f;
            if (DEG >= 1) {
                const float C1 = 0.4886025119029199f;
                vx -= C1 * gk[3]; vy -= C1 * gk[1]; vz += C1 * gk[2];
            }
            if (DEG >= 2) {
                const float a = 1.0925484305920792f, b = 0.31539156525252005f, e = 0.5462742152960396f;
                vx += a * y * gk[4] - 2.0f * b * x * gk[6] - a * z * gk[7] + 2.0f * e * x * gk[8];
                vy += a * x * gk[4] - a * z * gk[5] - 2.0f * b * y * gk[6] - 2.0f * e * y * gk[8];
                vz += -a * y * gk[5] + 4.0f * b * z * gk[6] - a * x * gk[7];
            }
            if (DEG >= 3) {
                const float a = 0.5900435899266435f, b = 2.890611442640554f, cc = 0.4570457994644658f,
                            d = 0.3731763325901154f, e = 1.445305721320277f;
                vx += -6.0f * a * xy * gk[9] + b * yz * gk[10] + 2.0f * cc * xy * gk[11] - 6.0f * d * xz * gk[12] -
                      cc * (4.0f * zz - 3.0f * xx - yy) * gk[13] + 2.0f * e * xz * gk[14] - 3.0f * a * (xx - yy) * gk[15];
                vy += -3.0f * a * (xx - yy) * gk[9] + b * xz * gk[10] - cc * (4.0f * zz - xx - 3.0f * yy) * gk[11] -
                      6.0f * d * yz * gk[12] + 2.0f * cc * xy * gk[13] - 2.0f * e * yz * gk[14] + 6.0f * a * xy * gk[15];
                vz += b * xy * gk[10] - 8.0f * cc * yz * gk[11] + d * (6.0f * zz - 3.0f * xx - 3.0f * yy) * gk[12] -
                      8.0f * cc * xz * gk[13] + e * (xx - yy) * gk[14];
            }
            // dir = d / |d|: v_d = (v_dir - dir (dir . v_dir)) / |d|
            const float dp = x * vx + y * vy + z * vz;
            v_means3d[3 * g] = (vx - x * dp) * inv;
            v_means3d[3 * g + 1] = (vy - y * dp) * inv;
            v_means3d[3 * g + 2] = (vz - z * dp) * inv;
        }
    }
    __syncthreads();
    for (int64_t i = tid; i < n4; i += kShThreads) reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(s_c)[i];
    for (int64_t i = (n4 << 2) + tid; i < words; i += kShThreads) dst[i] = s_c[i];
}

}  // namespace bsplat

using namespace bsplat;

// colors[N,3] = max(SH_degree(dir) . coeffs + 0.5, 0).  coeffs is [N, K_stored, 3] with
// K_stored >= (degree + 1)^2 (higher bands are ignored: progressive SH training).
extern "C" int bsplat_sh_eval(int64_t N, int32_t degree, int32_t K_stored, const float* coeffs,
                              const float* means3d, const float* campos_host, float* colors, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (N < 0 || degree < 0 || degree > 3 || K_stored < (degree + 1) * (degree + 1) || K_stored > 64) return BSPLAT_E_ARG;
    if (N == 0) return BSPLAT_OK;
    if (!coeffs || !colors || !campos_host || (degree > 0 && !means3d)) return BSPLAT_E_ARG;
    const unsigned grid = (unsigned)ceil_div(N, kShThreads);
    const size_t smem = (size_t)kShThreads * K_stored * 3 * sizeof(float);
    const float cx = campos_host[0], cy = campos_host[1], cz = campos_host[2];
#define BSPLAT_SH(D)                                                                                          \
    do {                                                                                                      \
        if (smem > 48 * 1024)                                                                                 \
            BSPLAT_CUDA_TRY(cudaFuncSetAttribute(sh_eval_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                                 (int)smem));                                                 \
        sh_eval_kernel<D><<<grid, kShThreads, smem, stream>>>(N, K_stored, coeffs, means3d, cx, cy, cz, colors); \
    } while (0)
    switch (degree) {
        case 0: BSPLAT_SH(0); break;
        case 1: BSPLAT_SH(1); break;
        case 2: BSPLAT_SH(2); break;
        default: BSPLAT_SH(3); break;
    }
#undef BSPLAT_SH
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}

// Backward of bsplat_sh_eval: writes v_coeffs [N, K_stored, 3] and (nullable) v_means3d [N, 3].
extern "C" int bsplat_sh_bwd(int64_t N, int32_t degree, int32_t K_stored, const float* coeffs, const float* means3d,
                             const float* campos_host, const float* v_colors, float* v_coeffs, float* v_means3d,
                             void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (N < 0 || degree < 0 || degree > 3 || K_stored < (degree + 1) * (degree + 1) || K_stored > 64) return BSPLAT_E_ARG;
    if (N == 0) return BSPLAT_OK;
    if (!coeffs || !v_colors || !v_coeffs || !campos_host || (degree > 0 && !means3d)) return BSPLAT_E_ARG;
    const unsigned grid = (unsigned)ceil_div(N, kShThreads);
    const size_t smem = (size_t)kShThreads * K_stored * 3 * sizeof(float);
    const float cx = campos_host[0], cy = campos_host[1], cz = campos_host[2];
#define BSPLAT_SH_BWD(D)                                                                                      \
    do {                                                                                                      \
        if (smem > 48 * 1024)                                                                                 \
            BSPLAT_CUDA_TRY(cudaFuncSetAttribute(sh_bwd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                                 (int)smem));                                                 \
        sh_bwd_kernel<D><<<grid, kShThreads, smem, stream>>>(N, K_stored, coeffs, means3d, cx, cy, cz, v_colors, \
                                                             v_coeffs, v_means3d);                            \
    } while (0)
    switch (degree) {
        case 0: BSPLAT_SH_BWD(0); break;
        case 1: BSPLAT_SH_BWD(1); break;
        case 2: BSPLAT_SH_BWD(2); break;
        default: BSPLAT_SH_BWD(3); break;
    }
#undef BSPLAT_SH_BWD
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}
