// 3DGS-MCMC densification (Kheradmand et al. 2024; gsplat's MCMCStrategy) on the GPU: the opacity-gated position
// noise of every step, and the relocation / sample-add of every refinement.  The draws (torch.multinomial, torch.randn)
// stay with the caller; these kernels turn them into the new rows.
//
// mcmc_noise_kernel: one thread per Gaussian, in place on means3d: mu += scale * sigma(100 ((1 - o) - 0.995)) *
// R S^2 R^T n, S = diag(exp(s)), quaternion normalisation and R as projection.cu.  56 B read, 12 B written.
//
// relocate / add: the sampled indices are counted with integer atomics (mcmc_count_kernel), then every row sampled
// c > 0 times gets its relocated opacity and log-scales once, in double (mcmc_values_kernel).  Relocate then rewrites
// those columns of the sampled rows and copies every dead row from its sampled row, in place (mcmc_relocate_kernel);
// add writes the N + n_add rows of every tensor out of place (mcmc_add_kernel).  No float atomics: the results are
// bit-identical from run to run.
#include "common.cuh"

namespace bsplat {

constexpr int kMcmcThreads = 256;
constexpr int kMcmcRows = 256;    // output rows per add CTA
constexpr int kMcmcUnroll = 4;    // output elements in flight per thread in the add loop
constexpr int kMcmcMaxTensors = 32;
constexpr int kMcmcMaxWidth = 256;
constexpr int kMcmcMaxCopies = 51;  // n = min(c + 1, 51): the size of gsplat's binomial table
static_assert((int64_t)kMcmcRows * kMcmcMaxWidth * kMcmcMaxWidth < (1ll << 32), "magic division is exact");

struct McmcWs {
    int32_t* cnt;    // [N] times each row was sampled
    float* opac;     // [N] relocated opacity, as stored (raw or logit); valid where cnt > 0
    float* scales;   // [N, 3] relocated log-scales; valid where cnt > 0
};

inline size_t mcmc_align(const size_t x) { return (x + 255) & ~(size_t)255; }

inline McmcWs carve_mcmc(void* base, const int64_t N, size_t* bytes) {
    char* p = static_cast<char*>(base);
    size_t off = 0;
    auto take = [&](size_t n) { char* r = p ? p + off : nullptr; off += mcmc_align(n); return r; };
    McmcWs w;
    w.cnt = (int32_t*)take((size_t)N * sizeof(int32_t));
    w.opac = (float*)take((size_t)N * sizeof(float));
    w.scales = (float*)take((size_t)N * 3 * sizeof(float));
    if (bytes) *bytes = off;
    return w;
}

// ---- noise ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kMcmcThreads)
mcmc_noise_kernel(const int64_t N, float* __restrict__ means, const float* __restrict__ log_scales,
                  const float4* __restrict__ quats, const float* __restrict__ opacities, const float* __restrict__ noise,
                  const float scale, const int logits) {
    const int64_t i = (int64_t)blockIdx.x * kMcmcThreads + threadIdx.x;
    if (i >= N) return;
    // the gate in double, rounded once with the scale: 1 - o = sigma(-x) for logits
    const double ov = (double)__ldg(opacities + i);
    const double one_m_o = logits ? 1.0 / (1.0 + exp(ov)) : 1.0 - ov;
    const float gs = (float)((double)scale / (1.0 + exp(-100.0 * (one_m_o - 0.995))));
    if (gs == 0.0f) return;  // (scale = 0: the means stay bit for bit, -0.0 included)
    const float4 q = __ldg(quats + i);  // (w, x, y, z)
    const float nrm = fmaxf(sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w), 1e-12f);
    const float w = q.x / nrm, x = q.y / nrm, y = q.z / nrm, z = q.w / nrm;
    const float R00 = 1.0f - 2.0f * (y * y + z * z), R01 = 2.0f * (x * y - w * z), R02 = 2.0f * (x * z + w * y);
    const float R10 = 2.0f * (x * y + w * z), R11 = 1.0f - 2.0f * (x * x + z * z), R12 = 2.0f * (y * z - w * x);
    const float R20 = 2.0f * (x * z - w * y), R21 = 2.0f * (y * z + w * x), R22 = 1.0f - 2.0f * (x * x + y * y);
    const float v0 = __ldg(noise + 3 * i) * gs, v1 = __ldg(noise + 3 * i + 1) * gs, v2 = __ldg(noise + 3 * i + 2) * gs;
    const float e0 = expf(__ldg(log_scales + 3 * i)), e1 = expf(__ldg(log_scales + 3 * i + 1)),
                e2 = expf(__ldg(log_scales + 3 * i + 2));
    // R (S^2 (R^T v))
    const float t0 = (R00 * v0 + R10 * v1 + R20 * v2) * (e0 * e0);
    const float t1 = (R01 * v0 + R11 * v1 + R21 * v2) * (e1 * e1);
    const float t2 = (R02 * v0 + R12 * v1 + R22 * v2) * (e2 * e2);
    means[3 * i] += R00 * t0 + R01 * t1 + R02 * t2;
    means[3 * i + 1] += R10 * t0 + R11 * t1 + R12 * t2;
    means[3 * i + 2] += R20 * t0 + R21 * t1 + R22 * t2;
}

// ---- relocation values ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kMcmcThreads)
mcmc_count_kernel(const int64_t n, const int64_t* __restrict__ idx, const int64_t N, int32_t* __restrict__ cnt) {
    const int64_t k = (int64_t)blockIdx.x * kMcmcThreads + threadIdx.x;
    if (k >= n) return;
    const int64_t r = __ldg(idx + k);
    BSPLAT_DASSERT(r >= 0 && r < N);
    atomicAdd(cnt + r, 1);
}

// A row sampled c times, n = min(c + 1, 51): o' = clamp(1 - (1 - o)^(1/n), min_opacity, 1 - 2^-23) and
// s' = s + log(o / D), D = sum_{k=0}^{n-1} C(n, k+1) (-1)^k o'^(k+1) / sqrt(k+1) (the hockey-stick form of gsplat's
// double sum).  All in double, rounded once: the alternating sum cancels up to ~5 digits for o near 1.  The binomials
// are exact (every C(n, j) * (n - j) < 2^53 for n <= 51).
__global__ void __launch_bounds__(kMcmcThreads)
mcmc_values_kernel(const int64_t N, const int32_t* __restrict__ cnt, const float* __restrict__ opacities,
                   const float* __restrict__ log_scales, const bsplat_mcmc_params p, float* __restrict__ v_opac,
                   float* __restrict__ v_scales) {
    const int64_t i = (int64_t)blockIdx.x * kMcmcThreads + threadIdx.x;
    if (i >= N) return;
    const int32_t c = __ldg(cnt + i);
    if (c == 0) return;
    const int n = min(c + 1, kMcmcMaxCopies);
    const float ov = __ldg(opacities + i);
    const double o = fmin(p.opacity_logits ? 1.0 / (1.0 + exp(-(double)ov)) : (double)ov, 1.0);
    double op = -expm1(log1p(-o) / n);
    op = fmin(fmax(op, (double)p.min_opacity), 1.0 - 0x1p-23);
    double binom = n, pw = op, D = 0.0;
    for (int k = 0; k < n; ++k) {
        const double term = binom * pw / sqrt((double)(k + 1));
        D += (k & 1) ? -term : term;
        binom = binom * (double)(n - k - 1) / (double)(k + 2);
        pw *= op;
    }
    const double ls = log(o / D);
    v_opac[i] = p.opacity_logits ? (float)log(op / (1.0 - op)) : (float)op;
#pragma unroll
    for (int j = 0; j < 3; ++j) v_scales[3 * i + j] = (float)((double)__ldg(log_scales + 3 * i + j) + ls);
}

// ---- apply ---------------------------------------------------------------------------------------------------------
struct McmcTensor {
    const float* src;
    float* dst;
    int32_t width, role;
    unsigned long long magic;  // ceil(2^32 / width): row = (e * magic) >> 32 for every element offset of an add CTA
};

struct McmcArgs {
    McmcTensor t[kMcmcMaxTensors];
    int32_t n;
};

// In place.  Thread j < N: row j, if sampled, gets its opacity and log-scale columns rewritten and its STATE rows zeroed.
// Thread N + k: dead row dead[k] becomes sampled row sampled[k] with the relocated values, STATE zero.  A dead row is
// never sampled, so no thread reads a row another thread writes.
__global__ void __launch_bounds__(kMcmcThreads)
mcmc_relocate_kernel(const int64_t N, const int64_t n_dead, const int64_t* __restrict__ dead,
                     const int64_t* __restrict__ sampled, const int32_t* __restrict__ cnt,
                     const float* __restrict__ v_opac, const float* __restrict__ v_scales,
                     const __grid_constant__ McmcArgs a) {
    const int64_t j = (int64_t)blockIdx.x * kMcmcThreads + threadIdx.x;
    int64_t row, from;
    if (j < N) {
        if (__ldg(cnt + j) == 0) return;
        row = from = j;
    } else {
        if (j - N >= n_dead) return;
        row = __ldg(dead + (j - N));
        from = __ldg(sampled + (j - N));
        BSPLAT_DASSERT(row >= 0 && row < N && from >= 0 && from < N);
        BSPLAT_DASSERT(__ldg(cnt + row) == 0 && __ldg(cnt + from) > 0);
    }
    for (int t = 0; t < a.n; ++t) {
        const McmcTensor d = a.t[t];
        const int w = d.width;
        float* __restrict__ dst = d.dst + row * w;
        if (d.role == BSPLAT_MCMC_STATE) {
            for (int c = 0; c < w; ++c) dst[c] = 0.0f;
        } else if (d.role == BSPLAT_MCMC_OPACITY) {
            dst[0] = __ldg(v_opac + from);
        } else if (d.role == BSPLAT_MCMC_LOG_SCALES) {
#pragma unroll
            for (int c = 0; c < 3; ++c) dst[c] = __ldg(v_scales + 3 * from + c);
        } else if (row != from) {
            const float* __restrict__ src = d.src + from * w;
            for (int c = 0; c < w; ++c) dst[c] = __ldg(src + c);
        }
    }
}

// Out of place, N + n_add output rows: row r < N is source row r (relocated values where sampled), row N + k the
// updated sampled row sampled[k]; STATE rows r < N are copied, appended STATE rows are zero.  Each CTA streams the
// contiguous output range of its kMcmcRows rows for every tensor: coalesced stores, 64-bit offsets.
__global__ void __launch_bounds__(kMcmcThreads)
mcmc_add_kernel(const int64_t N, const int64_t n_add, const int64_t* __restrict__ sampled,
                const int32_t* __restrict__ cnt, const float* __restrict__ v_opac, const float* __restrict__ v_scales,
                const __grid_constant__ McmcArgs a) {
    __shared__ int64_t s_src[kMcmcRows];
    __shared__ uint8_t s_flag[kMcmcRows];  // bit 0: relocated values, bit 1: appended row
    const int tid = threadIdx.x;
    const int64_t r0 = (int64_t)blockIdx.x * kMcmcRows;
    const int n_rows = (int)min((int64_t)kMcmcRows, N + n_add - r0);
    if (tid < n_rows) {
        const int64_t r = r0 + tid;
        BSPLAT_DASSERT(r < N + n_add);
        if (r < N) {
            s_src[tid] = r;
            s_flag[tid] = __ldg(cnt + r) > 0 ? 1 : 0;
        } else {
            const int64_t s = __ldg(sampled + (r - N));
            BSPLAT_DASSERT(s >= 0 && s < N && __ldg(cnt + s) > 0);
            s_src[tid] = s;
            s_flag[tid] = 3;
        }
    }
    __syncthreads();
    for (int t = 0; t < a.n; ++t) {
        const McmcTensor d = a.t[t];
        const int w = d.width;
        const uint32_t n_el = (uint32_t)n_rows * (uint32_t)w;
        float* __restrict__ dst = d.dst + r0 * w;
        for (uint32_t e0 = tid; e0 < n_el; e0 += kMcmcThreads * kMcmcUnroll) {
            float v[kMcmcUnroll];
#pragma unroll
            for (int u = 0; u < kMcmcUnroll; ++u) {
                const uint32_t e = e0 + u * kMcmcThreads;
                v[u] = 0.0f;
                if (e >= n_el) continue;
                const uint32_t lr = (uint32_t)(((unsigned long long)e * d.magic) >> 32);
                const int col = (int)(e - lr * (uint32_t)w);
                const int64_t s = s_src[lr];
                const uint32_t f = s_flag[lr];
                if (d.role == BSPLAT_MCMC_STATE) {
                    if (!(f & 2u)) v[u] = __ldg(d.src + s * w + col);
                } else if ((f & 1u) && d.role == BSPLAT_MCMC_OPACITY) {
                    v[u] = __ldg(v_opac + s);
                } else if ((f & 1u) && d.role == BSPLAT_MCMC_LOG_SCALES) {
                    v[u] = __ldg(v_scales + 3 * s + col);
                } else {
                    v[u] = __ldg(d.src + s * w + col);
                }
            }
#pragma unroll
            for (int u = 0; u < kMcmcUnroll; ++u) {
                const uint32_t e = e0 + u * kMcmcThreads;
                if (e < n_el) dst[e] = v[u];
            }
        }
    }
}

// Checks shared by relocate and add: the descriptors (1..32, width 1..256, exactly one OPACITY of width 1 and one
// LOG_SCALES of width 3, dst == src in place or dst != src out of place) and the workspace.
int mcmc_prepare(const int64_t N, const bsplat_mcmc_params* params, const int32_t n_tensors,
                 const bsplat_mcmc_tensor* tensors, const bool in_place, void* workspace, const size_t workspace_bytes,
                 size_t* needed_bytes, McmcArgs* a, const float** opac, const float** scales, McmcWs* w) {
    if (N < 0 || N > 0x7fffffffll || !params || n_tensors < 1 || n_tensors > kMcmcMaxTensors || !tensors)
        return BSPLAT_E_ARG;
    a->n = n_tensors;
    int n_opac = 0, n_scales = 0;
    for (int t = 0; t < n_tensors; ++t) {
        const bsplat_mcmc_tensor& d = tensors[t];
        if (d.width < 1 || d.width > kMcmcMaxWidth || d.role < BSPLAT_MCMC_COPY || d.role > BSPLAT_MCMC_STATE)
            return BSPLAT_E_ARG;
        if (!d.src || !d.dst || in_place != ((const float*)d.dst == d.src)) return BSPLAT_E_ARG;
        if (d.role == BSPLAT_MCMC_OPACITY) {
            if (d.width != 1) return BSPLAT_E_ARG;
            *opac = d.src;
            ++n_opac;
        }
        if (d.role == BSPLAT_MCMC_LOG_SCALES) {
            if (d.width != 3) return BSPLAT_E_ARG;
            *scales = d.src;
            ++n_scales;
        }
        a->t[t] = McmcTensor{d.src, d.dst, d.width, d.role,
                             ((1ull << 32) + (unsigned)d.width - 1) / (unsigned)d.width};
    }
    if (n_opac != 1 || n_scales != 1) return BSPLAT_E_ARG;
    size_t need = 0;
    carve_mcmc(nullptr, N, &need);
    if (needed_bytes) *needed_bytes = need;
    if (need > 0 && (!workspace || workspace_bytes < need)) return BSPLAT_E_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(workspace) & 15u) return BSPLAT_E_ARG;
    *w = carve_mcmc(workspace, N, nullptr);
    return BSPLAT_OK;
}

// Counts of `idx` and the relocated values of every sampled row, into the workspace.
int mcmc_values(const int64_t N, const int64_t n, const int64_t* idx, const float* opac, const float* scales,
                const bsplat_mcmc_params& p, const McmcWs& w, cudaStream_t stream) {
    BSPLAT_CUDA_TRY(cudaMemsetAsync(w.cnt, 0, (size_t)N * sizeof(int32_t), stream));
    if (n == 0) return BSPLAT_OK;
    mcmc_count_kernel<<<(unsigned)ceil_div(n, kMcmcThreads), kMcmcThreads, 0, stream>>>(n, idx, N, w.cnt);
    BSPLAT_LAUNCH_CHECK();
    mcmc_values_kernel<<<(unsigned)ceil_div(N, kMcmcThreads), kMcmcThreads, 0, stream>>>(N, w.cnt, opac, scales, p,
                                                                                         w.opac, w.scales);
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}

}  // namespace bsplat

using namespace bsplat;

extern "C" size_t bsplat_mcmc_workspace_bytes(int64_t N) {
    if (N < 0) return 0;
    size_t bytes = 0;
    carve_mcmc(nullptr, N, &bytes);
    return bytes;
}

extern "C" int bsplat_mcmc_noise(int64_t N, float* means3d, const float* log_scales, const float* quats,
                                 const float* opacities, const float* noise, float scale,
                                 const bsplat_mcmc_params* params, void* stream_) {
    if (N < 0 || N > 0x7fffffffll || !params) return BSPLAT_E_ARG;
    if (N == 0) return BSPLAT_OK;
    if (!means3d || !log_scales || !quats || !opacities || !noise) return BSPLAT_E_ARG;
    if (reinterpret_cast<uintptr_t>(quats) & 15u) return BSPLAT_E_ARG;
    mcmc_noise_kernel<<<(unsigned)ceil_div(N, kMcmcThreads), kMcmcThreads, 0, (cudaStream_t)stream_>>>(
        N, means3d, log_scales, reinterpret_cast<const float4*>(quats), opacities, noise, scale,
        params->opacity_logits ? 1 : 0);
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}

extern "C" int bsplat_mcmc_relocate(int64_t N, int64_t n_dead, const int64_t* dead, const int64_t* sampled,
                                    const bsplat_mcmc_params* params, int32_t n_tensors,
                                    const bsplat_mcmc_tensor* tensors, void* workspace, size_t workspace_bytes,
                                    size_t* needed_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    McmcArgs a;
    const float *opac = nullptr, *scales = nullptr;
    McmcWs w;
    const int rc = mcmc_prepare(N, params, n_tensors, tensors, true, workspace, workspace_bytes, needed_bytes, &a,
                                &opac, &scales, &w);
    if (rc != BSPLAT_OK) return rc;
    if (n_dead < 0 || n_dead > N) return BSPLAT_E_ARG;
    if (n_dead == 0) return BSPLAT_OK;
    if (!dead || !sampled) return BSPLAT_E_ARG;
    const int v = mcmc_values(N, n_dead, sampled, opac, scales, *params, w, stream);
    if (v != BSPLAT_OK) return v;
    mcmc_relocate_kernel<<<(unsigned)ceil_div(N + n_dead, kMcmcThreads), kMcmcThreads, 0, stream>>>(
        N, n_dead, dead, sampled, w.cnt, w.opac, w.scales, a);
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}

extern "C" int bsplat_mcmc_add(int64_t N, int64_t n_add, const int64_t* sampled, const bsplat_mcmc_params* params,
                               int32_t n_tensors, const bsplat_mcmc_tensor* tensors, void* workspace,
                               size_t workspace_bytes, size_t* needed_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    McmcArgs a;
    const float *opac = nullptr, *scales = nullptr;
    McmcWs w;
    const int rc = mcmc_prepare(N, params, n_tensors, tensors, false, workspace, workspace_bytes, needed_bytes, &a,
                                &opac, &scales, &w);
    if (rc != BSPLAT_OK) return rc;
    if (n_add < 0 || N + n_add > 0x7fffffffll || (n_add > 0 && N == 0)) return BSPLAT_E_ARG;
    if (n_add > 0 && !sampled) return BSPLAT_E_ARG;
    if (N == 0) return BSPLAT_OK;
    const int v = mcmc_values(N, n_add, sampled, opac, scales, *params, w, stream);
    if (v != BSPLAT_OK) return v;
    mcmc_add_kernel<<<(unsigned)ceil_div(N + n_add, kMcmcRows), kMcmcThreads, 0, stream>>>(
        N, n_add, sampled, w.cnt, w.opac, w.scales, a);
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}
