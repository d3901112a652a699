// Adaptive density control (3DGS's densify_and_prune) on the GPU: screen-space gradient statistics, the per-Gaussian
// clone / split / prune decision and one gather pass that writes every parameter and optimizer-state tensor of the
// densified set.
//
// densify_stats_kernel (every training step): one thread per Gaussian; a visible row (max radius > 0) adds the
// NDC-scaled norm of its means2d gradient, one view and its largest radius to the three stat arrays.
//
// densify_plan_kernel + densify_apply_kernel (every densification): the output keeps the input order, each parent
// replaced by 0, 1 or 2 rows, so the rows of any contiguous range of parents form one contiguous range of the output.
// The plan writes one code byte per parent and the per-chunk counts; the CTA that finishes last (ticket) turns the
// chunk counts into exclusive row / split offsets in a fixed order and stores the totals into the caller's
// host-visible counts block (the two-launch compaction of binning2.cu: no look-back, no CTA ever waits for another).
// The apply CTA of a chunk rebuilds the chunk's row map from the codes (block scan) and then streams every tensor's
// contiguous output range: coalesced stores, loads from the chunk's contiguous parent range, no atomics, every output
// element written exactly once.
#include "common.cuh"

namespace bsplat {

constexpr int kDensThreads = 256;
constexpr int kDensItems = 4;                          // consecutive parents per thread (one 32-bit word of codes)
constexpr int kDensChunk = kDensThreads * kDensItems;  // parents per plan / apply CTA
constexpr int kDensMaxRows = 2 * kDensChunk;
constexpr int kDensUnroll = 6;                         // output elements in flight per thread in the apply loop
constexpr int kDensMaxTensors = 32;
constexpr int kDensMaxWidth = 256;
static_assert((int64_t)kDensMaxRows * kDensMaxWidth * kDensMaxWidth < (1ll << 32), "magic division is exact");

// code byte of a parent: the decision (low two bits) and whether its output rows are pruned
constexpr uint32_t kCodeKeep = 0, kCodeClone = 1, kCodeSplit = 2, kCodePruned = 4;
// role of an output row
constexpr uint32_t kRoleSelf = 0, kRoleCopy = 1, kRoleChild0 = 2;

// (float)ln 1.6: a split child's log-scales are the parent's minus this, one fp32 subtraction
constexpr float kLn16 = 0.4700036292457356f;

__device__ __forceinline__ uint32_t code_rows(const uint32_t c) {
    return (c & kCodePruned) ? 0u : ((c & 3u) == kCodeKeep ? 1u : 2u);
}

// max of three with NaN propagation (torch's max): fmaxf would drop a NaN
__device__ __forceinline__ float max3_nan(const float a, const float b, const float c) {
    float m = a;
    m = (b > m || b != b) ? b : m;
    m = (c > m || c != c) ? c : m;
    return m;
}

struct DensWs {
    uint8_t* codes;                 // [n_chunks * kDensChunk]
    uint32_t* counts;               // [n_chunks][4]: output rows, split parents, clone parents, pruned rows
    unsigned long long* offs;       // [n_chunks][2]: exclusive output-row and split-rank offsets
    bsplat_densify_counts* totals;  // the totals, on the device (checked build: bounds of the apply kernel)
    uint32_t* ticket;
};

inline size_t dens_align(const size_t x) { return (x + 255) & ~(size_t)255; }

inline DensWs carve_dens(void* base, const int64_t N, size_t* bytes) {
    const int64_t n_chunks = ceil_div(N, kDensChunk);
    char* p = static_cast<char*>(base);
    size_t off = 0;
    auto take = [&](size_t n) { char* r = p ? p + off : nullptr; off += dens_align(n); return r; };
    DensWs w;
    w.codes = (uint8_t*)take((size_t)n_chunks * kDensChunk);
    w.counts = (uint32_t*)take((size_t)n_chunks * 4 * sizeof(uint32_t));
    w.offs = (unsigned long long*)take((size_t)n_chunks * 2 * sizeof(unsigned long long));
    w.totals = (bsplat_densify_counts*)take(sizeof(bsplat_densify_counts));
    w.ticket = (uint32_t*)take(sizeof(uint32_t));
    if (bytes) *bytes = off;
    return w;
}

// ---- statistics ----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kDensThreads)
densify_stats_kernel(const int64_t N, const float2* __restrict__ v_means2d, const int2* __restrict__ radii,
                     const float half_w, const float half_h, float* __restrict__ grad2d, int32_t* __restrict__ count,
                     int32_t* __restrict__ max_radius) {
    const int64_t i = (int64_t)blockIdx.x * kDensThreads + threadIdx.x;
    if (i >= N) return;
    const int2 r = __ldg(radii + i);
    const int rm = max(r.x, r.y);
    if (rm <= 0) return;
    const float2 g = __ldg(v_means2d + i);
    const float gx = __fmul_rn(g.x, half_w), gy = __fmul_rn(g.y, half_h);
    grad2d[i] = __fadd_rn(grad2d[i], __fsqrt_rn(__fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy))));
    count[i] += 1;
    max_radius[i] = max(max_radius[i], rm);
}

// ---- plan ----------------------------------------------------------------------------------------------------------
// Exclusive scan over the CTA of one value per thread (thread order); returns the exclusive prefix, *total the sum.
__device__ __forceinline__ unsigned long long block_excl_scan(unsigned long long v, unsigned long long* s_warp,
                                                              unsigned long long* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long u = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += u;
    }
    __syncthreads();  // s_warp of a previous scan is consumed
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    unsigned long long run = incl - v, t = 0;
#pragma unroll
    for (int w = 0; w < kDensThreads / 32; ++w) {
        if (w < warp) run += s_warp[w];
        t += s_warp[w];
    }
    *total = t;
    return run;
}

__global__ void __launch_bounds__(kDensThreads)
densify_plan_kernel(const int64_t N, const float* __restrict__ grad2d, const int32_t* __restrict__ count,
                    const int32_t* __restrict__ max_radius, const float* __restrict__ log_scales,
                    const float* __restrict__ opacities, const bsplat_densify_params p, uint32_t* __restrict__ codes,
                    uint32_t* __restrict__ counts, unsigned long long* __restrict__ offs, uint32_t* __restrict__ ticket,
                    bsplat_densify_counts* __restrict__ totals, bsplat_densify_counts* __restrict__ counts_host) {
    __shared__ uint32_t s_cnt[kDensThreads / 32][4];
    __shared__ unsigned long long s_scan[kDensThreads / 32];
    __shared__ bool s_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t base = (int64_t)blockIdx.x * kDensChunk + (int64_t)tid * kDensItems;
    uint32_t word = 0, c_rows = 0, c_split = 0, c_clone = 0, c_pruned = 0;
#pragma unroll
    for (int k = 0; k < kDensItems; ++k) {
        const int64_t i = base + k;
        uint32_t code = kCodePruned;  // (past the end: no rows)
        if (i < N) {
            const int32_t cnt = __ldg(count + i);
            const bool high = cnt > 0 && __fdiv_rn(__ldg(grad2d + i), (float)cnt) >= p.grad_threshold;
            const float smax = max3_nan(__ldg(log_scales + 3 * i), __ldg(log_scales + 3 * i + 1),
                                        __ldg(log_scales + 3 * i + 2));
            code = !high ? kCodeKeep : (smax <= p.log_clone_max_scale ? kCodeClone : kCodeSplit);
            const float row_smax = code == kCodeSplit ? __fsub_rn(smax, kLn16) : smax;
            const bool prune = __ldg(opacities + i) < p.min_opacity || row_smax > p.log_max_world_scale ||
                               __ldg(max_radius + i) > p.max_screen_radius;
            c_split += code == kCodeSplit;
            c_clone += code == kCodeClone;
            const uint32_t rows = code == kCodeKeep ? 1u : 2u;
            if (prune) {
                c_pruned += rows;
                code |= kCodePruned;
            } else {
                c_rows += rows;
            }
        }
        word |= code << (8 * k);
    }
    codes[(int64_t)blockIdx.x * kDensThreads + tid] = word;
    c_rows = __reduce_add_sync(0xffffffffu, c_rows);
    c_split = __reduce_add_sync(0xffffffffu, c_split);
    c_clone = __reduce_add_sync(0xffffffffu, c_clone);
    c_pruned = __reduce_add_sync(0xffffffffu, c_pruned);
    if (lane == 0) {
        s_cnt[warp][0] = c_rows; s_cnt[warp][1] = c_split; s_cnt[warp][2] = c_clone; s_cnt[warp][3] = c_pruned;
    }
    __syncthreads();
    if (tid == 0) {  // (the thread that writes the counts is the one that fences and draws the ticket)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            uint32_t s = 0;
#pragma unroll
            for (int w = 0; w < kDensThreads / 32; ++w) s += s_cnt[w][j];
            counts[(int64_t)blockIdx.x * 4 + j] = s;
        }
        __threadfence();
        s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    // ---- the last CTA: exclusive offsets of the output rows and split ranks, and the totals, in chunk order ----
    __threadfence();
    const int64_t n_chunks = gridDim.x;
    const int64_t per = ceil_div(n_chunks, kDensThreads);
    const int64_t c0 = tid * per;
    unsigned long long sum[4] = {0, 0, 0, 0};
    for (int64_t q = 0; q < per; ++q)
        if (c0 + q < n_chunks)
#pragma unroll
            for (int j = 0; j < 4; ++j) sum[j] += __ldcg(counts + (c0 + q) * 4 + j);
    unsigned long long tot[4];
    unsigned long long run_rows = block_excl_scan(sum[0], s_scan, &tot[0]);
    unsigned long long run_split = block_excl_scan(sum[1], s_scan, &tot[1]);
    block_excl_scan(sum[2], s_scan, &tot[2]);
    block_excl_scan(sum[3], s_scan, &tot[3]);
    for (int64_t q = 0; q < per; ++q)
        if (c0 + q < n_chunks) {
            offs[2 * (c0 + q)] = run_rows;
            offs[2 * (c0 + q) + 1] = run_split;
            run_rows += __ldcg(counts + (c0 + q) * 4);
            run_split += __ldcg(counts + (c0 + q) * 4 + 1);
        }
    if (tid == 0) {
        bsplat_densify_counts t;
        t.n_out = (int64_t)tot[0];
        t.n_split = (int64_t)tot[1];
        t.n_clone = (int64_t)tot[2];
        t.n_pruned = (int64_t)tot[3];
        *totals = t;
        // a direct store into the caller's host-visible block: no copy queued behind other device-to-host traffic
        volatile int64_t* h = reinterpret_cast<volatile int64_t*>(counts_host);
        h[0] = t.n_out; h[1] = t.n_clone; h[2] = t.n_split; h[3] = t.n_pruned;
    }
}

// ---- apply ---------------------------------------------------------------------------------------------------------
struct DensTensor {
    const float* src;
    float* dst;
    int32_t width, role;
    unsigned long long magic;  // ceil(2^32 / width): row = (e * magic) >> 32 for every element offset of a chunk
};

struct DensApplyArgs {
    DensTensor t[kDensMaxTensors];
    int32_t n;
};

// mu + R(q / |q|) (exp(s) * n) for output component `col` of a split child (quaternion (w, x, y, z) and rotation as
// projection.cu; n = the child's noise row).  Out of line: rare, and it would otherwise take registers from the loop.
__device__ __noinline__ float split_mean(const float mu, const int col, const float* __restrict__ q,
                                        const float* __restrict__ s, const float* __restrict__ n) {
    const float q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2), q3 = __ldg(q + 3);
    const float nrm = fmaxf(sqrtf(q0 * q0 + q1 * q1 + q2 * q2 + q3 * q3), 1e-12f);
    const float w = q0 / nrm, x = q1 / nrm, y = q2 / nrm, z = q3 / nrm;
    float r0, r1, r2;
    if (col == 0) {
        r0 = 1.0f - 2.0f * (y * y + z * z); r1 = 2.0f * (x * y - w * z); r2 = 2.0f * (x * z + w * y);
    } else if (col == 1) {
        r0 = 2.0f * (x * y + w * z); r1 = 1.0f - 2.0f * (x * x + z * z); r2 = 2.0f * (y * z - w * x);
    } else {
        r0 = 2.0f * (x * z - w * y); r1 = 2.0f * (y * z + w * x); r2 = 1.0f - 2.0f * (x * x + y * y);
    }
    return mu + (r0 * (expf(__ldg(s)) * __ldg(n)) + r1 * (expf(__ldg(s + 1)) * __ldg(n + 1)) +
                 r2 * (expf(__ldg(s + 2)) * __ldg(n + 2)));
}

__global__ void __launch_bounds__(kDensThreads, 4)
densify_apply_kernel(const uint32_t* __restrict__ codes, const unsigned long long* __restrict__ offs,
                     const bsplat_densify_counts* __restrict__ totals, const float* __restrict__ log_scales,
                     const float* __restrict__ quats, const float* __restrict__ noise,
                     const __grid_constant__ DensApplyArgs a) {
    __shared__ uint32_t s_row[kDensMaxRows];  // output row of the chunk -> split rank << 12 | local parent << 2 | role
    __shared__ unsigned long long s_scan[kDensThreads / 32];
    const int tid = threadIdx.x;
    const int64_t chunk = blockIdx.x;
    const int64_t p0 = chunk * kDensChunk;
    const uint32_t word = __ldg(codes + chunk * kDensThreads + tid);
    uint32_t rows = 0, splits = 0;
#pragma unroll
    for (int k = 0; k < kDensItems; ++k) {
        const uint32_t c = (word >> (8 * k)) & 0xffu;
        rows += code_rows(c);
        splits += (c & 3u) == kCodeSplit;
    }
    unsigned long long n_rows_ll, n_split_ll;
    uint32_t r = (uint32_t)block_excl_scan(rows, s_scan, &n_rows_ll);
    uint32_t rank = (uint32_t)block_excl_scan(splits, s_scan, &n_split_ll);
    const int n_rows = (int)n_rows_ll;
#pragma unroll
    for (int k = 0; k < kDensItems; ++k) {
        const uint32_t c = (word >> (8 * k)) & 0xffu;
        const uint32_t lp = (uint32_t)(tid * kDensItems + k);
        const uint32_t nr = code_rows(c);
        for (uint32_t j = 0; j < nr; ++j) {
            const uint32_t role = (c & 3u) == kCodeSplit ? kRoleChild0 + j : (j == 0 ? kRoleSelf : kRoleCopy);
            BSPLAT_DASSERT(r < (uint32_t)kDensMaxRows);
            s_row[r++] = rank << 12 | lp << 2 | role;
        }
        rank += (c & 3u) == kCodeSplit;
    }
    __syncthreads();
    const unsigned long long o0 = __ldg(offs + 2 * chunk), k0 = __ldg(offs + 2 * chunk + 1);
    BSPLAT_DASSERT(o0 + (unsigned long long)n_rows <= (unsigned long long)totals->n_out);
    for (int t = 0; t < a.n; ++t) {
        const DensTensor d = a.t[t];
        const int w = d.width;
        const uint32_t n_el = (uint32_t)n_rows * (uint32_t)w;
        float* __restrict__ dst = d.dst + (int64_t)o0 * w;
        for (uint32_t e0 = tid; e0 < n_el; e0 += kDensThreads * kDensUnroll) {
            float v[kDensUnroll];
#pragma unroll
            for (int u = 0; u < kDensUnroll; ++u) {
                const uint32_t e = e0 + u * kDensThreads;
                v[u] = 0.0f;
                if (e >= n_el) continue;
                const uint32_t row = (uint32_t)(((unsigned long long)e * d.magic) >> 32);
                const int col = (int)(e - row * (uint32_t)w);
                const uint32_t m = s_row[row];
                const uint32_t role = m & 3u;
                const int64_t parent = p0 + ((m >> 2) & 0x3ffu);
                if (d.role == BSPLAT_DENSIFY_STATE && role != kRoleSelf) continue;  // new rows start with zero moments
                float x = __ldg(d.src + parent * w + col);
                if (role >= kRoleChild0) {
                    if (d.role == BSPLAT_DENSIFY_LOG_SCALES) {
                        x = __fsub_rn(x, kLn16);
                    } else if (d.role == BSPLAT_DENSIFY_MEANS) {
                        const int64_t ks = (int64_t)k0 + (m >> 12);
                        BSPLAT_DASSERT(noise != nullptr && ks < totals->n_split);
                        const float* nz = noise + (ks * 2 + (role - kRoleChild0)) * 3;
                        x = split_mean(x, col, quats + 4 * parent, log_scales + 3 * parent, nz);
                    }
                }
                v[u] = x;
            }
#pragma unroll
            for (int u = 0; u < kDensUnroll; ++u) {
                const uint32_t e = e0 + u * kDensThreads;
                if (e < n_el) dst[e] = v[u];
            }
        }
    }
}

}  // namespace bsplat

using namespace bsplat;

extern "C" size_t bsplat_densify_workspace_bytes(int64_t N) {
    if (N < 0) return 0;
    size_t bytes = 0;
    carve_dens(nullptr, N, &bytes);
    return bytes;
}

extern "C" int bsplat_densify_stats(int64_t N, const float* v_means2d, const int32_t* radii, int32_t width,
                                    int32_t height, float* grad2d, int32_t* count, int32_t* max_radius,
                                    void* stream_) {
    if (N < 0 || N > 0x7fffffffll || width < 1 || height < 1) return BSPLAT_E_ARG;
    if (N == 0) return BSPLAT_OK;
    if (!v_means2d || !radii || !grad2d || !count || !max_radius) return BSPLAT_E_ARG;
    if ((reinterpret_cast<uintptr_t>(v_means2d) | reinterpret_cast<uintptr_t>(radii)) & 7u) return BSPLAT_E_ARG;
    densify_stats_kernel<<<(unsigned)ceil_div(N, kDensThreads), kDensThreads, 0, (cudaStream_t)stream_>>>(
        N, reinterpret_cast<const float2*>(v_means2d), reinterpret_cast<const int2*>(radii), 0.5f * (float)width,
        0.5f * (float)height, grad2d, count, max_radius);
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}

extern "C" int bsplat_densify_plan(int64_t N, const float* grad2d, const int32_t* count, const int32_t* max_radius,
                                   const float* log_scales, const float* opacities,
                                   const bsplat_densify_params* params, void* workspace, size_t workspace_bytes,
                                   size_t* needed_bytes, bsplat_densify_counts* counts_host, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (N < 0 || N > 0x7fffffffll || !params || !counts_host) return BSPLAT_E_ARG;
    size_t need = 0;
    carve_dens(nullptr, N, &need);
    if (needed_bytes) *needed_bytes = need;
    if (N == 0) {
        *counts_host = bsplat_densify_counts{0, 0, 0, 0};
        return BSPLAT_OK;
    }
    if (!grad2d || !count || !max_radius || !log_scales || !opacities) return BSPLAT_E_ARG;
    if (!workspace || workspace_bytes < need) return BSPLAT_E_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(workspace) & 15u) return BSPLAT_E_ARG;
    const DensWs w = carve_dens(workspace, N, nullptr);
    BSPLAT_CUDA_TRY(cudaMemsetAsync(w.ticket, 0, sizeof(uint32_t), stream));
    densify_plan_kernel<<<(unsigned)ceil_div(N, kDensChunk), kDensThreads, 0, stream>>>(
        N, grad2d, count, max_radius, log_scales, opacities, *params, reinterpret_cast<uint32_t*>(w.codes), w.counts,
        w.offs, w.ticket, w.totals, counts_host);
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}

extern "C" int bsplat_densify_apply(int64_t N, const void* workspace, const float* means3d, const float* log_scales,
                                    const float* quats, const float* noise, int32_t n_tensors,
                                    const bsplat_densify_tensor* tensors, void* stream_) {
    if (N < 0 || N > 0x7fffffffll || n_tensors < 1 || n_tensors > kDensMaxTensors || !tensors) return BSPLAT_E_ARG;
    DensApplyArgs a;
    a.n = n_tensors;
    int n_means = 0, n_scales = 0;
    for (int t = 0; t < n_tensors; ++t) {
        const bsplat_densify_tensor& d = tensors[t];
        if (d.width < 1 || d.width > kDensMaxWidth || d.role < BSPLAT_DENSIFY_COPY || d.role > BSPLAT_DENSIFY_STATE)
            return BSPLAT_E_ARG;
        if (N > 0 && (!d.src || !d.dst || (const float*)d.dst == d.src)) return BSPLAT_E_ARG;
        if (d.role == BSPLAT_DENSIFY_MEANS && (d.width != 3 || d.src != means3d)) return BSPLAT_E_ARG;
        if (d.role == BSPLAT_DENSIFY_LOG_SCALES && (d.width != 3 || d.src != log_scales)) return BSPLAT_E_ARG;
        n_means += d.role == BSPLAT_DENSIFY_MEANS;
        n_scales += d.role == BSPLAT_DENSIFY_LOG_SCALES;
        a.t[t] = DensTensor{d.src, d.dst, d.width, d.role, ((1ull << 32) + (unsigned)d.width - 1) / (unsigned)d.width};
    }
    if (n_means != 1 || n_scales != 1) return BSPLAT_E_ARG;
    if (N == 0) return BSPLAT_OK;
    if (!workspace || !means3d || !log_scales || !quats) return BSPLAT_E_ARG;
    if (reinterpret_cast<uintptr_t>(workspace) & 15u) return BSPLAT_E_ARG;
    const DensWs w = carve_dens(const_cast<void*>(workspace), N, nullptr);
    densify_apply_kernel<<<(unsigned)ceil_div(N, kDensChunk), kDensThreads, 0, (cudaStream_t)stream_>>>(
        reinterpret_cast<const uint32_t*>(w.codes), w.offs, w.totals, log_scales, quats, noise, a);
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}
