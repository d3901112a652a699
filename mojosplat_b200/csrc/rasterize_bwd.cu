// Stage 3, training side -- rasterization forward that keeps what the backward pass needs, and the
// backward pass itself (SURVEY.md 8f rank 1; BASELINE.json config 5 asks for it).
//
// The reference is forward-only (`@torch.no_grad`, mojosplat/render.py:11; README.md:145 lists the
// backward pass as future work), so there is no reference implementation to restate: the gradient is
// the derivative of the forward algorithm of mojosplat/kernels/rasterization.mojo:138-162,
//   out = sum_k c_k alpha_k T_k + T_end bg,  T_k = prod_{j<k} (1 - alpha_j),  alpha = min(0.999, o exp(-sigma)),
//   sigma = 0.5 (a dx^2 + c dy^2) + b dx dy,  d = mean - pixel,
// with the skip / stop tests treated as piecewise constant, and it is checked against torch autograd
// (fp64) through a pure-torch restatement of that forward (tests/test_gpu_raster_bwd.py).
//
//   raster_train_fwd_kernel  the faithful forward (same operation order as raster_faithful_kernel) that also
//                            stores, per pixel, the final transmittance and the list index of the last
//                            Gaussian that was composited.
//   Both kernels cull per warp like the fast forward kernel: the 32 lanes test 32 staged Gaussians at once against
//   the bounding box of the warp's pixels with the exact conservative bound (raster_common.cuh) and only the
//   survivors are walked.  A skipped Gaussian has alpha < 1/255 on every pixel of the warp, i.e. it is skipped by
//   the reference arithmetic as well: values and gradients are unchanged.
//   raster_bwd_kernel        one CTA per tile, one pixel per thread, the tile's list walked BACK to front
//                            from the furthest "last index" of the tile, 1 Gaussian staged per thread per
//                            batch; per Gaussian the 6 + C partial gradients are reduced over the warp
//                            (butterfly shuffles, skipped when no lane of the warp contributes) and added
//                            to the per-Gaussian gradient arrays with one atomic per value and warp.
//   Both backward kernels also come with kAbs = true (bsplat_rasterize_bwd[_fast]_abs): per Gaussian they then add the
//   sum over pixels of |d loss_p / d mean| (AbsGS's densification statistic, gsplat's absgrad; the absolute value taken
//   per pixel) into a second [N, 2] array.  kAbs = false is the plain kernel, instruction for instruction.
//   d out / d alpha_k = c_k T_k - (sum_{m>k} c_m alpha_m T_m + T_end bg) / (1 - alpha_k)
//   d alpha / d sigma = -alpha, d alpha / d o = exp(-sigma)        (zero through the 0.999 clamp)
//   d sigma / d(a, b, c) = (0.5 dx^2, dx dy, 0.5 dy^2),  d sigma / d mean = (a dx + b dy, b dx + c dy)
#include "raster_common.cuh"

namespace bsplat {

constexpr float kAlphaMin = 1.0f / 255.0f;

// Thread -> pixel of the tile.  Tile sizes that are multiples of 8 give every warp an 8x4 pixel block (a tighter
// culling box than the 16x2 strip of the row-major order: fewer Gaussians survive the per-warp test); other sizes keep
// the row-major order (threads past ts*ts idle).
__device__ __forceinline__ void tile_pixel_of(const int tid, const int ts, int& lx, int& ly) {
    if ((ts & 7) == 0) {
        const int w = tid >> 5, l = tid & 31, per_row = ts >> 3;
        lx = (w % per_row) * 8 + (l & 7);
        ly = (w / per_row) * 4 + (l >> 3);
    } else {
        ly = tid / ts;
        lx = tid - ly * ts;
    }
}

// Warp reduction of P (4, 8 or 16) values per lane in P + log2(32 / P) shuffles instead of 5 P: at every step a lane
// keeps one half of its values and sends the other half to its partner, so the sums end up SPREAD over the lanes --
// lane L holds the total of value L / (32 / P) in v[0] -- and P lanes can issue their atomics in one instruction
// instead of one lane issuing P.
template <int P>
__device__ __forceinline__ void warp_reduce_spread(float (&v)[P], const unsigned lane) {
    static_assert(P == 4 || P == 8 || P == 16, "4, 8 or 16 values");
    int d = 16;
#pragma unroll
    for (int half = P / 2; half >= 1; half >>= 1, d >>= 1) {
        const bool up = (lane & (unsigned)d) != 0u;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const float send = up ? v[i] : v[i + half];
            const float keep = up ? v[i + half] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, d);
        }
    }
#pragma unroll
    for (; d >= 1; d >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], d);
}

template <int CH>
__global__ void __launch_bounds__(1024)
raster_train_fwd_kernel(const int64_t N, const float* __restrict__ means2d, const float* __restrict__ conics,
                        const float* __restrict__ colors, const float* __restrict__ opacities,
                        const float* __restrict__ background, const int32_t* __restrict__ tile_ranges,
                        const int32_t* __restrict__ sorted_ids, const int W, const int H, const int ts,
                        const int tiles_w, float* __restrict__ image, float* __restrict__ final_T,
                        int32_t* __restrict__ last_idx) {
    extern __shared__ float s_buf[];
    const int nthreads = blockDim.x;  // ts*ts rounded up to a multiple of 32
    float* s_mx = s_buf;
    float* s_my = s_mx + nthreads;
    float* s_a = s_my + nthreads;
    float* s_b = s_a + nthreads;
    float* s_c = s_b + nthreads;
    float* s_o = s_c + nthreads;
    float* s_tau = s_o + nthreads;
    float* s_hy = s_tau + nthreads;
    float* s_hx = s_hy + nthreads;
    float* s_col = s_hx + nthreads;  // [nthreads][CH]

    const int tid = threadIdx.x;
    const unsigned lane = tid & 31u;
    int lx, ly;
    tile_pixel_of(tid, ts, lx, ly);
    const int tile = blockIdx.y * tiles_w + blockIdx.x;
    const int i = blockIdx.y * ts + ly;
    const int j = blockIdx.x * ts + lx;
    const bool inside = (ly < ts) && (i < H) && (j < W);
    bool done = !inside;
    const float px = (float)j + 0.5f, py = (float)i + 0.5f;
    // bounding box of this warp's pixels (any tile size: a warp is not always a rectangle of the tile)
    float X0 = inside ? px : INFINITY, X1 = inside ? px : -INFINITY;
    float Y0 = inside ? py : INFINITY, Y1 = inside ? py : -INFINITY;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        X0 = fminf(X0, __shfl_xor_sync(0xffffffffu, X0, d)); X1 = fmaxf(X1, __shfl_xor_sync(0xffffffffu, X1, d));
        Y0 = fminf(Y0, __shfl_xor_sync(0xffffffffu, Y0, d)); Y1 = fmaxf(Y1, __shfl_xor_sync(0xffffffffu, Y1, d));
    }

    const int32_t r0 = tile_ranges[2 * tile], r1 = tile_ranges[2 * tile + 1];
    float T = 1.0f;
    float acc[CH];
#pragma unroll
    for (int c = 0; c < CH; ++c) acc[c] = 0.0f;
    int32_t last = -1;

    for (int32_t b0 = r0; b0 < r1; b0 += nthreads) {
        if (__syncthreads_count(done) >= nthreads) break;
        const int32_t idx = b0 + tid;
        if (idx < r1) {
            const int32_t g = sorted_ids[idx];
            if (g >= 0 && (int64_t)g < N) {
                s_mx[tid] = means2d[2 * (int64_t)g];
                s_my[tid] = means2d[2 * (int64_t)g + 1];
                s_a[tid] = conics[3 * (int64_t)g];
                s_b[tid] = conics[3 * (int64_t)g + 1];
                s_c[tid] = conics[3 * (int64_t)g + 2];
                s_o[tid] = opacities[g];
                cull_constants(s_a[tid], s_b[tid], s_c[tid], s_o[tid], s_tau[tid], s_hy[tid], s_hx[tid]);
#pragma unroll
                for (int c = 0; c < CH; ++c) s_col[tid * CH + c] = colors[(int64_t)g * CH + c];
            } else {
                s_mx[tid] = s_my[tid] = s_a[tid] = s_b[tid] = s_c[tid] = 0.0f;
                s_o[tid] = __int_as_float(0x7fc00000);  // NaN marks "not a Gaussian"
                s_tau[tid] = -INFINITY; s_hy[tid] = s_hx[tid] = 0.0f;
            }
        }
        __syncthreads();
        const int bs = min(nthreads, (int)(r1 - b0));
        for (int c0 = 0; c0 < bs; c0 += 32) {  // warp-uniform
            if (__all_sync(0xffffffffu, done)) break;
            const int e = c0 + (int)lane;
            bool hit = false;
            if (e < bs && X0 <= X1)
                hit = pair_cull_hit(s_mx[e], s_my[e], 0.5f * kLog2e * s_a[e], kLog2e * s_b[e], 0.5f * kLog2e * s_c[e],
                                    s_tau[e], s_hy[e], s_hx[e], X0, X1, Y0, Y1);
            unsigned mask = __ballot_sync(0xffffffffu, hit);
            while (mask && !done) {
                const int t = c0 + __ffs(mask) - 1;
                mask &= mask - 1;
                const float op = s_o[t];
                if (op != op) continue;
                const float dx = __fsub_rn(s_mx[t], px), dy = __fsub_rn(s_my[t], py);
                const float a = s_a[t], b = s_b[t], c = s_c[t];
                const float q = __fadd_rn(__fmul_rn(__fmul_rn(a, dx), dx), __fmul_rn(__fmul_rn(c, dy), dy));
                const float sigma = __fadd_rn(__fmul_rn(0.5f, q), __fmul_rn(__fmul_rn(b, dx), dy));
                float alpha = __fmul_rn(op, expf(-sigma));
                alpha = fminf(alpha, 0.999f);
                if (sigma < 0.0f || alpha < kAlphaMin) continue;
                const float next_T = __fmul_rn(T, __fsub_rn(1.0f, alpha));
                if (next_T <= 1e-4f) { done = true; break; }
                const float vis = __fmul_rn(alpha, T);
#pragma unroll
                for (int ch = 0; ch < CH; ++ch) acc[ch] = __fadd_rn(acc[ch], __fmul_rn(s_col[t * CH + ch], vis));
                T = next_T;
                last = b0 + t;
            }
        }
    }
    if (inside) {
        const int64_t pix = (int64_t)i * W + j;
#pragma unroll
        for (int ch = 0; ch < CH; ++ch) image[pix * CH + ch] = __fadd_rn(acc[ch], __fmul_rn(T, background[ch]));
        final_T[pix] = T;
        last_idx[pix] = last;
    }
}

template <int CH, bool kAbs>
__global__ void __launch_bounds__(1024)
raster_bwd_kernel(const int64_t N, const float* __restrict__ means2d, const float* __restrict__ conics,
                  const float* __restrict__ colors, const float* __restrict__ opacities,
                  const float* __restrict__ background, const int32_t* __restrict__ tile_ranges,
                  const int32_t* __restrict__ sorted_ids, const int W, const int H, const int ts,
                  const int tiles_w, const float* __restrict__ final_T, const int32_t* __restrict__ last_idx,
                  const float* __restrict__ grad_image, float* __restrict__ g_means2d,
                  float* __restrict__ g_conics, float* __restrict__ g_colors, float* __restrict__ g_opac,
                  float* __restrict__ g_means2d_abs) {
    extern __shared__ float s_buf[];
    const int nthreads = blockDim.x;
    float* s_mx = s_buf;
    float* s_my = s_mx + nthreads;
    float* s_a = s_my + nthreads;
    float* s_b = s_a + nthreads;
    float* s_c = s_b + nthreads;
    float* s_o = s_c + nthreads;
    float* s_tau = s_o + nthreads;
    float* s_hy = s_tau + nthreads;
    float* s_hx = s_hy + nthreads;
    float* s_col = s_hx + nthreads;                                 // [nthreads][CH]
    int32_t* s_id = reinterpret_cast<int32_t*>(s_col + nthreads * CH);  // [nthreads]
    __shared__ int s_max_last;

    const int tid = threadIdx.x;
    const unsigned lane = tid & 31u;
    int lx, ly;
    tile_pixel_of(tid, ts, lx, ly);
    const int tile = blockIdx.y * tiles_w + blockIdx.x;
    const int i = blockIdx.y * ts + ly;
    const int j = blockIdx.x * ts + lx;
    const bool inside = (ly < ts) && (i < H) && (j < W);
    const float px = (float)j + 0.5f, py = (float)i + 0.5f;
    const int32_t r0 = tile_ranges[2 * tile];
    // bounding box of this warp's pixels
    float X0 = inside ? px : INFINITY, X1 = inside ? px : -INFINITY;
    float Y0 = inside ? py : INFINITY, Y1 = inside ? py : -INFINITY;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        X0 = fminf(X0, __shfl_xor_sync(0xffffffffu, X0, d)); X1 = fmaxf(X1, __shfl_xor_sync(0xffffffffu, X1, d));
        Y0 = fminf(Y0, __shfl_xor_sync(0xffffffffu, Y0, d)); Y1 = fmaxf(Y1, __shfl_xor_sync(0xffffffffu, Y1, d));
    }

    const int64_t pix = (int64_t)i * W + j;
    const float T_final = inside ? final_T[pix] : 0.0f;
    const int32_t last = inside ? last_idx[pix] : -1;
    float gout[CH], buffer[CH];
    float bg_dot = 0.0f;  // sum_ch bg_ch * dL/dout_ch
#pragma unroll
    for (int ch = 0; ch < CH; ++ch) {
        gout[ch] = inside ? grad_image[pix * CH + ch] : 0.0f;
        buffer[ch] = 0.0f;
        bg_dot += background[ch] * gout[ch];
    }
    float T = T_final;

    if (tid == 0) s_max_last = -1;
    __syncthreads();
    if (last >= 0) atomicMax(&s_max_last, last);
    __syncthreads();
    const int32_t hi_all = s_max_last;  // furthest composited entry of the tile
    if (hi_all < r0) return;

    for (int32_t hi = hi_all; hi >= r0; hi -= nthreads) {
        __syncthreads();  // previous batch fully consumed
        const int32_t idx = hi - tid;  // staged back to front: slot t holds entry hi - t
        if (idx >= r0) {
            const int32_t g = sorted_ids[idx];
            s_id[tid] = g;
            if (g >= 0 && (int64_t)g < N) {
                s_mx[tid] = means2d[2 * (int64_t)g];
                s_my[tid] = means2d[2 * (int64_t)g + 1];
                s_a[tid] = conics[3 * (int64_t)g];
                s_b[tid] = conics[3 * (int64_t)g + 1];
                s_c[tid] = conics[3 * (int64_t)g + 2];
                s_o[tid] = opacities[g];
                cull_constants(s_a[tid], s_b[tid], s_c[tid], s_o[tid], s_tau[tid], s_hy[tid], s_hx[tid]);
#pragma unroll
                for (int c = 0; c < CH; ++c) s_col[tid * CH + c] = colors[(int64_t)g * CH + c];
            } else {
                s_mx[tid] = s_my[tid] = s_a[tid] = s_b[tid] = s_c[tid] = 0.0f;
                s_o[tid] = __int_as_float(0x7fc00000);
                s_tau[tid] = -INFINITY; s_hy[tid] = s_hx[tid] = 0.0f;
            }
        }
        __syncthreads();
        const int bs = min(nthreads, (int)(hi - r0 + 1));
        // the furthest composited entry of THIS warp: slots in front of it are skipped without a test
        int warp_last = last;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) warp_last = max(warp_last, __shfl_xor_sync(0xffffffffu, warp_last, d));
        for (int c0 = 0; c0 < bs; c0 += 32) {  // warp-uniform; slot t holds entry hi - t (back to front)
          const int e = c0 + (int)lane;
          bool hit = false;
          if (e < bs && hi - e <= warp_last)
              hit = pair_cull_hit(s_mx[e], s_my[e], 0.5f * kLog2e * s_a[e], kLog2e * s_b[e], 0.5f * kLog2e * s_c[e],
                                  s_tau[e], s_hy[e], s_hx[e], X0, X1, Y0, Y1);
          unsigned mask = __ballot_sync(0xffffffffu, hit);
          while (mask) {  // warp-uniform: every lane walks the same survivors (shuffles below need all lanes)
            const int t = c0 + __ffs(mask) - 1;
            mask &= mask - 1;
            const float op = s_o[t];
            if (op != op) continue;  // uniform across the warp
            bool valid = inside && (hi - t <= last);
            float dx = 0.f, dy = 0.f, alpha = 0.f, vis = 0.f;
            const float a = s_a[t], b = s_b[t], c = s_c[t];
            if (valid) {
                dx = __fsub_rn(s_mx[t], px); dy = __fsub_rn(s_my[t], py);
                const float q = __fadd_rn(__fmul_rn(__fmul_rn(a, dx), dx), __fmul_rn(__fmul_rn(c, dy), dy));
                const float sigma = __fadd_rn(__fmul_rn(0.5f, q), __fmul_rn(__fmul_rn(b, dx), dy));
                vis = expf(-sigma);
                alpha = fminf(__fmul_rn(op, vis), 0.999f);
                if (sigma < 0.0f || alpha < kAlphaMin) valid = false;
            }
            if (!__any_sync(0xffffffffu, valid)) continue;  // nothing to reduce for this warp
            float v_rgb[CH];
            float v_ca = 0.f, v_cb = 0.f, v_cc = 0.f, v_mx = 0.f, v_my = 0.f, v_op = 0.f, v_ax = 0.f, v_ay = 0.f;
#pragma unroll
            for (int ch = 0; ch < CH; ++ch) v_rgb[ch] = 0.f;
            if (valid) {
                const float ra = 1.0f / (1.0f - alpha);
                T *= ra;  // transmittance in front of this Gaussian
                const float fac = alpha * T;
                float v_alpha = 0.0f;
#pragma unroll
                for (int ch = 0; ch < CH; ++ch) {
                    const float col = s_col[t * CH + ch];
                    v_rgb[ch] = fac * gout[ch];
                    v_alpha += (col * T - buffer[ch] * ra) * gout[ch];
                    buffer[ch] += col * fac;
                }
                v_alpha += -T_final * ra * bg_dot;
                if (op * vis <= 0.999f) {  // no gradient through the clamp
                    const float v_sigma = -op * vis * v_alpha;
                    v_ca = 0.5f * v_sigma * dx * dx;
                    v_cb = v_sigma * dx * dy;
                    v_cc = 0.5f * v_sigma * dy * dy;
                    v_mx = v_sigma * (a * dx + b * dy);
                    v_my = v_sigma * (b * dx + c * dy);
                    v_op = vis * v_alpha;
                    if constexpr (kAbs) { v_ax = fabsf(v_mx); v_ay = fabsf(v_my); }  // |.| of this pixel's term
                }
            }
            // spread reduction: lane L ends up with the total of value L >> kShift (colours first, then conic a, b,
            // c, mean x, y, opacity[, |mean x|, |mean y|]), and those lanes add it to the gradient arrays in one atomic
            // instruction
            constexpr int kVals = CH + (kAbs ? 8 : 6), P = kVals <= 8 ? 8 : 16, kShift = P == 16 ? 1 : 2;
            float v[P];
#pragma unroll
            for (int q = 0; q < P; ++q) v[q] = 0.0f;
#pragma unroll
            for (int ch = 0; ch < CH; ++ch) v[ch] = v_rgb[ch];
            v[CH] = v_ca; v[CH + 1] = v_cb; v[CH + 2] = v_cc; v[CH + 3] = v_mx; v[CH + 4] = v_my; v[CH + 5] = v_op;
            if constexpr (kAbs) { v[CH + 6] = v_ax; v[CH + 7] = v_ay; }
            warp_reduce_spread<P>(v, lane);
            const int which = (int)(lane >> kShift);
            if ((lane & ((1u << kShift) - 1u)) == 0u && which < kVals) {
                const int64_t g = s_id[t];
                float* dst;
                if (which < CH) dst = g_colors + g * CH + which;
                else if (which < CH + 3) dst = g_conics + 3 * g + (which - CH);
                else if (which < CH + 5) dst = g_means2d + 2 * g + (which - CH - 3);
                else if (!kAbs || which == CH + 5) dst = g_opac + g;
                else dst = g_means2d_abs + 2 * g + (which - CH - 6);
                atomicAdd(dst, v[0]);
            }
          }
        }
    }
}


// ------------------------------------------------------------------------------------------
// Backward in the layout of the fast forward kernel (16x16 tiles, RGB): 128 threads per tile, one warp per 8x8 pixel
// block, TWO pixels per lane ((x, y) and (x, y + 4)), the 48-byte records of raster_common.cuh staged back to front,
// per-warp culling with the exact conservative bound, packed FP32 pairs for the per-pixel arithmetic.  What makes it
// ~3x leaner than raster_bwd_kernel per (Gaussian, pixel):
//   * alpha = 2^(L - q) from the log2-folded record (one MUFU.EX2, as in the forward walk), 1 / (1 - alpha) from
//     MUFU.RCP; a pixel that fails a test gets alpha = 0, after which every term below is an exact zero -- no branches;
//   * only nine sums leave a lane -- sum v_sigma {dx^2, dx dy, dy^2, dx, dy, 1} and sum alpha T gout_{r,g,b} -- and the
//     two pixels of a lane are added before the warp reduction, so a reduction serves 64 pixels instead of 32; the
//     per-Gaussian factors (a, b, c in the mean gradient, 1 / opacity, the 0.5 of the conic gradient) are applied once
//     per Gaussian by the lanes that issue the atomics.
// d alpha / d sigma = -alpha (zero through the 0.999 clamp), sigma = q / log2e:
//   d sigma / d(a, b, c) = (dx^2 / 2, dx dy, dy^2 / 2),  d sigma / d mean = (a dx + b dy, b dx + c dy),
//   d alpha / d opacity = alpha / opacity.
constexpr int kBwdThreads = 128;
constexpr int kBwdBatch = 128;

__device__ __forceinline__ float ex2_approx_b(const float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx_b(const float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float2 dupb(const float v) { return make_float2(v, v); }

template <bool kAbs>
__global__ void __launch_bounds__(kBwdThreads)
raster_bwd_pair_kernel(const int64_t N, const float4* __restrict__ rec, const float* __restrict__ background,
                       const int32_t* __restrict__ tile_ranges, const int32_t* __restrict__ tile_order,
                       const int32_t* __restrict__ sorted_ids, const int W, const int H, const int tiles_w,
                       const float* __restrict__ final_T, const int32_t* __restrict__ last_idx,
                       const float* __restrict__ grad_image, float* __restrict__ g_means2d,
                       float* __restrict__ g_conics, float* __restrict__ g_colors, float* __restrict__ g_opac,
                       float* __restrict__ g_means2d_abs) {
    __shared__ float4 s_rec[2 * kBwdBatch * kPairRec];
    __shared__ int32_t s_id[2 * kBwdBatch];
    __shared__ int s_max_last;
    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int tile = tile_order ? __ldg(tile_order + blockIdx.x) : (int)blockIdx.x;
    const int tile_y = tile / tiles_w, tile_x = tile - tile_y * tiles_w;
    const int bx = tile_x * 16 + (warp & 1) * 8, by = tile_y * 16 + (warp >> 1) * 8;
    const int j = bx + (lane & 7);
    const int i0 = by + (lane >> 3), i1 = i0 + 4;
    const bool in0 = (i0 < H) && (j < W), in1 = (i1 < H) && (j < W);
    const float px = (float)j + 0.5f;
    const float2 npy = make_float2(-((float)i0 + 0.5f), -((float)i1 + 0.5f));
    const float X0 = (float)bx + 0.5f, X1 = (float)bx + 7.5f;
    const float Y0 = (float)by + 0.5f, Y1 = (float)by + 7.5f;
    const int32_t r0 = tile_ranges[2 * tile];

    const int64_t pix0 = (int64_t)i0 * W + j, pix1 = (int64_t)i1 * W + j;
    const int32_t last0 = in0 ? last_idx[pix0] : -1, last1 = in1 ? last_idx[pix1] : -1;
    float2 T2 = make_float2(in0 ? final_T[pix0] : 0.0f, in1 ? final_T[pix1] : 0.0f);
    float2 go_r, go_g, go_b;
    go_r.x = in0 ? grad_image[pix0 * 3] : 0.0f; go_g.x = in0 ? grad_image[pix0 * 3 + 1] : 0.0f;
    go_b.x = in0 ? grad_image[pix0 * 3 + 2] : 0.0f;
    go_r.y = in1 ? grad_image[pix1 * 3] : 0.0f; go_g.y = in1 ? grad_image[pix1 * 3 + 1] : 0.0f;
    go_b.y = in1 ? grad_image[pix1 * 3 + 2] : 0.0f;
    const float bgr = __ldg(background), bgg = __ldg(background + 1), bgb = __ldg(background + 2);
    // -T_final * sum_ch bg_ch gout_ch: the background's share of d out / d alpha, up to the factor 1 / (1 - alpha)
    const float2 ntfbg = make_float2(-T2.x * (bgr * go_r.x + bgg * go_g.x + bgb * go_b.x),
                                     -T2.y * (bgr * go_r.y + bgg * go_g.y + bgb * go_b.y));
    float2 behind = make_float2(-ntfbg.x, -ntfbg.y);  // (sum over the Gaussians behind: c alpha T) . gout + T_final bg . gout

    const uint32_t s_rec_addr = (uint32_t)__cvta_generic_to_shared(s_rec);
    const uint32_t s_id_addr = (uint32_t)__cvta_generic_to_shared(s_id);
    if (tid == 0) s_max_last = -1;
    __syncthreads();
    int warp_last = max(last0, last1);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) warp_last = max(warp_last, __shfl_xor_sync(0xffffffffu, warp_last, d));
    if (lane == 0 && warp_last >= 0) atomicMax(&s_max_last, warp_last);
    __syncthreads();
    const int32_t hi_all = s_max_last;  // furthest entry any pixel of the tile looked at
    if (hi_all < r0) return;

    // this thread's record of a batch goes into the other half of the staging ring with cp.async, one batch ahead of
    // the walk (slot t of batch `hi` holds entry hi - t)
    auto fetch = [&](const int32_t hi, const int half) {
        const int32_t idx = hi - tid;
        int32_t g = -1;
        if (idx >= r0) g = __ldg(sorted_ids + idx);
        float4* dst = s_rec + (half * kBwdBatch + tid) * kPairRec;
        if (g >= 0 && (int64_t)g < N) {
            const float4* src = rec + kPairRec * (int64_t)g;
#pragma unroll
            for (int q = 0; q < kPairRec; ++q) {
                const unsigned int d = (unsigned int)__cvta_generic_to_shared(dst + q);
                asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src + q) : "memory");
            }
        } else {
            g = -1;
            pair_record_none(dst[0], dst[1], dst[2]);
        }
        s_id[half * kBwdBatch + tid] = g;
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // loop-invariant roles of the lanes that issue the atomics: lane 4 k adds value k of the spread reduction (colours,
    // conic a b c, mean x y), lane 1 the opacity gradient[, lanes 9 and 17 the absolute mean gradient x and y] -- one
    // predicated RED instruction per Gaussian and warp
    const int which = lane >> 2;
    const bool role_mean = which >= 6, role_my = which == 7, role_op = lane == 1;
    const bool role_abs = kAbs && (lane == 9 || lane == 17);
    const bool issues = ((lane & 3) == 0) || role_op || role_abs;
    float* role_base;
    int role_stride;
    float role_scale = 1.0f;
    if (role_op) { role_base = g_opac; role_stride = 1; }
    else if (role_abs) { role_base = g_means2d_abs + (lane >> 4); role_stride = 2; }
    else if (which < 3) { role_base = g_colors + which; role_stride = 3; }
    else if (which < 6) { role_base = g_conics + (which - 3); role_stride = 3; role_scale = (which == 4) ? 1.0f : 0.5f; }
    else { role_base = g_means2d + (which - 6); role_stride = 2; }

    fetch(hi_all, 0);
    int half = 0;
    for (int32_t hi = hi_all; hi >= r0; hi -= kBwdBatch, half ^= 1) {
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncthreads();  // this batch has landed; everyone is done with the other half
        if (hi - kBwdBatch >= r0) fetch(hi - kBwdBatch, half ^ 1);  // in flight during the walk below
        const float4* s_cur = s_rec + half * kBwdBatch * kPairRec;
        const uint32_t a_cur = s_rec_addr + (uint32_t)(half * kBwdBatch * kPairRec * sizeof(float4));
        const uint32_t a_idc = s_id_addr + (uint32_t)(half * kBwdBatch * sizeof(int32_t));
        const int bs = min(kBwdBatch, (int)(hi - r0 + 1));
        if (hi - (bs - 1) > warp_last) continue;  // nothing of this batch was looked at by this warp's pixels
        for (int c0 = 0; c0 < bs; c0 += 32) {
            // lane l tests slot c0 + 31 - l: the first slot of the walk is the HIGHEST ballot bit
            const int gi = c0 + 31 - lane;
            bool hit = false, special = false;
            if (gi < bs && hi - gi <= warp_last) hit = pair_record_hit(s_cur + kPairRec * gi, X0, X1, Y0, Y1, &special);
            unsigned mask = __ballot_sync(0xffffffffu, hit);
            while (mask) {
                unsigned b_hi, below;
                asm("bfind.u32 %0, %1;" : "=r"(b_hi) : "r"(mask));
                asm("bmsk.clamp.b32 %0, 0, %1;" : "=r"(below) : "r"(b_hi));
                mask &= below;
                const int slot = c0 + 31 - (int)b_hi;
                const int32_t cur = hi - slot;
                BSPLAT_DASSERT(slot >= 0 && slot < bs && cur >= r0 && cur <= hi_all);
                const uint32_t ra_ = a_cur + (uint32_t)slot * (uint32_t)(kPairRec * sizeof(float4));
                const float4 p0 = lds_f4(ra_), p1 = lds_f4(ra_ + 16u);
                const float2 p2 = lds_f2(ra_ + 32u);  // {b, tau}
                const float2 dx2 = dupb(p0.x - px);
                const float2 dy2 = __fadd2_rn(dupb(p0.y), npy);
                const float2 nbdy = __fmul2_rn(dupb(p0.w), dy2);
                const float2 ncdy = __fmul2_rn(dupb(p1.x), dy2);
                const float2 lmc = __ffma2_rn(ncdy, dy2, dupb(p1.y));
                const float2 t = __ffma2_rn(dupb(p0.z), dx2, nbdy);
                const float2 pw = __ffma2_rn(t, dx2, lmc);
                // sigma >= 0 <=> power <= L: only special Gaussians can fail it (plain ones pass by construction)
                const float tau = p2.y;
                const float Lt = (__float_as_uint(tau) & 1u) ? p1.y : INFINITY;
                const bool pass0 = (pw.x >= kLog2AlphaThreshold) && (pw.x <= Lt) && (cur <= last0);
                const bool pass1 = (pw.y >= kLog2AlphaThreshold) && (pw.y <= Lt) && (cur <= last1);
                if (!__any_sync(0xffffffffu, pass0 || pass1)) continue;  // nothing to reduce for this warp
                float2 araw = make_float2(0.0f, 0.0f);
                if (pass0) araw.x = ex2_approx_b(pw.x);
                if (pass1) araw.y = ex2_approx_b(pw.y);
                const float2 alpha = make_float2(fminf(araw.x, 0.999f), fminf(araw.y, 0.999f));
                const float2 oma = __fadd2_rn(dupb(1.0f), make_float2(-alpha.x, -alpha.y));
                const float2 ra = make_float2(rcp_approx_b(oma.x), rcp_approx_b(oma.y));  // (alpha = 0: exactly 1)
                T2 = __fmul2_rn(T2, ra);  // transmittance in front of this Gaussian
                const float2 fac = __fmul2_rn(alpha, T2);
                const float cb = p2.x;
                // d out / d alpha = sum_ch (c_ch T - behind_ch / (1 - alpha)) gout_ch - T_final bg.gout / (1 - alpha)
                //                 = T (c . gout) - (behind . gout + T_final bg . gout) / (1 - alpha):
                // only the scalar behind . gout is carried per pixel (plus the constant background term), not the
                // three channel sums -- 6 packed instructions instead of 13
                float2 cgo = __fmul2_rn(dupb(p1.z), go_r);
                cgo = __ffma2_rn(dupb(p1.w), go_g, cgo);
                cgo = __ffma2_rn(dupb(cb), go_b, cgo);
                const float2 rb = __fmul2_rn(ra, behind);
                const float2 va = __ffma2_rn(T2, cgo, make_float2(-rb.x, -rb.y));
                behind = __ffma2_rn(fac, cgo, behind);
                const float2 vr = __fmul2_rn(fac, go_r), vg = __fmul2_rn(fac, go_g), vb = __fmul2_rn(fac, go_b);
                // v_sigma = -alpha v_alpha; no gradient through the clamp
                float2 vs = __fmul2_rn(make_float2(-araw.x, -araw.y), va);
                vs.x = (araw.x <= 0.999f) ? vs.x : 0.0f;
                vs.y = (araw.y <= 0.999f) ? vs.y : 0.0f;
                const float2 vsdx = __fmul2_rn(vs, dx2), vsdy = __fmul2_rn(vs, dy2);
                const float2 xx = __fmul2_rn(vsdx, dx2), xy = __fmul2_rn(vsdx, dy2), yy = __fmul2_rn(vsdy, dy2);
                float v[8];
                v[0] = vr.x + vr.y; v[1] = vg.x + vg.y; v[2] = vb.x + vb.y;
                v[3] = xx.x + xx.y; v[4] = xy.x + xy.y; v[5] = yy.x + yy.y;
                v[6] = vsdx.x + vsdx.y; v[7] = vsdy.x + vsdy.y;
                // conic of the record: (a, b, c) = (-2 nA, -nB, -2 nC) / log2e;  mean gradient = (a sx + b sy, b sx + c sy)
                constexpr float kInv = 1.0f / kLog2e;
                const float cb_ = -kInv * p0.w;
                float ss = vs.x + vs.y;
                if constexpr (kAbs) {
                    // each pixel's own mean gradient v_sigma (a dx + b dy, b dx + c dy), made absolute before any sum;
                    // reduced together with the opacity's sum: lanes 0-7 get sum v_sigma, 8-15 sum |x|, 16-23 sum |y|
                    const float ca = -2.0f * kInv * p0.z, cc = -2.0f * kInv * p1.x;
                    const float2 mx = __ffma2_rn(dupb(ca), vsdx, __fmul2_rn(dupb(cb_), vsdy));
                    const float2 my = __ffma2_rn(dupb(cb_), vsdx, __fmul2_rn(dupb(cc), vsdy));
                    float w[4] = {ss, fabsf(mx.x) + fabsf(mx.y), fabsf(my.x) + fabsf(my.y), 0.0f};
                    warp_reduce_spread<4>(w, (unsigned)lane);
                    ss = w[0];
                }
                warp_reduce_spread<8>(v, (unsigned)lane);  // lane 4 k holds the total of value k
                if constexpr (!kAbs) {
#pragma unroll
                    for (int d = 16; d > 0; d >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, d);
                }
                const float sx = __shfl_sync(0xffffffffu, v[0], 24), sy = __shfl_sync(0xffffffffu, v[0], 28);
                const int64_t g = lds_i32(a_idc + 4u * (uint32_t)slot);
                BSPLAT_DASSERT(g >= 0 && g < N);  // (a record that is not a Gaussian never passes the alpha test)
                const float c_first = role_my ? cb_ : -2.0f * kInv * p0.z;
                const float c_second = role_my ? -2.0f * kInv * p1.x : cb_;
                float val = role_mean ? (c_first * sx + c_second * sy) : role_scale * v[0];
                // d alpha / d opacity = alpha / opacity  =>  -sum v_sigma / opacity, opacity = 2^L
                val = role_op ? -ss * ex2_approx_b(-p1.y) : val;
                if constexpr (kAbs) val = role_abs ? ss : val;  // lanes 9 and 17 hold sum |x| and sum |y|
                if (issues) atomicAdd(role_base + g * role_stride, val);
            }
        }
    }
}

}  // namespace bsplat

using namespace bsplat;

namespace {
inline int round_up32(int v) { return (v + 31) / 32 * 32; }
}

extern "C" int bsplat_rasterize_fwd_train(int64_t N, int32_t channels, const float* means2d, const float* conics,
                                          const float* colors, const float* opacities, const float* background,
                                          const int32_t* tile_ranges, const int32_t* sorted_ids, int64_t M,
                                          int32_t width, int32_t height, int32_t tile_size, float* image,
                                          float* final_T, int32_t* last_idx, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (N < 0 || M < 0 || !tile_ranges || !image || !background || !final_T || !last_idx) return BSPLAT_E_ARG;
    if (M > 0 && (!sorted_ids || !means2d || !conics || !colors || !opacities)) return BSPLAT_E_ARG;
    if (width <= 0 || height <= 0 || tile_size <= 0 || tile_size > 32) return BSPLAT_E_ARG;
    if (channels < 1 || channels > 4) return BSPLAT_E_ARG;
    const int tiles_w = (width + tile_size - 1) / tile_size, tiles_h = (height + tile_size - 1) / tile_size;
    if (tiles_h > 65535) return BSPLAT_E_ARG;
    const int nthreads = round_up32(tile_size * tile_size);
    const dim3 grid(tiles_w, tiles_h);
    const size_t smem = (size_t)nthreads * (9 + channels) * sizeof(float);
    // tile sizes 31 / 32 need more than the 48 KB a kernel gets without opting in
#define BSPLAT_TRAIN_FWD(CH)                                                                                    \
    do {                                                                                                        \
        if (smem + 256 > 48 * 1024) /* (+ the kernel's static shared memory) */                                 \
            BSPLAT_CUDA_TRY(cudaFuncSetAttribute(raster_train_fwd_kernel<CH>,                                   \
                                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));      \
        raster_train_fwd_kernel<CH><<<grid, nthreads, smem, stream>>>(N, means2d, conics, colors, opacities,   \
            background, tile_ranges, sorted_ids, width, height, tile_size, tiles_w, image, final_T, last_idx);  \
    } while (0)
    switch (channels) {
        case 1: BSPLAT_TRAIN_FWD(1); break;
        case 2: BSPLAT_TRAIN_FWD(2); break;
        case 3: BSPLAT_TRAIN_FWD(3); break;
        default: BSPLAT_TRAIN_FWD(4); break;
    }
#undef BSPLAT_TRAIN_FWD
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}

namespace bsplat {
int rasterize_train_fast_launch(int64_t N, const float* means2d, const float* conics, const float* colors,
                                const float* opacities, const float* background_dev, const int32_t* tile_ranges,
                                const int32_t* tile_order, const int32_t* sorted_ids, int W, int H, float* image,
                                float* final_T, int32_t* last_idx, void* rec_ws, cudaStream_t stream);
size_t raster_workspace_bytes(int64_t N);
}

// The same through the fast forward kernel (16x16 tiles, RGB only): image bit-identical to bsplat_rasterize_fwd's
// default mode; last_idx holds, per pixel, the last list entry the backward pass has to look at.
extern "C" int bsplat_rasterize_fwd_train_fast(int64_t N, const float* means2d, const float* conics,
                                               const float* colors, const float* opacities, const float* background,
                                               const int32_t* tile_ranges, const int32_t* tile_order,
                                               const int32_t* sorted_ids, int64_t M, int32_t width, int32_t height,
                                               float* image, float* final_T, int32_t* last_idx, void* workspace,
                                               size_t workspace_bytes, void* stream_) {
    if (N < 0 || M < 0 || width <= 0 || height <= 0) return BSPLAT_E_ARG;
    if (M > 0 && !sorted_ids) return BSPLAT_E_ARG;
    if ((height + 15) / 16 > 65535) return BSPLAT_E_ARG;
    if (workspace && workspace_bytes < raster_workspace_bytes(N)) return BSPLAT_E_WORKSPACE;
    return rasterize_train_fast_launch(N, means2d, conics, colors, opacities, background, tile_ranges, tile_order,
                                       sorted_ids, width, height, image, final_T, last_idx, workspace,
                                       (cudaStream_t)stream_);
}

// Backward in the fast kernel's layout (16x16 tiles, RGB; see raster_bwd_pair_kernel).  workspace: the per-Gaussian
// records, bsplat_rasterize_workspace_bytes(N) (rewritten here: the caller's workspace need not survive from the
// forward call).  tile_order optional.
namespace bsplat {
int raster_records_launch(int64_t N, const float* means2d, const float* conics, const float* colors,
                          const float* opacities, void* rec_ws, cudaStream_t stream);
}
namespace {
// bsplat_rasterize_bwd_fast[_abs]: g_abs == nullptr launches the plain kernel
int rasterize_bwd_fast_impl(int64_t N, const float* means2d, const float* conics, const float* colors,
                            const float* opacities, const float* background, const int32_t* tile_ranges,
                            const int32_t* tile_order, const int32_t* sorted_ids, int64_t M, int32_t width,
                            int32_t height, const float* final_T, const int32_t* last_idx, const float* grad_image,
                            float* grad_means2d, float* grad_conics, float* grad_colors, float* grad_opacities,
                            float* g_abs, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    if (N < 0 || M < 0 || !tile_ranges || !background || !final_T || !last_idx || !grad_image) return BSPLAT_E_ARG;
    if (N > 0 && (!grad_means2d || !grad_conics || !grad_colors || !grad_opacities)) return BSPLAT_E_ARG;
    if (M > 0 && (!sorted_ids || !means2d || !conics || !colors || !opacities)) return BSPLAT_E_ARG;
    if (width <= 0 || height <= 0) return BSPLAT_E_ARG;
    if (N == 0 || M == 0) return BSPLAT_OK;
    if ((reinterpret_cast<uintptr_t>(means2d) & 7u) != 0) return BSPLAT_E_ARG;
    if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 15u) != 0 || workspace_bytes < raster_workspace_bytes(N))
        return BSPLAT_E_WORKSPACE;
    const int tiles_w = (width + 15) / 16, tiles_h = (height + 15) / 16;
    int rc = raster_records_launch(N, means2d, conics, colors, opacities, workspace, stream);
    if (rc != BSPLAT_OK) return rc;
    const unsigned grid = (unsigned)(tiles_w * tiles_h);
    if (g_abs)
        raster_bwd_pair_kernel<true><<<grid, kBwdThreads, 0, stream>>>(
            N, static_cast<const float4*>(workspace), background, tile_ranges, tile_order, sorted_ids, width, height,
            tiles_w, final_T, last_idx, grad_image, grad_means2d, grad_conics, grad_colors, grad_opacities, g_abs);
    else
        raster_bwd_pair_kernel<false><<<grid, kBwdThreads, 0, stream>>>(
            N, static_cast<const float4*>(workspace), background, tile_ranges, tile_order, sorted_ids, width, height,
            tiles_w, final_T, last_idx, grad_image, grad_means2d, grad_conics, grad_colors, grad_opacities, nullptr);
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}

// bsplat_rasterize_bwd[_abs]: g_abs == nullptr launches the plain kernels
int rasterize_bwd_impl(int64_t N, int32_t channels, const float* means2d, const float* conics, const float* colors,
                       const float* opacities, const float* background, const int32_t* tile_ranges,
                       const int32_t* sorted_ids, int64_t M, int32_t width, int32_t height, int32_t tile_size,
                       const float* final_T, const int32_t* last_idx, const float* grad_image, float* grad_means2d,
                       float* grad_conics, float* grad_colors, float* grad_opacities, float* g_abs,
                       cudaStream_t stream) {
    if (N < 0 || M < 0 || !tile_ranges || !background || !final_T || !last_idx || !grad_image) return BSPLAT_E_ARG;
    if (N > 0 && (!grad_means2d || !grad_conics || !grad_colors || !grad_opacities)) return BSPLAT_E_ARG;
    if (M > 0 && (!sorted_ids || !means2d || !conics || !colors || !opacities)) return BSPLAT_E_ARG;
    if (width <= 0 || height <= 0 || tile_size <= 0 || tile_size > 32) return BSPLAT_E_ARG;
    if (channels < 1 || channels > 4) return BSPLAT_E_ARG;
    if (N == 0 || M == 0) return BSPLAT_OK;  // gradients stay as the caller initialised them (zeros)
    const int tiles_w = (width + tile_size - 1) / tile_size, tiles_h = (height + tile_size - 1) / tile_size;
    if (tiles_h > 65535) return BSPLAT_E_ARG;
    const int nthreads = round_up32(tile_size * tile_size);
    const dim3 grid(tiles_w, tiles_h);
    const size_t smem = (size_t)nthreads * (10 + channels) * sizeof(float);
#define BSPLAT_BWD(CH, ABS)                                                                                     \
    do {                                                                                                        \
        if (smem + 256 > 48 * 1024) /* (+ the kernel's static shared memory) */                                 \
            BSPLAT_CUDA_TRY(cudaFuncSetAttribute(raster_bwd_kernel<CH, ABS>,                                    \
                                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));      \
        raster_bwd_kernel<CH, ABS><<<grid, nthreads, smem, stream>>>(N, means2d, conics, colors, opacities,    \
            background, tile_ranges, sorted_ids, width, height, tile_size, tiles_w, final_T, last_idx,          \
            grad_image, grad_means2d, grad_conics, grad_colors, grad_opacities, g_abs);                         \
    } while (0)
#define BSPLAT_BWD_CH(CH)                 \
    do {                                  \
        if (g_abs) BSPLAT_BWD(CH, true);  \
        else BSPLAT_BWD(CH, false);       \
    } while (0)
    switch (channels) {
        case 1: BSPLAT_BWD_CH(1); break;
        case 2: BSPLAT_BWD_CH(2); break;
        case 3: BSPLAT_BWD_CH(3); break;
        default: BSPLAT_BWD_CH(4); break;
    }
#undef BSPLAT_BWD_CH
#undef BSPLAT_BWD
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}
}  // namespace

extern "C" int bsplat_rasterize_bwd_fast(int64_t N, const float* means2d, const float* conics, const float* colors,
                                         const float* opacities, const float* background,
                                         const int32_t* tile_ranges, const int32_t* tile_order,
                                         const int32_t* sorted_ids, int64_t M, int32_t width, int32_t height,
                                         const float* final_T, const int32_t* last_idx, const float* grad_image,
                                         float* grad_means2d, float* grad_conics, float* grad_colors,
                                         float* grad_opacities, void* workspace, size_t workspace_bytes,
                                         void* stream_) {
    return rasterize_bwd_fast_impl(N, means2d, conics, colors, opacities, background, tile_ranges, tile_order,
                                   sorted_ids, M, width, height, final_T, last_idx, grad_image, grad_means2d,
                                   grad_conics, grad_colors, grad_opacities, nullptr, workspace, workspace_bytes,
                                   (cudaStream_t)stream_);
}

// ... that also ACCUMULATES, per Gaussian, the sum over pixels of |d loss_p / d means2d| into grad_means2d_abs [N, 2]
extern "C" int bsplat_rasterize_bwd_fast_abs(int64_t N, const float* means2d, const float* conics,
                                             const float* colors, const float* opacities, const float* background,
                                             const int32_t* tile_ranges, const int32_t* tile_order,
                                             const int32_t* sorted_ids, int64_t M, int32_t width, int32_t height,
                                             const float* final_T, const int32_t* last_idx, const float* grad_image,
                                             float* grad_means2d, float* grad_means2d_abs, float* grad_conics,
                                             float* grad_colors, float* grad_opacities, void* workspace,
                                             size_t workspace_bytes, void* stream_) {
    if (N > 0 && !grad_means2d_abs) return BSPLAT_E_ARG;
    return rasterize_bwd_fast_impl(N, means2d, conics, colors, opacities, background, tile_ranges, tile_order,
                                   sorted_ids, M, width, height, final_T, last_idx, grad_image, grad_means2d,
                                   grad_conics, grad_colors, grad_opacities, grad_means2d_abs, workspace,
                                   workspace_bytes, (cudaStream_t)stream_);
}

extern "C" int bsplat_rasterize_bwd(int64_t N, int32_t channels, const float* means2d, const float* conics,
                                    const float* colors, const float* opacities, const float* background,
                                    const int32_t* tile_ranges, const int32_t* sorted_ids, int64_t M,
                                    int32_t width, int32_t height, int32_t tile_size, const float* final_T,
                                    const int32_t* last_idx, const float* grad_image, float* grad_means2d,
                                    float* grad_conics, float* grad_colors, float* grad_opacities,
                                    void* stream_) {
    return rasterize_bwd_impl(N, channels, means2d, conics, colors, opacities, background, tile_ranges, sorted_ids,
                              M, width, height, tile_size, final_T, last_idx, grad_image, grad_means2d, grad_conics,
                              grad_colors, grad_opacities, nullptr, (cudaStream_t)stream_);
}

extern "C" int bsplat_rasterize_bwd_abs(int64_t N, int32_t channels, const float* means2d, const float* conics,
                                        const float* colors, const float* opacities, const float* background,
                                        const int32_t* tile_ranges, const int32_t* sorted_ids, int64_t M,
                                        int32_t width, int32_t height, int32_t tile_size, const float* final_T,
                                        const int32_t* last_idx, const float* grad_image, float* grad_means2d,
                                        float* grad_means2d_abs, float* grad_conics, float* grad_colors,
                                        float* grad_opacities, void* stream_) {
    if (N > 0 && !grad_means2d_abs) return BSPLAT_E_ARG;
    return rasterize_bwd_impl(N, channels, means2d, conics, colors, opacities, background, tile_ranges, sorted_ids,
                              M, width, height, tile_size, final_T, last_idx, grad_image, grad_means2d, grad_conics,
                              grad_colors, grad_opacities, grad_means2d_abs, (cudaStream_t)stream_);
}
