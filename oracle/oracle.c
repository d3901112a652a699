/*
 * oracle.c -- CPU restatement of the MojoSplat forward path.  TEST INFRASTRUCTURE ONLY.
 *
 * This file is the checker, never the product: only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load it.  The product path
 * (mojosplat_b200/) never imports, links or executes anything under oracle/.
 *
 * Each function restates one reference routine in plain fp32 C and cites the
 * reference lines it follows (paths relative to the reference checkout):
 *
 *   oracle_project        mojosplat/projection.py:51-346   (torch backend, "torch" semantics)
 *                         mojosplat/kernels/projection.mojo:13-257 ("gsplat" semantics)
 *   oracle_bin_*          mojosplat/binning.py:108-262     (torch backend, bit-exact target)
 *   oracle_rasterize      mojosplat/kernels/rasterization.mojo:75-162
 *
 * Pinning status:
 *   - projection + binning: PINNED against outputs of the unmodified reference torch
 *     backend run in the build container (oracle/make_golden.py -> tests/golden/*.npz):
 *     means2d, depths, radii, tile ranges bit for bit; conics bit for bit except where MKL's exp is
 *     1 ulp off the correctly rounded value (~3 % of the rows; within 1e-4 + 1e-4 |ref| there).
 *   - rasterization: the reference has no CPU rasterizer and gsplat is not installable
 *     offline, so gsplat parity is UNPINNED; the restatement is pinned only to the
 *     backend-independent known-answer checks of the reference's tests
 *     (tests/test_rasterization.py:154-248, tests/test_render.py:60-119) and to an
 *     independent numpy restatement (oracle/oracle_np.py).
 *
 * Error budgets (SURVEY 7 step 1d, H3/H4): oracle_project_f64 / oracle_rasterize_f64 evaluate the same
 * algorithms in double precision from the fp32 inputs; oracle_raster_audit explains out-of-tolerance pixels by
 * forced alpha-threshold / saturation flips.
 *
 * Build: oracle/build.sh  (gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC).
 * -ffp-contract=off keeps every multiply and add separately rounded, like the eager
 * torch ops the reference issues; where the reference's matmul kernels fuse, fmaf() is written out.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ORACLE_SEM_TORCH 0
#define ORACLE_SEM_GSPLAT 1

int oracle_num_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

void oracle_set_num_threads(int n) {
#ifdef _OPENMP
    if (n > 0) omp_set_num_threads(n);
#else
    (void)n;
#endif
}

/* How the reference's torch ops round (found by bisecting the unmodified reference against tests/golden, torch
 * 2.11 CPU; oracle/make_golden.py regenerates the evidence):
 *   - element-wise ops (quat -> R, R * s, the Jacobian entries, det, conic, radii): one rounding per operation;
 *   - einsum that lowers to the matmul kernel -- R . mu, (R Sigma) R^T, K . mu_c: a dot product is
 *     c = a0 b0; c = fma(a1, b1, c); c = fma(a2, b2, c);
 *   - einsum that lowers to product + sum -- M M^T ("ij,kj->ik") and (J Sigma_c) J^T: every product and every sum
 *     rounded, left to right;
 *   - torch.exp (MKL VML, high accuracy): the correctly rounded result for 98.9 % of the arguments, 1 ulp off
 *     otherwise -- not reproducible without MKL; exp_torch returns the correctly rounded value.
 * With these rules means2d, depths and radii of the oracle equal the reference's bit for bit on every fixture, and
 * so do the conics of every Gaussian whose three scales got the correctly rounded exp (tests/test_oracle_golden.py). */
static inline float dot3_mm(float a0, float b0, float a1, float b1, float a2, float b2) {
    float c = a0 * b0;
    c = fmaf(a1, b1, c);
    c = fmaf(a2, b2, c);
    return c;
}

static inline float exp_torch(float x) { return (float)exp((double)x); }

/* ------------------------------------------------------------------------------------
 * Projection.  projection.py:285-346 (wrapper), :72-102 (covariance), :51-69 (quat->R),
 * :163-196 (world->cam), :105-160 (pinhole), :199-283 (fused tail).
 *
 * semantics == ORACLE_SEM_TORCH : exactly the torch backend (opacity ignored, radius
 *   3.33 sigma, culled rows keep their computed means2d/conics/depths, det clamp 1e-10).
 * semantics == ORACLE_SEM_GSPLAT: the Mojo kernel's / gsplat's rules
 *   (projection.mojo:59-87 near + opacity cull with zeroed rows, :213-226 opacity-aware
 *   extent, :240-244 viewport cull, :246-251 conic without det clamp).  `near` comes from
 *   the caller (the Mojo kernel hard-codes 0.1, the gsplat call passes camera.near).
 * ---------------------------------------------------------------------------------- */
void oracle_project(
    int64_t N,
    const float* means3d,   /* [N,3] */
    const float* log_scales,/* [N,3] */
    const float* quats,     /* [N,4] wxyz */
    const float* opacities, /* [N] or NULL (only read in gsplat semantics) */
    const float* viewmat,   /* [4,4] row-major world->cam */
    float fx, float fy, float cx, float cy,
    int W, int H, float near_plane, float far_plane, float eps2d,
    int semantics,
    float* means2d,  /* [N,2] */
    float* conics,   /* [N,3] */
    float* depths,   /* [N] */
    int32_t* radii)  /* [N,2] */
{
    const float Rv[3][3] = {
        {viewmat[0], viewmat[1], viewmat[2]},
        {viewmat[4], viewmat[5], viewmat[6]},
        {viewmat[8], viewmat[9], viewmat[10]}};
    const float tv[3] = {viewmat[3], viewmat[7], viewmat[11]};

    /* projection.py:137-146 */
    const float tan_fovx = 0.5f * (float)W / fx;
    const float tan_fovy = 0.5f * (float)H / fy;
    const float lim_x_pos = ((float)W - cx) / fx + 0.3f * tan_fovx;
    const float lim_x_neg = cx / fx + 0.3f * tan_fovx;
    const float lim_y_pos = ((float)H - cy) / fy + 0.3f * tan_fovy;
    const float lim_y_neg = cy / fy + 0.3f * tan_fovy;

#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < N; ++i) {
        const float* mu = means3d + 3 * i;
        const float* ls = log_scales + 3 * i;
        const float* q = quats + 4 * i;

        /* world -> camera mean, projection.py:190-192 (einsum -> matmul kernel: FMA chain, then `+ t`) */
        float mc[3];
        for (int r = 0; r < 3; ++r)
            mc[r] = dot3_mm(Rv[r][0], mu[0], Rv[r][1], mu[1], Rv[r][2], mu[2]) + tv[r];

        if (semantics == ORACLE_SEM_GSPLAT) {
            /* projection.mojo:59-87 */
            float op = opacities ? opacities[i] : 1.0f;
            if (mc[2] <= near_plane || mc[2] >= far_plane || op < (1.0f / 255.0f)) {
                means2d[2 * i] = means2d[2 * i + 1] = 0.0f;
                conics[3 * i] = conics[3 * i + 1] = conics[3 * i + 2] = 0.0f;
                depths[i] = 0.0f;
                radii[2 * i] = radii[2 * i + 1] = 0;
                continue;
            }
        }

        /* quat -> rotation, projection.py:51-69 (F.normalize: x / max(||x||, 1e-12)) */
        float nrm = sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
        if (nrm < 1e-12f) nrm = 1e-12f;
        const float w = q[0] / nrm, x = q[1] / nrm, y = q[2] / nrm, z = q[3] / nrm;
        float R[3][3] = {
            {1.0f - 2.0f * (y * y + z * z), 2.0f * (x * y - w * z), 2.0f * (x * z + w * y)},
            {2.0f * (x * y + w * z), 1.0f - 2.0f * (x * x + z * z), 2.0f * (y * z - w * x)},
            {2.0f * (x * z - w * y), 2.0f * (y * z + w * x), 1.0f - 2.0f * (x * x + y * y)}};

        /* M = R * s ; Sigma = M M^T, projection.py:86-87 ("ij,kj->ik": product + sum, every operation rounded) */
        const float s[3] = {exp_torch(ls[0]), exp_torch(ls[1]), exp_torch(ls[2])};
        float M[3][3], S[3][3];
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) M[r][c] = R[r][c] * s[c];
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c)
                S[r][c] = M[r][0] * M[c][0] + M[r][1] * M[c][1] + M[r][2] * M[c][2];

        /* Sigma_c = (Rv Sigma) Rv^T, projection.py:193-195 (three-operand einsum, left to right, both products
         * through the matmul kernel: FMA chains) */
        float A[3][3], Sc[3][3];
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c)
                A[r][c] = dot3_mm(Rv[r][0], S[0][c], Rv[r][1], S[1][c], Rv[r][2], S[2][c]);
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c)
                Sc[r][c] = dot3_mm(A[r][0], Rv[c][0], A[r][1], Rv[c][1], A[r][2], Rv[c][2]);

        /* pinhole Jacobian, projection.py:134-159 */
        const float tz = mc[2];
        const float tz2 = tz * tz;
        float rx = mc[0] / tz, ry = mc[1] / tz;
        rx = fminf(fmaxf(rx, -lim_x_neg), lim_x_pos);
        ry = fminf(fmaxf(ry, -lim_y_neg), lim_y_pos);
        const float tx = tz * rx, ty = tz * ry;
        const float J[2][3] = {{fx / tz, 0.0f, -fx * tx / tz2}, {0.0f, fy / tz, -fy * ty / tz2}};
        float JS[2][3];
        for (int r = 0; r < 2; ++r)
            for (int c = 0; c < 3; ++c)
                JS[r][c] = J[r][0] * Sc[0][c] + J[r][1] * Sc[1][c] + J[r][2] * Sc[2][c];
        float c00 = JS[0][0] * J[0][0] + JS[0][1] * J[0][1] + JS[0][2] * J[0][2];
        float c01 = JS[0][0] * J[1][0] + JS[0][1] * J[1][1] + JS[0][2] * J[1][2];
        float c10 = JS[1][0] * J[0][0] + JS[1][1] * J[0][1] + JS[1][2] * J[0][2];
        float c11 = JS[1][0] * J[1][0] + JS[1][1] * J[1][1] + JS[1][2] * J[1][2];

        /* means2d = (K[:2,:3] . mu_c) / z, projection.py:156-159 (matmul kernel: FMA chain) */
        const float m2x = dot3_mm(fx, mc[0], 0.0f, mc[1], cx, mc[2]) / tz;
        const float m2y = dot3_mm(0.0f, mc[0], fy, mc[1], cy, mc[2]) / tz;

        c00 += eps2d; /* projection.py:242 */
        c11 += eps2d;
        float det = c00 * c11 - c01 * c10;

        if (semantics == ORACLE_SEM_TORCH) {
            if (!(det >= 1e-10f)) det = (det != det) ? det : 1e-10f; /* clamp(min=1e-10), :248 */
            const float k0 = c11 / det;
            const float k1 = -(c01 + c10) / 2.0f / det;
            const float k2 = c00 / det;
            float r_x = ceilf(3.33f * sqrtf(c00)); /* :266-267 */
            float r_y = ceilf(3.33f * sqrtf(c11));
            const int valid = (det > 0.0f) && (tz > near_plane) && (tz < far_plane); /* :271 */
            if (!valid) { r_x = 0.0f; r_y = 0.0f; }
            const int inside = (m2x + r_x > 0.0f) && (m2x - r_x < (float)W) &&
                               (m2y + r_y > 0.0f) && (m2y - r_y < (float)H); /* :274-279 */
            if (!inside) { r_x = 0.0f; r_y = 0.0f; }
            means2d[2 * i] = m2x; means2d[2 * i + 1] = m2y;
            conics[3 * i] = k0; conics[3 * i + 1] = k1; conics[3 * i + 2] = k2;
            depths[i] = tz;
            radii[2 * i] = (int32_t)r_x; radii[2 * i + 1] = (int32_t)r_y;
        } else {
            /* projection.mojo:213-257 */
            float extend = 3.33f;
            const float op = opacities ? opacities[i] : 1.0f;
            const float oe = sqrtf(2.0f * logf(op / (1.0f / 255.0f)));
            if (oe < extend) extend = oe;
            const float r_x = ceilf(extend * sqrtf(c00));
            const float r_y = ceilf(extend * sqrtf(c11));
            if ((r_x <= 0.0f && r_y <= 0.0f) ||
                m2x + r_x <= 0.0f || m2x - r_x >= (float)W ||
                m2y + r_y <= 0.0f || m2y - r_y >= (float)H) {
                means2d[2 * i] = means2d[2 * i + 1] = 0.0f;
                conics[3 * i] = conics[3 * i + 1] = conics[3 * i + 2] = 0.0f;
                depths[i] = 0.0f;
                radii[2 * i] = radii[2 * i + 1] = 0;
                continue;
            }
            const float inv_det = 1.0f / det;
            means2d[2 * i] = m2x; means2d[2 * i + 1] = m2y;
            conics[3 * i] = c11 * inv_det;
            conics[3 * i + 1] = -(c01 + c10) / 2.0f * inv_det;
            conics[3 * i + 2] = c00 * inv_det;
            depths[i] = tz;
            radii[2 * i] = (int32_t)r_x; radii[2 * i + 1] = (int32_t)r_y;
        }
    }
}

/* ------------------------------------------------------------------------------------
 * Binning.  binning.py:108-262.
 * ---------------------------------------------------------------------------------- */

/* Monotone float -> uint32 map used as the canonical depth order (SURVEY H2):
 * ascending float order, -0.0 == +0.0 (torch.argsort ties them), NaN last. */
static inline uint32_t depth_key(float d) {
    uint32_t b;
    memcpy(&b, &d, 4);
    if ((b & 0x7fffffffu) > 0x7f800000u) return 0xffffffffu; /* NaN sorts last */
    if (b == 0x80000000u) b = 0u;                             /* -0.0 -> +0.0 */
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

static inline float clampf(float v, float lo, float hi) {
    /* torch.clamp: min(max(v, lo), hi); NaN propagates */
    if (v != v) return v;
    v = v < lo ? lo : v;
    v = v > hi ? hi : v;
    return v;
}

static inline void tile_rect(
    const float* means2d, const float* radii_f, int64_t i, int W, int H, int tile_size,
    int tiles_w, int tiles_h, int semantics, int* x0, int* y0, int* x1, int* y1)
{
    const float mx = means2d[2 * i], my = means2d[2 * i + 1];
    const float rx = radii_f[2 * i], ry = radii_f[2 * i + 1];
    if (semantics == ORACLE_SEM_TORCH) {
        /* binning.py:139-155: pixel-space clamp, trunc-to-int32, INCLUSIVE max */
        const float ts = (float)tile_size;
        float ax = clampf(mx - rx, 0.0f, (float)(W - 1));
        float bx = clampf(mx + rx, 0.0f, (float)(W - 1));
        float ay = clampf(my - ry, 0.0f, (float)(H - 1));
        float by = clampf(my + ry, 0.0f, (float)(H - 1));
        int tx0 = (int)(ax / ts), tx1 = (int)(bx / ts);
        int ty0 = (int)(ay / ts), ty1 = (int)(by / ts);
        /* binning.py:181-184 second clamp in tile space (no-op for finite inputs) */
        tx0 = tx0 < 0 ? 0 : (tx0 > tiles_w - 1 ? tiles_w - 1 : tx0);
        tx1 = tx1 < 0 ? 0 : (tx1 > tiles_w - 1 ? tiles_w - 1 : tx1);
        ty0 = ty0 < 0 ? 0 : (ty0 > tiles_h - 1 ? tiles_h - 1 : ty0);
        ty1 = ty1 < 0 ? 0 : (ty1 > tiles_h - 1 ? tiles_h - 1 : ty1);
        *x0 = tx0; *x1 = tx1 + 1; *y0 = ty0; *y1 = ty1 + 1; /* exclusive ends */
    } else {
        /* gsplat isect_tiles [upstream-knowledge, SURVEY 8a-2]: tile-space floor/ceil,
         * exclusive max, nothing for radii <= 0 */
        if (rx <= 0.0f || ry <= 0.0f) { *x0 = *x1 = *y0 = *y1 = 0; return; }
        const float ts = (float)tile_size;
        float fx0 = floorf((mx - rx) / ts), fx1 = ceilf((mx + rx) / ts);
        float fy0 = floorf((my - ry) / ts), fy1 = ceilf((my + ry) / ts);
        fx0 = fminf(fmaxf(fx0, 0.0f), (float)tiles_w); fx1 = fminf(fmaxf(fx1, 0.0f), (float)tiles_w);
        fy0 = fminf(fmaxf(fy0, 0.0f), (float)tiles_h); fy1 = fminf(fmaxf(fy1, 0.0f), (float)tiles_h);
        *x0 = (int)fx0; *x1 = (int)fx1; *y0 = (int)fy0; *y1 = (int)fy1;
    }
}

/* Number of (gaussian, tile) intersections; also per-gaussian counts if `counts` != NULL.
 * binning.py:162-163.  radii are passed as float (the reference promotes int32 radii to
 * float in `means2d - radii`, binning.py:139). */
int64_t oracle_bin_count(
    int64_t N, const float* means2d, const float* radii_f, int W, int H, int tile_size,
    int semantics, int32_t* counts)
{
    const int tiles_w = (W + tile_size - 1) / tile_size, tiles_h = (H + tile_size - 1) / tile_size;
    int64_t total = 0;
    for (int64_t i = 0; i < N; ++i) {
        int x0, y0, x1, y1;
        tile_rect(means2d, radii_f, i, W, H, tile_size, tiles_w, tiles_h, semantics, &x0, &y0, &x1, &y1);
        int c = (x1 - x0) * (y1 - y0);
        if (c < 0) c = 0;
        if (counts) counts[i] = c;
        total += c;
    }
    return total;
}

static void radix_sort_u64_pairs(uint64_t* keys, int32_t* vals, int64_t n, int key_bits) {
    /* stable LSD radix sort, 11-bit digits */
    uint64_t* k2 = (uint64_t*)malloc(sizeof(uint64_t) * (size_t)(n > 0 ? n : 1));
    int32_t* v2 = (int32_t*)malloc(sizeof(int32_t) * (size_t)(n > 0 ? n : 1));
    const int RB = 11, NB = 1 << RB;
    int64_t* hist = (int64_t*)malloc(sizeof(int64_t) * NB);
    uint64_t* src = keys; uint64_t* dst = k2; int32_t* vs = vals; int32_t* vd = v2;
    for (int shift = 0; shift < key_bits; shift += RB) {
        memset(hist, 0, sizeof(int64_t) * NB);
        for (int64_t i = 0; i < n; ++i) hist[(src[i] >> shift) & (NB - 1)]++;
        int64_t acc = 0;
        for (int b = 0; b < NB; ++b) { int64_t c = hist[b]; hist[b] = acc; acc += c; }
        for (int64_t i = 0; i < n; ++i) {
            int64_t p = hist[(src[i] >> shift) & (NB - 1)]++;
            dst[p] = src[i]; vd[p] = vs[i];
        }
        uint64_t* tk = src; src = dst; dst = tk;
        int32_t* tv = vs; vs = vd; vd = tv;
    }
    if (src != keys) { memcpy(keys, src, sizeof(uint64_t) * (size_t)n); memcpy(vals, vs, sizeof(int32_t) * (size_t)n); }
    free(k2); free(v2); free(hist);
}

/* Full binning: emits (tile, depth, gaussian) in the reference's emission order
 * (binning.py:172-200: gaussian ascending, ty ascending, tx ascending), sorts by depth and
 * then STABLY by tile (binning.py:223-231; the depth argsort is made stable here, the
 * canonical tie order of SURVEY H2), and derives tile_ranges with searchsorted-left
 * (binning.py:252-260).
 *   sorted_ids  [M] int32, isect_keys [M] uint64 (tile<<32 | depth_key) or NULL,
 *   tile_ranges [tiles_h*tiles_w*2] int32.
 * Returns M (must equal oracle_bin_count). */
int64_t oracle_bin(
    int64_t N, const float* means2d, const float* radii_f, const float* depths,
    int W, int H, int tile_size, int semantics,
    int64_t M_capacity, int32_t* sorted_ids, uint64_t* isect_keys, int32_t* tile_ranges)
{
    const int tiles_w = (W + tile_size - 1) / tile_size, tiles_h = (H + tile_size - 1) / tile_size;
    const int64_t n_tiles = (int64_t)tiles_w * tiles_h;
    uint64_t* keys = (uint64_t*)malloc(sizeof(uint64_t) * (size_t)(M_capacity > 0 ? M_capacity : 1));
    int64_t m = 0;
    for (int64_t i = 0; i < N; ++i) {
        int x0, y0, x1, y1;
        tile_rect(means2d, radii_f, i, W, H, tile_size, tiles_w, tiles_h, semantics, &x0, &y0, &x1, &y1);
        const uint64_t dk = depth_key(depths[i]);
        for (int ty = y0; ty < y1; ++ty)
            for (int tx = x0; tx < x1; ++tx) {
                if (m >= M_capacity) { free(keys); return -1; }
                keys[m] = ((uint64_t)(ty * tiles_w + tx) << 32) | dk;
                sorted_ids[m] = (int32_t)i;
                ++m;
            }
    }
    int tile_bits = 1;
    while (((int64_t)1 << tile_bits) < n_tiles) ++tile_bits;
    radix_sort_u64_pairs(keys, sorted_ids, m, 32 + tile_bits);

    /* searchsorted(sorted_tile_ids, arange(n_tiles+1), side='left') */
    int64_t p = 0;
    for (int64_t t = 0; t < n_tiles; ++t) {
        while (p < m && (int64_t)(keys[p] >> 32) < t) ++p;
        int64_t e = p;
        while (e < m && (int64_t)(keys[e] >> 32) < t + 1) ++e;
        tile_ranges[2 * t] = (int32_t)p;
        tile_ranges[2 * t + 1] = (int32_t)e;
        p = e;
    }
    if (isect_keys) memcpy(isect_keys, keys, sizeof(uint64_t) * (size_t)m);
    free(keys);
    return m;
}

/* ------------------------------------------------------------------------------------
 * Rasterization.  kernels/rasterization.mojo:75-162.
 *   pixel centre +0.5 (:78-79); sigma (:138-142); alpha clamp and thresholds (:143-150);
 *   accumulate then update T (:152-157); background blend (:160-162).
 * stats[0] += evaluated (pixel, gaussian) pairs (every loop iteration reached),
 * stats[1] += contributing pairs (passed both tests).  stats may be NULL.
 * Out-of-range ids are skipped like the Mojo staging guard (:109).
 * ---------------------------------------------------------------------------------- */
void oracle_rasterize(
    int64_t N, int CDIM,
    const float* means2d, const float* conics, const float* colors, const float* opacities,
    const float* background,          /* [CDIM] */
    const int32_t* tile_ranges,       /* [tiles_h, tiles_w, 2] */
    const int32_t* sorted_ids,        /* [M] */
    int W, int H, int tile_size,
    float* image,                     /* [H, W, CDIM] */
    int64_t* stats)
{
    const int tiles_w = (W + tile_size - 1) / tile_size, tiles_h = (H + tile_size - 1) / tile_size;
    int64_t e_all = 0, e_pass = 0;
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : e_all, e_pass)
    for (int t = 0; t < tiles_w * tiles_h; ++t) {
        const int tr = t / tiles_w, tc = t % tiles_w;
        const int32_t r0 = tile_ranges[2 * t], r1 = tile_ranges[2 * t + 1];
        float pix[CDIM > 0 ? CDIM : 1];
        for (int ii = 0; ii < tile_size; ++ii) {
            const int i = tr * tile_size + ii;
            if (i >= H) break;
            for (int jj = 0; jj < tile_size; ++jj) {
                const int j = tc * tile_size + jj;
                if (j >= W) break;
                const float px = (float)j + 0.5f, py = (float)i + 0.5f;
                float T = 1.0f;
                for (int c = 0; c < CDIM; ++c) pix[c] = 0.0f;
                for (int32_t k = r0; k < r1; ++k) {
                    const int32_t g = sorted_ids[k];
                    if (g < 0 || g >= N) continue;
                    ++e_all;
                    const float dx = means2d[2 * g] - px, dy = means2d[2 * g + 1] - py;
                    const float a = conics[3 * g], b = conics[3 * g + 1], cc = conics[3 * g + 2];
                    const float sigma = 0.5f * (a * dx * dx + cc * dy * dy) + b * dx * dy;
                    float alpha = opacities[g] * expf(-sigma);
                    if (alpha > 0.999f) alpha = 0.999f;
                    if (sigma < 0.0f || alpha < (1.0f / 255.0f)) continue;
                    const float next_T = T * (1.0f - alpha);
                    if (next_T <= 1e-4f) break;
                    const float vis = alpha * T;
                    for (int c = 0; c < CDIM; ++c) pix[c] += colors[(int64_t)g * CDIM + c] * vis;
                    T = next_T;
                    ++e_pass;
                }
                float* out = image + ((int64_t)i * W + j) * CDIM;
                for (int c = 0; c < CDIM; ++c) out[c] = pix[c] + T * background[c];
            }
        }
    }
    if (stats) { stats[0] += e_all; stats[1] += e_pass; }
}

/* ------------------------------------------------------------------------------------
 * fp64 variants (SURVEY 7 step 1d, H3): the same algorithms evaluated in double precision
 * from the same fp32 inputs.  They are the yardstick of the error-budget tests: the error of
 * a GPU kernel against these must not exceed the error the reference's own fp32 arithmetic has
 * against them.  Thresholds are the reference's constants (rasterization.mojo:143-150).
 * ---------------------------------------------------------------------------------- */
void oracle_project_f64(
    int64_t N, const float* means3d, const float* log_scales, const float* quats,
    const float* viewmat, double fx, double fy, double cx, double cy, int W, int H,
    double near_plane, double far_plane, double eps2d,
    double* means2d, double* conics, double* depths, double* radii_real /* [N,2] 3.33 sqrt(c), 0 if culled */)
{
    const double Rv[3][3] = {
        {viewmat[0], viewmat[1], viewmat[2]},
        {viewmat[4], viewmat[5], viewmat[6]},
        {viewmat[8], viewmat[9], viewmat[10]}};
    const double tv[3] = {viewmat[3], viewmat[7], viewmat[11]};
    const double tan_fovx = 0.5 * (double)W / fx, tan_fovy = 0.5 * (double)H / fy;
    const double lim_x_pos = ((double)W - cx) / fx + 0.3 * tan_fovx, lim_x_neg = cx / fx + 0.3 * tan_fovx;
    const double lim_y_pos = ((double)H - cy) / fy + 0.3 * tan_fovy, lim_y_neg = cy / fy + 0.3 * tan_fovy;
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < N; ++i) {
        const float* mu = means3d + 3 * i;
        const float* ls = log_scales + 3 * i;
        const float* q = quats + 4 * i;
        double mc[3];
        for (int r = 0; r < 3; ++r) mc[r] = Rv[r][0] * mu[0] + Rv[r][1] * mu[1] + Rv[r][2] * mu[2] + tv[r];
        double nrm = sqrt((double)q[0] * q[0] + (double)q[1] * q[1] + (double)q[2] * q[2] + (double)q[3] * q[3]);
        if (nrm < 1e-12) nrm = 1e-12;
        const double w = q[0] / nrm, x = q[1] / nrm, y = q[2] / nrm, z = q[3] / nrm;
        const double R[3][3] = {
            {1.0 - 2.0 * (y * y + z * z), 2.0 * (x * y - w * z), 2.0 * (x * z + w * y)},
            {2.0 * (x * y + w * z), 1.0 - 2.0 * (x * x + z * z), 2.0 * (y * z - w * x)},
            {2.0 * (x * z - w * y), 2.0 * (y * z + w * x), 1.0 - 2.0 * (x * x + y * y)}};
        const double s[3] = {exp((double)ls[0]), exp((double)ls[1]), exp((double)ls[2])};
        double M[3][3], S[3][3], A[3][3], Sc[3][3];
        for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) M[r][c] = R[r][c] * s[c];
        for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c)
            S[r][c] = M[r][0] * M[c][0] + M[r][1] * M[c][1] + M[r][2] * M[c][2];
        for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c)
            A[r][c] = Rv[r][0] * S[0][c] + Rv[r][1] * S[1][c] + Rv[r][2] * S[2][c];
        for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c)
            Sc[r][c] = A[r][0] * Rv[c][0] + A[r][1] * Rv[c][1] + A[r][2] * Rv[c][2];
        const double tz = mc[2], tz2 = tz * tz;
        double rx = mc[0] / tz, ry = mc[1] / tz;
        rx = fmin(fmax(rx, -lim_x_neg), lim_x_pos);
        ry = fmin(fmax(ry, -lim_y_neg), lim_y_pos);
        const double tx = tz * rx, ty = tz * ry;
        const double J[2][3] = {{fx / tz, 0.0, -fx * tx / tz2}, {0.0, fy / tz, -fy * ty / tz2}};
        double JS[2][3];
        for (int r = 0; r < 2; ++r) for (int c = 0; c < 3; ++c)
            JS[r][c] = J[r][0] * Sc[0][c] + J[r][1] * Sc[1][c] + J[r][2] * Sc[2][c];
        double c00 = JS[0][0] * J[0][0] + JS[0][1] * J[0][1] + JS[0][2] * J[0][2];
        const double c01 = JS[0][0] * J[1][0] + JS[0][1] * J[1][1] + JS[0][2] * J[1][2];
        const double c10 = JS[1][0] * J[0][0] + JS[1][1] * J[0][1] + JS[1][2] * J[0][2];
        double c11 = JS[1][0] * J[1][0] + JS[1][1] * J[1][1] + JS[1][2] * J[1][2];
        const double m2x = (fx * mc[0] + cx * mc[2]) / tz, m2y = (fy * mc[1] + cy * mc[2]) / tz;
        c00 += eps2d; c11 += eps2d;
        double det = c00 * c11 - c01 * c10;
        if (!(det >= 1e-10)) det = (det != det) ? det : 1e-10;
        means2d[2 * i] = m2x; means2d[2 * i + 1] = m2y;
        conics[3 * i] = c11 / det; conics[3 * i + 1] = -(c01 + c10) / 2.0 / det; conics[3 * i + 2] = c00 / det;
        depths[i] = tz;
        double r_x = 3.33 * sqrt(c00), r_y = 3.33 * sqrt(c11);
        const int valid = (det > 0.0) && (tz > near_plane) && (tz < far_plane);
        if (!valid) { r_x = 0.0; r_y = 0.0; }
        const int inside = (m2x + ceil(r_x) > 0.0) && (m2x - ceil(r_x) < (double)W) &&
                           (m2y + ceil(r_y) > 0.0) && (m2y - ceil(r_y) < (double)H);
        if (!inside) { r_x = 0.0; r_y = 0.0; }
        radii_real[2 * i] = r_x; radii_real[2 * i + 1] = r_y;
    }
}

/* The rasterizer in double precision, fp32 inputs (kernels/rasterization.mojo:138-162). */
void oracle_rasterize_f64(
    int64_t N, int CDIM, const float* means2d, const float* conics, const float* colors,
    const float* opacities, const float* background, const int32_t* tile_ranges,
    const int32_t* sorted_ids, int W, int H, int tile_size, double* image)
{
    const int tiles_w = (W + tile_size - 1) / tile_size, tiles_h = (H + tile_size - 1) / tile_size;
#pragma omp parallel for schedule(dynamic, 1)
    for (int t = 0; t < tiles_w * tiles_h; ++t) {
        const int tr = t / tiles_w, tc = t % tiles_w;
        const int32_t r0 = tile_ranges[2 * t], r1 = tile_ranges[2 * t + 1];
        double pix[CDIM > 0 ? CDIM : 1];
        for (int ii = 0; ii < tile_size; ++ii) {
            const int i = tr * tile_size + ii;
            if (i >= H) break;
            for (int jj = 0; jj < tile_size; ++jj) {
                const int j = tc * tile_size + jj;
                if (j >= W) break;
                const double px = (double)j + 0.5, py = (double)i + 0.5;
                double T = 1.0;
                for (int c = 0; c < CDIM; ++c) pix[c] = 0.0;
                for (int32_t k = r0; k < r1; ++k) {
                    const int32_t g = sorted_ids[k];
                    if (g < 0 || g >= N) continue;
                    const double dx = (double)means2d[2 * g] - px, dy = (double)means2d[2 * g + 1] - py;
                    const double a = conics[3 * g], b = conics[3 * g + 1], cc = conics[3 * g + 2];
                    const double sigma = 0.5 * (a * dx * dx + cc * dy * dy) + b * dx * dy;
                    double alpha = (double)opacities[g] * exp(-sigma);
                    if (alpha > 0.999) alpha = 0.999;
                    if (sigma < 0.0 || alpha < (1.0 / 255.0)) continue;
                    const double next_T = T * (1.0 - alpha);
                    if (next_T <= 1e-4) break;
                    const double vis = alpha * T;
                    for (int c = 0; c < CDIM; ++c) pix[c] += (double)colors[(int64_t)g * CDIM + c] * vis;
                    T = next_T;
                }
                double* out = image + ((int64_t)i * W + j) * CDIM;
                for (int c = 0; c < CDIM; ++c) out[c] = pix[c] + T * (double)background[c];
            }
        }
    }
}

/* ------------------------------------------------------------------------------------
 * Compositing backward in double precision, fp32 inputs: the derivative of oracle_rasterize_f64's algorithm
 * (the decisions -- sigma >= 0, alpha >= 1/255, the 0.999 clamp, the T (1 - alpha) <= 1e-4 stop -- held fixed).
 * Every pixel walks its tile's list front to back, stores what it composited (alpha_k, exp(-sigma_k), T_k, d_k),
 * then walks that back to front with the upstream gradient g = grad_image[pixel]:
 *   d out / d alpha_k = T_k (c_k . g) - (behind_k . g + T_end bg . g) / (1 - alpha_k),
 *     behind_k = sum_{m > k} c_m alpha_m T_m;
 *   v_sigma = -alpha_k d out / d alpha_k (zero where o exp(-sigma) > 0.999, the clamp);
 *   colour: alpha_k T_k g;  conic: v_sigma (dx^2 / 2, dx dy, dy^2 / 2);  mean: v_sigma (a dx + b dy, b dx + c dy);
 *   opacity: exp(-sigma_k) d out / d alpha_k (zero through the clamp);  background: T_end g.
 * Besides the gradient, per value:
 *   mag   the same sum with every sum and product replaced by sums and products of absolute values: the scale of
 *         the rounding error of any evaluation order, immune to cancellation;
 *   wmag  the same sum with each pixel's term weighted by w_pk (below), in units of 2^-22: a fp32 kernel's error
 *         on the entry is at most rho * wmag + (fp32 additions) 2^-24 mag, rho a small multiple of 2^-22.
 *   count the number of pixels that composited the entry (bounds the fp32 additions, atomics included).
 * Per pixel: T_end, the last composited list index, kappa = sum alpha_k / (1 - alpha_k) (the condition number of
 * T recovered by dividing by (1 - alpha), as both CUDA backwards do), the weight W_p and the borderline flag.
 *
 * Error model (the fast kernel, raster_bwd_pair_kernel, is the coarser of the two CUDA backwards; units of u = 2^-22):
 *   alpha = 2^(L - q) with L = lg2.approx(o) (absolute error <= u), q from the log2-folded record by a chain of three
 *   fp32 FMAs (absolute error <= 4 2^-24 (A dx^2 + |B dx dy| + C dy^2 + |L|) = u log2e (s + |ln o|),
 *   s = a dx^2 / 2 + |b dx dy| + c dy^2 / 2), ex2.approx relative error <= u: the relative error of alpha is
 *     e_k u,  e_k = 2 + s_k + |ln o_k|   (ln2 (1 + s + |ln o|) + 1 <= e).
 *   The generic kernel (expf <= 2 ulp, separately rounded products) errs by <= 2^-24 (4 s + 5) <= e_k u as well.
 *   A relative error eps of alpha_j moves T past it by eps alpha_j / (1 - alpha_j); every step of the forward product
 *   and of the backward recovery (1 - alpha, rcp.approx or IEEE division, the product) adds <= u.  The forward and the
 *   backward each do that once, so the relative error of any recovered T_k, and of T_end, is at most
 *     W_p u,  W_p = sum_j (2 e_j alpha_j / (1 - alpha_j) + 2) + max_j e_j
 *   (the max covers the alphas inside behind_k), and a term of entry k carries at most w_pk = 2 e_k + W_p units:
 *   its own alpha enters at most twice (alpha and the factor 1 / (1 - alpha) of d out / d alpha, whose amplification
 *   alpha / (1 - alpha) is already in W_p), and each of the ~10 fp32 products of a term adds < 1/4 u.
 * Borderline flag: set when a decision lies within twice that error of its threshold, compared in log space (the
 *   error is an absolute error of the exponent: for far-away Gaussians e_k u can exceed 1 while alpha is 0 on both
 *   sides) --
 *   |ln(255 alpha)| <= 2 e_k u;  |ln(o exp(-sigma) / 0.999)| <= 2 e_k u;  |sigma| <= 2 u s_k (s_k > 0);
 *   |ln(T (1 - alpha) / 1e-4)| <= 2 W u, W the weight of the entries up to and including this one.
 * With mask_borderline set, flagged pixels get g = 0 (the backward is linear in g: their terms vanish exactly).
 * Outputs (zeroed here): grad / mag / wmag [N, 6 + C] columns (mean x, y, conic a, b, c, colour 0..C-1, opacity);
 * count [N]; bg [3, C] (grad, mag, wmag); final_T, kappa, weight [H, W]; last_idx [H, W]; border [H, W].
 * Accumulation: per tile into per-list-entry partials, then one omp atomic per entry and value.
 * ---------------------------------------------------------------------------------- */
typedef struct {
    int32_t k;
    int clamped;
    double alpha, vis, T, dx, dy, e;
} bwd_entry_t;

#define BWD_U (1.0 / 4194304.0) /* 2^-22 */

void oracle_raster_bwd_f64(
    int64_t N, int CDIM, const float* means2d, const float* conics, const float* colors,
    const float* opacities, const float* background, const int32_t* tile_ranges,
    const int32_t* sorted_ids, int W, int H, int tile_size, const float* grad_image, int mask_borderline,
    double* grad, double* mag, double* wmag, int64_t* count, double* bg,
    double* final_T, int32_t* last_idx, double* kappa, double* weight, uint8_t* border)
{
    const int tiles_w = (W + tile_size - 1) / tile_size, tiles_h = (H + tile_size - 1) / tile_size;
    const int V = 6 + CDIM;
    const int S = 3 * V + 1; /* per list entry: grad[V], mag[V], wmag[V], count */
    if (CDIM < 1 || CDIM > 16) return;
    memset(grad, 0, sizeof(double) * (size_t)N * V);
    memset(mag, 0, sizeof(double) * (size_t)N * V);
    memset(wmag, 0, sizeof(double) * (size_t)N * V);
    memset(count, 0, sizeof(int64_t) * (size_t)N);
    memset(bg, 0, sizeof(double) * 3 * (size_t)CDIM);
#pragma omp parallel for schedule(dynamic, 1)
    for (int t = 0; t < tiles_w * tiles_h; ++t) {
        const int tr = t / tiles_w, tc = t % tiles_w;
        const int32_t r0 = tile_ranges[2 * t], r1 = tile_ranges[2 * t + 1];
        const int64_t len = r1 > r0 ? (int64_t)(r1 - r0) : 0;
        double* loc = (double*)calloc((size_t)(len > 0 ? len : 1) * S, sizeof(double));
        bwd_entry_t* ent = (bwd_entry_t*)malloc(sizeof(bwd_entry_t) * (size_t)(len > 0 ? len : 1));
        double bg_loc[3 * 16];
        double gp[16], gabs[16];
        for (int q = 0; q < 3 * CDIM; ++q) bg_loc[q] = 0.0;
        for (int ii = 0; ii < tile_size; ++ii) {
            const int i = tr * tile_size + ii;
            if (i >= H) break;
            for (int jj = 0; jj < tile_size; ++jj) {
                const int j = tc * tile_size + jj;
                if (j >= W) break;
                const int64_t pix = (int64_t)i * W + j;
                const double px = (double)j + 0.5, py = (double)i + 0.5;
                /* forward walk: what the pixel composites, and how close each decision is to its threshold */
                double T = 1.0, kap = 0.0, Wrun = 0.0, emax = 0.0;
                int nent = 0, flag = 0;
                int32_t last = -1;
                for (int32_t k = r0; k < r1; ++k) {
                    const int32_t g = sorted_ids[k];
                    if (g < 0 || g >= N) continue;
                    const double dx = (double)means2d[2 * g] - px, dy = (double)means2d[2 * g + 1] - py;
                    const double a = conics[3 * g], b = conics[3 * g + 1], cc = conics[3 * g + 2];
                    const double sigma = 0.5 * (a * dx * dx + cc * dy * dy) + b * dx * dy;
                    const double s = 0.5 * fabs(a) * dx * dx + fabs(b * dx * dy) + 0.5 * fabs(cc) * dy * dy;
                    const double o = opacities[g];
                    const double vis = exp(-sigma);
                    const double araw = o * vis;
                    const double alpha = araw > 0.999 ? 0.999 : araw;
                    const double e = 2.0 + s + (o > 0.0 ? fabs(log(o)) : 0.0);
                    if (s > 0.0 && fabs(sigma) <= 2.0 * BWD_U * s) flag = 1;
                    if (fabs(log(alpha * 255.0)) <= 2.0 * e * BWD_U) flag = 1;
                    if (sigma < 0.0 || alpha < (1.0 / 255.0)) continue;
                    if (fabs(log(araw / 0.999)) <= 2.0 * e * BWD_U) flag = 1;
                    const double next_T = T * (1.0 - alpha);
                    const double Wnext = Wrun + 2.0 * e * alpha / (1.0 - alpha) + 2.0;
                    if (fabs(log(next_T / 1e-4)) <= 2.0 * Wnext * BWD_U) flag = 1;
                    if (next_T <= 1e-4) break;
                    bwd_entry_t* en = &ent[nent++];
                    en->k = k; en->clamped = araw > 0.999; en->alpha = alpha; en->vis = vis; en->T = T;
                    en->dx = dx; en->dy = dy; en->e = e;
                    kap += alpha / (1.0 - alpha);
                    Wrun = Wnext;
                    if (e > emax) emax = e;
                    T = next_T;
                    last = k;
                }
                const double Wp = Wrun + emax;
                final_T[pix] = T; last_idx[pix] = last; kappa[pix] = kap; weight[pix] = Wp;
                border[pix] = (uint8_t)flag;
                const int zero = mask_borderline && flag;
                double bg_dot = 0.0, bg_abs = 0.0;
                for (int c = 0; c < CDIM; ++c) {
                    gp[c] = zero ? 0.0 : (double)grad_image[pix * CDIM + c];
                    gabs[c] = fabs(gp[c]);
                    bg_dot += (double)background[c] * gp[c];
                    bg_abs += fabs((double)background[c] * gp[c]);
                    bg_loc[c] += T * gp[c];
                    bg_loc[CDIM + c] += T * gabs[c];
                    bg_loc[2 * CDIM + c] += (2.0 + Wp) * T * gabs[c];
                }
                /* backward walk */
                double behind = 0.0, behind_abs = 0.0;
                for (int n = nent - 1; n >= 0; --n) {
                    const bwd_entry_t* en = &ent[n];
                    const int32_t g = sorted_ids[en->k];
                    const float* col = colors + (int64_t)g * CDIM;
                    const double a = conics[3 * g], b = conics[3 * g + 1], cc = conics[3 * g + 2];
                    const double Tk = en->T, al = en->alpha, ra = 1.0 / (1.0 - al), fac = al * Tk;
                    const double dx = en->dx, dy = en->dy;
                    double cg = 0.0, cg_abs = 0.0;
                    for (int c = 0; c < CDIM; ++c) {
                        cg += (double)col[c] * gp[c];
                        cg_abs += fabs((double)col[c] * gp[c]);
                    }
                    const double v_alpha = Tk * cg - (behind + T * bg_dot) * ra;
                    const double m_alpha = Tk * cg_abs + (behind_abs + T * bg_abs) * ra;
                    double gv[6 + 16], mv[6 + 16];
                    for (int q = 0; q < V; ++q) gv[q] = mv[q] = 0.0;
                    for (int c = 0; c < CDIM; ++c) { gv[5 + c] = fac * gp[c]; mv[5 + c] = fac * gabs[c]; }
                    if (!en->clamped) {
                        const double vs = -al * v_alpha, ms = al * m_alpha;
                        gv[0] = vs * (a * dx + b * dy);       mv[0] = ms * (fabs(a * dx) + fabs(b * dy));
                        gv[1] = vs * (b * dx + cc * dy);      mv[1] = ms * (fabs(b * dx) + fabs(cc * dy));
                        gv[2] = 0.5 * vs * dx * dx;           mv[2] = 0.5 * ms * dx * dx;
                        gv[3] = vs * dx * dy;                 mv[3] = ms * fabs(dx * dy);
                        gv[4] = 0.5 * vs * dy * dy;           mv[4] = 0.5 * ms * dy * dy;
                        gv[5 + CDIM] = en->vis * v_alpha;     mv[5 + CDIM] = en->vis * m_alpha;
                    }
                    const double w = 2.0 * en->e + Wp;
                    double* L = loc + (int64_t)(en->k - r0) * S;
                    for (int q = 0; q < V; ++q) { L[q] += gv[q]; L[V + q] += mv[q]; L[2 * V + q] += w * mv[q]; }
                    L[3 * V] += 1.0;
                    behind += fac * cg;
                    behind_abs += fac * cg_abs;
                }
            }
        }
        for (int64_t k = 0; k < len; ++k) {
            const double* L = loc + k * S;
            if (L[3 * V] == 0.0) continue;
            const int64_t g = sorted_ids[r0 + k];
            for (int q = 0; q < V; ++q) {
#pragma omp atomic
                grad[g * V + q] += L[q];
#pragma omp atomic
                mag[g * V + q] += L[V + q];
#pragma omp atomic
                wmag[g * V + q] += L[2 * V + q];
            }
#pragma omp atomic
            count[g] += (int64_t)L[3 * V];
        }
        for (int q = 0; q < 3 * CDIM; ++q) {
#pragma omp atomic
            bg[q] += bg_loc[q];
        }
        free(loc);
        free(ent);
    }
}

/* ------------------------------------------------------------------------------------
 * Outlier audit (SURVEY H4).  The alpha >= 1/255 test and the T (1 - alpha) <= 1e-4 stop make a pixel
 * discontinuous in exp(): two correct fp32 implementations may take a different branch when a value sits
 * within rounding distance of a threshold, and the pixel then differs by up to alpha T colour.  That is the
 * ONLY legitimate cause of a value outside the tolerance.  For every listed pixel this routine re-composites
 * the pixel (fp32, the oracle's arithmetic) with each borderline decision forced the other way -- one flip at
 * a time, then pairs -- and reports whether some variant reproduces the observed value within atol + rtol |v|.
 * A decision is borderline when |alpha - 1/255| <= rel_window / 255 or |next_T - 1e-4| <= 10 rel_window * 1e-4
 * (or sigma within rel_window of 0).
 *   pixels[n][2] = (row, col); observed[n][CDIM]; explained[n] (out) = 0 unexplained, 1 one flip, 2 two flips,
 *   3 = the unflipped oracle value is already within tolerance; n_borderline[n] (out).
 * ---------------------------------------------------------------------------------- */
#define AUDIT_MAX_BORDER 24

static void audit_composite(
    int CDIM, const float* means2d, const float* conics, const float* colors, const float* opacities,
    const float* background, const int32_t* sorted_ids, int64_t N, int32_t r0, int32_t r1, float px, float py,
    const int32_t* flip_at, int n_flip, float rel_window, int32_t* border, int* n_border, float* out)
{
    float T = 1.0f;
    float pix[16];
    for (int c = 0; c < CDIM; ++c) pix[c] = 0.0f;
    int nb = 0;
    for (int32_t k = r0; k < r1; ++k) {
        const int32_t g = sorted_ids[k];
        if (g < 0 || g >= N) continue;
        const float dx = means2d[2 * g] - px, dy = means2d[2 * g + 1] - py;
        const float a = conics[3 * g], b = conics[3 * g + 1], cc = conics[3 * g + 2];
        const float sigma = 0.5f * (a * dx * dx + cc * dy * dy) + b * dx * dy;
        float alpha = opacities[g] * expf(-sigma);
        if (alpha > 0.999f) alpha = 0.999f;
        int skip = (sigma < 0.0f || alpha < (1.0f / 255.0f));
        const int near_alpha = fabsf(alpha - (1.0f / 255.0f)) <= rel_window * (1.0f / 255.0f) ||
                               fabsf(sigma) <= rel_window;
        int flipped = 0;
        for (int f = 0; f < n_flip; ++f) if (flip_at[f] == k) flipped = 1;
        if (near_alpha) {
            if (border && nb < AUDIT_MAX_BORDER) border[nb] = k;
            ++nb;
            if (flipped) { skip = !skip; flipped = 0; }
        }
        if (skip) continue;
        const float next_T = T * (1.0f - alpha);
        int stop = next_T <= 1e-4f;
        const int near_T = fabsf(next_T - 1e-4f) <= 10.0f * rel_window * 1e-4f;  /* T carries the error of every earlier alpha */
        if (near_T) {
            if (!near_alpha) {  /* (a Gaussian borderline on both tests is listed once) */
                if (border && nb < AUDIT_MAX_BORDER) border[nb] = k;
                ++nb;
            }
            if (flipped) stop = !stop;
        }
        if (stop) break;
        const float vis = alpha * T;
        for (int c = 0; c < CDIM; ++c) pix[c] += colors[(int64_t)g * CDIM + c] * vis;
        T = next_T;
    }
    for (int c = 0; c < CDIM; ++c) out[c] = pix[c] + T * background[c];
    if (n_border) *n_border = nb;
}

void oracle_raster_audit(
    int64_t N, int CDIM, const float* means2d, const float* conics, const float* colors,
    const float* opacities, const float* background, const int32_t* tile_ranges,
    const int32_t* sorted_ids, int W, int H, int tile_size,
    int64_t n_pixels, const int32_t* pixels, const float* observed, float atol, float rtol, float rel_window,
    int32_t* explained, int32_t* n_borderline)
{
    (void)H;
    const int tiles_w = (W + tile_size - 1) / tile_size;
    if (CDIM > 16) { for (int64_t n = 0; n < n_pixels; ++n) { explained[n] = 0; n_borderline[n] = -1; } return; }
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t n = 0; n < n_pixels; ++n) {
        const int i = pixels[2 * n], j = pixels[2 * n + 1];
        const int t = (i / tile_size) * tiles_w + (j / tile_size);
        const int32_t r0 = tile_ranges[2 * t], r1 = tile_ranges[2 * t + 1];
        const float px = (float)j + 0.5f, py = (float)i + 0.5f;
        const float* obs = observed + n * CDIM;
        int32_t border[AUDIT_MAX_BORDER];
        int nb = 0;
        float out[16];
        audit_composite(CDIM, means2d, conics, colors, opacities, background, sorted_ids, N, r0, r1, px, py,
                        NULL, 0, rel_window, border, &nb, out);
        n_borderline[n] = nb;
        int ok = 1;
        for (int c = 0; c < CDIM; ++c) if (fabsf(out[c] - obs[c]) > atol + rtol * fabsf(obs[c])) ok = 0;
        if (ok) { explained[n] = 3; continue; }
        explained[n] = 0;
        const int m = nb < AUDIT_MAX_BORDER ? nb : AUDIT_MAX_BORDER;
        for (int f = 0; f < m && !explained[n]; ++f) {
            audit_composite(CDIM, means2d, conics, colors, opacities, background, sorted_ids, N, r0, r1, px, py,
                            &border[f], 1, rel_window, NULL, NULL, out);
            ok = 1;
            for (int c = 0; c < CDIM; ++c) if (fabsf(out[c] - obs[c]) > atol + rtol * fabsf(obs[c])) ok = 0;
            if (ok) explained[n] = 1;
        }
        /* a flip can make a later decision borderline that was not before (T changed): pairs re-enumerate */
        for (int f = 0; f < m && !explained[n]; ++f) {
            int32_t border2[AUDIT_MAX_BORDER];
            int nb2 = 0;
            audit_composite(CDIM, means2d, conics, colors, opacities, background, sorted_ids, N, r0, r1, px, py,
                            &border[f], 1, rel_window, border2, &nb2, out);
            const int m2 = nb2 < AUDIT_MAX_BORDER ? nb2 : AUDIT_MAX_BORDER;
            for (int f2 = 0; f2 < m2 && !explained[n]; ++f2) {
                if (border2[f2] == border[f]) continue;
                int32_t two[2] = {border[f], border2[f2]};
                audit_composite(CDIM, means2d, conics, colors, opacities, background, sorted_ids, N, r0, r1, px, py,
                                two, 2, rel_window, NULL, NULL, out);
                ok = 1;
                for (int c = 0; c < CDIM; ++c) if (fabsf(out[c] - obs[c]) > atol + rtol * fabsf(obs[c])) ok = 0;
                if (ok) explained[n] = 2;
            }
        }
    }
}
