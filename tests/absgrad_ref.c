/* fp64 reference of AbsGS's absolute screen-space gradient (gsplat's `absgrad`), for the tests.
 *
 * abs_means2d[g, k] = sum over the pixels p where Gaussian g was composited of |d L_p / d means2d[g, k]|, the term of
 * pixel p being v_sigma (a dx + b dy) for x and v_sigma (b dx + c dy) for y, the absolute value taken per pixel.
 *
 * The walk is oracle_raster_bwd_f64's (oracle/oracle.c), in double precision on fp32 inputs, with the same decisions
 * held fixed (sigma >= 0, alpha >= 1/255, no gradient through the 0.999 clamp, the T (1 - alpha) <= 1e-4 stop) and the
 * same operation order for the signed term, so sum_p of the signed terms equals that function's grad_means2d.  Pixels
 * to leave out (its borderline flag) are left out by zeroing them in grad_image: the backward is linear in it.
 * Output: abs_means2d [N, 2] (zeroed here) and signed_means2d [N, 2] (the same sums without |.|, zeroed here).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
    int32_t k;
    int clamped;
    double alpha, T, dx, dy;
} absgrad_entry_t;

void absgrad_ref_f64(int64_t N, int CDIM, const float* means2d, const float* conics, const float* colors,
                     const float* opacities, const float* background, const int32_t* tile_ranges,
                     const int32_t* sorted_ids, int W, int H, int tile_size, const float* grad_image,
                     double* abs_means2d, double* signed_means2d)
{
    const int tiles_w = (W + tile_size - 1) / tile_size, tiles_h = (H + tile_size - 1) / tile_size;
    memset(abs_means2d, 0, sizeof(double) * (size_t)N * 2);
    memset(signed_means2d, 0, sizeof(double) * (size_t)N * 2);
    if (CDIM < 1 || CDIM > 16) return;
#pragma omp parallel for schedule(dynamic, 1)
    for (int t = 0; t < tiles_w * tiles_h; ++t) {
        const int tr = t / tiles_w, tc = t % tiles_w;
        const int32_t r0 = tile_ranges[2 * t], r1 = tile_ranges[2 * t + 1];
        const int64_t len = r1 > r0 ? (int64_t)(r1 - r0) : 0;
        double* loc = (double*)calloc((size_t)(len > 0 ? len : 1) * 4, sizeof(double)); /* |x|, |y|, x, y */
        absgrad_entry_t* ent = (absgrad_entry_t*)malloc(sizeof(absgrad_entry_t) * (size_t)(len > 0 ? len : 1));
        double gp[16];
        for (int ii = 0; ii < tile_size; ++ii) {
            const int i = tr * tile_size + ii;
            if (i >= H) break;
            for (int jj = 0; jj < tile_size; ++jj) {
                const int j = tc * tile_size + jj;
                if (j >= W) break;
                const int64_t pix = (int64_t)i * W + j;
                const double px = (double)j + 0.5, py = (double)i + 0.5;
                double T = 1.0;
                int nent = 0;
                for (int32_t k = r0; k < r1; ++k) {
                    const int32_t g = sorted_ids[k];
                    if (g < 0 || g >= N) continue;
                    const double dx = (double)means2d[2 * g] - px, dy = (double)means2d[2 * g + 1] - py;
                    const double a = conics[3 * g], b = conics[3 * g + 1], cc = conics[3 * g + 2];
                    const double sigma = 0.5 * (a * dx * dx + cc * dy * dy) + b * dx * dy;
                    const double araw = (double)opacities[g] * exp(-sigma);
                    const double alpha = araw > 0.999 ? 0.999 : araw;
                    if (sigma < 0.0 || alpha < (1.0 / 255.0)) continue;
                    const double next_T = T * (1.0 - alpha);
                    if (next_T <= 1e-4) break;
                    absgrad_entry_t* en = &ent[nent++];
                    en->k = k; en->clamped = araw > 0.999; en->alpha = alpha; en->T = T; en->dx = dx; en->dy = dy;
                    T = next_T;
                }
                double bg_dot = 0.0;
                for (int c = 0; c < CDIM; ++c) {
                    gp[c] = (double)grad_image[pix * CDIM + c];
                    bg_dot += (double)background[c] * gp[c];
                }
                double behind = 0.0;
                for (int n = nent - 1; n >= 0; --n) {
                    const absgrad_entry_t* en = &ent[n];
                    const int32_t g = sorted_ids[en->k];
                    const float* col = colors + (int64_t)g * CDIM;
                    const double a = conics[3 * g], b = conics[3 * g + 1], cc = conics[3 * g + 2];
                    const double Tk = en->T, al = en->alpha, ra = 1.0 / (1.0 - al), fac = al * Tk;
                    double cg = 0.0;
                    for (int c = 0; c < CDIM; ++c) cg += (double)col[c] * gp[c];
                    const double v_alpha = Tk * cg - (behind + T * bg_dot) * ra;
                    if (!en->clamped) {
                        const double vs = -al * v_alpha;
                        const double mx = vs * (a * en->dx + b * en->dy), my = vs * (b * en->dx + cc * en->dy);
                        double* L = loc + (int64_t)(en->k - r0) * 4;
                        L[0] += fabs(mx); L[1] += fabs(my); L[2] += mx; L[3] += my;
                    }
                    behind += fac * cg;
                }
            }
        }
        for (int64_t k = 0; k < len; ++k) {
            const double* L = loc + k * 4;
            const int64_t g = sorted_ids[r0 + k];
            if (g < 0 || g >= N) continue;
            for (int q = 0; q < 2; ++q) {
#pragma omp atomic
                abs_means2d[g * 2 + q] += L[q];
#pragma omp atomic
                signed_means2d[g * 2 + q] += L[2 + q];
            }
        }
        free(loc);
        free(ent);
    }
}
