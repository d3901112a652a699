// Stage 1, backward -- gradients of the EWA projection (projection.cu: project_core) with respect to the 3D
// parameters: d loss / d (means3d, log_scales, raw quats) from d loss / d (means2d, conics, depths).
//
// Same shape as the forward: one thread per Gaussian, the 3-wide AoS rows (means3d, log_scales, v_conics in;
// v_means3d, v_log_scales out) staged through shared memory so that every global access is coalesced, the 2- and
// 4-wide rows as 64 / 128-bit accesses.  The forward intermediates are recomputed in fp32 from the inputs (nothing is
// saved by the forward): 72 B read + 40 B written per Gaussian, HBM-bound.  This file is not bound by the reference's
// rounding (the gradient is checked against fp64 autograd), so it is built with FMA contraction allowed.
//
// Differentiated chain (both rule sets): s = exp(log_scales); quaternion -> F.normalize (eps 1e-12) -> R;
// Sigma = (R S)(R S)^T; Sigma_c = Rv Sigma Rv^T; pinhole Jacobian J with x/z, y/z clamped to [-lim_neg, lim_pos]
// (torch.clamp: the gradient passes inside the bounds, bounds included); cov2d = J Sigma_c J^T + eps2d I;
// BSPLAT_SEM_TORCH clamps det at 1e-10 (no gradient where clamped); conic = (c11, -(c01 + c10) / 2, c00) / det;
// means2d = (K mu_c) / z; depth = z.  Rows with radii == (0, 0) (culled by the forward) are written as zeros.
#include "projection.cuh"

namespace bsplat {

constexpr int kProjBwdThreads = 256;

struct Grad3 {
    float v[3];
};

// One visible Gaussian: reads the inputs, writes d loss / d (mu, log_scales, quat).
template <int SEM>
__device__ __forceinline__ void project_bwd_one(const ProjCam& cam, const float mux, const float muy, const float muz,
                                                const float ls0, const float ls1, const float ls2, const float4 q,
                                                const float2 vm2, const float vk0, const float vk1, const float vk2,
                                                const float vdepth, Grad3& v_mu, Grad3& v_ls, float4& v_q) {
    const float* rv = cam.r;
    // ---- forward, recomputed ----
    const float mcx = rv[0] * mux + rv[1] * muy + rv[2] * muz + cam.t[0];
    const float mcy = rv[3] * mux + rv[4] * muy + rv[5] * muz + cam.t[1];
    const float tz = rv[6] * mux + rv[7] * muy + rv[8] * muz + cam.t[2];
    const float s[3] = {expf(ls0), expf(ls1), expf(ls2)};
    const float nrm_raw = sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w);
    const float inv_n = 1.0f / fmaxf(nrm_raw, 1e-12f);
    const float w = q.x * inv_n, x = q.y * inv_n, y = q.z * inv_n, z = q.w * inv_n;
    const float R[3][3] = {{1.0f - 2.0f * (y * y + z * z), 2.0f * (x * y - w * z), 2.0f * (x * z + w * y)},
                           {2.0f * (x * y + w * z), 1.0f - 2.0f * (x * x + z * z), 2.0f * (y * z - w * x)},
                           {2.0f * (x * z - w * y), 2.0f * (y * z + w * x), 1.0f - 2.0f * (x * x + y * y)}};
    float M[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) M[r][c] = R[r][c] * s[c];
    float S[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = r; c < 3; ++c) S[r][c] = S[c][r] = M[r][0] * M[c][0] + M[r][1] * M[c][1] + M[r][2] * M[c][2];
    float A[3][3], Sc[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) A[r][c] = rv[3 * r] * S[0][c] + rv[3 * r + 1] * S[1][c] + rv[3 * r + 2] * S[2][c];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) Sc[r][c] = A[r][0] * rv[3 * c] + A[r][1] * rv[3 * c + 1] + A[r][2] * rv[3 * c + 2];
    const float rz = 1.0f / tz;
    const float rxz_raw = mcx * rz, ryz_raw = mcy * rz;
    const bool x_in = rxz_raw >= -cam.lim_x_neg && rxz_raw <= cam.lim_x_pos;
    const bool y_in = ryz_raw >= -cam.lim_y_neg && ryz_raw <= cam.lim_y_pos;
    const float rxz = fminf(fmaxf(rxz_raw, -cam.lim_x_neg), cam.lim_x_pos);
    const float ryz = fminf(fmaxf(ryz_raw, -cam.lim_y_neg), cam.lim_y_pos);
    const float tx = tz * rxz, ty = tz * ryz;
    const float rz2 = rz * rz;
    const float J00 = cam.fx * rz, J11 = cam.fy * rz, J02 = -cam.fx * tx * rz2, J12 = -cam.fy * ty * rz2;
    float JS[2][3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        JS[0][c] = J00 * Sc[0][c] + J02 * Sc[2][c];
        JS[1][c] = J11 * Sc[1][c] + J12 * Sc[2][c];
    }
    const float c00 = JS[0][0] * J00 + JS[0][2] * J02 + cam.eps2d;
    const float c01 = JS[0][1] * J11 + JS[0][2] * J12;
    const float c10 = JS[1][0] * J00 + JS[1][2] * J02;
    const float c11 = JS[1][1] * J11 + JS[1][2] * J12 + cam.eps2d;
    float det = c00 * c11 - c01 * c10;
    const bool det_pass = (SEM != BSPLAT_SEM_TORCH) || det >= 1e-10f;
    if (!det_pass) det = 1e-10f;
    const float idet = 1.0f / det;
    const float k0 = c11 * idet, k1 = -0.5f * (c01 + c10) * idet, k2 = c00 * idet;

    // ---- backward ----
    // conic = n / det: v_n = v_k / det, v_det = -(v_k . k) / det
    float v_c00 = vk2 * idet, v_c11 = vk0 * idet;
    float v_c01 = -0.5f * vk1 * idet, v_c10 = v_c01;
    if (det_pass) {
        const float v_det = -(vk0 * k0 + vk1 * k1 + vk2 * k2) * idet;
        v_c00 += v_det * c11; v_c11 += v_det * c00;
        v_c01 -= v_det * c10; v_c10 -= v_det * c01;
    }
    // cov = J Sc J^T with W = V + V^T: v_J = W (J Sc), and v_Sc + v_Sc^T = J^T W J
    const float W00 = 2.0f * v_c00, W01 = v_c01 + v_c10, W11 = 2.0f * v_c11;
    const float vJ00 = W00 * JS[0][0] + W01 * JS[1][0];
    const float vJ02 = W00 * JS[0][2] + W01 * JS[1][2];
    const float vJ11 = W01 * JS[0][1] + W11 * JS[1][1];
    const float vJ12 = W01 * JS[0][2] + W11 * JS[1][2];
    const float u02 = W00 * J02 + W01 * J12, u12 = W01 * J02 + W11 * J12;
    float G[3][3];
    G[0][0] = J00 * J00 * W00; G[0][1] = G[1][0] = J00 * W01 * J11; G[0][2] = G[2][0] = J00 * u02;
    G[1][1] = J11 * J11 * W11; G[1][2] = G[2][1] = J11 * u12;  G[2][2] = J02 * u02 + J12 * u12;
    // v_Sigma + v_Sigma^T = Rv^T G Rv =: H; v_M = H M
    float B[3][3], H[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) B[r][c] = G[r][0] * rv[c] + G[r][1] * rv[3 + c] + G[r][2] * rv[6 + c];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = r; c < 3; ++c) H[r][c] = H[c][r] = rv[r] * B[0][c] + rv[3 + r] * B[1][c] + rv[6 + r] * B[2][c];
    float vR[3][3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float vs = 0.0f;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float vM = H[r][0] * M[0][c] + H[r][1] * M[1][c] + H[r][2] * M[2][c];
            vR[r][c] = vM * s[c];
            vs += vM * R[r][c];
        }
        v_ls.v[c] = vs * s[c];
    }
    // R(w, x, y, z) -> normalised quaternion
    const float vw = 2.0f * (-z * vR[0][1] + y * vR[0][2] + z * vR[1][0] - x * vR[1][2] - y * vR[2][0] + x * vR[2][1]);
    const float vx = 2.0f * (y * vR[0][1] + z * vR[0][2] + y * vR[1][0] - 2.0f * x * vR[1][1] - w * vR[1][2] +
                             z * vR[2][0] + w * vR[2][1] - 2.0f * x * vR[2][2]);
    const float vy = 2.0f * (-2.0f * y * vR[0][0] + x * vR[0][1] + w * vR[0][2] + x * vR[1][0] + z * vR[1][2] -
                             w * vR[2][0] + z * vR[2][1] - 2.0f * y * vR[2][2]);
    const float vz = 2.0f * (-2.0f * z * vR[0][0] - w * vR[0][1] + x * vR[0][2] + w * vR[1][0] - 2.0f * z * vR[1][1] +
                             y * vR[1][2] + x * vR[2][0] + y * vR[2][1]);
    // F.normalize: q / max(|q|, eps); the norm's gradient passes where |q| >= eps
    const float dot = nrm_raw >= 1e-12f ? (w * vw + x * vx + y * vy + z * vz) : 0.0f;
    v_q = make_float4((vw - w * dot) * inv_n, (vx - x * dot) * inv_n, (vy - y * dot) * inv_n, (vz - z * dot) * inv_n);

    // camera-space mean: J (through tx = z * clamp(x / z), ty), means2d, depth
    const float v_tx = -cam.fx * rz2 * vJ02, v_ty = -cam.fy * rz2 * vJ12;
    float v_tz = -J00 * rz * vJ00 - J11 * rz * vJ11 - 2.0f * J02 * rz * vJ02 - 2.0f * J12 * rz * vJ12;
    v_tz += rxz * v_tx + ryz * v_ty;
    float v_mcx = 0.0f, v_mcy = 0.0f;
    if (x_in) {
        const float v_r = tz * v_tx;
        v_mcx += v_r * rz;
        v_tz -= rxz_raw * rz * v_r;
    }
    if (y_in) {
        const float v_r = tz * v_ty;
        v_mcy += v_r * rz;
        v_tz -= ryz_raw * rz * v_r;
    }
    v_mcx += cam.fx * rz * vm2.x;
    v_mcy += cam.fy * rz * vm2.y;
    v_tz -= (cam.fx * mcx * vm2.x + cam.fy * mcy * vm2.y) * rz2;
    v_tz += vdepth;
    // mu_c = Rv mu + t
#pragma unroll
    for (int c = 0; c < 3; ++c) v_mu.v[c] = rv[c] * v_mcx + rv[3 + c] * v_mcy + rv[6 + c] * v_tz;
}

// vec_ok bits: 1 quats, 2 v_quats (16-byte aligned); 4 radii, 8 v_means2d (8-byte aligned)
template <int SEM>
__global__ void __launch_bounds__(kProjBwdThreads, 4)
project_bwd_kernel(const int64_t N, const float* __restrict__ means3d, const float* __restrict__ log_scales,
                   const float* __restrict__ quats, const ProjCam cam, const int32_t* __restrict__ radii,
                   const float* __restrict__ v_means2d, const float* __restrict__ v_conics,
                   const float* __restrict__ v_depths, float* __restrict__ v_means3d,
                   float* __restrict__ v_log_scales, float* __restrict__ v_quats, const int vec_ok) {
    // 3-wide rows: means3d -> v_means3d, log_scales -> v_log_scales in place (each thread reads and then overwrites
    // its own row), v_conics in
    __shared__ float s_mean[kProjBwdThreads * 3];
    __shared__ float s_scale[kProjBwdThreads * 3];
    __shared__ float s_vcon[kProjBwdThreads * 3];
    const int tid = threadIdx.x;
    const int64_t base = (int64_t)blockIdx.x * kProjBwdThreads;
    const int n_here = (int)min((int64_t)kProjBwdThreads, N - base);
    const int n3 = n_here * 3;
    const float* gm = means3d + base * 3;
    const float* gs = log_scales + base * 3;
    const float* gc = v_conics + base * 3;
    if (n_here == kProjBwdThreads) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            s_mean[tid + k * kProjBwdThreads] = __ldg(gm + tid + k * kProjBwdThreads);
            s_scale[tid + k * kProjBwdThreads] = __ldg(gs + tid + k * kProjBwdThreads);
            s_vcon[tid + k * kProjBwdThreads] = __ldg(gc + tid + k * kProjBwdThreads);
        }
    } else {
        for (int j = tid; j < n3; j += kProjBwdThreads) {
            s_mean[j] = __ldg(gm + j);
            s_scale[j] = __ldg(gs + j);
            s_vcon[j] = __ldg(gc + j);
        }
    }
    __syncthreads();
    if (tid < n_here) {
        const int64_t i = base + tid;
        const int2 rad = (vec_ok & 4) ? __ldg(reinterpret_cast<const int2*>(radii) + i)
                                      : make_int2(__ldg(radii + 2 * i), __ldg(radii + 2 * i + 1));
        Grad3 v_mu = {{0.0f, 0.0f, 0.0f}}, v_ls = {{0.0f, 0.0f, 0.0f}};
        float4 v_q = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (rad.x != 0 || rad.y != 0) {
            const float4 q = (vec_ok & 1) ? __ldg(reinterpret_cast<const float4*>(quats) + i)
                                          : make_float4(__ldg(quats + 4 * i), __ldg(quats + 4 * i + 1),
                                                        __ldg(quats + 4 * i + 2), __ldg(quats + 4 * i + 3));
            const float2 vm2 = (vec_ok & 8) ? __ldg(reinterpret_cast<const float2*>(v_means2d) + i)
                                            : make_float2(__ldg(v_means2d + 2 * i), __ldg(v_means2d + 2 * i + 1));
            const float vd = v_depths != nullptr ? __ldg(v_depths + i) : 0.0f;
            project_bwd_one<SEM>(cam, s_mean[3 * tid], s_mean[3 * tid + 1], s_mean[3 * tid + 2], s_scale[3 * tid],
                                 s_scale[3 * tid + 1], s_scale[3 * tid + 2], q, vm2, s_vcon[3 * tid],
                                 s_vcon[3 * tid + 1], s_vcon[3 * tid + 2], vd, v_mu, v_ls, v_q);
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            s_mean[3 * tid + k] = v_mu.v[k];
            s_scale[3 * tid + k] = v_ls.v[k];
        }
        if (vec_ok & 2) {
            reinterpret_cast<float4*>(v_quats)[i] = v_q;
        } else {
            v_quats[4 * i] = v_q.x; v_quats[4 * i + 1] = v_q.y; v_quats[4 * i + 2] = v_q.z; v_quats[4 * i + 3] = v_q.w;
        }
    }
    __syncthreads();
    float* om = v_means3d + base * 3;
    float* os = v_log_scales + base * 3;
    if (n_here == kProjBwdThreads) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            om[tid + k * kProjBwdThreads] = s_mean[tid + k * kProjBwdThreads];
            os[tid + k * kProjBwdThreads] = s_scale[tid + k * kProjBwdThreads];
        }
    } else {
        for (int j = tid; j < n3; j += kProjBwdThreads) {
            om[j] = s_mean[j];
            os[j] = s_scale[j];
        }
    }
}

}  // namespace bsplat

using namespace bsplat;

extern "C" int bsplat_project_bwd(int64_t N, const float* means3d, const float* log_scales, const float* quats,
                                  const bsplat_camera* cam_host, float eps2d, int32_t semantics, const int32_t* radii,
                                  const float* v_means2d, const float* v_conics, const float* v_depths,
                                  float* v_means3d, float* v_log_scales, float* v_quats, void* stream) {
    if (N < 0 || !cam_host) return BSPLAT_E_ARG;
    if (semantics != BSPLAT_SEM_TORCH && semantics != BSPLAT_SEM_GSPLAT) return BSPLAT_E_ARG;
    if (N == 0) return BSPLAT_OK;
    if (!means3d || !log_scales || !quats || !radii || !v_means2d || !v_conics || !v_means3d || !v_log_scales ||
        !v_quats)
        return BSPLAT_E_ARG;
    const ProjCam pc = make_proj_cam(*cam_host, eps2d);
    int vec_ok = 0;
    if ((reinterpret_cast<uintptr_t>(quats) & 15u) == 0) vec_ok |= 1;
    if ((reinterpret_cast<uintptr_t>(v_quats) & 15u) == 0) vec_ok |= 2;
    if ((reinterpret_cast<uintptr_t>(radii) & 7u) == 0) vec_ok |= 4;
    if ((reinterpret_cast<uintptr_t>(v_means2d) & 7u) == 0) vec_ok |= 8;
    const unsigned grid = (unsigned)ceil_div(N, kProjBwdThreads);
    cudaStream_t s = (cudaStream_t)stream;
    if (semantics == BSPLAT_SEM_TORCH)
        project_bwd_kernel<BSPLAT_SEM_TORCH><<<grid, kProjBwdThreads, 0, s>>>(
            N, means3d, log_scales, quats, pc, radii, v_means2d, v_conics, v_depths, v_means3d, v_log_scales, v_quats,
            vec_ok);
    else
        project_bwd_kernel<BSPLAT_SEM_GSPLAT><<<grid, kProjBwdThreads, 0, s>>>(
            N, means3d, log_scales, quats, pc, radii, v_means2d, v_conics, v_depths, v_means3d, v_log_scales, v_quats,
            vec_ok);
    BSPLAT_LAUNCH_CHECK();
    return BSPLAT_OK;
}
