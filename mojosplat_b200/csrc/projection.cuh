// Camera constants of the projection, shared by the forward (projection.cu) and its backward (projection_bwd.cu).
#pragma once

#include "common.cuh"

namespace bsplat {

struct ProjCam {
    float r[9];
    float t[3];
    float fx, fy, cx, cy;
    float lim_x_pos, lim_x_neg, lim_y_pos, lim_y_neg;
    float near_plane, far_plane, eps2d;
    int W, H;
};

__host__ __device__ inline ProjCam make_proj_cam(const bsplat_camera& c, float eps2d) {
    ProjCam p;
    for (int r = 0; r < 3; ++r) {
        for (int k = 0; k < 3; ++k) p.r[3 * r + k] = c.viewmat[4 * r + k];
        p.t[r] = c.viewmat[4 * r + 3];
    }
    p.fx = c.fx; p.fy = c.fy; p.cx = c.cx; p.cy = c.cy;
    p.W = c.width; p.H = c.height;
    // projection.py:137-146, evaluated in fp32 like the reference tensors
    const float W = (float)c.width, H = (float)c.height;
    const float tan_fovx = 0.5f * W / c.fx, tan_fovy = 0.5f * H / c.fy;
    p.lim_x_pos = (W - c.cx) / c.fx + 0.3f * tan_fovx;
    p.lim_x_neg = c.cx / c.fx + 0.3f * tan_fovx;
    p.lim_y_pos = (H - c.cy) / c.fy + 0.3f * tan_fovy;
    p.lim_y_neg = c.cy / c.fy + 0.3f * tan_fovy;
    p.near_plane = c.near_plane; p.far_plane = c.far_plane; p.eps2d = eps2d;
    return p;
}

}  // namespace bsplat
