// LiDAR beam direction of pixel id p = j*W + i (column i, row j), in the sensor frame.  Shared by ray
// generation (k_lidar_rays, scene.cu) and range image -> point cloud (eval.cu), so a synthesized point is
// exactly the generated ray direction times the range.
#pragma once
#include <stdint.h>

// dataset_utils.py:512-530: beta = -(i - W/2)/W * fov_hoz/180*pi, alpha = (fov_up - j/H*fov)/180*pi,
// d = (cos a cos b, cos a sin b, sin a).  Every product / quotient is rounded on its own (no FMA contraction).
__device__ __forceinline__ void lidar_dir(int64_t p, uint32_t H, uint32_t W, float fov_up, float fov,
                                          float fov_hoz, float& x, float& y, float& z) {
    const float i = (float)(p % W), j = (float)(p / W);
    const float kPi = 3.14159265358979323846f;
    float beta = __fdiv_rn(-(i - (float)W * 0.5f), (float)W);
    beta = __fmul_rn(__fdiv_rn(__fmul_rn(beta, fov_hoz), 180.0f), kPi);
    float alpha = __fsub_rn(fov_up, __fmul_rn(__fdiv_rn(j, (float)H), fov));
    alpha = __fmul_rn(__fdiv_rn(alpha, 180.0f), kPi);
    float sa, ca, sb, cb;
    sincosf(alpha, &sa, &ca);
    sincosf(beta, &sb, &cb);
    x = __fmul_rn(ca, cb);
    y = __fmul_rn(ca, sb);
    z = sa;
}
