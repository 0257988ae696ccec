// Per-ray core of the surface-hit step of prior extraction (reference: scripts/extract_priors.py:100-126): the hit of a
// camera ray at its threshold depth, in scene units and in metres, and the range / height selector.
//   points_scaled = o + d * depth          one fmaf per component
//   points_m      = points_scaled / pose_scale_factor
//   keep          = depth / pose_scale_factor <= max_range_m  and  z_min_m <= points_m.z <= z_max_m
// A bound that is not finite (inf or NaN) is not applied.
// Plain C++ shared by the CUDA kernel (csrc/hits.cu) and the host harness of tests/test_extract_host.py.
#pragma once

#ifndef PS_HD
#define PS_HD
#endif
#ifndef PS_FMAF
#include <cmath>
#define PS_FMAF(a, b, c) (std::fmaf((a), (b), (c)))
#define PS_FDIV(a, b) ((a) / (b))
#define PS_ISFINITE(a) (std::isfinite(a))
#endif

namespace ps {
namespace hits {

// o, d: the ray's origin / direction (3 floats); writes points_scaled[3], points_m[3]; returns keep
PS_HD inline bool surface_hit(const float* o, const float* d, float depth, float pose_scale, float max_range_m, float z_min_m,
                              float z_max_m, float* points_scaled, float* points_m) {
    for (int k = 0; k < 3; ++k) {
        points_scaled[k] = PS_FMAF(d[k], depth, o[k]);
        points_m[k] = PS_FDIV(points_scaled[k], pose_scale);
    }
    const float range_m = PS_FDIV(depth, pose_scale);
    const bool in_range = !PS_ISFINITE(max_range_m) || range_m <= max_range_m;
    const bool above = !PS_ISFINITE(z_min_m) || z_min_m <= points_m[2];
    const bool below = !PS_ISFINITE(z_max_m) || points_m[2] <= z_max_m;
    return in_range && above && below;
}

}  // namespace hits
}  // namespace ps
