// Surface hits of camera rays at their threshold depth (prior extraction, scripts/extract_priors.py:100-126): one thread
// per ray, the arithmetic of hits_core.h.
#include <cmath>

#include "common.cuh"

#define PS_HD __device__
#define PS_FMAF(a, b, c) fmaf((a), (b), (c))
#define PS_FDIV(a, b) __fdiv_rn((a), (b))
#define PS_ISFINITE(a) isfinite(a)
#include "hits_core.h"

namespace ps {
namespace {

__global__ void surface_hits_kernel(const float* __restrict__ origins, const float* __restrict__ dirs,
                                    const float* __restrict__ depth, int64_t N, float pose_scale, float max_range_m,
                                    float z_min_m, float z_max_m, float* __restrict__ points_scaled,
                                    float* __restrict__ points_m, uint8_t* __restrict__ keep) {
    for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
        const float o[3] = {__ldg(origins + 3 * n), __ldg(origins + 3 * n + 1), __ldg(origins + 3 * n + 2)};
        const float d[3] = {__ldg(dirs + 3 * n), __ldg(dirs + 3 * n + 1), __ldg(dirs + 3 * n + 2)};
        float ps[3], pm[3];
        const bool k = hits::surface_hit(o, d, __ldg(depth + n), pose_scale, max_range_m, z_min_m, z_max_m, ps, pm);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            points_scaled[3 * n + c] = ps[c];
            points_m[3 * n + c] = pm[c];
        }
        keep[n] = k ? 1 : 0;
    }
}

}  // namespace
}  // namespace ps

extern "C" int ps_surface_hits(const float* origins, const float* dirs, const float* depth, int64_t N, float pose_scale,
                               float max_range_m, float z_min_m, float z_max_m, float* points_scaled, float* points_m,
                               uint8_t* keep, void* stream) {
    if (N == 0) return 0;
    PS_REQUIRE(origins && dirs && depth && points_scaled && points_m && keep, "surface_hits: null pointer");
    PS_REQUIRE(pose_scale > 0.f && std::isfinite(pose_scale), "surface_hits: pose scale factor %g is not a positive number",
               (double)pose_scale);
    int64_t blocks = ps::cdiv(N, 256);
    if (blocks > (int64_t)ps::kNumSMs * 16) blocks = (int64_t)ps::kNumSMs * 16;
    ps::surface_hits_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(origins, dirs, depth, N, pose_scale,
                                                                               max_range_m, z_min_m, z_max_m,
                                                                               points_scaled, points_m, keep);
    return ps::check_launch("surface_hits");
}
