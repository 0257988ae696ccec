// Host harness around presight_b200/csrc/hits_core.h: the per-ray surface-hit arithmetic compiled with g++ so that
// tests/test_extract_host.py can check it without a GPU.  (The product reaches the same code only through the CUDA
// kernel in csrc/hits.cu.)
#include <cstdint>

#include "../../presight_b200/csrc/hits_core.h"

extern "C" int surface_hits_host(const float* origins, const float* dirs, const float* depth, int64_t N, float pose_scale,
                                 float max_range_m, float z_min_m, float z_max_m, float* points_scaled, float* points_m,
                                 uint8_t* keep) {
    for (int64_t n = 0; n < N; ++n)
        keep[n] = ps::hits::surface_hit(origins + 3 * n, dirs + 3 * n, depth[n], pose_scale, max_range_m, z_min_m, z_max_m,
                                        points_scaled + 3 * n, points_m + 3 * n) ? 1 : 0;
    return 0;
}
