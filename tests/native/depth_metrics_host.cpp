// Host harness around presight_b200/csrc/depth_metrics_core.h: the depth metrics of M maps against one target image
// with the per-pixel arithmetic the CUDA kernels run, compiled with g++ so that tests/test_geometry_host.py can check it
// against the numpy oracle without a GPU.  The sums over pixels are plain loops here; csrc/depth_metrics.cu sums the
// same fp64 per-pixel terms in a different fixed order.
#include <cstdint>

#include "../../presight_b200/csrc/depth_metrics_core.h"

using namespace ps::depthmetrics;

// pred [M][HW], target [HW] -> out [M][8]; returns 1 for M outside [1, 4] (as ps_depth_metrics does)
extern "C" int depth_metrics_host(const float* pred, int M, int64_t HW, const float* target, float pose_scale,
                                  float min_m, float max_m, double* out) {
    if (M < 1 || M > kMaxMaps) return 1;
    for (int m = 0; m < M; ++m) {
        Acc acc;
        acc_zero(acc);
        unsigned long long n = 0;
        for (int64_t i = 0; i < HW; ++i) {
            const float t = target[i];
            if (!pixel_valid(t, min_m, max_m)) continue;
            ++n;
            acc_pixel(acc, clamp_pred(pred_metres(pred[m * HW + i], pose_scale), min_m, max_m), t);
        }
        finish(acc.s, acc.c, n, out + m * kOut);
    }
    return 0;
}
