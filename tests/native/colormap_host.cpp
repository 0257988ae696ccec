// Host harness around presight_b200/csrc/colormap_core.h: the colormapped accumulation image and depth-like images of
// one image with the per-pixel arithmetic the CUDA kernels run, compiled with g++ (-ffp-contract=off) so that
// tests/test_colormap_host.py can check it against a numpy restatement without a GPU.  The min / max run as one
// sequential loop here; the kernels in csrc/colormap.cu reduce in a different fixed order, which cannot change an exact
// min / max, NaN included.
#include <cmath>
#include <cstdint>

#include "../../presight_b200/csrc/colormap_core.h"

using namespace ps::colormap;

// maps [M][HW], acc [HW], lut [256][3] -> out [M+1][HW][3]
extern "C" void colormap_host(const float* maps, int M, int64_t HW, const float* acc, const float* lut, float* out) {
    for (int64_t p = 0; p < HW; ++p)
        for (int c = 0; c < 3; ++c) out[3 * p + c] = lut[3 * lut_index(acc[p]) + c];
    for (int m = 0; m < M; ++m) {
        const float* d = maps + (int64_t)m * HW;
        float near = INFINITY, far = -INFINITY;
        for (int64_t p = 0; p < HW; ++p) near = nan_min(near, d[p]), far = nan_max(far, d[p]);
        const float inv = depth_inv_range(near, far);
        float* o = out + (int64_t)(m + 1) * HW * 3;
        for (int64_t p = 0; p < HW; ++p) {
            const int i = depth_index(d[p], near, inv);
            for (int c = 0; c < 3; ++c) o[3 * p + c] = blend(lut[3 * i + c], acc[p]);
        }
    }
}
