// Host harness around presight_b200/csrc/metrics_core.h: PSNR and SSIM of one channels-last image pair with the per-window
// arithmetic the CUDA kernels run (separable 11-tap window, rows first), compiled with g++ so that
// tests/test_metrics_host.py can check it against the numpy oracle without a GPU.  The sums over pixels are plain fp64
// loops here; the kernels in csrc/metrics.cu sum the same fp32 per-pixel values in a different fixed order.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <vector>

#include "../../presight_b200/csrc/metrics_core.h"

using namespace ps::metrics;

// pred, gt [H,W,3]; returns 1 for images below 11 x 11 (as ps_image_metrics does)
extern "C" int image_metrics_host(const float* pred, const float* gt, int H, int W, float data_range_psnr, double* sse,
                                  float* psnr, double* ssim) {
    if (H < kWin || W < kWin) return 1;
    const int64_t n = (int64_t)H * W * 3;
    double e = 0.0;
    float mn_p = INFINITY, mx_p = -INFINITY, mn_g = INFINITY, mx_g = -INFINITY;
    for (int64_t i = 0; i < n; ++i) {
        const float d = pred[i] - gt[i];
        e += (double)d * (double)d;
        mn_p = std::min(mn_p, pred[i]), mx_p = std::max(mx_p, pred[i]);
        mn_g = std::min(mn_g, gt[i]), mx_g = std::max(mx_g, gt[i]);
    }
    *sse = e;
    const double dr_psnr = data_range_psnr;
    *psnr = (float)(10.0 * std::log10(dr_psnr * dr_psnr / (e / (double)n)));
    const float dr = std::max(mx_p - mn_p, mx_g - mn_g);
    float c1, c2;
    ssim_constants(dr, c1, c2);
    const float g[kWin] = PS_GAUSS_TAPS;
    const int HO = H - 2 * kHalf, WO = W - 2 * kHalf;
    std::vector<float> x((size_t)H * W), y((size_t)H * W), h((size_t)kMoments * H * WO);
    double s = 0.0;
    for (int c = 0; c < 3; ++c) {
        for (int64_t p = 0; p < (int64_t)H * W; ++p) x[p] = pred[3 * p + c], y[p] = gt[3 * p + c];
        for (int r = 0; r < H; ++r)
            for (int col = 0; col < WO; ++col) {
                float m[kMoments];
                window_moments(&x[(size_t)r * W + col], &y[(size_t)r * W + col], 1, g, m);
                for (int k = 0; k < kMoments; ++k) h[((size_t)k * H + r) * WO + col] = m[k];
            }
        for (int r = 0; r < HO; ++r)
            for (int col = 0; col < WO; ++col) {
                float m[kMoments];
                window_sum(&h[(size_t)r * WO + col], WO, H * WO, g, m);
                s += (double)ssim_pixel(m, c1, c2);
            }
    }
    *ssim = dr == 0.f ? NAN : s / ((double)HO * WO * 3);
    return 0;
}
