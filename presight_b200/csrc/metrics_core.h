// Per-window core of the image metrics nerfstudio's nerfacto reports (models/nerfacto.py get_image_metrics_and_images):
// torchmetrics' PeakSignalNoiseRatio(data_range=1.0) and structural_similarity_index_measure with its defaults, on one
// image [1,3,H,W] at a time.
//   PSNR = 10 log10(data_range^2 / (sse / 3HW)), sse accumulated in fp64; +inf for equal images
//   SSIM = mean over channels and the (H-10) x (W-10) interior of
//          ((2 mx my + c1)(2 sxy + c2)) / ((mx^2 + my^2 + c1)(sxx + syy + c2))
//     mx, my, E[x^2], E[y^2], E[xy]: 11 x 11 Gaussian window (sigma 1.5), the outer product of kGauss with itself
//     sxx = E[x^2] - mx^2 and so on, not clamped (torchmetrics 1.0's form)
//     c1 = (0.01 dr)^2, c2 = (0.03 dr)^2, dr = max(max(x) - min(x), max(y) - min(y)) over the whole image
// torchmetrics reflect-pads by 5, convolves and crops 5 from every side, so every window it keeps lies inside the image:
// the windows here are the valid ones and no padding is formed.  Two constant images give dr = 0 and 0/0 = NaN, as
// torchmetrics does.  The window runs separably (11 taps along a row, then 11 along a column), in fp32 as torchmetrics
// computes.
// Plain C++ shared by the CUDA kernels (csrc/metrics.cu) and the host harness of tests/test_metrics_host.py.
#pragma once

#ifndef PS_HD
#define PS_HD
#endif
#ifndef PS_FMAF
#include <cmath>
#define PS_FMAF(a, b, c) (std::fmaf((a), (b), (c)))
#define PS_MUL(a, b) ((a) * (b))
#define PS_ADD(a, b) ((a) + (b))
#define PS_SUB(a, b) ((a) - (b))
#define PS_DIV(a, b) ((a) / (b))
#endif

namespace ps {
namespace metrics {

constexpr int kWin = 11;              // Gaussian window taps
constexpr int kHalf = kWin / 2;       // torchmetrics' reflect pad and crop
constexpr int kMoments = 5;           // x, y, x^2, y^2, xy

// exp(-(d / 1.5)^2 / 2) / sum for d = -5..5, computed in fp64 and rounded to fp32 (torchmetrics' _gaussian, which
// computes in fp32, gives the same values to within a few ulp)
#define PS_GAUSS_TAPS                                                                                            \
    {0.00102838012f, 0.00759875821f, 0.0360007733f, 0.109360687f, 0.213005543f, 0.266011715f, 0.213005543f,     \
     0.109360687f,   0.0360007733f,  0.00759875821f, 0.00102838012f}

// the five weighted sums of 11 samples of x and y, `stride` floats apart
PS_HD inline void window_moments(const float* x, const float* y, int stride, const float* g, float (&m)[kMoments]) {
    for (int k = 0; k < kMoments; ++k) m[k] = 0.f;
    for (int t = 0; t < kWin; ++t) {
        const float a = x[t * stride], b = y[t * stride], w = g[t];
        m[0] = PS_FMAF(w, a, m[0]);
        m[1] = PS_FMAF(w, b, m[1]);
        m[2] = PS_FMAF(w, PS_MUL(a, a), m[2]);
        m[3] = PS_FMAF(w, PS_MUL(b, b), m[3]);
        m[4] = PS_FMAF(w, PS_MUL(a, b), m[4]);
    }
}

// the same weighted sums over 11 row-filtered moments (the vertical pass): moment k of tap t at h[k * plane + t * stride]
PS_HD inline void window_sum(const float* h, int stride, int plane, const float* g, float (&m)[kMoments]) {
    for (int k = 0; k < kMoments; ++k) m[k] = 0.f;
    for (int t = 0; t < kWin; ++t)
        for (int k = 0; k < kMoments; ++k) m[k] = PS_FMAF(g[t], h[k * plane + t * stride], m[k]);
}

PS_HD inline void ssim_constants(float data_range, float& c1, float& c2) {
    const float a = PS_MUL(0.01f, data_range), b = PS_MUL(0.03f, data_range);
    c1 = PS_MUL(a, a);
    c2 = PS_MUL(b, b);
}

// SSIM of one window from its five moments.  PS_MUL / PS_ADD / PS_SUB / PS_DIV are un-fused fp32 operations (`__fmul_rn`
// ... on the device), so that host and device round alike and two equal images give numerator == denominator, SSIM 1
PS_HD inline float ssim_pixel(const float (&m)[kMoments], float c1, float c2) {
    const float mxx = PS_MUL(m[0], m[0]), myy = PS_MUL(m[1], m[1]), mxy = PS_MUL(m[0], m[1]);
    const float sxx = PS_SUB(m[2], mxx), syy = PS_SUB(m[3], myy), sxy = PS_SUB(m[4], mxy);
    const float upper = PS_ADD(PS_MUL(2.f, sxy), c2), lower = PS_ADD(PS_ADD(sxx, syy), c2);
    return PS_DIV(PS_MUL(PS_ADD(PS_MUL(2.f, mxy), c1), upper), PS_MUL(PS_ADD(PS_ADD(mxx, myy), c1), lower));
}

}  // namespace metrics
}  // namespace ps
