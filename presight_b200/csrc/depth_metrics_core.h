// Per-pixel core of the depth metrics of rendered images against LiDAR depth (the Eigen et al. / Monodepth evaluation
// convention, as KITTI depth benchmarks report it):
//   pred_m = pred / pose_scale_factor                      fp32, IEEE division (as csrc/depth_loss.cu brings the
//                                                            rendered depth to metres); depth along the ray
//   valid  = min_m < target < max_m                          target in metres, 0 = no LiDAR return (the depth mask of
//                                                            depthloss::ray_supervised without the sky term)
//   p      = pred_m clamped to [min_m, max_m]                (a NaN prediction stays NaN)
//   per valid pixel, in fp64 from the fp32 p and t:
//     abs_rel  += |p - t| / t          sq_rel += (p - t)^2 / t
//     se       += (p - t)^2            sle    += (ln p - ln t)^2
//     a_k      += max(p / t, t / p) < 1.25^k  (k = 1, 2, 3; integer counts)
//   metrics = abs_rel / n, sq_rel / n, sqrt(se / n), sqrt(sle / n), a1 / n, a2 / n, a3 / n, n  (NaN for n == 0)
// Plain C++ shared by the CUDA kernels (csrc/depth_metrics.cu) and the host harness of tests/test_geometry_host.py.
#pragma once

#include <cmath>

#ifndef PS_HD
#define PS_HD
#endif
#ifndef PS_FDIV
#define PS_FDIV(a, b) ((a) / (b))   // fp32 IEEE division (the host harness builds with -ffp-contract=off)
#define PS_DMUL(a, b) ((a) * (b))   // fp64 product never contracted into the following sum (`__dmul_rn` on the device)
#endif

namespace ps {
namespace depthmetrics {

constexpr int kOut = 8;          // abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3, n_valid
constexpr int kSums = 4;         // fp64 sums per map: abs_rel, sq_rel, se, sle
constexpr int kCounts = 3;       // integer counts per map: a1, a2, a3
constexpr int kMaxMaps = 4;

// 1.25, 1.25^2, 1.25^3: exact in binary
constexpr double kDelta1 = 1.25, kDelta2 = 1.5625, kDelta3 = 1.953125;

PS_HD inline float pred_metres(float pred, float pose_scale) { return PS_FDIV(pred, pose_scale); }

PS_HD inline bool pixel_valid(float target_m, float min_m, float max_m) { return target_m > min_m && target_m < max_m; }

PS_HD inline float clamp_pred(float pred_m, float min_m, float max_m) {
    return pred_m < min_m ? min_m : (pred_m > max_m ? max_m : pred_m);
}

struct Acc {
    double s[kSums];
    unsigned long long c[kCounts];
};

PS_HD inline void acc_zero(Acc& a) {
    for (int k = 0; k < kSums; ++k) a.s[k] = 0.0;
    for (int k = 0; k < kCounts; ++k) a.c[k] = 0ull;
}

// one valid pixel: p the clamped prediction, t the target (both metres)
PS_HD inline void acc_pixel(Acc& a, float p, float t) {
    const double pd = (double)p, td = (double)t;
    const double d = pd - td, d2 = PS_DMUL(d, d);
    a.s[0] += (d < 0.0 ? -d : d) / td;
    a.s[1] += d2 / td;
    a.s[2] += d2;
    const double lg = log(pd) - log(td);
    a.s[3] += PS_DMUL(lg, lg);
    const double r1 = pd / td, r2 = td / pd;
    const double ratio = r1 > r2 ? r1 : r2;
    a.c[0] += ratio < kDelta1 ? 1ull : 0ull;
    a.c[1] += ratio < kDelta2 ? 1ull : 0ull;
    a.c[2] += ratio < kDelta3 ? 1ull : 0ull;
}

// the eight outputs of one map from its summed accumulator and valid-pixel count
PS_HD inline void finish(const double (&s)[kSums], const unsigned long long (&c)[kCounts], unsigned long long n,
                         double* out) {
    if (n == 0) {
        for (int k = 0; k < kOut - 1; ++k) out[k] = NAN;
        out[kOut - 1] = 0.0;
        return;
    }
    const double nd = (double)n;
    out[0] = s[0] / nd;
    out[1] = s[1] / nd;
    out[2] = sqrt(s[2] / nd);
    out[3] = sqrt(s[3] / nd);
    for (int k = 0; k < kCounts; ++k) out[4 + k] = (double)c[k] / nd;
    out[7] = nd;
}

}  // namespace depthmetrics
}  // namespace ps
