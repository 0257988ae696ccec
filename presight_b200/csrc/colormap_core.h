// Per-pixel core of the evaluation images nerfacto returns (models/nerfacto.py get_image_metrics_and_images), as
// nerfstudio 0.3.3's utils/colormaps.py computes them with default ColormapOptions (turbo, no normalisation, range
// [0,1], not inverted):
//   accumulation  apply_colormap(acc):            lut[idx(acc)]
//   depth-like    apply_depth_colormap(d, acc):   c = lut[idx(clip((d - near) / (far - near + 1e-10), 0, 1))]
//                                                 c * acc + (1 - acc)
//   idx(x) = long(nan_to_num(clip(x, 0, 1), 0) * 255)     (clip propagates NaN; nan_to_num sends it to 0)
//   near, far = min(d), max(d) over the map, NaN if the map holds one (torch.min / torch.max propagate NaN)
// torch's rounding is reproduced operation by operation:
//   - `far - near + 1e-10` is Python float (fp64) arithmetic on the two fp32 extremes;
//   - a CUDA tensor divided by a Python float is multiplied by the scalar's reciprocal, taken in fp64 and rounded to
//     fp32 once: the map is (d - near) * float(1.0 / divisor), each operation rounded on its own (neither an fp32
//     division nor 1.f / float(divisor) matches torch on the device);
//   - `c * acc + (1 - acc)` and `x * 255` are separate kernels in torch, so nothing here may be fused into an FMA:
//     PS_MUL / PS_ADD / PS_SUB are un-fused fp32 operations (`__fmul_rn` ... on the device).
// `x * (1.0 - 0.0) + 0.0` of apply_colormap changes at most the sign of a zero, which no index depends on.
// Plain C++ shared by the CUDA kernels (csrc/colormap.cu) and the host harness of tests/test_colormap_host.py.
#pragma once

#ifndef PS_HD
#define PS_HD
#endif
#ifndef PS_MUL
#define PS_MUL(a, b) ((a) * (b))
#define PS_ADD(a, b) ((a) + (b))
#define PS_SUB(a, b) ((a) - (b))
#endif

namespace ps {
namespace colormap {

constexpr int kLutSize = 256;  // entries of the [256,3] table (matplotlib's listed colormaps)

// NaN-propagating min / max: once either argument is NaN the result is NaN, in any order of reduction
PS_HD inline float nan_min(float a, float b) { return (a != a || a < b) ? a : b; }
PS_HD inline float nan_max(float a, float b) { return (a != a || a > b) ? a : b; }

// the fp32 factor torch multiplies (d - near) by: float(1.0 / (double(far) - double(near) + 1e-10)), IEEE fp64
// division (correctly rounded on the device and the host alike)
PS_HD inline float depth_inv_range(float near, float far) {
    const double divisor = ((double)far - (double)near) + 1e-10;
    return (float)(1.0 / divisor);
}

// LUT row of a value: clip to [0,1] (NaN stays NaN), NaN -> 0, times 255, truncated
PS_HD inline int lut_index(float x) {
    x = x != x ? x : (x < 0.f ? 0.f : (x > 1.f ? 1.f : x));
    if (x != x) x = 0.f;
    return (int)PS_MUL(x, 255.f);
}

PS_HD inline int depth_index(float d, float near, float inv) { return lut_index(PS_MUL(PS_SUB(d, near), inv)); }

// a colour channel blended with the accumulation: c * acc + (1 - acc), two roundings
PS_HD inline float blend(float c, float acc) { return PS_ADD(PS_MUL(c, acc), PS_SUB(1.f, acc)); }

}  // namespace colormap
}  // namespace ps
