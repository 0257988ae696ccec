// Colormapped evaluation images: nerfacto's accumulation image and its depth-like images (depth, prop_depth_i), as
// nerfstudio's utils/colormaps.py computes them with a caller's [256,3] LUT; the arithmetic of colormap_core.h, bit for
// bit what torch gives for the same definition.  Two kernels, no floating-point atomics and no host read:
//   1. minmax: per map, nb blocks each write the NaN-propagating (min, max) of a fixed strided slice
//   2. map:    every CTA reduces each map's nb partials in a fixed order to (near, 1 / range), stages the LUT in shared
//              memory and runs a grid-stride loop over pixels; a pixel's accumulation is read once and all M + 1
//              colours are written: out[0] the accumulation image, out[1 + m] map m blended with the accumulation
// Bytes (memory-bound): 8 M HW read for the maps (two passes), 4 HW for the accumulation, 12 (M + 1) HW written.
// ptxas (sm_100a, CUDA 12.9): minmax 26 registers, map 32 registers (8 CTAs of 256 threads per SM), no spills, no stack
// frame.
#include <algorithm>

#include "common.cuh"

#define PS_HD __device__
#define PS_MUL(a, b) __fmul_rn((a), (b))
#define PS_ADD(a, b) __fadd_rn((a), (b))
#define PS_SUB(a, b) __fsub_rn((a), (b))
#include "colormap_core.h"

namespace ps {
namespace {

using colormap::kLutSize;
using colormap::nan_max;
using colormap::nan_min;

constexpr int kThreads = 256;
constexpr int kMaxMaps = 1024;                 // bounds the map kernel's shared memory (2 floats per map)
constexpr int kMapCtasPerSM = 8;

struct MinMax {
    float mn, mx;
};

// partial blocks per map: about four waves of CTAs over all maps, at least 2048 pixels per block, at most 256
int minmax_blocks(int M, int64_t HW) {
    const int64_t want = std::max<int64_t>(1, cdiv(4 * kNumSMs, std::max(M, 1)));
    return (int)std::max<int64_t>(1, std::min<int64_t>({256, want, cdiv(HW, kThreads * 8)}));
}

__device__ __forceinline__ void warp_minmax(float& mn, float& mx) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = nan_min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = nan_max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
}

__global__ void __launch_bounds__(kThreads) colormap_minmax_kernel(const float* __restrict__ maps, int64_t HW, int nb,
                                                                   MinMax* __restrict__ part) {
    const float* p = maps + (int64_t)blockIdx.y * HW;
    const int64_t step = (int64_t)nb * kThreads;
    float mn = INFINITY, mx = -INFINITY;
    int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    for (; i + 3 * step < HW; i += 4 * step) {                 // four independent loads in flight
        const float a = __ldg(p + i), b = __ldg(p + i + step), c = __ldg(p + i + 2 * step), d = __ldg(p + i + 3 * step);
        mn = nan_min(nan_min(mn, a), nan_min(nan_min(b, c), d));
        mx = nan_max(nan_max(mx, a), nan_max(nan_max(b, c), d));
    }
    for (; i < HW; i += step) {
        const float a = __ldg(p + i);
        mn = nan_min(mn, a), mx = nan_max(mx, a);
    }
    __shared__ MinMax red[kThreads / 32];
    warp_minmax(mn, mx);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = {mn, mx};
    __syncthreads();
    if (threadIdx.x == 0) {
        MinMax s = red[0];
        for (int w = 1; w < kThreads / 32; ++w) s.mn = nan_min(s.mn, red[w].mn), s.mx = nan_max(s.mx, red[w].mx);
        part[(int64_t)blockIdx.y * nb + blockIdx.x] = s;
    }
}

__global__ void __launch_bounds__(kThreads) colormap_map_kernel(const float* __restrict__ maps, int M, int64_t HW,
                                                                const float* __restrict__ acc,
                                                                const float* __restrict__ lut,
                                                                const MinMax* __restrict__ part, int nb,
                                                                float* __restrict__ out) {
    extern __shared__ float sm[];
    float* s_lut = sm;                         // [256][3]
    float* s_near = sm + kLutSize * 3;         // [M]
    float* s_inv = s_near + M;                 // [M]
    for (int e = threadIdx.x; e < kLutSize * 3; e += kThreads) s_lut[e] = __ldg(lut + e);
    const int lane = threadIdx.x & 31;
    for (int m = threadIdx.x >> 5; m < M; m += kThreads / 32) {
        float mn = INFINITY, mx = -INFINITY;
        for (int i = lane; i < nb; i += 32) {
            const MinMax v = part[(int64_t)m * nb + i];
            mn = nan_min(mn, v.mn), mx = nan_max(mx, v.mx);
        }
        warp_minmax(mn, mx);
        if (lane == 0) s_near[m] = mn, s_inv[m] = colormap::depth_inv_range(mn, mx);
    }
    __syncthreads();
    const int64_t plane = HW * 3;
    for (int64_t p = (int64_t)blockIdx.x * kThreads + threadIdx.x; p < HW; p += (int64_t)gridDim.x * kThreads) {
        const float a = __ldg(acc + p);
        const float* c = s_lut + 3 * colormap::lut_index(a);
        float* o = out + 3 * p;
        o[0] = c[0], o[1] = c[1], o[2] = c[2];
        for (int m = 0; m < M; ++m) {
            const float d = __ldg(maps + (int64_t)m * HW + p);
            const float* cd = s_lut + 3 * colormap::depth_index(d, s_near[m], s_inv[m]);
            o += plane;
            o[0] = colormap::blend(cd[0], a), o[1] = colormap::blend(cd[1], a), o[2] = colormap::blend(cd[2], a);
        }
    }
}

}  // namespace
}  // namespace ps

extern "C" int ps_colormap_workspace(int M, int64_t HW, int64_t* bytes) {
    PS_REQUIRE(bytes, "colormap_workspace: null pointer");
    PS_REQUIRE(M >= 0 && M <= ps::kMaxMaps, "colormap_workspace: M must be in [0, %d], got %d", ps::kMaxMaps, M);
    PS_REQUIRE(HW > 0, "colormap_workspace: HW must be positive, got %lld", (long long)HW);
    *bytes = M == 0 ? 0 : (int64_t)sizeof(ps::MinMax) * M * ps::minmax_blocks(M, HW);
    return 0;
}

extern "C" int ps_colormap(const float* maps, int M, int64_t HW, const float* acc, const float* lut, void* workspace,
                           float* out, void* stream) {
    PS_REQUIRE(M >= 0 && M <= ps::kMaxMaps, "colormap: M must be in [0, %d], got %d", ps::kMaxMaps, M);
    PS_REQUIRE(HW > 0, "colormap: HW must be positive, got %lld", (long long)HW);
    PS_REQUIRE(acc && lut && out, "colormap: null pointer (acc, lut or out)");
    PS_REQUIRE(M == 0 || (maps && workspace), "colormap: null pointer (maps or workspace with M = %d)", M);
    cudaStream_t st = (cudaStream_t)stream;
    const int nb = ps::minmax_blocks(M, HW);
    ps::MinMax* part = (ps::MinMax*)workspace;
    if (M > 0) {
        ps::colormap_minmax_kernel<<<dim3(nb, M), ps::kThreads, 0, st>>>(maps, HW, nb, part);
        if (int rc = ps::check_launch("colormap minmax")) return rc;
    }
    const int grid = (int)std::min<int64_t>(ps::cdiv(HW, ps::kThreads), (int64_t)ps::kNumSMs * ps::kMapCtasPerSM);
    const size_t smem = sizeof(float) * (ps::kLutSize * 3 + 2 * (size_t)M);
    ps::colormap_map_kernel<<<grid, ps::kThreads, smem, st>>>(maps, M, HW, acc, lut, part, nb, out);
    return ps::check_launch("colormap map");
}
