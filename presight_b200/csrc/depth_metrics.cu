// Depth metrics of rendered depth maps against LiDAR depth, the arithmetic of depth_metrics_core.h.  Two kernels, no
// floating-point atomics, and a grid that depends on the image size only, so two runs give bit-identical results:
//   1. stats: up to 512 CTAs grid-stride over the pixels; every thread reads the target once for all M maps and keeps
//             fp64 sums and integer counts per map; each CTA writes its partials (fixed-order block reduction)
//   2. final: one CTA sums the partials of every quantity in a fixed order and writes [M, 8] f64
// Registers (sm_100a, ptxas -v): stats<1> 56, stats<2> 74, stats<3> 94, stats<4> 113, final 32; no spills.
#include <algorithm>

#include "common.cuh"

#define PS_HD __device__
#define PS_FDIV(a, b) __fdiv_rn((a), (b))
#define PS_DMUL(a, b) __dmul_rn((a), (b))
#include "depth_metrics_core.h"

namespace ps {
namespace {

using depthmetrics::kCounts;
using depthmetrics::kMaxMaps;
using depthmetrics::kOut;
using depthmetrics::kSums;

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxBlocks = 512;

int stat_blocks(int64_t n) { return (int)std::min<int64_t>(kMaxBlocks, std::max<int64_t>(1, cdiv(n, kThreads * 16))); }

size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

// partials of one CTA: sums [M][kSums] f64, counts [M][kCounts] + n_valid u64
size_t sums_bytes(int M, int nb) { return align256(sizeof(double) * (size_t)nb * M * kSums); }

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// fixed-order block sums; the result is valid in thread 0
__device__ __forceinline__ double block_sum(double v, double* red) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < kWarps; ++w) s += red[w];
    __syncthreads();
    return s;
}
__device__ __forceinline__ unsigned long long block_sum(unsigned long long v, unsigned long long* red) {
    v = warp_sum_u64(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    unsigned long long s = 0;
    if (threadIdx.x == 0)
        for (int w = 0; w < kWarps; ++w) s += red[w];
    __syncthreads();
    return s;
}

template <int M>
__global__ void __launch_bounds__(kThreads) depth_stats_kernel(const float* __restrict__ pred, int64_t HW,
                                                               const float* __restrict__ target, float pose_scale,
                                                               const float* __restrict__ pose_scale_dev, float min_m,
                                                               float max_m, double* __restrict__ psums,
                                                               unsigned long long* __restrict__ pcounts) {
    __shared__ double red[kWarps];
    __shared__ unsigned long long redu[kWarps];
    if (pose_scale_dev) pose_scale = __ldg(pose_scale_dev);
    depthmetrics::Acc acc[M];
#pragma unroll
    for (int m = 0; m < M; ++m) depthmetrics::acc_zero(acc[m]);
    unsigned long long n = 0;
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < HW; i += stride) {
        const float t = __ldg(target + i);
        if (!depthmetrics::pixel_valid(t, min_m, max_m)) continue;
        ++n;
#pragma unroll
        for (int m = 0; m < M; ++m) {
            const float p = depthmetrics::clamp_pred(depthmetrics::pred_metres(__ldg(pred + m * HW + i), pose_scale),
                                                     min_m, max_m);
            depthmetrics::acc_pixel(acc[m], p, t);
        }
    }
    const int b = blockIdx.x;
#pragma unroll
    for (int m = 0; m < M; ++m) {
#pragma unroll
        for (int k = 0; k < kSums; ++k) {
            const double s = block_sum(acc[m].s[k], red);
            if (threadIdx.x == 0) psums[((int64_t)b * M + m) * kSums + k] = s;
        }
#pragma unroll
        for (int k = 0; k < kCounts; ++k) {
            const unsigned long long c = block_sum(acc[m].c[k], redu);
            if (threadIdx.x == 0) pcounts[(int64_t)b * (M * kCounts + 1) + m * kCounts + k] = c;
        }
    }
    const unsigned long long c = block_sum(n, redu);
    if (threadIdx.x == 0) pcounts[(int64_t)b * (M * kCounts + 1) + M * kCounts] = c;
}

__global__ void __launch_bounds__(kThreads) depth_final_kernel(const double* __restrict__ psums,
                                                               const unsigned long long* __restrict__ pcounts, int M,
                                                               int nb, double* __restrict__ out) {
    __shared__ double red[kWarps];
    __shared__ unsigned long long redu[kWarps];
    __shared__ double s_sum[kMaxMaps][kSums];
    __shared__ unsigned long long s_cnt[kMaxMaps * kCounts + 1];
    const int nc = M * kCounts + 1;
    for (int q = 0; q < M * kSums; ++q) {
        double v = 0.0;
        for (int b = threadIdx.x; b < nb; b += kThreads) v += psums[(int64_t)b * M * kSums + q];
        const double s = block_sum(v, red);
        if (threadIdx.x == 0) s_sum[q / kSums][q % kSums] = s;
    }
    for (int q = 0; q < nc; ++q) {
        unsigned long long v = 0;
        for (int b = threadIdx.x; b < nb; b += kThreads) v += pcounts[(int64_t)b * nc + q];
        const unsigned long long s = block_sum(v, redu);
        if (threadIdx.x == 0) s_cnt[q] = s;
    }
    __syncthreads();
    if (threadIdx.x < M) {
        const int m = threadIdx.x;
        unsigned long long c[kCounts];
        for (int k = 0; k < kCounts; ++k) c[k] = s_cnt[m * kCounts + k];
        depthmetrics::finish(s_sum[m], c, s_cnt[M * kCounts], out + (int64_t)m * kOut);
    }
}

}  // namespace
}  // namespace ps

extern "C" int ps_depth_metrics_workspace(int M, int64_t HW, int64_t* bytes) {
    PS_REQUIRE(bytes, "depth_metrics_workspace: null pointer");
    PS_REQUIRE(M >= 1 && M <= ps::kMaxMaps, "depth_metrics_workspace: M must be in [1, %d], got %d", ps::kMaxMaps, M);
    PS_REQUIRE(HW > 0, "depth_metrics_workspace: HW must be positive, got %lld", (long long)HW);
    const int nb = ps::stat_blocks(HW);
    *bytes = (int64_t)(ps::sums_bytes(M, nb) + sizeof(unsigned long long) * (size_t)nb * (M * ps::kCounts + 1));
    return 0;
}

extern "C" int ps_depth_metrics(const float* pred, int M, int64_t HW, const float* target_m, float pose_scale,
                                const float* pose_scale_dev, float min_m, float max_m, void* workspace, double* out,
                                void* stream) {
    PS_REQUIRE(M >= 1 && M <= ps::kMaxMaps, "depth_metrics: M must be in [1, %d], got %d", ps::kMaxMaps, M);
    PS_REQUIRE(HW > 0, "depth_metrics: HW must be positive, got %lld", (long long)HW);
    PS_REQUIRE(pred && target_m && workspace && out, "depth_metrics: null pointer");
    PS_REQUIRE(pose_scale_dev != nullptr || pose_scale > 0.f, "depth_metrics: pose scale must be positive");
    PS_REQUIRE(min_m > 0.f && min_m < max_m && max_m < INFINITY,
               "depth_metrics: need 0 < min_m < max_m < inf, got min_m %g, max_m %g", (double)min_m, (double)max_m);
    cudaStream_t st = (cudaStream_t)stream;
    const int nb = ps::stat_blocks(HW);
    double* psums = (double*)workspace;
    unsigned long long* pcounts = (unsigned long long*)((char*)workspace + ps::sums_bytes(M, nb));
#define PS_DEPTH_STATS(MM)                                                                                              \
    ps::depth_stats_kernel<MM><<<nb, ps::kThreads, 0, st>>>(pred, HW, target_m, pose_scale, pose_scale_dev, min_m, max_m, \
                                                           psums, pcounts)
    switch (M) {
        case 1: PS_DEPTH_STATS(1); break;
        case 2: PS_DEPTH_STATS(2); break;
        case 3: PS_DEPTH_STATS(3); break;
        default: PS_DEPTH_STATS(4); break;
    }
#undef PS_DEPTH_STATS
    if (int rc = ps::check_launch("depth_metrics stats")) return rc;
    ps::depth_final_kernel<<<1, ps::kThreads, 0, st>>>(psums, pcounts, M, nb, out);
    return ps::check_launch("depth_metrics final");
}
