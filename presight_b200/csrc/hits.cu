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

// ---- kept hits -> the extractor's hit store ----------------------------------------------------------------------------
// An order-preserving compaction in two launches over G <= kAppendMaxBlocks blocks, each owning one contiguous span of
// rays: (1) every block counts its kept rows into ws[b], and block 0 snapshots the store cursor into ws[G]; (2) every
// block sums the counts before its own (its output offset) and all counts (the call's total), then walks its span in
// tiles of 256 rays with a ballot scan.  Only block G-1 of launch 2 writes the cursor, and nothing in launch 2 reads it,
// so the call needs no host round trip and no spin-wait.  A call whose rows do not all fit writes none of them.
constexpr int kAppendThreads = 256;
constexpr int kAppendMaxBlocks = 1024;
constexpr int64_t kAppendMinSpan = 2048;

__device__ __forceinline__ bool hit_kept(const uint8_t* __restrict__ keep, const float* __restrict__ dens, int64_t i) {
    return __ldg(keep + i) != 0 && __ldg(dens + i) > 1.0f;          // extract_priors.py:157
}

__device__ __forceinline__ long long block_sum_i64(long long v, long long* s_red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    long long t = 0;
#pragma unroll
    for (int w = 0; w < kAppendThreads / 32; ++w) t += s_red[w];
    __syncthreads();
    return t;
}

__global__ void __launch_bounds__(kAppendThreads) hits_count_kernel(const uint8_t* __restrict__ keep,
                                                                    const float* __restrict__ dens, int64_t N, int64_t span,
                                                                    const long long* __restrict__ cursor,
                                                                    long long* __restrict__ ws) {
    __shared__ long long s_red[kAppendThreads / 32];
    const int64_t lo = (int64_t)blockIdx.x * span, hi = min(N, lo + span);
    long long c = 0;
    for (int64_t i = lo + threadIdx.x; i < hi; i += kAppendThreads) c += hit_kept(keep, dens, i) ? 1 : 0;
    c = block_sum_i64(c, s_red);
    if (threadIdx.x == 0) {
        ws[blockIdx.x] = c;
        if (blockIdx.x == 0) ws[gridDim.x] = *cursor;
    }
}

__global__ void __launch_bounds__(kAppendThreads) hits_scatter_kernel(
    const float* __restrict__ points_scaled, const float* __restrict__ points_m, const uint8_t* __restrict__ keep,
    const float* __restrict__ dens, const float* __restrict__ colors, int64_t N, int64_t span,
    const long long* __restrict__ ws, float* __restrict__ store_points, float* __restrict__ store_colors,
    int64_t capacity, long long* __restrict__ cursor, float* __restrict__ min_out, int* __restrict__ status) {
    __shared__ long long s_red[kAppendThreads / 32];
    __shared__ int s_warp[kAppendThreads / 32];
    const int G = gridDim.x, b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long pre = 0, tot = 0;
    for (int j = threadIdx.x; j < G; j += kAppendThreads) {
        const long long c = ws[j];
        tot += c;
        if (j < b) pre += c;
    }
    pre = block_sum_i64(pre, s_red);
    tot = block_sum_i64(tot, s_red);
    const long long base = ws[G];
    if (base + tot > capacity) {                                  // block-uniform: the whole call is refused
        if (b == 0 && threadIdx.x == 0) atomicOr(status, 1);
        return;
    }
    if (b == G - 1 && threadIdx.x == 0) *cursor = base + tot;
    long long row = base + pre;
    float m[3] = {INFINITY, INFINITY, INFINITY};
    const int64_t lo = (int64_t)b * span, hi = min(N, lo + span);
    for (int64_t t0 = lo; t0 < hi; t0 += kAppendThreads) {
        const int64_t i = t0 + threadIdx.x;
        const bool sel = i < hi && hit_kept(keep, dens, i);
        const unsigned bal = __ballot_sync(0xffffffffu, sel);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        int woff = 0, ttot = 0;
#pragma unroll
        for (int w = 0; w < kAppendThreads / 32; ++w) {
            woff += w < warp ? s_warp[w] : 0;
            ttot += s_warp[w];
        }
        if (sel) {
            const long long r = row + woff + __popc(bal & ((1u << lane) - 1u));
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                store_points[3 * r + a] = __ldg(points_scaled + 3 * i + a);
                store_colors[3 * r + a] = colors ? __ldg(colors + 3 * i + a) : 0.0f;
                m[a] = fminf(m[a], __ldg(points_m + 3 * i + a));
            }
        }
        row += ttot;
        __syncthreads();                                           // s_warp is rewritten by the next tile
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        m[a] = warp_min(m[a]);
        if (lane == 0 && m[a] != INFINITY) atomic_min_float(min_out + a, m[a]);
    }
}

int64_t append_blocks(int64_t N) {
    int64_t g = cdiv(N, kAppendMinSpan);
    return g < 1 ? 1 : (g > kAppendMaxBlocks ? kAppendMaxBlocks : g);
}

}  // namespace
}  // namespace ps

extern "C" int ps_hits_append_workspace(int64_t N, int64_t* bytes) {
    PS_REQUIRE(bytes, "hits_append_workspace: null pointer");
    PS_REQUIRE(N >= 0, "hits_append_workspace: negative row count %lld", (long long)N);
    *bytes = (ps::append_blocks(N) + 1) * (int64_t)sizeof(long long);
    return 0;
}

extern "C" int ps_hits_append(const float* points_scaled, const float* points_m, const uint8_t* keep,
                              const float* density, const float* colors, int64_t N, float* store_points,
                              float* store_colors, int64_t capacity, int64_t* cursor, float* min_out, int* status,
                              void* workspace, void* stream) {
    PS_REQUIRE(N >= 0 && capacity >= 0, "hits_append: negative size (N %lld, capacity %lld)", (long long)N,
               (long long)capacity);
    if (N == 0) return 0;
    PS_REQUIRE(points_scaled && points_m && keep && density && store_points && store_colors && cursor && min_out &&
                   status && workspace,
               "hits_append: null pointer");
    const int64_t G = ps::append_blocks(N);
    const int64_t span = ps::cdiv(ps::cdiv(N, G), ps::kAppendThreads) * ps::kAppendThreads;
    auto* ws = reinterpret_cast<long long*>(workspace);
    auto* cur = reinterpret_cast<long long*>(cursor);
    ps::hits_count_kernel<<<(unsigned)G, ps::kAppendThreads, 0, (cudaStream_t)stream>>>(keep, density, N, span, cur, ws);
    if (int e = ps::check_launch("hits_append(count)")) return e;
    ps::hits_scatter_kernel<<<(unsigned)G, ps::kAppendThreads, 0, (cudaStream_t)stream>>>(
        points_scaled, points_m, keep, density, colors, N, span, ws, store_points, store_colors, capacity, cur, min_out,
        status);
    return ps::check_launch("hits_append");
}

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
