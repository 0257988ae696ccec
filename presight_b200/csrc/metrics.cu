// Image metrics of rendered camera images against the photographs: PSNR and SSIM as nerfstudio's nerfacto computes them
// (torchmetrics, one image at a time), the arithmetic of metrics_core.h.  Three kernels, no floating-point atomics, so two
// runs give bit-identical results:
//   1. stats: per image, up to 512 blocks each write (fp64 SSE, min / max of pred, min / max of gt) for a fixed slice
//   2. ssim:  one CTA per 32 x 16 output tile; it reduces the image's stats partials to the data range (min / max are
//             exact in any order), stages the tile and its 10-pixel halo of both images in shared memory, runs the 11-tap
//             window along rows into shared memory and then along columns, and writes the tile's fp64 sum of SSIM
//   3. final: one CTA per image sums both partial arrays in a fixed order -> sse, psnr, ssim
#include <algorithm>
#include <cmath>

#include "common.cuh"

#define PS_HD __device__
#define PS_FMAF(a, b, c) fmaf((a), (b), (c))
#define PS_MUL(a, b) __fmul_rn((a), (b))
#define PS_ADD(a, b) __fadd_rn((a), (b))
#define PS_SUB(a, b) __fsub_rn((a), (b))
#define PS_DIV(a, b) __fdiv_rn((a), (b))
#include "metrics_core.h"

namespace ps {
namespace {

using metrics::kHalf;
using metrics::kMoments;
using metrics::kWin;

constexpr int kThreads = 256;
constexpr int kTileX = 32, kTileY = 16;                          // SSIM output tile
constexpr int kInX = kTileX + kWin - 1, kInY = kTileY + kWin - 1; // staged input: tile + halo
constexpr int kMaxStatBlocks = 512;

__constant__ float c_gauss[kWin] = PS_GAUSS_TAPS;

struct Stat {
    double sse;
    float mn_p, mx_p, mn_g, mx_g;
};

struct Workspace {
    Stat* stats;        // [B][nb1]
    double* ssim_part;  // [B][tiles]
};

int stat_blocks(int64_t n) { return (int)std::min<int64_t>(kMaxStatBlocks, std::max<int64_t>(1, cdiv(n, kThreads * 16))); }

size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

Workspace carve(void* ws, int B, int nb1) {
    char* p = (char*)ws;
    return {(Stat*)p, (double*)(p + align256(sizeof(Stat) * (size_t)B * nb1))};
}

__device__ __forceinline__ double block_sum(double v, double* red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < kThreads / 32; ++w) s += red[w];
    __syncthreads();
    return s;  // valid in thread 0
}

__global__ void __launch_bounds__(kThreads) stats_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                         int64_t n, int nb1, Stat* __restrict__ stats) {
    const int b = blockIdx.y;
    const float* p = pred + (int64_t)b * n;
    const float* g = gt + (int64_t)b * n;
    double sse = 0.0;
    float mn_p = INFINITY, mx_p = -INFINITY, mn_g = INFINITY, mx_g = -INFINITY;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (int64_t)nb1 * kThreads) {
        const float a = __ldg(p + i), c = __ldg(g + i);
        const float d = a - c;
        sse += (double)d * (double)d;
        mn_p = fminf(mn_p, a), mx_p = fmaxf(mx_p, a);
        mn_g = fminf(mn_g, c), mx_g = fmaxf(mx_g, c);
    }
    __shared__ double red[kThreads / 32];
    __shared__ float redf[4][kThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    mn_p = warp_min(mn_p), mx_p = warp_max(mx_p), mn_g = warp_min(mn_g), mx_g = warp_max(mx_g);
    if (lane == 0) redf[0][warp] = mn_p, redf[1][warp] = mx_p, redf[2][warp] = mn_g, redf[3][warp] = mx_g;
    sse = block_sum(sse, red);
    if (threadIdx.x == 0) {
        Stat s{sse, INFINITY, -INFINITY, INFINITY, -INFINITY};
        for (int w = 0; w < kThreads / 32; ++w) {
            s.mn_p = fminf(s.mn_p, redf[0][w]), s.mx_p = fmaxf(s.mx_p, redf[1][w]);
            s.mn_g = fminf(s.mn_g, redf[2][w]), s.mx_g = fmaxf(s.mx_g, redf[3][w]);
        }
        stats[(int64_t)b * nb1 + blockIdx.x] = s;
    }
}

// the image's data range from its stats partials; called by a whole warp, the result in every lane
__device__ __forceinline__ float data_range_of(const Stat* s, int nb1) {
    float mn_p = INFINITY, mx_p = -INFINITY, mn_g = INFINITY, mx_g = -INFINITY;
    for (int i = threadIdx.x & 31; i < nb1; i += 32) {
        mn_p = fminf(mn_p, s[i].mn_p), mx_p = fmaxf(mx_p, s[i].mx_p);
        mn_g = fminf(mn_g, s[i].mn_g), mx_g = fmaxf(mx_g, s[i].mx_g);
    }
    return fmaxf(warp_max(mx_p) - warp_min(mn_p), warp_max(mx_g) - warp_min(mn_g));
}

__global__ void __launch_bounds__(kThreads) ssim_tile_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                             int H, int W, const Stat* __restrict__ stats, int nb1,
                                                             double* __restrict__ ssim_part) {
    __shared__ float xs[3][kInY][kInX], ys[3][kInY][kInX];   // both images, planar per channel
    __shared__ float hs[kMoments][kInY][kTileX];              // row-filtered moments of one channel
    __shared__ float cs[2];
    __shared__ double red[kThreads / 32];
    const int b = blockIdx.z, ox0 = blockIdx.x * kTileX, oy0 = blockIdx.y * kTileY;
    const int HO = H - 2 * kHalf, WO = W - 2 * kHalf;        // valid windows
    if (threadIdx.x < 32) {
        float c1, c2;
        metrics::ssim_constants(data_range_of(stats + (int64_t)b * nb1, nb1), c1, c2);
        if (threadIdx.x == 0) cs[0] = c1, cs[1] = c2;
    }
    // stage: each staged row is kInX * 3 contiguous floats of the channels-last image
    const int64_t img = (int64_t)b * H * W * 3;
    for (int e = threadIdx.x; e < kInY * kInX * 3; e += kThreads) {
        const int r = e / (kInX * 3), q = e - r * (kInX * 3), col = q / 3, c = q - col * 3;
        const int y = oy0 + r, x = ox0 + col;
        float a = 0.f, v = 0.f;
        if (y < H && x < W) {
            const int64_t o = img + ((int64_t)y * W + x) * 3 + c;
            a = __ldg(pred + o), v = __ldg(gt + o);
        }
        xs[c][r][col] = a, ys[c][r][col] = v;
    }
    __syncthreads();
    const float c1 = cs[0], c2 = cs[1];
    double acc = 0.0;                                         // this thread's pixels, 2 per channel
    for (int c = 0; c < 3; ++c) {
        for (int e = threadIdx.x; e < kInY * kTileX; e += kThreads) {
            const int r = e / kTileX, col = e - r * kTileX;
            float m[kMoments];
            metrics::window_moments(&xs[c][r][col], &ys[c][r][col], 1, c_gauss, m);
#pragma unroll
            for (int k = 0; k < kMoments; ++k) hs[k][r][col] = m[k];
        }
        __syncthreads();
        for (int e = threadIdx.x; e < kTileY * kTileX; e += kThreads) {
            const int r = e / kTileX, col = e - r * kTileX;
            if (oy0 + r < HO && ox0 + col < WO) {
                float m[kMoments];
                metrics::window_sum(&hs[0][r][col], kTileX, kInY * kTileX, c_gauss, m);
                acc += (double)metrics::ssim_pixel(m, c1, c2);
            }
        }
        __syncthreads();
    }
    const double s = block_sum(acc, red);
    if (threadIdx.x == 0)
        ssim_part[((int64_t)b * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x] = s;
}

__global__ void __launch_bounds__(kThreads) final_kernel(const Stat* __restrict__ stats, int nb1,
                                                         const double* __restrict__ ssim_part, int tiles, int64_t n,
                                                         int64_t n_ssim, float data_range_psnr, double* __restrict__ sse,
                                                         float* __restrict__ psnr, double* __restrict__ ssim) {
    __shared__ double red[kThreads / 32];
    const int b = blockIdx.x;
    double v = 0.0;
    for (int i = threadIdx.x; i < nb1; i += kThreads) v += stats[(int64_t)b * nb1 + i].sse;
    const double e = block_sum(v, red);
    if (threadIdx.x == 0) {
        if (sse) sse[b] = e;
        const double dr = (double)data_range_psnr;
        psnr[b] = (float)(10.0 * log10(dr * dr / (e / (double)n)));
    }
    if (!ssim) return;
    v = 0.0;
    for (int i = threadIdx.x; i < tiles; i += kThreads) v += ssim_part[(int64_t)b * tiles + i];
    const double s = block_sum(v, red);
    if (threadIdx.x < 32) {
        // two constant images: data range 0, and the definition's 0 / 0 (rounding in the window sums of a non-zero
        // constant can leave a tiny variance, so the NaN is set rather than left to the arithmetic)
        const float dr = data_range_of(stats + (int64_t)b * nb1, nb1);
        if (threadIdx.x == 0) ssim[b] = dr == 0.f ? (double)NAN : s / (double)n_ssim;
    }
}

}  // namespace
}  // namespace ps

extern "C" int ps_image_metrics_workspace(int B, int H, int W, int64_t* bytes) {
    PS_REQUIRE(bytes, "image_metrics_workspace: null pointer");
    PS_REQUIRE(B >= 0 && H >= 0 && W >= 0, "image_metrics_workspace: negative size");
    const int64_t n = (int64_t)H * W * 3;
    const int nb1 = ps::stat_blocks(n);
    const int64_t tiles = H > 2 * ps::kHalf && W > 2 * ps::kHalf
                              ? ps::cdiv(W - 2 * ps::kHalf, ps::kTileX) * ps::cdiv(H - 2 * ps::kHalf, ps::kTileY)
                              : 0;
    *bytes = (int64_t)(ps::align256(sizeof(ps::Stat) * (size_t)B * nb1) + sizeof(double) * (size_t)B * tiles);
    return 0;
}

extern "C" int ps_image_metrics(const float* pred, const float* gt, int B, int H, int W, float data_range_psnr,
                                void* workspace, double* sse, float* psnr, double* ssim, void* stream) {
    PS_REQUIRE(B >= 0 && H >= 0 && W >= 0, "image_metrics: negative size (B %d, H %d, W %d)", B, H, W);
    if (ssim)
        PS_REQUIRE(H >= ps::metrics::kWin && W >= ps::metrics::kWin,
                   "image_metrics: SSIM needs images of at least 11 x 11 pixels, got %d x %d", H, W);
    if (B == 0) return 0;
    PS_REQUIRE((int64_t)H * W > 0, "image_metrics: empty image (%d x %d)", H, W);
    PS_REQUIRE(pred && gt && workspace && psnr, "image_metrics: null pointer");
    PS_REQUIRE(B <= 65535, "image_metrics: at most 65535 images per call, got %d", B);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = (int64_t)H * W * 3;
    const int nb1 = ps::stat_blocks(n);
    const ps::Workspace ws = ps::carve(workspace, B, nb1);
    ps::stats_kernel<<<dim3(nb1, B), ps::kThreads, 0, st>>>(pred, gt, n, nb1, ws.stats);
    if (int rc = ps::check_launch("image_metrics stats")) return rc;
    int tiles = 0;
    int64_t n_ssim = 0;
    if (ssim) {
        const int HO = H - 2 * ps::kHalf, WO = W - 2 * ps::kHalf;
        const dim3 grid((unsigned)ps::cdiv(WO, ps::kTileX), (unsigned)ps::cdiv(HO, ps::kTileY), B);
        tiles = (int)(grid.x * grid.y);
        n_ssim = (int64_t)HO * WO * 3;
        ps::ssim_tile_kernel<<<grid, ps::kThreads, 0, st>>>(pred, gt, H, W, ws.stats, nb1, ws.ssim_part);
        if (int rc = ps::check_launch("image_metrics ssim")) return rc;
    }
    ps::final_kernel<<<B, ps::kThreads, 0, st>>>(ws.stats, nb1, ws.ssim_part, tiles, n, n_ssim, data_range_psnr, sse, psnr,
                                                 ssim);
    return ps::check_launch("image_metrics final");
}
