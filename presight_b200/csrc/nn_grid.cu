// Nearest-neighbour distances within a radius r between two point clouds (accuracy / completeness of extracted priors
// against LiDAR), on a uniform grid of cells of side r over the reference set:
//   build  1. bounds: per-axis min / max of the reference points (exact in any order)
//          2. keys:   cell of every point, floor(((double)p - (double)min) / r) per axis, 21 bits per axis in an int64
//          (the caller sorts (key, index); presight_b200.geometry uses torch.sort)
//          3. count:  number of occupied cells (the caller sizes the table from it)
//          4. cells:  every run of equal sorted keys -> its [start, end) in an open-addressing table (key_table.cuh), and
//                     the points gathered into cell order
//   query  one thread per query point scans the 27 cells around its own and keeps the exact minimum of
//          ((qx - px)^2 + (qy - py)^2) + (qz - pz)^2 in fp64 from the fp32 coordinates (no contraction), then sqrt; a
//          distance that is not < r becomes r.  Any point closer than r lies in one of those cells: the cell index of a
//          coordinate is a monotone function of it and two coordinates less than r apart get indices at most one apart.
//          Every CTA scores a fixed block of 1024 consecutive queries (global index), so the partials, and the scores
//          reduced from them in a fixed order, do not depend on how the caller splits the queries into chunks.
//   reduce one CTA: mean clamped distance and the number of distances below each threshold.
// No floating-point atomics: repeated calls give bit-identical results.
// Registers (sm_100a, ptxas -v): bounds 32, keys 32, count 34, cells 20, cell_ends 18, query 40 (8.3 KB smem),
// reduce 32; no spills.
#include <algorithm>
#include <cmath>

#include "key_table.cuh"

namespace ps {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kQueriesPerThread = 4;
constexpr int kBlockQueries = PS_NN_BLOCK_QUERIES;      // kThreads * kQueriesPerThread
static_assert(kBlockQueries == kThreads * kQueriesPerThread, "query block size");
constexpr int kCellBits = 21;
constexpr long long kCells = 1ll << kCellBits;
constexpr double kMinCell = 1e-6, kMaxCell = 1e6;

struct Taus {
    double v[PS_NN_MAX_TAUS];
};

// (x / cell) rounded to nearest as IEEE division rounds it, from inv = 1 / cell (IEEE, computed on the host): with a
// correctly rounded reciprocal, q0 = x inv within an ulp and the exact residual r = x - q0 cell, q0 + r inv rounds to
// the correctly rounded quotient (Markstein).  Avoids the call to the fp64 division's slow path, whose register saves
// would spill; cell in [kMinCell, kMaxCell] and fp32 coordinates keep every step away from underflow and overflow.
__device__ __forceinline__ double div_rn(double x, double cell, double inv) {
    const double q0 = x * inv;
    return __fma_rn(__fma_rn(-q0, cell, x), inv, q0);
}

// cell coordinate of a coordinate x along an axis whose grid starts at o
__device__ __forceinline__ double cell_of(float x, float o, double cell, double inv) {
    return floor(div_rn((double)x - (double)o, cell, inv));
}

__device__ __forceinline__ long long pack_cell(long long cx, long long cy, long long cz) {
    return (cx << (2 * kCellBits)) | (cy << kCellBits) | cz;
}

__global__ void __launch_bounds__(kThreads) nn_bounds_kernel(const float* __restrict__ pts, int64_t M,
                                                             float* __restrict__ bounds) {
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < M; i += stride) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float v = __ldg(pts + 3 * i + a);
            mn[a] = fminf(mn[a], v), mx[a] = fmaxf(mx[a], v);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        mn[a] = warp_min(mn[a]), mx[a] = warp_max(mx[a]);
        if ((threadIdx.x & 31) == 0) {
            if (mn[a] != INFINITY) atomic_min_float(bounds + a, mn[a]);
            if (mx[a] != -INFINITY) atomic_max_float(bounds + 3 + a, mx[a]);
        }
    }
}

__global__ void __launch_bounds__(kThreads) nn_keys_kernel(const float* __restrict__ pts, int64_t M, float ox, float oy,
                                                           float oz, double cell, double inv, long long* __restrict__ keys) {
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < M; i += stride)
        keys[i] = pack_cell((long long)cell_of(__ldg(pts + 3 * i), ox, cell, inv),
                            (long long)cell_of(__ldg(pts + 3 * i + 1), oy, cell, inv),
                            (long long)cell_of(__ldg(pts + 3 * i + 2), oz, cell, inv));
}

__device__ __forceinline__ bool run_start(const long long* __restrict__ k, int64_t i) { return i == 0 || k[i] != k[i - 1]; }

__global__ void __launch_bounds__(kThreads) nn_count_cells_kernel(const long long* __restrict__ sorted_keys, int64_t M,
                                                                  unsigned long long* __restrict__ n_cells) {
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    unsigned long long n = 0;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < M; i += stride) n += run_start(sorted_keys, i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if ((threadIdx.x & 31) == 0 && n) atomicAdd(n_cells, n);
}

// gathers the points into cell order and inserts every cell with its start; status |= 1 when the table is full
__global__ void __launch_bounds__(kThreads) nn_cells_kernel(const float* __restrict__ pts, const long long* __restrict__ perm,
                                                            const long long* __restrict__ sorted_keys, int64_t M,
                                                            long long* __restrict__ cell_keys, int2* __restrict__ ranges,
                                                            uint64_t cap_mask, float* __restrict__ sorted_pts,
                                                            int* __restrict__ status) {
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < M; i += stride) {
        const long long j = __ldg(perm + i);
#pragma unroll
        for (int a = 0; a < 3; ++a) sorted_pts[3 * i + a] = __ldg(pts + 3 * j + a);
        if (!run_start(sorted_keys, i)) continue;
        bool fresh;
        const long long s = table_insert(cell_keys, cap_mask, sorted_keys[i], fresh);
        if (s < 0) atomicOr(status, 1);
        else ranges[s].x = (int)i;
    }
}

// the end of every cell (after nn_cells_kernel has inserted them all); status |= 2 for a cell missing from the table
__global__ void __launch_bounds__(kThreads) nn_cell_ends_kernel(const long long* __restrict__ sorted_keys, int64_t M,
                                                                const long long* __restrict__ cell_keys,
                                                                int2* __restrict__ ranges, uint64_t cap_mask,
                                                                int* __restrict__ status) {
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < M; i += stride) {
        if (i + 1 < M && sorted_keys[i + 1] == sorted_keys[i]) continue;
        const long long s = table_find(cell_keys, cap_mask, sorted_keys[i]);
        if (s < 0) atomicOr(status, 2);
        else ranges[s].y = (int)(i + 1);
    }
}

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

__device__ __forceinline__ long long block_sum_i64(long long v, long long* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    long long s = 0;
    if (threadIdx.x == 0)
        for (int w = 0; w < kWarps; ++w) s += red[w];
    __syncthreads();
    return s;
}

// squared distance to the nearest grid point, +inf when no point lies in the 27 cells around q
__device__ __forceinline__ double nearest_sq(const float (&q)[3], const ps_nn_grid& g, double inv) {
    const double qd[3] = {(double)q[0], (double)q[1], (double)q[2]};
    long long c[3];
#pragma unroll
    for (int a = 0; a < 3; ++a)   // clamped to [-2, 2^21 + 1]: beyond that no neighbour cell exists
        c[a] = (long long)fmin(fmax(cell_of(q[a], g.origin[a], g.cell, inv), -2.0), (double)kCells + 1.0);
    const uint64_t cap_mask = (uint64_t)g.capacity - 1;
    const long long* __restrict__ keys = reinterpret_cast<const long long*>(g.cell_keys);
    const int2* __restrict__ ranges = reinterpret_cast<const int2*>(g.cell_ranges);
    double best = INFINITY;
    for (int dz = -1; dz <= 1; ++dz) {
        const long long cz = c[2] + dz;
        if (cz < 0 || cz >= kCells) continue;
        for (int dy = -1; dy <= 1; ++dy) {
            const long long cy = c[1] + dy;
            if (cy < 0 || cy >= kCells) continue;
            for (int dx = -1; dx <= 1; ++dx) {
                const long long cx = c[0] + dx;
                if (cx < 0 || cx >= kCells) continue;
                const long long s = table_find(keys, cap_mask, pack_cell(cx, cy, cz));
                if (s < 0) continue;
                const int2 r = __ldg(ranges + s);
                for (int j = r.x; j < r.y; ++j) {
                    const double ex = qd[0] - (double)__ldg(g.points + 3 * (int64_t)j);
                    const double ey = qd[1] - (double)__ldg(g.points + 3 * (int64_t)j + 1);
                    const double ez = qd[2] - (double)__ldg(g.points + 3 * (int64_t)j + 2);
                    const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)), __dmul_rn(ez, ez));
                    best = fmin(best, d2);
                }
            }
        }
    }
    return best;
}

__global__ void __launch_bounds__(kThreads) nn_query_kernel(ps_nn_grid g, const float* __restrict__ queries, int64_t N,
                                                            int64_t first_block, double inv, Taus taus, int K,
                                                            double* __restrict__ dist_out,
                                                            double* __restrict__ block_sums,
                                                            long long* __restrict__ block_counts) {
    __shared__ double red[kWarps];
    __shared__ long long redi[kWarps];
    // squared distances first, square roots in a pass of their own: little is live across the call to the fp64 sqrt's
    // slow path, so nothing spills
    __shared__ double dist[kBlockQueries];
    const int64_t base = (int64_t)blockIdx.x * kBlockQueries;
    const int n = (int)(N - base < kBlockQueries ? N - base : kBlockQueries);
#pragma unroll 1
    for (int j = threadIdx.x; j < n; j += kThreads) {
        const int64_t i = base + j;
        const float q[3] = {__ldg(queries + 3 * i), __ldg(queries + 3 * i + 1), __ldg(queries + 3 * i + 2)};
        dist[j] = nearest_sq(q, g, inv);
    }
#pragma unroll 1
    for (int j = threadIdx.x; j < n; j += kThreads) {
        double d = sqrt(dist[j]);
        if (!(d < g.cell)) d = g.cell;
        dist[j] = d;
        if (dist_out) dist_out[base + j] = d;
    }
    double sum = 0.0;
    int cnt[PS_NN_MAX_TAUS];
#pragma unroll
    for (int k = 0; k < PS_NN_MAX_TAUS; ++k) cnt[k] = 0;
    for (int j = threadIdx.x; j < n; j += kThreads) {        // the entries this thread wrote: no barrier needed
        const double d = dist[j];
        sum += d;
#pragma unroll
        for (int k = 0; k < PS_NN_MAX_TAUS; ++k) cnt[k] += (k < K && d < taus.v[k]) ? 1 : 0;
    }
    const int64_t b = first_block + blockIdx.x;
    const double s = block_sum(sum, red);
    if (threadIdx.x == 0) block_sums[b] = s;
#pragma unroll
    for (int k = 0; k < PS_NN_MAX_TAUS; ++k) {
        if (k >= K) break;                                     // uniform over the CTA
        const long long c = block_sum_i64(cnt[k], redi);
        if (threadIdx.x == 0) block_counts[b * K + k] = c;
    }
}

__global__ void __launch_bounds__(kThreads) nn_reduce_kernel(const double* __restrict__ block_sums,
                                                             const long long* __restrict__ block_counts,
                                                             int64_t nblocks, int K, int64_t n, double* __restrict__ mean,
                                                             long long* __restrict__ counts) {
    __shared__ double red[kWarps];
    __shared__ long long redi[kWarps];
    double v = 0.0;
    for (int64_t b = threadIdx.x; b < nblocks; b += kThreads) v += block_sums[b];
    const double s = block_sum(v, red);
    if (threadIdx.x == 0) mean[0] = s / (double)n;
    for (int k = 0; k < K; ++k) {
        long long c = 0;
        for (int64_t b = threadIdx.x; b < nblocks; b += kThreads) c += block_counts[b * K + k];
        const long long t = block_sum_i64(c, redi);
        if (threadIdx.x == 0) counts[k] = t;
    }
}

unsigned grid_for(int64_t n, int per_sm) {
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>(cdiv(n, kThreads), (int64_t)kNumSMs * per_sm));
}

bool pow2_capacity(int64_t c) { return c >= 2 && (c & (c - 1)) == 0; }

}  // namespace
}  // namespace ps

extern "C" int ps_nn_grid_bounds(const float* points, int64_t M, float* bounds, void* stream) {
    PS_REQUIRE(M >= 1, "nn_grid_bounds: empty point set");
    PS_REQUIRE(points && bounds, "nn_grid_bounds: null pointer");
    ps::nn_bounds_kernel<<<ps::grid_for(M, 8), ps::kThreads, 0, (cudaStream_t)stream>>>(points, M, bounds);
    return ps::check_launch("nn_grid_bounds");
}

extern "C" int ps_nn_grid_cells_per_axis(const float* bounds_host, double cell, int64_t* cells) {
    PS_REQUIRE(bounds_host && cells, "nn_grid_cells_per_axis: null pointer");
    PS_REQUIRE(cell >= ps::kMinCell && cell <= ps::kMaxCell, "nn_grid: cell size (radius) %g outside [%g, %g]", cell,
               ps::kMinCell, ps::kMaxCell);
    for (int a = 0; a < 3; ++a) {
        const double lo = (double)bounds_host[a], hi = (double)bounds_host[3 + a];
        PS_REQUIRE(std::isfinite(lo) && std::isfinite(hi) && lo <= hi,
                   "nn_grid_cells_per_axis: bounds of axis %d are [%g, %g]", a, lo, hi);
        const double top = std::floor((hi - lo) / cell);                  // the cell of the maximum, as nn_keys_kernel
        PS_REQUIRE(top < (double)ps::kCells,
                   "nn_grid: the points span %.9g m on axis %d, which needs %.0f cells of %.9g m; at most 2^21 = %lld "
                   "cells per axis fit the packed key (use a larger radius or crop the points)",
                   hi - lo, a, top + 1.0, cell, (long long)ps::kCells);
        cells[a] = (int64_t)top + 1;
    }
    return 0;
}

extern "C" int ps_nn_grid_keys(const float* points, int64_t M, const float* bounds_host, double cell, int64_t* keys,
                               void* stream) {
    PS_REQUIRE(M >= 1, "nn_grid_keys: empty point set");
    PS_REQUIRE(points && keys, "nn_grid_keys: null pointer");
    int64_t cells[3];
    if (int rc = ps_nn_grid_cells_per_axis(bounds_host, cell, cells)) return rc;
    ps::nn_keys_kernel<<<ps::grid_for(M, 16), ps::kThreads, 0, (cudaStream_t)stream>>>(
        points, M, bounds_host[0], bounds_host[1], bounds_host[2], cell, 1.0 / cell, reinterpret_cast<long long*>(keys));
    return ps::check_launch("nn_grid_keys");
}

extern "C" int ps_nn_grid_count_cells(const int64_t* sorted_keys, int64_t M, int64_t* n_cells, void* stream) {
    PS_REQUIRE(M >= 1, "nn_grid_count_cells: empty point set");
    PS_REQUIRE(sorted_keys && n_cells, "nn_grid_count_cells: null pointer");
    ps::nn_count_cells_kernel<<<ps::grid_for(M, 8), ps::kThreads, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const long long*>(sorted_keys), M, reinterpret_cast<unsigned long long*>(n_cells));
    return ps::check_launch("nn_grid_count_cells");
}

extern "C" int ps_nn_grid_cells(const float* points, const int64_t* perm, const int64_t* sorted_keys, int64_t M,
                                int64_t* cell_keys, int32_t* cell_ranges, int64_t capacity, float* points_sorted,
                                int* status, void* stream) {
    PS_REQUIRE(M >= 1 && M < (1ll << 31), "nn_grid_cells: %lld points outside [1, 2^31)", (long long)M);
    PS_REQUIRE(points && perm && sorted_keys && cell_keys && cell_ranges && points_sorted && status,
               "nn_grid_cells: null pointer");
    PS_REQUIRE(ps::pow2_capacity(capacity), "nn_grid_cells: capacity %lld is not a power of two", (long long)capacity);
    cudaStream_t st = (cudaStream_t)stream;
    const uint64_t mask = (uint64_t)capacity - 1;
    ps::nn_cells_kernel<<<ps::grid_for(M, 16), ps::kThreads, 0, st>>>(
        points, reinterpret_cast<const long long*>(perm), reinterpret_cast<const long long*>(sorted_keys), M,
        reinterpret_cast<long long*>(cell_keys), reinterpret_cast<int2*>(cell_ranges), mask, points_sorted, status);
    if (int rc = ps::check_launch("nn_grid_cells")) return rc;
    ps::nn_cell_ends_kernel<<<ps::grid_for(M, 16), ps::kThreads, 0, st>>>(
        reinterpret_cast<const long long*>(sorted_keys), M, reinterpret_cast<const long long*>(cell_keys),
        reinterpret_cast<int2*>(cell_ranges), mask, status);
    return ps::check_launch("nn_grid_cell_ends");
}

extern "C" int ps_nn_grid_query(const ps_nn_grid* grid, const float* queries, int64_t N, int64_t first_block,
                                const double* taus_host, int K, double* dist_out, double* block_sums,
                                int64_t* block_counts, void* stream) {
    PS_REQUIRE(grid && grid->points && grid->cell_keys && grid->cell_ranges, "nn_grid_query: null grid pointer");
    PS_REQUIRE(ps::pow2_capacity(grid->capacity), "nn_grid_query: capacity %lld is not a power of two",
               (long long)grid->capacity);
    PS_REQUIRE(grid->cell >= ps::kMinCell && grid->cell <= ps::kMaxCell, "nn_grid: cell size (radius) %g outside [%g, %g]",
               grid->cell, ps::kMinCell, ps::kMaxCell);
    PS_REQUIRE(N >= 0 && first_block >= 0, "nn_grid_query: negative size");
    PS_REQUIRE(K >= 0 && K <= PS_NN_MAX_TAUS, "nn_grid_query: K must be in [0, %d], got %d", PS_NN_MAX_TAUS, K);
    if (N == 0) return 0;
    PS_REQUIRE(queries && block_sums && (K == 0 || (taus_host && block_counts)), "nn_grid_query: null pointer");
    ps::Taus taus{};
    for (int k = 0; k < K; ++k) {
        PS_REQUIRE(taus_host[k] > 0.0 && taus_host[k] <= grid->cell,
                   "nn_grid_query: threshold %d = %g outside (0, r = %g]", k, taus_host[k], grid->cell);
        taus.v[k] = taus_host[k];
    }
    const int64_t blocks = ps::cdiv(N, ps::kBlockQueries);
    PS_REQUIRE(blocks < (1ll << 31), "nn_grid_query: %lld queries in one call", (long long)N);
    ps::nn_query_kernel<<<(unsigned)blocks, ps::kThreads, 0, (cudaStream_t)stream>>>(
        *grid, queries, N, first_block, 1.0 / grid->cell, taus, K, dist_out, block_sums, reinterpret_cast<long long*>(block_counts));
    return ps::check_launch("nn_grid_query");
}

extern "C" int ps_nn_grid_reduce(const double* block_sums, const int64_t* block_counts, int64_t nblocks, int K, int64_t n,
                                 double* mean, int64_t* counts, void* stream) {
    PS_REQUIRE(nblocks >= 1 && n >= 1, "nn_grid_reduce: empty input");
    PS_REQUIRE(K >= 0 && K <= PS_NN_MAX_TAUS, "nn_grid_reduce: K must be in [0, %d], got %d", PS_NN_MAX_TAUS, K);
    PS_REQUIRE(block_sums && mean && (K == 0 || (block_counts && counts)), "nn_grid_reduce: null pointer");
    ps::nn_reduce_kernel<<<1, ps::kThreads, 0, (cudaStream_t)stream>>>(
        block_sums, reinterpret_cast<const long long*>(block_counts), nblocks, K, n, mean,
        reinterpret_cast<long long*>(counts));
    return ps::check_launch("nn_grid_reduce");
}
