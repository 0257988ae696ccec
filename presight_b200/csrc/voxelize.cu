// Prior post-processing on the GPU (SURVEY 8f-4): voxel down-sampling of the extracted hit points with per-voxel means.
// Replaces, for the points of one tile resident in HBM (156 B per point: 1 G points fit one B200),
//   scripts/extract_priors.py:156-165   density filter (density > 1)
//   scripts/extract_priors.py:216-245   open3d PointCloud.voxel_down_sample_and_trace (bounds min - 1 / max + 1, index =
//                                        floor((p - (min_bound - voxel/2)) / voxel) in double precision)
//   scripts/extract_priors.py:175-191   per-voxel hit count, colour mean, fp64 feature mean -> fp16, hit quantile
// — the step the reference does on the host with ~300 GB of RAM (docs/building_priors.md:65).
//
// Design: an open-addressing hash table in HBM keyed by the packed voxel index (3 x 21 bits), one WARP per point:
// lane 0 claims / finds the slot (atomicCAS), the slot is broadcast, and the lanes add the point's coordinates, colour
// and features to the slot's fp64 accumulators with native double atomics.  Sums of fp16 features in fp64 are exact
// (11-bit mantissas, < 2^40 points), so the feature means are independent of the accumulation order; coordinates and
// colours are order-independent to ~1e-16 relative.  The table lives in caller-owned buffers.
#include "key_table.cuh"

#include <cmath>

#include <cuda_fp16.h>

namespace ps {

__device__ __forceinline__ bool point_selected(const float* __restrict__ dens, int64_t i) {
    return dens == nullptr || __ldg(dens + i) > 1.0f;
}

// min over the selected points, per axis (float atomics through the int ordering trick); out[3] preset to +inf
__global__ void __launch_bounds__(256) voxel_min_kernel(const float* __restrict__ pts, const float* __restrict__ dens,
                                                        int64_t N, float* __restrict__ out) {
    float m[3] = {INFINITY, INFINITY, INFINITY};
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
        if (!point_selected(dens, i)) continue;
#pragma unroll
        for (int a = 0; a < 3; ++a) m[a] = fminf(m[a], __ldg(pts + 3 * i + a));
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        m[a] = warp_min(m[a]);
        if ((threadIdx.x & 31) == 0 && m[a] != INFINITY) atomic_min_float(out + a, m[a]);
    }
}

// voxel index of a point exactly as open3d computes it: doubles, bound shifted by half a voxel, floor
__device__ __forceinline__ long long voxel_key(const float* __restrict__ p, const float* __restrict__ min_pt,
                                               double voxel, bool& ok) {
    long long key = 0;
    ok = true;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const double vmb = (double)__fsub_rn(min_pt[a], 1.0f) - voxel * 0.5;     // (min - 1) in float32 as numpy does
        const double ref = ((double)p[a] - vmb) / voxel;
        const long long idx = (long long)floor(ref);
        if (idx < 0 || idx >= (1ll << 21)) ok = false;
        key = (key << 21) | (idx & ((1ll << 21) - 1));
    }
    return key;
}

__global__ void __launch_bounds__(256) voxel_accumulate_kernel(
    const float* __restrict__ pts, const __half* __restrict__ feat, const float* __restrict__ col,
    const float* __restrict__ dens, int64_t N, int C, const float* __restrict__ min_pt, double voxel,
    long long* __restrict__ keys, uint64_t cap_mask, unsigned int* __restrict__ cnt, double* __restrict__ sum_xyz,
    double* __restrict__ sum_col, double* __restrict__ sum_feat, int* __restrict__ status) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < N; i += warps) {
        if (!point_selected(dens, i)) continue;                       // warp-uniform
        float p[3] = {__ldg(pts + 3 * i), __ldg(pts + 3 * i + 1), __ldg(pts + 3 * i + 2)};
        long long slot = -1;
        if (lane == 0) {
            bool ok;
            const long long key = voxel_key(p, min_pt, voxel, ok);
            if (!ok) {
                atomicOr(status, 2);                                  // voxel index outside 21 bits per axis
            } else {
                uint64_t s = mix64((uint64_t)key) & cap_mask;
                for (uint64_t probe = 0; probe <= cap_mask; ++probe) {
                    const long long prev = (long long)atomicCAS(reinterpret_cast<unsigned long long*>(keys + s),
                                                                (unsigned long long)kEmptyKey, (unsigned long long)key);
                    if (prev == kEmptyKey || prev == key) { slot = (long long)s; break; }
                    s = (s + 1) & cap_mask;
                }
                if (slot < 0) atomicOr(status, 1);                    // table full
            }
        }
        slot = __shfl_sync(0xffffffffu, slot, 0);
        if (slot < 0) continue;
        if (lane == 0) atomicAdd(cnt + slot, 1u);
        if (lane < 3) atomicAdd(sum_xyz + slot * 3 + lane, (double)p[lane]);
        else if (lane < 6 && col) atomicAdd(sum_col + slot * 3 + (lane - 3), (double)__ldg(col + 3 * i + (lane - 3)));
        if (feat)
            for (int c = lane; c < C; c += 32)
                atomicAdd(sum_feat + slot * C + c, (double)__half2float(feat[i * C + c]));
    }
}

// centre of mass, colour mean, feature mean (fp64 mean rounded once to fp16, as numpy's astype does) of accumulator row
// `s` into output row `row`; one warp
__device__ __forceinline__ void write_means(uint64_t s, unsigned long long row, int lane, unsigned int count,
                                           const double* __restrict__ sum_xyz, const double* __restrict__ sum_col,
                                           const double* __restrict__ sum_feat, int C, float* __restrict__ out_xyz,
                                           float* __restrict__ out_col, __half* __restrict__ out_feat) {
    const double n = (double)count;
    if (lane < 3) out_xyz[row * 3 + lane] = (float)(sum_xyz[s * 3 + lane] / n);
    else if (lane < 6 && out_col) out_col[row * 3 + (lane - 3)] = (float)(sum_col[s * 3 + (lane - 3)] / n);
    if (out_feat)
        for (int c = lane; c < C; c += 32) out_feat[row * C + c] = __double2half(sum_feat[s * C + c] / n);
}

// occupied slots -> dense rows (arbitrary order; the caller orders them by key): key, means, hits
__global__ void __launch_bounds__(256) voxel_finalize_kernel(
    const long long* __restrict__ keys, uint64_t cap, const unsigned int* __restrict__ cnt,
    const double* __restrict__ sum_xyz, const double* __restrict__ sum_col, const double* __restrict__ sum_feat, int C,
    unsigned long long* __restrict__ n_out, long long* __restrict__ out_keys, float* __restrict__ out_xyz,
    float* __restrict__ out_col, __half* __restrict__ out_feat, long long* __restrict__ out_hits) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t s = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; s < cap; s += warps) {
        const long long key = keys[s];
        if (key == kEmptyKey) continue;
        unsigned long long row = 0;
        if (lane == 0) row = atomicAdd(n_out, 1ull);
        row = __shfl_sync(0xffffffffu, row, 0);
        if (lane == 0) {
            out_keys[row] = key;
            out_hits[row] = (long long)cnt[s];
        }
        write_means(s, row, lane, cnt[s], sum_xyz, sum_col, sum_feat, C, out_xyz, out_col, out_feat);
    }
}

// ---- the tile voxelizer: a key table sized by the voxels, then dense rows in ascending key order ---------------------
// Pass 1 inserts keys only (8 B per slot; the caller keeps the load factor <= 1/2 and grows the table with
// ps_voxel_rehash).  Sealing ranks the sorted keys into a row array beside the table (4 B per slot).  Pass 2 looks each
// point's row up and adds it to dense fp64 rows with the accumulate kernel's warp-per-point scheme.
// status: |= 1 table full, |= 2 voxel index outside 21 bits per axis, |= 4 a point's voxel is not in the table.

__global__ void __launch_bounds__(256) voxel_insert_kernel(const float* __restrict__ pts, int64_t N,
                                                           const float* __restrict__ min_pt, double voxel,
                                                           long long* __restrict__ keys, uint64_t cap_mask,
                                                           unsigned long long* __restrict__ n_voxels,
                                                           int* __restrict__ status) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
        const float p[3] = {__ldg(pts + 3 * i), __ldg(pts + 3 * i + 1), __ldg(pts + 3 * i + 2)};
        bool ok, fresh;
        const long long key = voxel_key(p, min_pt, voxel, ok);
        if (!ok) { atomicOr(status, 2); continue; }
        if (table_insert(keys, cap_mask, key, fresh) < 0) atomicOr(status, 1);
        else if (fresh) atomicAdd(n_voxels, 1ull);
    }
}

__global__ void __launch_bounds__(256) voxel_rehash_kernel(const long long* __restrict__ old_keys, uint64_t old_cap,
                                                           long long* __restrict__ keys, uint64_t cap_mask,
                                                           int* __restrict__ status) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < old_cap; s += stride) {
        const long long key = old_keys[s];
        bool fresh;
        if (key != kEmptyKey && table_insert(keys, cap_mask, key, fresh) < 0) atomicOr(status, 1);
    }
}

__global__ void __launch_bounds__(256) voxel_assign_rows_kernel(const long long* __restrict__ sorted_keys, int64_t V,
                                                                const long long* __restrict__ keys, uint64_t cap_mask,
                                                                int* __restrict__ rows, int* __restrict__ status) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < V; r += stride) {
        const long long s = table_find(keys, cap_mask, sorted_keys[r]);
        if (s < 0) atomicOr(status, 4);
        else rows[s] = (int)r;
    }
}

__global__ void __launch_bounds__(256) voxel_accumulate_rows_kernel(
    const float* __restrict__ pts, const __half* __restrict__ feat, const float* __restrict__ col, int64_t N, int C,
    const float* __restrict__ min_pt, double voxel, const long long* __restrict__ keys, const int* __restrict__ rows,
    uint64_t cap_mask, unsigned int* __restrict__ cnt, double* __restrict__ sum_xyz, double* __restrict__ sum_col,
    double* __restrict__ sum_feat, int* __restrict__ status) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < N; i += warps) {
        const float p[3] = {__ldg(pts + 3 * i), __ldg(pts + 3 * i + 1), __ldg(pts + 3 * i + 2)};
        long long row = -1;
        if (lane == 0) {
            bool ok;
            const long long key = voxel_key(p, min_pt, voxel, ok);
            const long long s = ok ? table_find(keys, cap_mask, key) : -1;
            if (!ok) atomicOr(status, 2);
            else if (s < 0) atomicOr(status, 4);
            else row = rows[s];
        }
        row = __shfl_sync(0xffffffffu, row, 0);
        if (row < 0) continue;
        if (lane == 0) atomicAdd(cnt + row, 1u);
        if (lane < 3) atomicAdd(sum_xyz + row * 3 + lane, (double)(lane == 0 ? p[0] : lane == 1 ? p[1] : p[2]));
        else if (lane < 6 && col) atomicAdd(sum_col + row * 3 + (lane - 3), (double)__ldg(col + 3 * i + (lane - 3)));
        if (feat)
            for (int c = lane; c < C; c += 32) atomicAdd(sum_feat + row * C + c, (double)__half2float(feat[i * C + c]));
    }
}

__global__ void __launch_bounds__(256) voxel_finalize_rows_kernel(
    const unsigned int* __restrict__ cnt, const double* __restrict__ sum_xyz, const double* __restrict__ sum_col,
    const double* __restrict__ sum_feat, int64_t V, int C, float* __restrict__ out_xyz, float* __restrict__ out_col,
    __half* __restrict__ out_feat, long long* __restrict__ out_hits) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < (uint64_t)V; r += warps) {
        if (lane == 0) out_hits[r] = (long long)cnt[r];
        write_means(r, r, lane, cnt[r], sum_xyz, sum_col, sum_feat, C, out_xyz, out_col, out_feat);
    }
}

// ---- owner partition of stored hits (one tile's extraction over several GPUs) ---------------------------------------
// A stable counting sort of the extractor's stored hits by owner rank, in two launches over G <= kPartMaxBlocks blocks,
// each owning one contiguous span of hits (the pattern of ps_hits_append): (1) every block counts its hits per owner
// into ws[r * G + b]; (2) every block sums, per owner, the counts of all blocks (the segment sizes, which block 0 writes
// out) and of the blocks before it, then walks its span in tiles of 256 hits, ranking each owner's hits within a tile by
// a warp match and per-warp counts.  Nothing reads a value written by the same launch: no host round trip, no spin-wait.
constexpr int kPartThreads = 256;
constexpr int kPartWarps = kPartThreads / 32;
constexpr int kPartMaxBlocks = 1024;
constexpr int64_t kPartMinSpan = 2048;
constexpr int kPartMaxWorld = 64;

// Owner rank of a voxel key: the high 32 bits of splitmix64(key), mod world.  Not the low bits: every rank's key table
// places its keys by the low bits of the same hash, and a rank owns only keys of one residue.
__device__ __forceinline__ int owner_of(long long key, int world) {
    return (int)((mix64((uint64_t)key) >> 32) % (uint64_t)world);
}

// owner of stored hit i: its voxel key from the metre value TileVoxelizer.insert receives (an IEEE division of the
// scene-unit point by the pose scale, as PriorExtractor.finalize computes it)
__device__ __forceinline__ int hit_owner(const float* __restrict__ pts, int64_t i, float pose_scale,
                                         const float* __restrict__ min_pt, double voxel, int world, bool& ok) {
    const float p[3] = {__fdiv_rn(__ldg(pts + 3 * i), pose_scale), __fdiv_rn(__ldg(pts + 3 * i + 1), pose_scale),
                        __fdiv_rn(__ldg(pts + 3 * i + 2), pose_scale)};
    return owner_of(voxel_key(p, min_pt, voxel, ok), world);
}

__global__ void __launch_bounds__(kPartThreads) partition_count_kernel(
    const float* __restrict__ pts, int64_t N, int64_t span, float pose_scale, const float* __restrict__ min_pt,
    double voxel, int world, long long* __restrict__ ws, int* __restrict__ status) {
    __shared__ int s_cnt[kPartMaxWorld];
    const int G = gridDim.x, b = blockIdx.x, lane = threadIdx.x & 31;
    for (int r = threadIdx.x; r < world; r += kPartThreads) s_cnt[r] = 0;
    __syncthreads();
    const int64_t lo = (int64_t)b * span, hi = min(N, lo + span);
    bool bad = false;
    for (int64_t t0 = lo; t0 < hi; t0 += kPartThreads) {         // block-uniform trip count: full-warp matches
        const int64_t i = t0 + threadIdx.x;
        bool ok = true;
        const int o = i < hi ? hit_owner(pts, i, pose_scale, min_pt, voxel, world, ok) : -1;
        bad |= !ok;
        const unsigned peers = __match_any_sync(0xffffffffu, o);
        if (o >= 0 && lane == __ffs(peers) - 1) atomicAdd(s_cnt + o, __popc(peers));
    }
    if (bad) atomicOr(status, 2);                                  // voxel index outside 21 bits per axis
    __syncthreads();
    for (int r = threadIdx.x; r < world; r += kPartThreads) ws[(int64_t)r * G + b] = s_cnt[r];
}

__global__ void __launch_bounds__(kPartThreads) partition_scatter_kernel(
    const float* __restrict__ pts, const float* __restrict__ cols, int64_t N, int64_t span, float pose_scale,
    const float* __restrict__ min_pt, double voxel, int world, const long long* __restrict__ ws,
    float* __restrict__ out_pts, float* __restrict__ out_cols, long long* __restrict__ counts) {
    __shared__ long long s_pre[kPartMaxWorld], s_tot[kPartMaxWorld];
    __shared__ long long s_base[kPartMaxWorld];                    // next output row of each owner in this block
    __shared__ int s_warp[kPartWarps][kPartMaxWorld];              // hits of each owner in each warp of the tile
    const int G = gridDim.x, b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int r = warp; r < world; r += kPartWarps) {               // one warp per owner: its column of the counts
        long long pre = 0, tot = 0;
        for (int j = lane; j < G; j += 32) {
            const long long c = ws[(int64_t)r * G + j];
            tot += c;
            pre += j < b ? c : 0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            pre += __shfl_xor_sync(0xffffffffu, pre, o);
            tot += __shfl_xor_sync(0xffffffffu, tot, o);
        }
        if (lane == 0) s_pre[r] = pre, s_tot[r] = tot;
    }
    for (int k = threadIdx.x; k < kPartWarps * kPartMaxWorld; k += kPartThreads) (&s_warp[0][0])[k] = 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long seg = 0;                                         // owner r's segment starts after owners < r
        for (int r = 0; r < world; ++r) {
            s_base[r] = seg + s_pre[r];
            if (b == 0) counts[r] = s_tot[r];
            seg += s_tot[r];
        }
    }
    __syncthreads();
    const int64_t lo = (int64_t)b * span, hi = min(N, lo + span);
    for (int64_t t0 = lo; t0 < hi; t0 += kPartThreads) {
        const int64_t i = t0 + threadIdx.x;
        bool ok = true;
        const int o = i < hi ? hit_owner(pts, i, pose_scale, min_pt, voxel, world, ok) : -1;
        const unsigned peers = __match_any_sync(0xffffffffu, o);
        if (o >= 0 && lane == __ffs(peers) - 1) s_warp[warp][o] = __popc(peers);
        __syncthreads();
        if (o >= 0) {
            long long row = s_base[o] + __popc(peers & ((1u << lane) - 1u));
            for (int w = 0; w < warp; ++w) row += s_warp[w][o];
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                out_pts[3 * row + a] = __ldg(pts + 3 * i + a);
                out_cols[3 * row + a] = __ldg(cols + 3 * i + a);
            }
        }
        __syncthreads();
        for (int r = threadIdx.x; r < world; r += kPartThreads) {
            long long t = 0;
#pragma unroll
            for (int w = 0; w < kPartWarps; ++w) {
                t += s_warp[w][r];
                s_warp[w][r] = 0;
            }
            s_base[r] += t;
        }
        __syncthreads();
    }
}

int64_t partition_blocks(int64_t N) {
    const int64_t g = cdiv(N, kPartMinSpan);
    return g < 1 ? 1 : (g > kPartMaxBlocks ? kPartMaxBlocks : g);
}

// np.quantile(hits, q) (linear interpolation, numpy's _lerp) from a histogram of the hit counts; one CTA.
__global__ void __launch_bounds__(1024) hits_hist_kernel(const long long* __restrict__ hits, int64_t M,
                                                          unsigned int* __restrict__ hist, int64_t bins,
                                                          int* __restrict__ status) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += stride) {
        const long long h = hits[i];
        if (h < 0 || h >= bins) atomicOr(status, 4);
        else atomicAdd(hist + h, 1u);
    }
}
__global__ void hits_quantile_kernel(const unsigned int* __restrict__ hist, int64_t bins, int64_t M, double q,
                                     double* __restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    // virtual index (n - 1) q; order statistics k0 = floor, k1 = k0 + 1 (clamped)
    const double vi = (double)(M - 1) * q;
    int64_t k0 = (int64_t)floor(vi);
    if (k0 < 0) k0 = 0;
    if (k0 > M - 1) k0 = M - 1;
    const int64_t k1 = k0 + 1 > M - 1 ? M - 1 : k0 + 1;
    const double t = vi - (double)k0;
    double a = 0.0, b = 0.0;
    int64_t seen = 0;
    bool have_a = false;
    for (int64_t v = 0; v < bins; ++v) {
        seen += hist[v];
        if (!have_a && seen > k0) { a = (double)v; have_a = true; }
        if (seen > k1) { b = (double)v; break; }
    }
    const double diff = b - a;
    double r = a + diff * t;
    if (t >= 0.5) r = b - diff * (1.0 - t);                 // numpy/lib/function_base.py:_lerp
    if (diff == 0.0) r = a;
    out[0] = r;
}

}  // namespace ps

using namespace ps;

extern "C" int ps_voxel_min_bound(const float* points, const float* densities, int64_t N, float* min_out, void* stream) {
    if (N == 0) return 0;
    PS_REQUIRE(points && min_out, "voxel_min_bound: null pointer");
    int64_t blocks = cdiv(N, 256 * 8);
    if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
    voxel_min_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(points, densities, N, min_out);
    return check_launch("voxel_min_bound");
}

extern "C" int ps_voxel_accumulate(const float* points, const void* features_f16, const float* colors,
                                   const float* densities, int64_t N, int C, const float* min_point, double voxel_size,
                                   int64_t* keys, int64_t capacity, uint32_t* counts, double* sum_xyz, double* sum_col,
                                   double* sum_feat, int* status, void* stream) {
    if (N == 0) return 0;
    PS_REQUIRE(points && min_point && keys && counts && sum_xyz && status, "voxel_accumulate: null pointer");
    PS_REQUIRE(capacity >= 2 && (capacity & (capacity - 1)) == 0, "voxel_accumulate: capacity %lld is not a power of two",
               (long long)capacity);
    PS_REQUIRE(voxel_size > 0.0, "voxel_accumulate: voxel size must be positive");
    PS_REQUIRE((features_f16 == nullptr) == (sum_feat == nullptr), "voxel_accumulate: features and sum_feat go together");
    PS_REQUIRE((colors == nullptr) == (sum_col == nullptr), "voxel_accumulate: colors and sum_col go together");
    PS_REQUIRE(features_f16 == nullptr || C >= 1, "voxel_accumulate: bad feature width %d", C);
    int64_t blocks = cdiv(N, 8);                                       // 8 warps (points) per CTA per pass
    if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
    voxel_accumulate_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        points, reinterpret_cast<const __half*>(features_f16), colors, densities, N, C, min_point, voxel_size,
        reinterpret_cast<long long*>(keys), (uint64_t)capacity - 1, counts, sum_xyz, sum_col, sum_feat, status);
    return check_launch("voxel_accumulate");
}

extern "C" int ps_voxel_finalize(const int64_t* keys, int64_t capacity, const uint32_t* counts, const double* sum_xyz,
                                 const double* sum_col, const double* sum_feat, int C, uint64_t* n_out, int64_t* out_keys,
                                 float* out_xyz, float* out_col, void* out_feat_f16, int64_t* out_hits, void* stream) {
    PS_REQUIRE(keys && counts && sum_xyz && n_out && out_keys && out_xyz && out_hits, "voxel_finalize: null pointer");
    PS_REQUIRE((sum_col == nullptr) == (out_col == nullptr) && (sum_feat == nullptr) == (out_feat_f16 == nullptr),
               "voxel_finalize: accumulators and outputs go together");
    int64_t blocks = cdiv(capacity, 8);
    if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
    voxel_finalize_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const long long*>(keys), (uint64_t)capacity, counts, sum_xyz, sum_col, sum_feat, C,
        reinterpret_cast<unsigned long long*>(n_out), reinterpret_cast<long long*>(out_keys), out_xyz, out_col,
        reinterpret_cast<__half*>(out_feat_f16), reinterpret_cast<long long*>(out_hits));
    return check_launch("voxel_finalize");
}

static bool pow2_capacity(int64_t capacity) { return capacity >= 2 && (capacity & (capacity - 1)) == 0; }

extern "C" int ps_voxel_insert(const float* points, int64_t N, const float* min_point, double voxel_size, int64_t* keys,
                               int64_t capacity, uint64_t* n_voxels, int* status, void* stream) {
    PS_REQUIRE(N >= 0, "voxel_insert: negative point count %lld", (long long)N);
    if (N == 0) return 0;
    PS_REQUIRE(points && min_point && keys && n_voxels && status, "voxel_insert: null pointer");
    PS_REQUIRE(pow2_capacity(capacity), "voxel_insert: capacity %lld is not a power of two", (long long)capacity);
    PS_REQUIRE(voxel_size > 0.0, "voxel_insert: voxel size must be positive");
    int64_t blocks = cdiv(N, 256);
    if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
    voxel_insert_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        points, N, min_point, voxel_size, reinterpret_cast<long long*>(keys), (uint64_t)capacity - 1,
        reinterpret_cast<unsigned long long*>(n_voxels), status);
    return check_launch("voxel_insert");
}

extern "C" int ps_voxel_rehash(const int64_t* old_keys, int64_t old_capacity, int64_t* keys, int64_t capacity, int* status,
                               void* stream) {
    PS_REQUIRE(old_keys && keys && status, "voxel_rehash: null pointer");
    PS_REQUIRE(pow2_capacity(old_capacity) && pow2_capacity(capacity) && capacity >= old_capacity,
               "voxel_rehash: capacities %lld -> %lld must be powers of two that do not shrink", (long long)old_capacity,
               (long long)capacity);
    int64_t blocks = cdiv(old_capacity, 256);
    if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
    voxel_rehash_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const long long*>(old_keys), (uint64_t)old_capacity, reinterpret_cast<long long*>(keys),
        (uint64_t)capacity - 1, status);
    return check_launch("voxel_rehash");
}

extern "C" int ps_voxel_assign_rows(const int64_t* sorted_keys, int64_t V, const int64_t* keys, int64_t capacity,
                                    int32_t* rows, int* status, void* stream) {
    PS_REQUIRE(V >= 0 && V < (1ll << 31), "voxel_assign_rows: %lld voxels outside [0, 2^31)", (long long)V);
    if (V == 0) return 0;
    PS_REQUIRE(sorted_keys && keys && rows && status, "voxel_assign_rows: null pointer");
    PS_REQUIRE(pow2_capacity(capacity) && capacity >= 2 * V, "voxel_assign_rows: capacity %lld for %lld voxels",
               (long long)capacity, (long long)V);
    int64_t blocks = cdiv(V, 256);
    if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
    voxel_assign_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const long long*>(sorted_keys), V, reinterpret_cast<const long long*>(keys),
        (uint64_t)capacity - 1, rows, status);
    return check_launch("voxel_assign_rows");
}

extern "C" int ps_voxel_accumulate_rows(const float* points, const void* features_f16, const float* colors, int64_t N,
                                        int C, const float* min_point, double voxel_size, const int64_t* keys,
                                        const int32_t* rows, int64_t capacity, uint32_t* counts, double* sum_xyz,
                                        double* sum_col, double* sum_feat, int* status, void* stream) {
    PS_REQUIRE(N >= 0, "voxel_accumulate_rows: negative point count %lld", (long long)N);
    if (N == 0) return 0;
    PS_REQUIRE(points && min_point && keys && rows && counts && sum_xyz && status, "voxel_accumulate_rows: null pointer");
    PS_REQUIRE(pow2_capacity(capacity), "voxel_accumulate_rows: capacity %lld is not a power of two", (long long)capacity);
    PS_REQUIRE(voxel_size > 0.0, "voxel_accumulate_rows: voxel size must be positive");
    PS_REQUIRE((features_f16 == nullptr) == (sum_feat == nullptr), "voxel_accumulate_rows: features and sum_feat go together");
    PS_REQUIRE((colors == nullptr) == (sum_col == nullptr), "voxel_accumulate_rows: colors and sum_col go together");
    PS_REQUIRE(features_f16 == nullptr || C >= 1, "voxel_accumulate_rows: bad feature width %d", C);
    int64_t blocks = cdiv(N, 8);                                       // 8 warps (points) per CTA per pass
    if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
    voxel_accumulate_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        points, reinterpret_cast<const __half*>(features_f16), colors, N, C, min_point, voxel_size,
        reinterpret_cast<const long long*>(keys), rows, (uint64_t)capacity - 1, counts, sum_xyz, sum_col, sum_feat,
        status);
    return check_launch("voxel_accumulate_rows");
}

extern "C" int ps_voxel_finalize_rows(const uint32_t* counts, const double* sum_xyz, const double* sum_col,
                                      const double* sum_feat, int64_t V, int C, float* out_xyz, float* out_col,
                                      void* out_feat_f16, int64_t* out_hits, void* stream) {
    PS_REQUIRE(V >= 0, "voxel_finalize_rows: negative row count %lld", (long long)V);
    if (V == 0) return 0;
    PS_REQUIRE(counts && sum_xyz && out_xyz && out_hits, "voxel_finalize_rows: null pointer");
    PS_REQUIRE((sum_col == nullptr) == (out_col == nullptr) && (sum_feat == nullptr) == (out_feat_f16 == nullptr),
               "voxel_finalize_rows: accumulators and outputs go together");
    PS_REQUIRE(sum_feat == nullptr || C >= 1, "voxel_finalize_rows: bad feature width %d", C);
    int64_t blocks = cdiv(V, 8);
    if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
    voxel_finalize_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        counts, sum_xyz, sum_col, sum_feat, V, C, out_xyz, out_col, reinterpret_cast<__half*>(out_feat_f16),
        reinterpret_cast<long long*>(out_hits));
    return check_launch("voxel_finalize_rows");
}

extern "C" int ps_hits_histogram(const int64_t* hits, int64_t M, uint32_t* hist, int64_t bins, int* status,
                                 void* stream) {
    PS_REQUIRE(M >= 0, "hits_histogram: negative count %lld", (long long)M);
    if (M == 0) return 0;
    PS_REQUIRE(hits && hist && status, "hits_histogram: null pointer");
    PS_REQUIRE(bins >= 1, "hits_histogram: no bins");
    int64_t blocks = cdiv(M, 1024);
    if (blocks > kNumSMs * 2) blocks = kNumSMs * 2;
    hits_hist_kernel<<<(unsigned)blocks, 1024, 0, (cudaStream_t)stream>>>(reinterpret_cast<const long long*>(hits), M, hist,
                                                                        bins, status);
    return check_launch("hits_histogram");
}

extern "C" int ps_hits_quantile_from_histogram(const uint32_t* hist, int64_t bins, int64_t M, double q, double* out,
                                               void* stream) {
    PS_REQUIRE(hist && out, "hits_quantile_from_histogram: null pointer");
    PS_REQUIRE(M >= 1 && bins >= 1, "hits_quantile_from_histogram: empty input");
    PS_REQUIRE(q >= 0.0 && q <= 1.0, "hits_quantile_from_histogram: q = %f outside [0, 1]", q);
    hits_quantile_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(hist, bins, M, q, out);
    return check_launch("hits_quantile_from_histogram");
}

extern "C" int ps_hits_quantile(const int64_t* hits, int64_t M, double q, uint32_t* hist, int64_t bins, double* out,
                                int* status, void* stream) {
    PS_REQUIRE(hits && hist && out && status, "hits_quantile: null pointer");
    PS_REQUIRE(M >= 1 && bins >= 2, "hits_quantile: empty input");
    PS_REQUIRE(q >= 0.0 && q <= 1.0, "hits_quantile: q = %f outside [0, 1]", q);
    if (int e = ps_hits_histogram(hits, M, hist, bins, status, stream)) return e;
    return ps_hits_quantile_from_histogram(hist, bins, M, q, out, stream);
}

extern "C" int ps_voxel_partition_workspace(int64_t N, int world, int64_t* bytes) {
    PS_REQUIRE(bytes, "voxel_partition_workspace: null pointer");
    PS_REQUIRE(N >= 0, "voxel_partition_workspace: negative hit count %lld", (long long)N);
    PS_REQUIRE(world >= 1 && world <= kPartMaxWorld, "voxel_partition_workspace: world %d outside [1, %d]", world,
               kPartMaxWorld);
    *bytes = partition_blocks(N) * world * (int64_t)sizeof(long long);
    return 0;
}

extern "C" int ps_voxel_partition(const float* points_scaled, const float* colors, int64_t N, float pose_scale,
                                  const float* min_point, double voxel_size, int world, float* out_points,
                                  float* out_colors, int64_t* counts, int* status, void* workspace, void* stream) {
    PS_REQUIRE(N >= 0, "voxel_partition: negative hit count %lld", (long long)N);
    PS_REQUIRE(world >= 1 && world <= kPartMaxWorld, "voxel_partition: world %d outside [1, %d]", world, kPartMaxWorld);
    PS_REQUIRE(counts && status && workspace, "voxel_partition: null pointer");
    PS_REQUIRE(N == 0 || (points_scaled && colors && min_point && out_points && out_colors),
               "voxel_partition: null pointer");
    PS_REQUIRE(pose_scale > 0.f && std::isfinite(pose_scale), "voxel_partition: pose scale factor %g is not a positive "
               "number", (double)pose_scale);
    PS_REQUIRE(voxel_size > 0.0, "voxel_partition: voxel size must be positive");
    const int64_t G = partition_blocks(N);                          // N == 0: one block writes zero counts
    const int64_t span = cdiv(cdiv(N, G), kPartThreads) * kPartThreads;
    auto* ws = reinterpret_cast<long long*>(workspace);
    partition_count_kernel<<<(unsigned)G, kPartThreads, 0, (cudaStream_t)stream>>>(
        points_scaled, N, span, pose_scale, min_point, voxel_size, world, ws, status);
    if (int e = check_launch("voxel_partition(count)")) return e;
    partition_scatter_kernel<<<(unsigned)G, kPartThreads, 0, (cudaStream_t)stream>>>(
        points_scaled, colors, N, span, pose_scale, min_point, voxel_size, world, ws, out_points, out_colors,
        reinterpret_cast<long long*>(counts));
    return check_launch("voxel_partition");
}
