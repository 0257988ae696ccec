// Fused proposal level: bin edges -> sample positions -> contraction -> multiresolution hash gather -> density MLP ->
// weights, ONE kernel; backward = ONE kernel (recompute, compositing backward, MLP backward, hash scatter-add).
// Reference: model_components/ray_samplers.py:600-609 (density_fn + get_weights per proposal level),
// fields/PreSight/prop_density_field.py:129-153, field_components/encodings.py:343-384, cameras/rays.py:49-58,128-150.
//
// CTA = 128 threads = one 128-point tile (128 / S rays), one thread per sample, several CTAs per SM so that the gather /
// scatter latency of one tile hides behind the MMA + epilogue of another.  The hash arithmetic is the bit-exact code of
// hash_grid.cuh; the first MLP layer runs on tcgen05.mma (bf16, fp32 accumulate in TMEM), the 1-wide output layer is a
// per-thread dot product over the bf16-rounded hidden row; in the backward the input-gradient GEMM, both weight-gradient
// GEMMs and the hidden bias gradient (a GEMM against a ones tile) run on the tensor core with accumulators resident in
// TMEM for the whole kernel.  The scatter-add keeps the warp pre-aggregation and x-pair merge of the stand-alone kernel.
//
// The forward kernels also serve the density head of the main field (ps_density_level_fwd / _ms: base0 [64, L*F] + ReLU,
// row 0 of base1, trunc_exp * selector — the same network shape with a wider input), instantiated for hidden 64,
// F in {1, 2, 4} and the padded input width K0 = 16 / 32 / 48; they write each pair of levels straight into the bf16 X0
// tile (gather_to_tile).  The proposal instantiations (K0 = 16, F <= 2) keep their register path and compile to the same
// SASS as before the widening (prop_fwd_kernel<64, 1> up to register numbering).  ptxas -v, sm_100a, CUDA 12.9, forward
// only, no spills in any of them; registers (ray mode / routed mode) and dynamic shared memory:
//   F = 1  K0 = 32: 62 / 52 regs     F = 2  K0 = 32: 68 / 72 regs     F = 4  K0 = 16: 92 / 94 regs
//          K0 = 48: 62 / 52 regs            K0 = 48: 67 / 72 regs            K0 = 32: 92 / 94 regs
//                                                                            K0 = 48: 96 / 94 regs
//   shared memory 21.1 KB (K0 = 32) / 27.2 KB (K0 = 48); resident CTAs per SM (registers / shared memory / 64 TMEM
//   columns): 8 up to 64 registers, 7 up to 72, 5 for the F = 4 kernels.
#include <cuda_bf16.h>
#include <stdlib.h>

#include "composite.cuh"
#include "hash_grid.cuh"
#include "position.cuh"
#include "tc5.cuh"

namespace ps {
namespace ptc5 {

using namespace tc5;

constexpr int kThreads = 128;
constexpr int kK0 = 16;   // padded input width (L * F <= 16)

struct PropArgs {
    const float *W0, *b0, *W1, *b1;   // [H, in], [H], [1, H], [1]
    float *dW0, *db0, *dW1, *db1;
    int in_dim;
    const float* origins;   // [N,3]
    const float* dirs;      // [N,3]
    const float* eu;        // [N,S+1]
    int64_t N;
    int S;
    Aabb box;
    int contract;
    const float* table;     // [L*T, F]
    float* dtable;
    HashParams hp;
    int F;
    float* weights;         // [N,S] forward output
    __nv_bfloat16* feat;    // [N*S, feat_stride] bf16 features (forward: nullable output; backward: input)
    int feat_stride;        // 8 or 16
    const float* d_w;       // [N,S]
};

// K0: padded input width of the first layer.  The backward kernels exist for K0 = 16 only; the forward kernels are
// also instantiated for K0 = 32 / 48 (the main field's density head, ps_density_level_fwd*).
template <int H, int K0 = kK0>
struct Smem {
    // tiles used as the M = 128 "X" operand of a weight-gradient GEMM (H1, DZ0) are followed by >= 32 KB - own size
    static constexpr uint32_t h1 = 0;                                  // [128 x H]   (backward)
    static constexpr uint32_t dz0 = h1 + cm_bytes(kRows, H);           // [128 x H]   (backward)
    static constexpr uint32_t x0 = dz0 + cm_bytes(kRows, H);           // [128 x K0]
    static constexpr uint32_t dz1 = x0 + cm_bytes(kRows, K0);          // [128 x 16]  (backward)
    static constexpr uint32_t ones = dz1 + cm_bytes(kRows, kK0);       // [128 x 16] of 1.0 (backward)
    static constexpr uint32_t w0 = ones + cm_bytes(kRows, kK0);        // [H x K0]
    static constexpr uint32_t fl = w0 + cm_bytes(H, K0);              // float: b0[H] | w1[H] (bf16-rounded) | b1
    static constexpr uint32_t tails = fl + (2 * H + 4) * 4;            // double [4][2]
    static constexpr uint32_t bars = ((tails + 64 + 15) / 16) * 16;
    static constexpr uint32_t used = bars + 32;
    static constexpr uint32_t bwd_total = (dz0 + 32 * 1024 > used) ? dz0 + 32 * 1024 : used;
    // forward only needs x0 .. bars; it uses the same offsets (the unused front part is simply not touched)
    static constexpr uint32_t fwd_base = x0;
    static constexpr uint32_t fwd_total = used - fwd_base;
};

struct RowCtx {
    int q, s;
    int64_t ray, p;
    bool valid;
    float t0, t1, x[3];
    bool inside;
};

__device__ __forceinline__ RowCtx make_row(const PropArgs& a, int64_t tile, int r, int rpt, int rows_used) {
    RowCtx c;
    c.q = r / a.S;
    c.s = r - c.q * a.S;
    c.ray = tile * rpt + c.q;
    c.valid = r < rows_used && c.ray < a.N;
    c.p = c.ray * a.S + c.s;
    c.t0 = c.t1 = 0.f;
    c.x[0] = c.x[1] = c.x[2] = 0.f;
    c.inside = false;
    if (c.valid) {
        c.t0 = __ldg(a.eu + c.ray * (a.S + 1) + c.s);
        c.t1 = __ldg(a.eu + c.ray * (a.S + 1) + c.s + 1);
        const float o[3] = {__ldg(a.origins + 3 * c.ray), __ldg(a.origins + 3 * c.ray + 1), __ldg(a.origins + 3 * c.ray + 2)};
        const float d[3] = {__ldg(a.dirs + 3 * c.ray), __ldg(a.dirs + 3 * c.ray + 1), __ldg(a.dirs + 3 * c.ray + 2)};
        frustum_midpoint(o, d, c.t0, c.t1, c.x);
        c.inside = normalize_point(c.x, a.box, a.contract != 0);
    }
    return c;
}

template <int H, int K0 = kK0>
__device__ __forceinline__ void load_net_raw(const float* W0, const float* b0, const float* W1, const float* b1, int in_dim,
                                             unsigned char* smem, int tid) {
    using SM = Smem<H, K0>;
    load_weight_cm(W0, H, in_dim, H, K0, smem + SM::w0, nullptr, tid, kThreads);
    float* fl = reinterpret_cast<float*>(smem + SM::fl);
    for (int i = tid; i < H; i += kThreads) {
        fl[i] = b0 ? __ldg(b0 + i) : 0.f;
        fl[H + i] = __bfloat162float(__float2bfloat16_rn(__ldg(W1 + i)));
    }
    if (tid == 0) fl[2 * H] = b1 ? __ldg(b1) : 0.f;
}
template <int H, int K0 = kK0>
__device__ __forceinline__ void load_net(const PropArgs& a, unsigned char* smem, int tid) {
    load_net_raw<H, K0>(a.W0, a.b0, a.W1, a.b1, a.in_dim, smem, tid);
}

// hidden row of this thread: accumulator -> +bias -> ReLU; returns raw = b1 + <h, w1> (fp32 h) and the ReLU mask.
// STORE: also write the bf16 row into the H1 tile (backward).
template <int H, bool STORE>
__device__ __forceinline__ float hidden_row(uint32_t trow, const float* fl, unsigned char* h1_tile, int r,
                                            uint32_t (&mask)[2]) {
    float raw = fl[2 * H];
    mask[0] = mask[1] = 0u;
#pragma unroll
    for (int c = 0; c < H; c += 16) {
        float v[16];
        tmem_ld16_nowait(trow + c, v);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const float x = v[i] + fl[c + i];
            if (x > 0.f) mask[(c + i) >> 5] |= 1u << ((c + i) & 31);
            v[i] = fmaxf(x, 0.f);
            raw = fmaf(v[i], fl[H + c + i], raw);
        }
        if (STORE) {
            store_chunk(h1_tile, kRows, r, c, v);
            store_chunk(h1_tile, kRows, r, c + 8, v + 8);
        }
    }
    return raw;
}

// Hash features of one point for the density-head instantiations (bit-exact encodings.py:343-384, two levels per loop trip as in the K0 = 16
// code): every pair of levels goes straight into row r of the bf16 X0 tile as one 2F-wide store (16 / 8 / 4 bytes for
// F = 4 / 2 / 1), so no K0-entry feature array is held in registers; the padding columns [L*F, K0) are zeroed.
template <int F, int K0>
constexpr bool kRegFeat = K0 == kK0 && F <= 2;     // the proposal levels' instantiations: features in registers

template <int F, int K0>
__device__ __forceinline__ void gather_to_tile(const float* table, const float (&x)[3], const HashParams& hp,
                                               uint32_t mask_t, unsigned char* X0, int r) {
    static_assert(K0 % (2 * F) == 0, "level pairs tile the padded width");
    const int L = hp.L;
#pragma unroll 1
    for (int l0 = 0; l0 < L; l0 += 2) {
        float v[2][8][F];
        Corner8 cr[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int l = min(l0 + j, L - 1);
            cr[j] = hash_corners(x[0], x[1], x[2], hp.scale[l], mask_t);
            const float* lt = table + ((size_t)l << hp.log2_T) * F;
#pragma unroll
            for (int k = 0; k < 8; ++k) gather_row<F>(lt, cr[j].row[k], v[j][k]);
        }
        float pair[2 * F];
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int f = 0; f < F; ++f) {
                const float t[8] = {v[j][0][f], v[j][1][f], v[j][2][f], v[j][3][f],
                                    v[j][4][f], v[j][5][f], v[j][6][f], v[j][7][f]};
                pair[j * F + f] = l0 + j < L ? trilerp_ref(t, cr[j].ox, cr[j].oy, cr[j].oz) : 0.f;
            }
        unsigned char* dst = X0 + cm_off(kRows, r, l0 * F);
        if constexpr (F == 4) {
            *reinterpret_cast<uint4*>(dst) = pack8(pair);
        } else if constexpr (F == 2) {
            *reinterpret_cast<uint2*>(dst) = make_uint2(pack_bf16x2(pair[0], pair[1]), pack_bf16x2(pair[2], pair[3]));
        } else {
            *reinterpret_cast<uint32_t*>(dst) = pack_bf16x2(pair[0], pair[1]);
        }
    }
#pragma unroll 1
    for (int c = (L + 1) / 2 * 2 * F; c < K0; c += 2 * F) {
        unsigned char* dst = X0 + cm_off(kRows, r, c);
        if constexpr (F == 4) {
            *reinterpret_cast<uint4*>(dst) = make_uint4(0u, 0u, 0u, 0u);
        } else if constexpr (F == 2) {
            *reinterpret_cast<uint2*>(dst) = make_uint2(0u, 0u);
        } else {
            *reinterpret_cast<uint32_t*>(dst) = 0u;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
template <int H, int F, int K0 = kK0>
__global__ void __launch_bounds__(kThreads) prop_fwd_kernel(PropArgs a) {
    using SM = Smem<H, K0>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned char* smem = smem_raw - SM::fwd_base;     // forward allocates only [fwd_base, used)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    unsigned char* X0 = smem + SM::x0;
    const float* fl = reinterpret_cast<const float*>(smem + SM::fl);
    double* tails = reinterpret_cast<double*>(smem + SM::tails);
    uint64_t* bar_ptr = reinterpret_cast<uint64_t*>(smem + SM::bars);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM::bars + 16);
    constexpr uint32_t kCols = H < 32 ? 32 : H;

    load_net<H, K0>(a, smem, tid);
    if (warp == 0) tmem_alloc(tmem_slot, kCols);
    if (tid == 0) {
        mbar_init(smem_u32(bar_ptr), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem = *tmem_slot;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);      // provably warp-uniform (MMA issue branch, tc5::elect_one)
    const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
    const uint32_t bar = smem_u32(bar_ptr);
    uint32_t phase = 0;
    const int S = a.S, rpt = kRows / S, rows_used = rpt * S, wpr = S / 32;
    const int64_t ntiles = (a.N + rpt - 1) / rpt;
    const uint32_t mask_t = (1u << a.hp.log2_T) - 1u;
    const int L = a.hp.L;

    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const RowCtx c = make_row(a, tile, tid, rpt, rows_used);
        if constexpr (kRegFeat<F, K0>) {
            // ---- hash gather: bit-exact encodings.py:343-384 -----------------------------------------------------
            // (two levels per loop trip: 16 independent gathers in flight per thread, compact code)
            float feat[kK0];
    #pragma unroll
            for (int i = 0; i < kK0; ++i) feat[i] = 0.f;
    #pragma unroll 1
            for (int l0 = 0; l0 < L; l0 += 2) {
                float v[2][8][F];
                Corner8 cr[2];
    #pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int l = min(l0 + j, L - 1);
                    cr[j] = hash_corners(c.x[0], c.x[1], c.x[2], a.hp.scale[l], mask_t);
                    const float* lt = a.table + ((size_t)l << a.hp.log2_T) * F;
    #pragma unroll
                    for (int k = 0; k < 8; ++k) gather_row<F>(lt, cr[j].row[k], v[j][k]);
                }
    #pragma unroll
                for (int j = 0; j < 2; ++j) {
                    if (l0 + j < L) {
    #pragma unroll
                        for (int f = 0; f < F; ++f) {
                            const float t[8] = {v[j][0][f], v[j][1][f], v[j][2][f], v[j][3][f],
                                                v[j][4][f], v[j][5][f], v[j][6][f], v[j][7][f]};
                            const float val = trilerp_ref(t, cr[j].ox, cr[j].oy, cr[j].oz);
                            // feat[(l0 + j) * F + f] with a compile-time register index
    #pragma unroll
                            for (int i = 0; i < kK0; ++i)
                                if (i == (l0 + j) * F + f) feat[i] = val;
                        }
                    }
                }
            }
            {
                const uint4 lo = pack8(feat), hi = pack8(feat + 8);
                *reinterpret_cast<uint4*>(X0 + cm_off(kRows, tid, 0)) = lo;
                *reinterpret_cast<uint4*>(X0 + cm_off(kRows, tid, 8)) = hi;
                if (a.feat && c.valid) {
                    uint4* dst = reinterpret_cast<uint4*>(a.feat + c.p * a.feat_stride);
                    dst[0] = lo;
                    if (a.feat_stride > 8) dst[1] = hi;
                }
            }
        } else {
            gather_to_tile<F, K0>(a.table, c.x, a.hp, mask_t, X0, tid);
        }
        fence_async_smem();
        fence_before();
        __syncthreads();
        if (warp_u == 0) {
            if (elect_one()) {
                fence_after();
                gemm_kk(tmem, smem_u32(X0), kRows, smem_u32(smem + SM::w0), H, H, K0, false);
                umma_commit(bar);
            }
            __syncwarp();
        }
        mbar_wait(bar, phase);
        phase ^= 1;
        fence_after();
        uint32_t mask[2];
        const float raw = hidden_row<H, false>(trow, fl, nullptr, tid, mask);
        // ---- density and weights (prop_density_field.py:148-152, rays.py:138-148) -------------------------------
        const float density = c.valid ? expf(raw) * (c.inside ? 1.f : 0.f) : 0.f;
        const float dd = __fmul_rn(__fsub_rn(c.t1, c.t0), density);
        const double dd_incl = warp_scan_incl((double)dd, lane);
        if (lane == 31) tails[warp * 2] = dd_incl;
        fence_before();
        __syncthreads();      // also orders this tile's TMEM reads before the next tile's MMA
        const int w_first = (warp / wpr) * wpr;
        double carry = 0.0;
        for (int k = w_first; k < warp; ++k) carry += tails[k * 2];
        const double incl = dd_incl + carry;
        const double prev = __shfl_up_sync(0xffffffffu, incl, 1);
        const double excl = lane == 0 ? carry : prev;
        const float T = expf(-(float)excl);
        const float alpha = __fsub_rn(1.f, expf(-dd));
        const float w = nan_to_num(__fmul_rn(alpha, T));
        if (c.valid) a.weights[c.p] = w;
        __syncthreads();      // tails consumed before the next tile rewrites them
    }
    fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, kCols);
}

// ------------------------------------------------------------------------------------------------------------------
template <int H>
struct BwdTmem {
    static constexpr int acc = 0;            // [128 x H] forward accumulator; columns 0..15 reused for d feat
    static constexpr int dw0 = H < 32 ? 32 : H;   // [H x 16]
    static constexpr int dw1 = dw0 + 16;     // transposed [H (k) x 16 (n, column 0 real)]
    static constexpr int db0 = dw1 + 16;     // [H x 16] (every column = bias gradient)
    static constexpr int end = db0 + 16;
    static constexpr uint32_t alloc = end <= 64 ? 64 : (end <= 128 ? 128 : 256);
};

template <int H, int F>
__global__ void __launch_bounds__(kThreads) prop_bwd_kernel(PropArgs a) {
    using SM = Smem<H>;
    using TM = BwdTmem<H>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    unsigned char* H1 = smem + SM::h1;
    unsigned char* DZ0 = smem + SM::dz0;
    unsigned char* X0 = smem + SM::x0;
    unsigned char* DZ1 = smem + SM::dz1;
    unsigned char* ONES = smem + SM::ones;
    const float* fl = reinterpret_cast<const float*>(smem + SM::fl);
    double* tails = reinterpret_cast<double*>(smem + SM::tails);
    uint64_t* bar_ptr = reinterpret_cast<uint64_t*>(smem + SM::bars);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM::bars + 16);

    load_net<H>(a, smem, tid);
    {
        float one[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) one[i] = 1.f;
        store_chunk(ONES, kRows, tid, 0, one);
        store_chunk(ONES, kRows, tid, 8, one);
    }
    if (warp == 0) tmem_alloc(tmem_slot, TM::alloc);
    if (tid == 0) {
        mbar_init(smem_u32(bar_ptr), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem = *tmem_slot;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);      // provably warp-uniform (MMA issue branch, tc5::elect_one)
    const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
    const uint32_t bar = smem_u32(bar_ptr);
    const uint32_t aH1 = smem_u32(H1), aDZ0 = smem_u32(DZ0), aX0 = smem_u32(X0), aDZ1 = smem_u32(DZ1),
                   aONES = smem_u32(ONES), aW0 = smem_u32(smem + SM::w0);
    uint32_t phase = 0;
    const int S = a.S, rpt = kRows / S, rows_used = rpt * S, wpr = S / 32;
    const int64_t ntiles = (a.N + rpt - 1) / rpt;
    const uint32_t mask_t = (1u << a.hp.log2_T) - 1u;
    const int L = a.hp.L;
    float db1 = 0.f;
    bool first = true;

    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const bool acc_dw = !first;
        first = false;
        const RowCtx c = make_row(a, tile, tid, rpt, rows_used);
        {
            uint4 lo = make_uint4(0, 0, 0, 0), hi = make_uint4(0, 0, 0, 0);
            if (c.valid) {
                const uint4* src = reinterpret_cast<const uint4*>(a.feat + c.p * a.feat_stride);
                lo = __ldg(src);
                if (a.feat_stride > 8) hi = __ldg(src + 1);
            }
            *reinterpret_cast<uint4*>(X0 + cm_off(kRows, tid, 0)) = lo;
            *reinterpret_cast<uint4*>(X0 + cm_off(kRows, tid, 8)) = hi;
        }
        const float gw_in = c.valid ? __ldg(a.d_w + c.p) : 0.f;
        fence_async_smem();
        fence_before();
        __syncthreads();
        if (warp_u == 0) {
            if (elect_one()) {
                fence_after();
                gemm_kk(tmem + TM::acc, aX0, kRows, aW0, H, H, kK0, false);
                umma_commit(bar);
            }
            __syncwarp();
        }
        mbar_wait(bar, phase);
        phase ^= 1;
        fence_after();
        uint32_t mask[2];
        const float raw = hidden_row<H, true>(trow + TM::acc, fl, H1, tid, mask);
        // ---- weights forward ---------------------------------------------------------------------------------
        const float selv = c.inside ? 1.f : 0.f;
        const float density = c.valid ? expf(raw) * selv : 0.f;
        const float dl = __fsub_rn(c.t1, c.t0);
        const float dd = __fmul_rn(dl, density);
        const double dd_incl = warp_scan_incl((double)dd, lane);
        if (lane == 31) tails[warp * 2] = dd_incl;
        __syncthreads();
        const int w_first = (warp / wpr) * wpr;
        float w, T, g;
        {
            double carry = 0.0;
            for (int k = w_first; k < warp; ++k) carry += tails[k * 2];
            const double incl = dd_incl + carry;
            const double prev = __shfl_up_sync(0xffffffffu, incl, 1);
            const double excl = lane == 0 ? carry : prev;
            T = expf(-(float)excl);
            const float alpha = __fsub_rn(1.f, expf(-dd));
            const float rawp = __fmul_rn(alpha, T);
            w = nan_to_num(rawp);
            g = (isfinite(rawp) && c.valid) ? gw_in : 0.f;
        }
        // ---- weights backward (see composite.cu): d sigma_i = delta_i (g_i T_{i+1} - sum_{k>i} g_k w_k) ----------
        const double gw_incl = warp_scan_incl((double)g * (double)w, lane);
        if (lane == 31) tails[warp * 2 + 1] = gw_incl;
        __syncthreads();
        float d_raw;
        {
            double pc = 0.0, G = 0.0;
            for (int k = w_first; k < w_first + wpr; ++k) {
                if (k < warp) pc += tails[k * 2 + 1];
                G += tails[k * 2 + 1];
            }
            const double Pi = gw_incl + pc;
            const float d_sigma = dl * (float)((double)g * (double)(T * expf(-dd)) - (G - Pi));
            d_raw = c.valid ? d_sigma * selv * expf(fminf(fmaxf(raw, -15.f), 15.f)) : 0.f;
        }
        db1 += d_raw;
        // ---- MLP backward: dz1 = d_raw (column 0), dz0 = d_raw * w1 under the ReLU mask -----------------------------
        {
            float z[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) z[i] = 0.f;
            z[0] = d_raw;
            store_chunk(DZ1, kRows, tid, 0, z);
            store_chunk(DZ1, kRows, tid, 8, z + 8);
#pragma unroll
            for (int c0 = 0; c0 < H; c0 += 8) {
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    v[i] = ((mask[(c0 + i) >> 5] >> ((c0 + i) & 31)) & 1u) ? d_raw * fl[H + c0 + i] : 0.f;
                store_chunk(DZ0, kRows, tid, c0, v);
            }
        }
        fence_async_smem();
        fence_before();
        __syncthreads();
        if (warp_u == 0) {
            if (elect_one()) {
                fence_after();
                gemm_dgrad(tmem + TM::acc, aDZ0, kRows, aW0, H, kK0, H, false);     // d feat [128 x 16]
                gemm_wgrad(tmem + TM::dw0, aDZ0, aX0, kK0, acc_dw);                // dW0 [H x 16]
                gemm_wgrad(tmem + TM::dw1, aH1, aDZ1, 16, acc_dw);                 // dW1^T [H x 16], column 0
                gemm_wgrad(tmem + TM::db0, aDZ0, aONES, 16, acc_dw);               // hidden bias gradient = dZ0^T 1
                umma_commit(bar);     // one commit: the tiles these GEMMs read are rewritten by the next tile
            }
            __syncwarp();
        }
        mbar_wait(bar, phase);
        phase ^= 1;
        fence_after();
        float gfeat[kK0];
        tmem_ld16_nowait(trow + TM::acc, gfeat);
        tmem_wait_ld();
        // ---- hash scatter-add ------------------------------------------------------------------------------------
#pragma unroll 1
        for (int l = 0; l < L; ++l) {
            const float scale = a.hp.scale[l];
            const Corner8 cr = hash_corners(c.x[0], c.x[1], c.x[2], scale, mask_t);
            float gl[F];
#pragma unroll
            for (int f = 0; f < F; ++f) {
                gl[f] = 0.f;
#pragma unroll
                for (int i = 0; i < kK0; ++i)
                    if (i == l * F + f) gl[f] = gfeat[i];
            }
            scatter_level_preagg<F>(a.dtable + ((size_t)l << a.hp.log2_T) * F, cr, c.x[0], c.x[1], c.x[2], scale, gl,
                                    c.valid, lane);
        }
        fence_before();       // orders this tile's TMEM reads before the next tile's MMA (issued behind its barrier)
    }
    // ---- flush ---------------------------------------------------------------------------------------------------
    db1 = warp_sum(db1);
    if (lane == 0 && a.db1) atomicAdd(a.db1, db1);
    if (!first) {
        const int n = warp * 32 + lane;          // hidden unit owned by this thread (TMEM lane)
        if (warp * 32 < H) {
            float u[16];
            tmem_ld16_nowait(trow + TM::dw0, u);
            tmem_wait_ld();
            if (n < H)
#pragma unroll
                for (int k = 0; k < 16; ++k)
                    if (k < a.in_dim && u[k] != 0.f) atomicAdd(a.dW0 + (size_t)n * a.in_dim + k, u[k]);
            tmem_ld16_nowait(trow + TM::dw1, u);
            tmem_wait_ld();
            if (n < H) atomicAdd(a.dW1 + n, u[0]);
            tmem_ld16_nowait(trow + TM::db0, u);
            tmem_wait_ld();
            if (n < H && a.db0) atomicAdd(a.db0 + n, u[0]);
        }
    }
    fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, TM::alloc);
}

// kHasBwd<H, F, K0>: a backward kernel exists (K0 = 16, F <= 2); the other instantiations are forward only, and
// referencing prop_bwd_kernel for them would instantiate a backward nobody calls.
template <int F, int K0>
constexpr bool kHasBwd = K0 == kK0 && F <= 2;

template <int H, int F, int K0 = kK0>
static int launch(const PropArgs& a, bool bwd, cudaStream_t stream, const char* what_fwd = "prop_level_fwd") {
    using SM = Smem<H, K0>;
    const void* fwd_kernel = reinterpret_cast<const void*>(prop_fwd_kernel<H, F, K0>);
    const void* kernel = fwd_kernel;
    if constexpr (kHasBwd<F, K0>) {
        if (bwd) kernel = reinterpret_cast<const void*>(prop_bwd_kernel<H, F>);
    } else {
        bwd = false;
    }
    const size_t smem = bwd ? SM::bwd_total : SM::fwd_total;
    static int ctas_fwd = 0, ctas_bwd = 0;
    int& ctas = bwd ? ctas_bwd : ctas_fwd;
    if (ctas == 0) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) {
            set_error("prop_level: cannot reserve %zu bytes of shared memory", smem);
            return 2;
        }
        // resident CTAs per SM.  cudaOccupancyMaxActiveBlocksPerMultiprocessor answers 1 for kernels that allocate tensor
        // memory (it cannot know the column count), so the limit is derived here: registers, shared memory (+1 KB
        // reserved per CTA), tensor-memory columns, and a cap of 8 (the hardware blocks in tcgen05.alloc otherwise).
        cudaFuncAttributes fa{};
        e = cudaFuncGetAttributes(&fa, kernel);
        const int regs = (e == cudaSuccess && fa.numRegs > 0) ? fa.numRegs : 128;
        const int regs_alloc = ((regs + 7) / 8) * 8;
        const int by_regs = 65536 / (regs_alloc * kThreads);
        const int by_smem = (int)((227 * 1024) / (smem + fa.sharedSizeBytes + 1024));
        const int tmem_cols = bwd ? (int)BwdTmem<H>::alloc : (H < 32 ? 32 : H);
        const int by_tmem = 512 / tmem_cols;
        int occ = by_regs < by_smem ? by_regs : by_smem;
        if (occ > 8) occ = 8;
        if (occ < 1) occ = 1;
        ctas = occ < by_tmem ? occ : by_tmem;
        if (getenv("PS_DEBUG"))
            fprintf(stderr, "[prop_level %s H=%d F=%d K0=%d] smem %zu occ %d (%s) by_tmem %d -> %d CTAs/SM\n",
                    bwd ? "bwd" : "fwd", H, F, K0, smem, occ, cudaGetErrorString(e), by_tmem, ctas);
    }
    const int rpt = kRows / a.S;
    const int64_t ntiles = (a.N + rpt - 1) / rpt;
    const int64_t cap = (int64_t)kNumSMs * ctas;
    const int grid = (int)(ntiles < cap ? ntiles : cap);
    if constexpr (kHasBwd<F, K0>) {
        if (bwd) {
            prop_bwd_kernel<H, F><<<grid, kThreads, smem, stream>>>(a);
            return check_launch("prop_level_bwd");
        }
    }
    prop_fwd_kernel<H, F, K0><<<grid, kThreads, smem, stream>>>(a);
    return check_launch(what_fwd);
}

static int dispatch(const PropArgs& a, int H, bool bwd, cudaStream_t s) {
    if (H == 64 && a.F == 1) return launch<64, 1>(a, bwd, s);
    if (H == 64 && a.F == 2) return launch<64, 2>(a, bwd, s);
    if (H == 16 && a.F == 1) return launch<16, 1>(a, bwd, s);
    if (H == 16 && a.F == 2) return launch<16, 2>(a, bwd, s);
    set_error("prop_level: hidden width %d / features per level %d not instantiated", H, a.F);
    return 3;
}


// ------------------------------------------------------------------------------------------------------------------
// Sub-field mode (SURVEY §8 a10; routers: fields/PreSight/prop_density_field_ms.py:86-105).  The level's points arrive
// grouped by sub-field (ms_route.cu): row i of tile t is point perm[i] (-1 = padding) with its unit-cube position already
// normalised by its sub-field's aabb; every 128-row tile belongs to ONE sub-field (tile_sf), whose hash table and MLP the
// tile uses.  CTAs take tiles round-robin and restage the (tiny) network when the sub-field
// changes — in the backward it then also flushes the TMEM-resident weight-gradient accumulators to that sub-field's
// gradient buffers.  Rays are no longer contiguous in a tile, so the kernels stop at the density (forward) and start
// from d loss / d density (backward); weights and their backward run in ps_composite_fwd / ps_composite_bwd.
struct PropNetDev {                      // one per sub-field, array in device memory
    const float *W0, *b0, *W1, *b1;
    float *dW0, *db0, *dW1, *db1;
};

struct PropMsArgs {
    const PropNetDev* nets;
    int in_dim;
    const float* x01s;          // [rows, 3] unit-cube positions in sub-field order
    const uint8_t* sels;        // [rows]
    const int32_t* perm;        // [rows] point index or -1
    const uint8_t* tile_sf;     // [rows / 128], 255 = unused
    int64_t rows;
    const float* const* tables;
    float* const* dtables;
    HashParams hp;
    int F;
    float* density;             // [P] forward output (written at the point's own index)
    __nv_bfloat16* feat;        // [rows, feat_stride] bf16 features in sub-field order (forward output / backward input)
    int feat_stride;
    const float* d_density;     // [P]
};

template <int H, int F, int K0 = kK0>
__global__ void __launch_bounds__(kThreads) prop_fwd_ms_kernel(PropMsArgs a) {
    using SM = Smem<H, K0>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned char* smem = smem_raw - SM::fwd_base;
    const int tid = threadIdx.x, warp = tid >> 5;
    unsigned char* X0 = smem + SM::x0;
    const float* fl = reinterpret_cast<const float*>(smem + SM::fl);
    uint64_t* bar_ptr = reinterpret_cast<uint64_t*>(smem + SM::bars);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM::bars + 16);
    constexpr uint32_t kCols = H < 32 ? 32 : H;
    if (warp == 0) tmem_alloc(tmem_slot, kCols);
    if (tid == 0) {
        mbar_init(smem_u32(bar_ptr), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem = *tmem_slot;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
    const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
    const uint32_t bar = smem_u32(bar_ptr);
    uint32_t phase = 0;
    // Tiles are taken round-robin, so at any moment all CTAs work on neighbouring tiles, i.e. (mostly) on the SAME sub-field:
    // the live hash-table working set is one sub-field's tables, which fit the 126 MB L2, instead of all of them.
    const int64_t ntiles = a.rows / kRows;
    const uint32_t mask_t = (1u << a.hp.log2_T) - 1u;
    const int L = a.hp.L;
    int cur = -1;

    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int sf = a.tile_sf[tile];
        if (sf == 255) break;                                   // the used tiles are a prefix
        if (sf != cur) {
            __syncthreads();                                    // everybody is done with the previous network's constants
            const PropNetDev n = a.nets[sf];
            load_net_raw<H, K0>(n.W0, n.b0, n.W1, n.b1, a.in_dim, smem, tid);
            cur = sf;                                           // (published by the barrier in front of the MMA below)
        }
        const int64_t i = tile * kRows + tid;
        const int32_t p = a.perm[i];
        const bool valid = p >= 0;
        const float x[3] = {valid ? __ldg(a.x01s + 3 * i) : 0.f, valid ? __ldg(a.x01s + 3 * i + 1) : 0.f,
                            valid ? __ldg(a.x01s + 3 * i + 2) : 0.f};
        const bool inside = valid && a.sels[i] != 0;
        const float* table = a.tables[sf];
        if constexpr (kRegFeat<F, K0>) {
            float feat[kK0];
    #pragma unroll
            for (int k = 0; k < kK0; ++k) feat[k] = 0.f;
    #pragma unroll 1
            for (int l0 = 0; l0 < L; l0 += 2) {
                float v[2][8][F];
                Corner8 cr[2];
    #pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int l = min(l0 + j, L - 1);
                    cr[j] = hash_corners(x[0], x[1], x[2], a.hp.scale[l], mask_t);
                    const float* lt = table + ((size_t)l << a.hp.log2_T) * F;
    #pragma unroll
                    for (int k = 0; k < 8; ++k) gather_row<F>(lt, cr[j].row[k], v[j][k]);
                }
    #pragma unroll
                for (int j = 0; j < 2; ++j) {
                    if (l0 + j < L) {
    #pragma unroll
                        for (int f = 0; f < F; ++f) {
                            const float t[8] = {v[j][0][f], v[j][1][f], v[j][2][f], v[j][3][f],
                                                v[j][4][f], v[j][5][f], v[j][6][f], v[j][7][f]};
                            const float val = trilerp_ref(t, cr[j].ox, cr[j].oy, cr[j].oz);
    #pragma unroll
                            for (int k = 0; k < kK0; ++k)
                                if (k == (l0 + j) * F + f) feat[k] = val;
                        }
                    }
                }
            }
            {
                const uint4 lo = pack8(feat), hi = pack8(feat + 8);
                *reinterpret_cast<uint4*>(X0 + cm_off(kRows, tid, 0)) = lo;
                *reinterpret_cast<uint4*>(X0 + cm_off(kRows, tid, 8)) = hi;
                if (a.feat) {
                    uint4* dst = reinterpret_cast<uint4*>(a.feat + i * a.feat_stride);
                    dst[0] = lo;
                    if (a.feat_stride > 8) dst[1] = hi;
                }
            }
        } else {
            gather_to_tile<F, K0>(table, x, a.hp, mask_t, X0, tid);
        }
        fence_async_smem();
        fence_before();
        __syncthreads();
        if (warp_u == 0) {
            if (elect_one()) {
                fence_after();
                gemm_kk(tmem, smem_u32(X0), kRows, smem_u32(smem + SM::w0), H, H, K0, false);
                umma_commit(bar);
            }
            __syncwarp();
        }
        mbar_wait(bar, phase);
        phase ^= 1;
        fence_after();
        uint32_t mask[2];
        const float raw = hidden_row<H, false>(trow, fl, nullptr, tid, mask);
        if (valid) a.density[p] = expf(raw) * (inside ? 1.f : 0.f);          // prop_density_field.py:148-152
        fence_before();
        __syncthreads();      // this tile's TMEM reads before the next tile's MMA; X0 free for restaging
    }
    fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, kCols);
}

template <int H, int F>
__global__ void __launch_bounds__(kThreads) prop_bwd_ms_kernel(PropMsArgs a) {
    using SM = Smem<H>;
    using TM = BwdTmem<H>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    unsigned char* H1 = smem + SM::h1;
    unsigned char* DZ0 = smem + SM::dz0;
    unsigned char* X0 = smem + SM::x0;
    unsigned char* DZ1 = smem + SM::dz1;
    unsigned char* ONES = smem + SM::ones;
    const float* fl = reinterpret_cast<const float*>(smem + SM::fl);
    uint64_t* bar_ptr = reinterpret_cast<uint64_t*>(smem + SM::bars);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM::bars + 16);
    {
        float one[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) one[k] = 1.f;
        store_chunk(ONES, kRows, tid, 0, one);
        store_chunk(ONES, kRows, tid, 8, one);
    }
    if (warp == 0) tmem_alloc(tmem_slot, TM::alloc);
    if (tid == 0) {
        mbar_init(smem_u32(bar_ptr), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem = *tmem_slot;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
    const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
    const uint32_t bar = smem_u32(bar_ptr);
    const uint32_t aH1 = smem_u32(H1), aDZ0 = smem_u32(DZ0), aX0 = smem_u32(X0), aDZ1 = smem_u32(DZ1),
                   aONES = smem_u32(ONES), aW0 = smem_u32(smem + SM::w0);
    uint32_t phase = 0;
    // Tiles are taken round-robin, so at any moment all CTAs work on neighbouring tiles, i.e. (mostly) on the SAME sub-field:
    // the live hash-table working set is one sub-field's tables, which fit the 126 MB L2, instead of all of them.
    const int64_t ntiles = a.rows / kRows;
    const uint32_t mask_t = (1u << a.hp.log2_T) - 1u;
    const int L = a.hp.L;
    float db1 = 0.f;
    bool first = true;
    int cur = -1;

    // weight / bias gradients of the current sub-field: TMEM accumulators + the register sum -> its gradient buffers
    auto flush = [&](int sf) {
        const PropNetDev n = a.nets[sf];
        db1 = warp_sum(db1);
        if (lane == 0 && n.db1) atomicAdd(n.db1, db1);
        db1 = 0.f;
        if (!first) {
            fence_after();
            const int u_row = warp * 32 + lane;
            if (warp * 32 < H) {
                float u[16];
                tmem_ld16_nowait(trow + TM::dw0, u);
                tmem_wait_ld();
                if (u_row < H)
#pragma unroll
                    for (int k = 0; k < 16; ++k)
                        if (k < a.in_dim && u[k] != 0.f) atomicAdd(n.dW0 + (size_t)u_row * a.in_dim + k, u[k]);
                tmem_ld16_nowait(trow + TM::dw1, u);
                tmem_wait_ld();
                if (u_row < H) atomicAdd(n.dW1 + u_row, u[0]);
                tmem_ld16_nowait(trow + TM::db0, u);
                tmem_wait_ld();
                if (u_row < H && n.db0) atomicAdd(n.db0 + u_row, u[0]);
            }
            fence_before();
        }
        first = true;
    };

    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int sf = a.tile_sf[tile];
        if (sf == 255) break;
        if (sf != cur) {
            if (cur >= 0) flush(cur);
            __syncthreads();
            const PropNetDev n = a.nets[sf];
            load_net_raw<H>(n.W0, n.b0, n.W1, n.b1, a.in_dim, smem, tid);
            cur = sf;
        }
        const bool acc_dw = !first;
        first = false;
        const int64_t i = tile * kRows + tid;
        const int32_t p = a.perm[i];
        const bool valid = p >= 0;
        const float x[3] = {valid ? __ldg(a.x01s + 3 * i) : 0.f, valid ? __ldg(a.x01s + 3 * i + 1) : 0.f,
                            valid ? __ldg(a.x01s + 3 * i + 2) : 0.f};
        const float selv = (valid && a.sels[i] != 0) ? 1.f : 0.f;
        {
            uint4 lo = make_uint4(0, 0, 0, 0), hi = make_uint4(0, 0, 0, 0);
            if (valid) {
                const uint4* src = reinterpret_cast<const uint4*>(a.feat + i * a.feat_stride);
                lo = __ldg(src);
                if (a.feat_stride > 8) hi = __ldg(src + 1);
            }
            *reinterpret_cast<uint4*>(X0 + cm_off(kRows, tid, 0)) = lo;
            *reinterpret_cast<uint4*>(X0 + cm_off(kRows, tid, 8)) = hi;
        }
        const float g_den = valid ? __ldg(a.d_density + p) : 0.f;
        fence_async_smem();
        fence_before();
        __syncthreads();
        if (warp_u == 0) {
            if (elect_one()) {
                fence_after();
                gemm_kk(tmem + TM::acc, aX0, kRows, aW0, H, H, kK0, false);
                umma_commit(bar);
            }
            __syncwarp();
        }
        mbar_wait(bar, phase);
        phase ^= 1;
        fence_after();
        uint32_t mask[2];
        const float raw = hidden_row<H, true>(trow + TM::acc, fl, H1, tid, mask);
        // density = exp(raw) * sel, gradient through the clamped exponential (activations.py:28-41)
        const float d_raw = valid ? g_den * selv * expf(fminf(fmaxf(raw, -15.f), 15.f)) : 0.f;
        db1 += d_raw;
        {
            float z[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) z[k] = 0.f;
            z[0] = d_raw;
            store_chunk(DZ1, kRows, tid, 0, z);
            store_chunk(DZ1, kRows, tid, 8, z + 8);
#pragma unroll
            for (int c0 = 0; c0 < H; c0 += 8) {
                float v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    v[k] = ((mask[(c0 + k) >> 5] >> ((c0 + k) & 31)) & 1u) ? d_raw * fl[H + c0 + k] : 0.f;
                store_chunk(DZ0, kRows, tid, c0, v);
            }
        }
        fence_async_smem();
        fence_before();
        __syncthreads();
        if (warp_u == 0) {
            if (elect_one()) {
                fence_after();
                gemm_dgrad(tmem + TM::acc, aDZ0, kRows, aW0, H, kK0, H, false);
                gemm_wgrad(tmem + TM::dw0, aDZ0, aX0, kK0, acc_dw);
                gemm_wgrad(tmem + TM::dw1, aH1, aDZ1, 16, acc_dw);
                gemm_wgrad(tmem + TM::db0, aDZ0, aONES, 16, acc_dw);
                umma_commit(bar);
            }
            __syncwarp();
        }
        mbar_wait(bar, phase);
        phase ^= 1;
        fence_after();
        float gfeat[kK0];
        tmem_ld16_nowait(trow + TM::acc, gfeat);
        tmem_wait_ld();
        float* dtable = a.dtables[sf];
#pragma unroll 1
        for (int l = 0; l < L; ++l) {
            const float scale = a.hp.scale[l];
            const Corner8 cr = hash_corners(x[0], x[1], x[2], scale, mask_t);
            float gl[F];
#pragma unroll
            for (int f = 0; f < F; ++f) {
                gl[f] = 0.f;
#pragma unroll
                for (int k = 0; k < kK0; ++k)
                    if (k == l * F + f) gl[f] = gfeat[k];
            }
            scatter_level_preagg<F>(dtable + ((size_t)l << a.hp.log2_T) * F, cr, x[0], x[1], x[2], scale, gl, valid, lane);
        }
        fence_before();
    }
    if (cur >= 0) flush(cur);
    fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, TM::alloc);
}

template <int H, int F, int K0 = kK0>
static int launch_ms(const PropMsArgs& a, bool bwd, cudaStream_t stream, const char* what_fwd = "prop_level_fwd_ms") {
    using SM = Smem<H, K0>;
    const void* kernel = reinterpret_cast<const void*>(prop_fwd_ms_kernel<H, F, K0>);
    if constexpr (kHasBwd<F, K0>) {
        if (bwd) kernel = reinterpret_cast<const void*>(prop_bwd_ms_kernel<H, F>);
    } else {
        bwd = false;
    }
    const size_t smem = bwd ? SM::bwd_total : SM::fwd_total;
    static bool conf_f = false, conf_b = false;
    bool& conf = bwd ? conf_b : conf_f;
    if (!conf) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) {
            set_error("prop_level_ms: cannot reserve %zu bytes of shared memory", smem);
            return 2;
        }
        conf = true;
    }
    const int ctas = bwd ? 4 : 8;                      // resident CTAs per SM (TMEM columns / shared memory, see launch())
    const int64_t ntiles = a.rows / kRows;
    const int64_t cap = (int64_t)kNumSMs * ctas;
    const int grid = (int)(ntiles < cap ? ntiles : cap);
    if constexpr (kHasBwd<F, K0>) {
        if (bwd) {
            prop_bwd_ms_kernel<H, F><<<grid, kThreads, smem, stream>>>(a);
            return check_launch("prop_level_bwd_ms");
        }
    }
    prop_fwd_ms_kernel<H, F, K0><<<grid, kThreads, smem, stream>>>(a);
    return check_launch(what_fwd);
}

// Density head of the main field (ps_density_level_fwd*): hidden width 64, F in {1, 2, 4}, K0 = L*F rounded up to 16.
template <int F>
static int dispatch_density_f(const PropArgs* a, const PropMsArgs* m, int in_dim, cudaStream_t s) {
    const int k0 = (in_dim + 15) / 16 * 16;
    if (k0 == 16) return a ? launch<64, F, 16>(*a, false, s, "density_level_fwd") : launch_ms<64, F, 16>(*m, false, s, "density_level_fwd_ms");
    if (k0 == 32) return a ? launch<64, F, 32>(*a, false, s, "density_level_fwd") : launch_ms<64, F, 32>(*m, false, s, "density_level_fwd_ms");
    return a ? launch<64, F, 48>(*a, false, s, "density_level_fwd") : launch_ms<64, F, 48>(*m, false, s, "density_level_fwd_ms");
}
static int dispatch_density(const PropArgs* a, const PropMsArgs* m, int F, int in_dim, cudaStream_t s) {
    if (F == 1) return dispatch_density_f<1>(a, m, in_dim, s);
    if (F == 2) return dispatch_density_f<2>(a, m, in_dim, s);
    return dispatch_density_f<4>(a, m, in_dim, s);
}

static int dispatch_ms(const PropMsArgs& a, int H, bool bwd, cudaStream_t s) {
    if (H == 64 && a.F == 1) return launch_ms<64, 1>(a, bwd, s);
    if (H == 64 && a.F == 2) return launch_ms<64, 2>(a, bwd, s);
    if (H == 16 && a.F == 1) return launch_ms<16, 1>(a, bwd, s);
    if (H == 16 && a.F == 2) return launch_ms<16, 2>(a, bwd, s);
    set_error("prop_level_ms: hidden width %d / features per level %d not instantiated", H, a.F);
    return 3;
}

// density = true: the main field's density head (ps_density_level_fwd*): hidden 64, F in {1, 2, 4}, L*F <= 48
static int check_shape(int hidden, int L, int F, bool density, const char* what) {
    if (density) {
        PS_REQUIRE(hidden == 64, "%s: hidden width %d is not 64", what, hidden);
        PS_REQUIRE(F == 1 || F == 2 || F == 4, "%s: features_per_level %d not in {1,2,4}", what, F);
        PS_REQUIRE(L >= 1 && L * F <= 48 && L <= PS_MAX_LEVELS, "%s: L*F = %d exceeds %d", what, L * F, 48);
        return 0;
    }
    PS_REQUIRE(hidden == 16 || hidden == 64, "%s: hidden width %d not in {16, 64}", what, hidden);
    PS_REQUIRE(F == 1 || F == 2, "%s: features_per_level %d not in {1,2}", what, F);
    PS_REQUIRE(L >= 1 && L * F <= kK0 && L <= PS_MAX_LEVELS, "%s: L*F = %d exceeds %d", what, L * F, kK0);
    return 0;
}

static int fill(PropArgs& a, const ps_prop_net* net, const float* origins, const float* dirs, const float* eu_bins, int64_t N,
                int S, const float* aabb_host, int contract, const float* scalings_host, int L, int F, int log2_T,
                const char* what, bool density = false) {
    PS_REQUIRE(net && net->W0 && net->W1, "%s: network is null", what);
    if (int e = check_shape(net->hidden, L, F, density, what)) return e;
    PS_REQUIRE(log2_T >= 1 && log2_T <= 31, "%s: log2_hashmap_size %d out of range", what, log2_T);
    PS_REQUIRE(S >= 32 && S <= 128 && S % 32 == 0, "%s: samples per ray %d must be 32, 64, 96 or 128", what, S);
    PS_REQUIRE(N > 0 && N * (int64_t)S < (1ll << 31), "%s: too many points", what);
    PS_REQUIRE(origins && dirs && eu_bins && aabb_host && scalings_host, "%s: null pointer", what);
    a.W0 = net->W0; a.b0 = net->b0; a.W1 = net->W1; a.b1 = net->b1;
    a.dW0 = net->dW0; a.db0 = net->db0; a.dW1 = net->dW1; a.db1 = net->db1;
    a.in_dim = L * F;
    a.origins = origins; a.dirs = dirs; a.eu = eu_bins; a.N = N; a.S = S;
    for (int k = 0; k < 3; ++k) { a.box.lo[k] = aabb_host[k]; a.box.hi[k] = aabb_host[3 + k]; }
    a.contract = contract;
    for (int l = 0; l < L; ++l) a.hp.scale[l] = scalings_host[l];
    a.hp.L = L; a.hp.log2_T = log2_T;
    a.F = F;
    a.feat_stride = L * F <= 8 ? 8 : 16;
    return 0;
}

}  // namespace ptc5
}  // namespace ps

using namespace ps;
using namespace ps::ptc5;

extern "C" int ps_prop_level_feat_stride(int L, int F) { return L * F <= 8 ? 8 : 16; }

extern "C" int ps_prop_level_fwd(const ps_prop_net* net, const float* origins, const float* dirs, const float* eu_bins,
                                 int64_t N, int S, const float* aabb_host, int contract, const float* table,
                                 const float* scalings_host, int L, int F, int log2_T, float* weights, void* feat_bf16,
                                 void* stream) {
    if (N == 0) return 0;
    PropArgs a{};
    if (int e = fill(a, net, origins, dirs, eu_bins, N, S, aabb_host, contract, scalings_host, L, F, log2_T, "prop_level_fwd"))
        return e;
    PS_REQUIRE(table && weights, "prop_level_fwd: null pointer");
    a.table = table; a.weights = weights; a.feat = reinterpret_cast<__nv_bfloat16*>(feat_bf16);
    return dispatch(a, net->hidden, false, (cudaStream_t)stream);
}

extern "C" int ps_prop_level_bwd(const ps_prop_net* net, const float* origins, const float* dirs, const float* eu_bins,
                                 int64_t N, int S, const float* aabb_host, int contract, const float* scalings_host, int L,
                                 int F, int log2_T, const void* feat_bf16, const float* d_weights, float* dtable,
                                 void* stream) {
    if (N == 0) return 0;
    PropArgs a{};
    if (int e = fill(a, net, origins, dirs, eu_bins, N, S, aabb_host, contract, scalings_host, L, F, log2_T, "prop_level_bwd"))
        return e;
    PS_REQUIRE(feat_bf16 && d_weights && dtable && net->dW0 && net->dW1, "prop_level_bwd: null pointer");
    a.dtable = dtable; a.d_w = d_weights;
    a.feat = reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(feat_bf16));
    return dispatch(a, net->hidden, true, (cudaStream_t)stream);
}

static_assert(sizeof(ps_prop_net_dev) == sizeof(ps::ptc5::PropNetDev), "ps_prop_net_dev layout");

static int fill_ms(PropMsArgs& a, const ps_prop_net_dev* nets, int hidden, const float* x01s, const uint8_t* sels,
                   const int32_t* perm, const uint8_t* tile_sf, int64_t rows, const float* scalings_host, int L, int F,
                   int log2_T, const char* what, bool density = false) {
    PS_REQUIRE(nets != nullptr, "%s: nets is null", what);
    if (int e = check_shape(hidden, L, F, density, what)) return e;
    PS_REQUIRE(log2_T >= 1 && log2_T <= 31, "%s: log2_hashmap_size %d out of range", what, log2_T);
    PS_REQUIRE(rows > 0 && rows % kRows == 0 && rows < (1ll << 31), "%s: rows must be a positive multiple of 128", what);
    PS_REQUIRE(x01s && sels && perm && tile_sf && scalings_host, "%s: null pointer", what);
    a.nets = reinterpret_cast<const PropNetDev*>(nets);
    a.in_dim = L * F;
    a.x01s = x01s; a.sels = sels; a.perm = perm; a.tile_sf = tile_sf; a.rows = rows;
    for (int l = 0; l < L; ++l) a.hp.scale[l] = scalings_host[l];
    a.hp.L = L; a.hp.log2_T = log2_T;
    a.F = F;
    a.feat_stride = L * F <= 8 ? 8 : 16;
    return 0;
}

extern "C" int ps_prop_level_fwd_ms(const ps_prop_net_dev* nets_dev, int hidden, const float* x01_sorted,
                                    const uint8_t* sel_sorted, const int32_t* perm, const uint8_t* tile_sf, int64_t rows,
                                    const float* const* tables_dev, const float* scalings_host, int L, int F, int log2_T,
                                    float* density, void* feat_bf16, void* stream) {
    PropMsArgs a{};
    if (int e = fill_ms(a, nets_dev, hidden, x01_sorted, sel_sorted, perm, tile_sf, rows, scalings_host, L, F, log2_T,
                        "prop_level_fwd_ms"))
        return e;
    PS_REQUIRE(tables_dev && density, "prop_level_fwd_ms: null pointer");
    a.tables = tables_dev; a.density = density; a.feat = reinterpret_cast<__nv_bfloat16*>(feat_bf16);
    return dispatch_ms(a, hidden, false, (cudaStream_t)stream);
}

extern "C" int ps_prop_level_bwd_ms(const ps_prop_net_dev* nets_dev, int hidden, const float* x01_sorted,
                                    const uint8_t* sel_sorted, const int32_t* perm, const uint8_t* tile_sf, int64_t rows,
                                    float* const* dtables_dev, const float* scalings_host, int L, int F, int log2_T,
                                    const void* feat_bf16, const float* d_density, void* stream) {
    PropMsArgs a{};
    if (int e = fill_ms(a, nets_dev, hidden, x01_sorted, sel_sorted, perm, tile_sf, rows, scalings_host, L, F, log2_T,
                        "prop_level_bwd_ms"))
        return e;
    PS_REQUIRE(dtables_dev && feat_bf16 && d_density, "prop_level_bwd_ms: null pointer");
    a.dtables = dtables_dev; a.d_density = d_density;
    a.feat = reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(feat_bf16));
    return dispatch_ms(a, hidden, true, (cudaStream_t)stream);
}

// ---- density head of the main field (forward only) -----------------------------------------------------------------
extern "C" int ps_density_level_fwd(const ps_prop_net* net, const float* origins, const float* dirs, const float* eu_bins,
                                    int64_t N, int S, const float* aabb_host, int contract, const float* table,
                                    const float* scalings_host, int L, int F, int log2_T, float* weights, void* stream) {
    if (N == 0) return 0;
    PropArgs a{};
    if (int e = fill(a, net, origins, dirs, eu_bins, N, S, aabb_host, contract, scalings_host, L, F, log2_T,
                     "density_level_fwd", true))
        return e;
    PS_REQUIRE(table && weights, "density_level_fwd: null pointer");
    a.table = table; a.weights = weights;
    return dispatch_density(&a, nullptr, F, a.in_dim, (cudaStream_t)stream);
}

extern "C" int ps_density_level_fwd_ms(const ps_prop_net_dev* nets_dev, int hidden, const float* x01_sorted,
                                       const uint8_t* sel_sorted, const int32_t* perm, const uint8_t* tile_sf, int64_t rows,
                                       const float* const* tables_dev, const float* scalings_host, int L, int F, int log2_T,
                                       float* density, void* stream) {
    PropMsArgs a{};
    if (int e = fill_ms(a, nets_dev, hidden, x01_sorted, sel_sorted, perm, tile_sf, rows, scalings_host, L, F, log2_T,
                        "density_level_fwd_ms", true))
        return e;
    PS_REQUIRE(tables_dev && density, "density_level_fwd_ms: null pointer");
    a.tables = tables_dev; a.density = density;
    return dispatch_density(nullptr, &a, F, a.in_dim, (cudaStream_t)stream);
}
