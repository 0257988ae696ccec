// LPIPS (AlexNet, v0.1) of rendered images against the photographs, as nerfacto's
// LearnedPerceptualImagePatchSimilarity(normalize=True) defines it (torchmetrics functional/image/lpips.py, lpips 0.1
// pretrained_networks.alexnet and normalize_tensor).  Per call, B pairs run as 2B images (pred 0..B-1, then gt 0..B-1):
//   1. conv1:  implicit-GEMM convolution straight from the [H,W,3] image; 2x - 1 and the scaling layer are applied as
//              the operands are gathered, so the zero padding is that of the scaled image, as F.conv2d pads it
//   2. pool -> conv2, pool -> conv3, conv4, conv5: max-pool 3x3/2 (floor) kernels and the same implicit-GEMM kernel
//              on NHWC fp32 activations; every conv applies bias + ReLU in its epilogue
//   3. head:   per layer and pixel, fp32 channel norms of both images, the lin-weighted squared difference of the
//              normalised vectors; each CTA writes one fp64 partial sum per (pair, layer)
//   4. final:  one CTA per pair sums each layer's partials in a fixed order -> the five means and their sum
// No floating-point atomics, and an image's arithmetic does not depend on its slot or on B: repeated calls are
// bit-identical, lpips(x, x) == 0, lpips(a, b) == lpips(b, a) and a batch equals its pairs one at a time, bit for bit.
//
// Convolution: M = output pixels of one image, N = C_out, K = kh * kw * C_in in (ky, kx, ci) order (the packed weight
// layout, [C_out][K_pad] with K_pad a multiple of 32, TF32-rounded (RNA) and zero-padded by presight_b200.metrics).
// CTA tile 128 x 64 x 32, 8 warps of 32 x 32, mma.sync m16n8k8 TF32 with fp32 accumulation, activations rounded with
// cvt.rna as they are read; a 3-stage cp.async pipeline (conv1 gathers its 3-channel taps through registers instead).
// Grid: (M tiles, N tiles, images), every image of the call in one launch.
// ptxas (sm_100a, CUDA 12.9): conv2-5 98 registers, conv1 88 registers + 1 KB static shared memory, 0 spills, all with
// 82 944 B dynamic shared memory (2 CTAs per SM); pool 38 / head 48 / final 32 registers, no spills, no stack frame.
#include <algorithm>
#include <climits>
#include <cmath>

#include "common.cuh"
#include "mlp_mma.cuh"

namespace ps {
namespace {

using mma::mma_tf32;
using mma::to_tf32;

constexpr int kLayers = 5;
constexpr int kThreads = 256;
constexpr int kBM = 128, kBN = 64, kBK = 32, kStages = 3;
constexpr int kLd = kBK + 4;                       // smem row stride (floats): fragment loads are bank-conflict free
constexpr int kStageFloats = (kBM + kBN) * kLd;
constexpr size_t kConvSmem = sizeof(float) * kStages * kStageFloats;
constexpr int kMaxHeadBlocks = 256;
constexpr int kMinSide = 31;                       // 30 leaves nothing after the second pool

constexpr int kCout[kLayers] = {64, 192, 384, 256, 256};

__constant__ float c_shift[3] = {-0.030f, -0.088f, -0.188f};
__constant__ float c_scale[3] = {0.458f, 0.448f, 0.450f};

struct Dims {
    int h[kLayers], w[kLayers];                    // output size of conv k (= the head's layer k)
    int ph[2], pw[2];                              // after pool 1 and pool 2
};

Dims dims_of(int H, int W) {
    Dims d;
    d.h[0] = (H + 4 - 11) / 4 + 1, d.w[0] = (W + 4 - 11) / 4 + 1;
    d.ph[0] = (d.h[0] - 3) / 2 + 1, d.pw[0] = (d.w[0] - 3) / 2 + 1;
    d.h[1] = d.ph[0], d.w[1] = d.pw[0];
    d.ph[1] = (d.h[1] - 3) / 2 + 1, d.pw[1] = (d.w[1] - 3) / 2 + 1;
    for (int k = 2; k < kLayers; ++k) d.h[k] = d.ph[1], d.w[k] = d.pw[1];
    return d;
}

size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

int head_blocks(int64_t pixels) { return (int)std::min<int64_t>(kMaxHeadBlocks, cdiv(pixels, 64)); }

struct Workspace {
    float* act[kLayers];                           // [2B][h_k * w_k][C_out k]
    float* pool[2];                                // [2B][ph * pw][C]
    double* part;                                  // [B][5][kMaxHeadBlocks]
    size_t bytes;
};

Workspace carve(void* ws, int B, const Dims& d) {
    char* p = (char*)ws;
    size_t off = 0;
    Workspace w;
    for (int k = 0; k < kLayers; ++k) {
        w.act[k] = (float*)(p + off);
        off += align256(sizeof(float) * 2 * (size_t)B * d.h[k] * d.w[k] * kCout[k]);
        if (k < 2) {
            w.pool[k] = (float*)(p + off);
            off += align256(sizeof(float) * 2 * (size_t)B * d.ph[k] * d.pw[k] * kCout[k]);
        }
    }
    w.part = (double*)(p + off);
    off += sizeof(double) * (size_t)B * kLayers * kMaxHeadBlocks;
    w.bytes = off;
    return w;
}

__device__ __forceinline__ void cp_async16(float* smem, const float* gmem, bool valid) {
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(valid ? 16 : 0) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// out[img][Ho*Wo][COUT] = ReLU(conv(in[img]) + bias).  FIRST: `in` is the pred images and `in2` the gt images
// ([H,W,3], values in [0,1]), image z < B reads in + z * H * W * 3, else in2 + (z - B) * H * W * 3.
template <int KS, int STRIDE, int PAD, int CIN, int COUT, bool FIRST>
__global__ void __launch_bounds__(kThreads, 2)
    lpips_conv_kernel(const float* __restrict__ in, const float* __restrict__ in2, int B, int H, int W, int Ho, int Wo,
                      const float* __restrict__ wgt, const float* __restrict__ bias, float* __restrict__ out) {
    constexpr int K = KS * KS * CIN;
    constexpr int KPAD = (K + kBK - 1) / kBK * kBK;
    constexpr int KT = KPAD / kBK;
    static_assert(FIRST || CIN % kBK == 0, "a K tile must lie inside one filter tap");
    static_assert(COUT % kBN == 0, "C_out must be a multiple of the N tile");
    extern __shared__ __align__(16) float smem[];
    __shared__ int2 rowbase[kBM];                  // FIRST: top-left input tap of each tile row, or (INT_MIN, 0)

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp & 3, wn = warp >> 2;
    const int m0 = blockIdx.x * kBM, n0 = blockIdx.y * kBN, z = blockIdx.z;
    const int M = Ho * Wo;
    const float* img = FIRST ? (z < B ? in + (int64_t)z * H * W * 3 : in2 + (int64_t)(z - B) * H * W * 3)
                             : in + (int64_t)z * H * W * CIN;

    // non-first layers: each thread gathers 16-byte segments of 4 fixed tile rows (row = tid / 8 + 32 j)
    int iy0[4], ix0[4];
    if constexpr (FIRST) {
        for (int r = tid; r < kBM; r += kThreads) {
            const int m = m0 + r;
            const int oy = m / Wo, ox = m - oy * Wo;
            rowbase[r] = m < M ? make_int2(oy * STRIDE - PAD, ox * STRIDE - PAD) : make_int2(INT_MIN, 0);
        }
        __syncthreads();
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int m = m0 + (tid >> 3) + 32 * j;
            const int oy = m / Wo, ox = m - oy * Wo;
            iy0[j] = m < M ? oy * STRIDE - PAD : INT_MIN / 2;
            ix0[j] = ox * STRIDE - PAD;
        }
    }

    auto load_stage = [&](int kt, int s) {
        float* As = smem + s * kStageFloats;
        float* Bs = As + kBM * kLd;
        const int k0 = kt * kBK;
        if constexpr (FIRST) {
            // one k column per lane, 16 rows per thread: k -> (ky, kx, c) once per stage
            const int k = k0 + lane;
            const int ky = k / (KS * 3), rem = k - ky * (KS * 3), kx = rem / 3, c = rem - kx * 3;
            const float sh = c_shift[c], sc = c_scale[c];
#pragma unroll 4
            for (int j = 0; j < kBM / 8; ++j) {
                const int r = warp + 8 * j;
                const int2 rb = rowbase[r];
                const int iy = rb.x + ky, ix = rb.y + kx;
                float v = 0.f;
                if (k < K && iy >= 0 && iy < H && ix >= 0 && ix < W)
                    v = (fmaf(2.f, __ldg(img + ((int64_t)iy * W + ix) * 3 + c), -1.f) - sh) / sc;
                As[r * kLd + lane] = v;
            }
        } else {
            const int tap = k0 / CIN, c0 = k0 - tap * CIN;
            const int ky = tap / KS, kx = tap - ky * KS;
            const int seg = tid & 7;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int r = (tid >> 3) + 32 * j;
                const int iy = iy0[j] + ky, ix = ix0[j] + kx;
                const bool ok = iy >= 0 && iy < H && ix >= 0 && ix < W;
                const float* src = ok ? img + ((int64_t)iy * W + ix) * CIN + c0 + 4 * seg : img;
                cp_async16(As + r * kLd + 4 * seg, src, ok);
            }
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int q = tid + kThreads * j, r = q >> 3, seg = q & 7;
            cp_async16(Bs + r * kLd + 4 * seg, wgt + (int64_t)(n0 + r) * KPAD + k0 + 4 * seg, true);
        }
    };

    float acc[2][4][4];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = acc[i][j][2] = acc[i][j][3] = 0.f;

#pragma unroll
    for (int s = 0; s < kStages - 1; ++s) {
        if (s < KT) load_stage(s, s);
        cp_async_commit();
    }
    for (int kt = 0; kt < KT; ++kt) {
        cp_async_wait<kStages - 2>();
        __syncthreads();                           // stage kt landed everywhere; stage kt - 1 is free again
        if (kt + kStages - 1 < KT) load_stage(kt + kStages - 1, (kt + kStages - 1) % kStages);
        cp_async_commit();
        const float* As = smem + (kt % kStages) * kStageFloats + (32 * wm) * kLd;
        const float* Bs = smem + (kt % kStages) * kStageFloats + kBM * kLd + (32 * wn) * kLd;
#pragma unroll
        for (int ks = 0; ks < kBK / 8; ++ks) {
            uint32_t a[2][4], b[4][2];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const float* p = As + (16 * i + g) * kLd + 8 * ks + t;
                a[i][0] = to_tf32(p[0]);
                a[i][1] = to_tf32(p[8 * kLd]);
                a[i][2] = to_tf32(p[4]);
                a[i][3] = to_tf32(p[8 * kLd + 4]);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {             // weights are TF32-rounded when packed
                const float* p = Bs + (8 * j + g) * kLd + 8 * ks + t;
                b[j][0] = __float_as_uint(p[0]);
                b[j][1] = __float_as_uint(p[4]);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) mma_tf32(acc[i][j], a[i], b[j][0], b[j][1]);
        }
    }
    cp_async_wait<0>();

    float* o = out + (int64_t)z * M * COUT;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int col = n0 + 32 * wn + 8 * j + 2 * t;
        const float b0 = __ldg(bias + col), b1 = __ldg(bias + col + 1);
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int m = m0 + 32 * wm + 16 * i + g + 8 * h;
                if (m < M)
                    *reinterpret_cast<float2*>(o + (int64_t)m * COUT + col) =
                        make_float2(fmaxf(acc[i][j][2 * h] + b0, 0.f), fmaxf(acc[i][j][2 * h + 1] + b1, 0.f));
            }
    }
}

// max-pool 3x3, stride 2, floor mode (every window lies inside the input): [imgs][H][W][C] -> [imgs][Ho][Wo][C]
__global__ void __launch_bounds__(kThreads) lpips_pool_kernel(const float4* __restrict__ in, int H, int W, int C4,
                                                              int Ho, int Wo, float4* __restrict__ out, int64_t n) {
    for (int64_t e = (int64_t)blockIdx.x * kThreads + threadIdx.x; e < n; e += (int64_t)gridDim.x * kThreads) {
        const int c = (int)(e % C4);
        const int64_t p = e / C4;
        const int ox = (int)(p % Wo), oy = (int)(p / Wo % Ho);
        const int64_t img = p / ((int64_t)Wo * Ho);
        const float4* src = in + ((img * H + 2 * oy) * W + 2 * ox) * C4 + c;
        float4 m = __ldg(src);
#pragma unroll
        for (int dy = 0; dy < 3; ++dy)
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) {
                const float4 v = __ldg(src + ((int64_t)dy * W + dx) * C4);
                m.x = fmaxf(m.x, v.x), m.y = fmaxf(m.y, v.y), m.z = fmaxf(m.z, v.z), m.w = fmaxf(m.w, v.w);
            }
        out[e] = m;
    }
}

struct HeadArgs {
    const float* act[kLayers];
    const float* lin[kLayers];
    int pixels[kLayers];
    int blocks[kLayers];
};

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

// One warp per pixel; lane l holds channels l + 32 j.
template <int C>
__device__ __forceinline__ float head_pixel(const float* __restrict__ f0, const float* __restrict__ f1,
                                            const float* __restrict__ lin, int lane) {
    constexpr int J = C / 32;
    float a[J], b[J];
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int j = 0; j < J; ++j) {
        a[j] = __ldg(f0 + lane + 32 * j), b[j] = __ldg(f1 + lane + 32 * j);
        s0 = fmaf(a[j], a[j], s0), s1 = fmaf(b[j], b[j], s1);
    }
    const float n0 = sqrtf(warp_sum(s0)) + 1e-10f, n1 = sqrtf(warp_sum(s1)) + 1e-10f;
    float d = 0.f;
#pragma unroll
    for (int j = 0; j < J; ++j) {
        const float e = a[j] / n0 - b[j] / n1;     // (x - y)^2 == (y - x)^2: symmetric bit for bit
        d = fmaf(__ldg(lin + lane + 32 * j), e * e, d);
    }
    return warp_sum(d);
}

// this CTA's share of layer K (constant, so the kernel argument arrays are indexed statically)
template <int K>
__device__ __forceinline__ void head_layer(const HeadArgs& h, int B, int pair, double* __restrict__ part) {
    constexpr int C = kCout[K];
    const int P = h.pixels[K], nb = h.blocks[K];
    if ((int)blockIdx.x >= nb) return;
    const float* f0 = h.act[K] + (int64_t)pair * P * C;
    const float* f1 = h.act[K] + (int64_t)(pair + B) * P * C;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double acc = 0.0;
    for (int p = blockIdx.x * (kThreads / 32) + warp; p < P; p += nb * (kThreads / 32))
        acc += (double)head_pixel<C>(f0 + (int64_t)p * C, f1 + (int64_t)p * C, h.lin[K], lane);
    __shared__ double red[kThreads / 32];
    const double s = block_sum(lane == 0 ? acc : 0.0, red);
    if (threadIdx.x == 0) part[((int64_t)pair * kLayers + K) * kMaxHeadBlocks + blockIdx.x] = s;
}

// grid (kMaxHeadBlocks, layer, pair); CTAs beyond a layer's block count return at once
__global__ void __launch_bounds__(kThreads) lpips_head_kernel(HeadArgs h, int B, double* __restrict__ part) {
    const int pair = blockIdx.z;
    switch (blockIdx.y) {
        case 0: head_layer<0>(h, B, pair, part); break;
        case 1: head_layer<1>(h, B, pair, part); break;
        case 2: head_layer<2>(h, B, pair, part); break;
        case 3: head_layer<3>(h, B, pair, part); break;
        default: head_layer<4>(h, B, pair, part); break;
    }
}

__global__ void __launch_bounds__(kThreads) lpips_final_kernel(const double* __restrict__ part, HeadArgs h,
                                                               double* __restrict__ per_layer,
                                                               double* __restrict__ out) {
    __shared__ double red[kThreads / 32];
    const int pair = blockIdx.x;
    double total = 0.0;
#pragma unroll
    for (int k = 0; k < kLayers; ++k) {
        const double* p = part + ((int64_t)pair * kLayers + k) * kMaxHeadBlocks;
        const double v = threadIdx.x < h.blocks[k] ? p[threadIdx.x] : 0.0;
        const double s = block_sum(v, red);
        if (threadIdx.x == 0) {
            const double mean = s / (double)h.pixels[k];
            if (per_layer) per_layer[(int64_t)pair * kLayers + k] = mean;
            total += mean;
        }
    }
    if (threadIdx.x == 0) out[pair] = total;
}
static_assert(kMaxHeadBlocks <= kThreads, "the final reduction reads one partial per thread");

template <int KS, int STRIDE, int PAD, int CIN, int COUT, bool FIRST>
int launch_conv(const float* in, const float* in2, int B, int H, int W, int Ho, int Wo, const float* wgt,
                const float* bias, float* out, cudaStream_t st, const char* what) {
    auto kern = lpips_conv_kernel<KS, STRIDE, PAD, CIN, COUT, FIRST>;
    const cudaError_t attr = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kConvSmem);
    if (attr != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(attr));
        return 2;
    }
    const dim3 grid((unsigned)cdiv((int64_t)Ho * Wo, kBM), COUT / kBN, 2 * B);
    kern<<<grid, kThreads, kConvSmem, st>>>(in, in2, B, H, W, Ho, Wo, wgt, bias, out);
    return check_launch(what);
}

int launch_pool(const float* in, int imgs, int H, int W, int C, int Ho, int Wo, float* out, cudaStream_t st,
                const char* what) {
    const int64_t n = (int64_t)imgs * Ho * Wo * (C / 4);
    const int blocks = (int)std::min<int64_t>(cdiv(n, kThreads), 16 * kNumSMs);
    lpips_pool_kernel<<<blocks, kThreads, 0, st>>>((const float4*)in, H, W, C / 4, Ho, Wo, (float4*)out, n);
    return check_launch(what);
}

// the sizes the call checks: every per-image index (input and largest activation) fits an int
bool sizes_ok(int H, int W) {
    if (H < kMinSide || W < kMinSide) return false;
    const Dims d = dims_of(H, W);
    return (int64_t)H * W * 3 <= INT32_MAX && (int64_t)d.h[0] * d.w[0] * kCout[0] <= INT32_MAX &&
           (int64_t)d.h[1] * d.w[1] * kCout[1] <= INT32_MAX;
}

}  // namespace
}  // namespace ps

extern "C" int ps_lpips_workspace(int B, int H, int W, int64_t* bytes) {
    PS_REQUIRE(bytes, "lpips_workspace: null pointer");
    PS_REQUIRE(B >= 1 && B <= 32767, "lpips_workspace: B must be in [1, 32767], got %d", B);
    PS_REQUIRE(H >= ps::kMinSide && W >= ps::kMinSide, "lpips_workspace: images need at least 31 x 31 pixels, got %d x %d",
               H, W);
    PS_REQUIRE(ps::sizes_ok(H, W), "lpips_workspace: %d x %d images overflow the kernels' 32-bit indices", H, W);
    *bytes = (int64_t)ps::carve(nullptr, B, ps::dims_of(H, W)).bytes;
    return 0;
}

extern "C" int ps_lpips(const float* pred, const float* gt, int B, int H, int W, const ps_lpips_net* net,
                        void* workspace, double* per_layer, double* out, void* stream) {
    PS_REQUIRE(B >= 1 && B <= 32767, "lpips: B must be in [1, 32767], got %d", B);
    PS_REQUIRE(H >= ps::kMinSide && W >= ps::kMinSide, "lpips: images need at least 31 x 31 pixels, got %d x %d", H, W);
    PS_REQUIRE(ps::sizes_ok(H, W), "lpips: %d x %d images overflow the kernels' 32-bit indices", H, W);
    PS_REQUIRE(pred && gt && net && workspace && out, "lpips: null pointer (pred, gt, net, workspace or out)");
    for (int k = 0; k < ps::kLayers; ++k)
        PS_REQUIRE(net->conv_w[k] && net->conv_b[k] && net->lin[k], "lpips: null weight pointer in layer %d", k);
    cudaStream_t st = (cudaStream_t)stream;
    const ps::Dims d = ps::dims_of(H, W);
    const ps::Workspace ws = ps::carve(workspace, B, d);
    const int imgs = 2 * B;
    int rc;
    if ((rc = ps::launch_conv<11, 4, 2, 3, 64, true>(pred, gt, B, H, W, d.h[0], d.w[0], net->conv_w[0], net->conv_b[0],
                                                     ws.act[0], st, "lpips conv1")))
        return rc;
    if ((rc = ps::launch_pool(ws.act[0], imgs, d.h[0], d.w[0], 64, d.ph[0], d.pw[0], ws.pool[0], st, "lpips pool1")))
        return rc;
    if ((rc = ps::launch_conv<5, 1, 2, 64, 192, false>(ws.pool[0], nullptr, B, d.ph[0], d.pw[0], d.h[1], d.w[1],
                                                       net->conv_w[1], net->conv_b[1], ws.act[1], st, "lpips conv2")))
        return rc;
    if ((rc = ps::launch_pool(ws.act[1], imgs, d.h[1], d.w[1], 192, d.ph[1], d.pw[1], ws.pool[1], st, "lpips pool2")))
        return rc;
    if ((rc = ps::launch_conv<3, 1, 1, 192, 384, false>(ws.pool[1], nullptr, B, d.ph[1], d.pw[1], d.h[2], d.w[2],
                                                        net->conv_w[2], net->conv_b[2], ws.act[2], st, "lpips conv3")))
        return rc;
    if ((rc = ps::launch_conv<3, 1, 1, 384, 256, false>(ws.act[2], nullptr, B, d.h[2], d.w[2], d.h[3], d.w[3],
                                                        net->conv_w[3], net->conv_b[3], ws.act[3], st, "lpips conv4")))
        return rc;
    if ((rc = ps::launch_conv<3, 1, 1, 256, 256, false>(ws.act[3], nullptr, B, d.h[3], d.w[3], d.h[4], d.w[4],
                                                        net->conv_w[4], net->conv_b[4], ws.act[4], st, "lpips conv5")))
        return rc;
    ps::HeadArgs h;
    for (int k = 0; k < ps::kLayers; ++k) {
        h.act[k] = ws.act[k];
        h.lin[k] = net->lin[k];
        h.pixels[k] = d.h[k] * d.w[k];
        h.blocks[k] = ps::head_blocks(h.pixels[k]);
    }
    ps::lpips_head_kernel<<<dim3(ps::kMaxHeadBlocks, ps::kLayers, B), ps::kThreads, 0, st>>>(h, B, ws.part);
    if ((rc = ps::check_launch("lpips head"))) return rc;
    ps::lpips_final_kernel<<<B, ps::kThreads, 0, st>>>(ws.part, h, per_layer, out);
    return ps::check_launch("lpips final");
}
