// C-ABI of kernel #2 (fused MLP): argument validation and shape dispatch.
#include "mlp_dispatch.cuh"

using namespace ps;
using namespace ps::mma;

static int pad16(int v) { return (v + 15) / 16 * 16; }

static int resolve(const int* dims, int n_layers, int& K0, int& H, int& NHID, int& NOUT) {
    PS_REQUIRE(dims != nullptr, "mlp: dims_host is null");
    PS_REQUIRE(n_layers >= 1 && n_layers <= 4, "mlp: %d layers unsupported (1..4)", n_layers);
    for (int i = 0; i <= n_layers; ++i) PS_REQUIRE(dims[i] >= 1, "mlp: dims[%d] = %d", i, dims[i]);
    K0 = pad16(dims[0]);
    NOUT = pad16(dims[n_layers]);
    NHID = n_layers - 1;
    H = NHID > 0 ? dims[1] : 16;
    for (int i = 1; i < n_layers; ++i)
        PS_REQUIRE(dims[i] == H, "mlp: hidden widths must be equal (got %d and %d)", H, dims[i]);
    PS_REQUIRE(H % 16 == 0, "mlp: hidden width %d must be a multiple of 16", H);
    return 0;
}

static int run(int K0, int H, int NHID, int NOUT, int prec, bool bwd, const MlpArgs& a, cudaStream_t s,
               const int* dims, int n_layers) {
    PS_REQUIRE(prec >= 0 && prec <= 1, "mlp: precision %d (0 = tf32x3 fp32-grade, 1 = bf16 mma.sync)", prec);
    int r = dispatch_group0(K0, H, NHID, NOUT, prec, bwd, a, s);
    if (r < 0) r = dispatch_group1(K0, H, NHID, NOUT, prec, bwd, a, s);
    if (r < 0) r = dispatch_group2(K0, H, NHID, NOUT, prec, bwd, a, s);
    if (r < 0) {
        set_error("mlp: no kernel instantiated for %d -> %d x%d -> %d (padded %d/%d/%d); add it to mlp_dispatch.cuh",
                  dims[0], H, NHID, dims[n_layers], K0, H, NOUT);
        return 3;
    }
    return r;
}

static int fill_segments(MlpArgs& a, const ps_row_segment* segs, int n_seg, int in_dim, bool bwd, int64_t P) {
    PS_REQUIRE(P >= 0 && P < (1ll << 31), "mlp: number of points %lld out of range", (long long)P);
    PS_REQUIRE(segs != nullptr && n_seg >= 1 && n_seg <= PS_MLP_MAX_SEGMENTS, "mlp: %d input segments (1..%d)", n_seg,
               PS_MLP_MAX_SEGMENTS);
    int col = 0;
    a.nseg = n_seg;
    a.any_group_dst = 0;
    a.want_dx = 0;
    for (int s = 0; s < n_seg; ++s) {
        PS_REQUIRE(segs[s].src != nullptr, "mlp: segment %d has no source", s);
        PS_REQUIRE(segs[s].width >= 1 && segs[s].group >= 1, "mlp: segment %d width/group invalid", s);
        PS_REQUIRE(segs[s].group == 1 || segs[s].group % 16 == 0,
                   "mlp: segment %d group %d must be 1 or a multiple of 16 (a warp's 16 rows share one group)", s,
                   segs[s].group);
        a.seg[s].src = segs[s].src;
        a.seg[s].dst = bwd ? segs[s].dst : nullptr;
        a.seg[s].stride = segs[s].stride;
        a.seg[s].col0 = segs[s].col0;
        a.seg[s].begin = col;
        a.seg[s].end = col + segs[s].width;
        a.seg[s].group = segs[s].group;
        col += segs[s].width;
        if (a.seg[s].dst) {
            a.want_dx = 1;
            if (segs[s].group > 1) a.any_group_dst = 1;
        }
    }
    PS_REQUIRE(col == in_dim, "mlp: segments cover %d columns but the first layer expects %d", col, in_dim);
    a.lm_F = 0;
    if (segs[0].feat_per_level > 0) {
        const int F = segs[0].feat_per_level;
        PS_REQUIRE(n_seg == 1 && segs[0].group == 1 && segs[0].col0 == 0, "mlp: level-major features need one plain segment");
        PS_REQUIRE((F == 1 || F == 2 || F == 4 || F == 8) && in_dim % F == 0, "mlp: feat_per_level %d invalid for %d columns",
                   F, in_dim);
        PS_REQUIRE((reinterpret_cast<uintptr_t>(segs[0].src) & 7u) == 0 && (reinterpret_cast<uintptr_t>(a.seg[0].dst) & 7u) == 0,
                   "mlp: level-major features must be 8-byte aligned");
        a.lm_F = F;
    }
    auto aligned8 = [](const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 7u) == 0; };
    a.vec2_x = n_seg == 1 && segs[0].group == 1 && in_dim % 2 == 0 && segs[0].stride % 2 == 0 && segs[0].col0 % 2 == 0 &&
               aligned8(segs[0].src) && aligned8(a.seg[0].dst);
    return 0;
}

extern "C" int ps_mlp_fwd_ex(const ps_row_segment* segs_host, int n_seg, int64_t P, const float* const* W_host,
                             const float* const* b_host, const int* dims_host, int n_layers, int out_act,
                             int precision, float* y, const uint8_t* sel, float* density_out, void* stream) {
    int K0, H, NHID, NOUT;
    if (int e = resolve(dims_host, n_layers, K0, H, NHID, NOUT)) return e;
    MlpArgs a{};
    if (P == 0) return 0;   // empty batches are a no-op (their tensors have null data pointers)
    if (int e = fill_segments(a, segs_host, n_seg, dims_host[0], false, P)) return e;
    PS_REQUIRE((y || density_out) && W_host && b_host, "mlp_fwd: null pointer");
    a.y = y; a.P = P; a.in_dim = dims_host[0]; a.out_dim = dims_host[n_layers]; a.out_act = out_act;
    a.sel = sel; a.density_out = density_out;
    a.vec2_y = a.out_dim % 2 == 0 && (reinterpret_cast<uintptr_t>(y) & 7u) == 0;
    for (int i = 0; i < n_layers; ++i) {
        PS_REQUIRE(W_host[i] != nullptr, "mlp_fwd: weight %d is null", i);
        a.W[i] = W_host[i];
        a.b[i] = b_host[i];
    }
    return run(K0, H, NHID, NOUT, precision, false, a, (cudaStream_t)stream, dims_host, n_layers);
}

extern "C" int ps_mlp_bwd_ex(const ps_row_segment* segs_host, int n_seg, const float* dy, int64_t P,
                             const float* const* W_host, const float* const* b_host, const int* dims_host,
                             int n_layers, int out_act, int precision, float* const* dW_host, float* const* db_host,
                             const uint8_t* sel, const float* d_density, void* stream) {
    int K0, H, NHID, NOUT;
    if (int e = resolve(dims_host, n_layers, K0, H, NHID, NOUT)) return e;
    MlpArgs a{};
    if (P == 0) return 0;
    if (int e = fill_segments(a, segs_host, n_seg, dims_host[0], true, P)) return e;
    PS_REQUIRE((dy || d_density) && W_host && b_host && dW_host && db_host, "mlp_bwd: null pointer");
    a.dy = dy; a.P = P; a.in_dim = dims_host[0]; a.out_dim = dims_host[n_layers]; a.out_act = out_act;
    a.sel = sel; a.d_density = d_density;
    a.vec2_y = a.out_dim % 2 == 0 && (reinterpret_cast<uintptr_t>(dy) & 7u) == 0;
    for (int i = 0; i < n_layers; ++i) {
        PS_REQUIRE(W_host[i] != nullptr && dW_host[i] != nullptr, "mlp_bwd: weight/grad %d is null", i);
        a.W[i] = W_host[i];
        a.b[i] = b_host[i];
        a.dW[i] = dW_host[i];
        a.db[i] = db_host[i];
    }
    return run(K0, H, NHID, NOUT, precision, true, a, (cudaStream_t)stream, dims_host, n_layers);
}

extern "C" int ps_mlp_fwd(const float* x, int64_t P, const float* const* W_host, const float* const* b_host,
                          const int* dims_host, int n_layers, int out_act, int precision, float* y, void* stream) {
    PS_REQUIRE(dims_host != nullptr, "mlp: dims_host is null");
    PS_REQUIRE(P == 0 || x != nullptr, "mlp_fwd: x is null");
    static const float dummy = 0.f;
    ps_row_segment seg{x ? x : &dummy, nullptr, dims_host[0], 0, dims_host[0], 1};
    return ps_mlp_fwd_ex(&seg, 1, P, W_host, b_host, dims_host, n_layers, out_act, precision, y, nullptr, nullptr,
                         stream);
}

extern "C" int ps_mlp_bwd(const float* x, const float* y, const float* dy, int64_t P, const float* const* W_host,
                          const float* const* b_host, const int* dims_host, int n_layers, int out_act, int precision,
                          float* dx, float* const* dW_host, float* const* db_host, void* stream) {
    (void)y;  // the forward is recomputed on chip
    PS_REQUIRE(dims_host != nullptr, "mlp: dims_host is null");
    PS_REQUIRE(P == 0 || x != nullptr, "mlp_bwd: x is null");
    static const float dummy = 0.f;
    ps_row_segment seg{x ? x : &dummy, dx, dims_host[0], 0, dims_host[0], 1};
    return ps_mlp_bwd_ex(&seg, 1, dy, P, W_host, b_host, dims_host, n_layers, out_act, precision, dW_host, db_host,
                         nullptr, nullptr, stream);
}
