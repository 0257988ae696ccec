// Shape registry of the fused MLP kernels.  Each group is compiled in its own translation unit
// (mlp_group{0,1,2}.cu) so nvcc can build them in parallel.
#pragma once
#include "mlp_kernels.cuh"

namespace ps {
namespace mma {

// (K0, H, NHID, NOUT), padded sizes.  Reference networks covered:
//   proposal nets    8|10 -> 16|64 -> 1, or a single Linear            (prop_density_field.py:85-98)
//   base MLP         12|32|40 -> 64 -> 16|80                          (ingp_field.py:130-138)
//   semantic head    64 -> 64 -> 64 -> 64                             (ingp_field.py:142-151)
//   colour head      31|47|63 -> 64 -> 64 -> 3                        (ingp_field.py:153-161)
//   sky heads        32 -> 32 -> 32 -> 3, 16 -> 32 -> 32 -> 64        (sky_field.py:75-93)
#define PS_MLP_GROUP0(X) X(16, 16, 0, 16) X(16, 16, 1, 16) X(16, 64, 1, 16) X(16, 64, 1, 80) X(32, 64, 1, 16)
#define PS_MLP_GROUP1(X) X(32, 64, 1, 80) X(48, 64, 1, 16) X(48, 64, 1, 80) X(64, 64, 2, 64) X(32, 32, 2, 16)
#define PS_MLP_GROUP2(X) X(32, 64, 2, 16) X(48, 64, 2, 16) X(64, 64, 2, 16) X(16, 32, 2, 64) X(64, 64, 1, 64)

// returns -1 when the shape is not in this group
int dispatch_group0(int K0, int H, int NHID, int NOUT, int prec, bool bwd, const MlpArgs& a, cudaStream_t s);
int dispatch_group1(int K0, int H, int NHID, int NOUT, int prec, bool bwd, const MlpArgs& a, cudaStream_t s);
int dispatch_group2(int K0, int H, int NHID, int NOUT, int prec, bool bwd, const MlpArgs& a, cudaStream_t s);

#define PS_MLP_CASE(k0, h, nhid, nout)                                                       \
    if (K0 == k0 && H == h && NHID == nhid && NOUT == nout) {                                \
        using S = Shape<k0, h, nhid, nout>;                                                  \
        if (prec == kBF16) return bwd ? launch_bwd<S, kBF16>(a, s) : launch_fwd<S, kBF16>(a, s); \
        return bwd ? launch_bwd<S, kTF32x3>(a, s) : launch_fwd<S, kTF32x3>(a, s);            \
    }

}  // namespace mma
}  // namespace ps
