// zuko_b200 — device helpers shared by the fully fused layer kernels
// (fused_layer.cu: hidden width <= 256, one CTA per tile; fused_wide.cu / fused_dual.cu: CTA pairs on
// cta_group::2 MMAs) and the host-side preparation they have in common (fused_layer.cu, fused_plan.cu).
#pragma once

#include <type_traits>
#include <utility>
#include <vector>

#include "bijector_math.cuh"
#include "fused_layer.cuh"
#include "tc_common.cuh"

namespace zk {

// D[tmem] (+)= A[tmem] * B[smem]^T
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}

// compile-time loop: f(integral_constant<int, Start>), ..., f(integral_constant<int, Start + N - 1>)
template <int Start, class F, int... I>
__device__ __forceinline__ void for_range_impl(F& f, std::integer_sequence<int, I...>) {
    (f(std::integral_constant<int, Start + I>{}), ...);
}
template <int Start, int N, class F>
__device__ __forceinline__ void for_range(F& f) {
    for_range_impl<Start>(f, std::make_integer_sequence<int, N>{});
}

// per-(UNI, K) chunking of the last layer: DPC dims per accumulator chunk
template <int UNI, int KT>
struct LastCfg;
template <>
struct LastCfg<ZK_UNI_RQS, 8> { static constexpr int P = 23, DPC = 4; };
template <>
struct LastCfg<ZK_UNI_RQS, 16> { static constexpr int P = 47, DPC = 2; };
template <>
struct LastCfg<ZK_UNI_AFFINE, 0> { static constexpr int P = 2, DPC = 64; };

inline int fused_dpc(int univariate, int bins) { return (univariate == ZK_UNI_RQS) ? (bins == 8 ? 4 : 2) : 64; }
inline int fused_p(int univariate, int bins) { return (univariate == ZK_UNI_RQS) ? 3 * bins - 1 : 2; }

// Host-side state both preparations start from: the masks (host copies; dense layers = all ones)
// and, per hidden layer, the permutation that sorts its units by dependency degree
// (perm[l][new] = old index).  fused_host_prepare also (re)builds f.w / f.bias: the bf16 hi / lo
// planes [2][N][Kp] and biases with rows (hidden layers) and columns (the layer after) permuted.
struct FusedHostPrep {
    std::vector<std::vector<uint8_t>> Mk;
    std::vector<std::vector<int>> perm;
};
void fused_degree_perm(const int* dims, int L, const std::vector<std::vector<uint8_t>>& Mk,
                       std::vector<std::vector<int>>& perm);
zk_status fused_host_prepare(zk_mlp* m, const uint8_t* const* mask_dev, FusedPack& f, FusedHostPrep& hp);

// Which (chunk, K block) tiles of the degree-permuted masked matrices hold a non-zero weight.  Hidden
// layers are cut into chunks of `cw` rows (64 or 128), the output layer into ceil(D / DPC) chunks of
// DPC dims (DPC * P rows).
struct FusedTileMap {
    std::vector<std::vector<uint32_t>> kbmask;  // [layer][chunk]: bit kb = K block kb is read (at least bit 0)
    std::vector<std::vector<int>> kmax;         // [layer][chunk * 8 + kb]: last column of the block any row of the chunk reads
};
FusedTileMap fused_tile_map(const int* dims, int L, const std::vector<std::vector<uint8_t>>& Mk,
                            const std::vector<std::vector<int>>& perm, int cw, int univariate, int bins, int D);
// Builds the pack `wp` of a pair kernel with S sub-tiles per CTA (pk->wide: S = 1, pk->dual: S = 2):
// tensor maps, issue schedule and its bookkeeping.  wp.ready stays false when the dry run rejects the
// schedule.  The shape is the caller's to check.
zk_status fused_pair_prepare(zk_mlp* m, const uint8_t* const* mask_dev, int univariate, int bins, int D, int C,
                             WidePack& wp, int S);

}  // namespace zk
