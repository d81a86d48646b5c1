// zuko_b200 — tcgen05 / TMA / TMEM PTX wrappers and the packed-weight structures shared by the
// per-layer GEMM kernel (mlp_tcgen05.cu) and the fused layer kernel (fused_layer.cu).
#pragma once

#include <cuda.h>  // CUtensorMap types only; the encoder is fetched through the runtime
#include <cuda_bf16.h>

#include <vector>

#include "mlp.cuh"

namespace zk {

// ---------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                            int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

// multicast variant: the box lands at the same CTA-relative offset in every CTA of `mask`, and each
// destination CTA's mbarrier (same offset) receives the complete_tx
__device__ __forceinline__ void tma_load_3d_mc(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                               int c0, int c1, int c2, uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
        " [%0], [%1, {%3, %4, %5}], [%2], %6;"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "h"(mask)
        : "memory");
}
// commit that arrives on the mbarrier at the same offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
// one leader lane of a converged warp (PTX elect.sync); lets the single-thread tcgen05 / TMA issue
// sit inside warp-uniform control flow so that its operands stay in uniform registers
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
        "elect.sync rx|px, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, px;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
// descriptor of the k-th 16-element K step inside a 64-wide swizzled K block: +32 bytes = +2 units
__device__ __forceinline__ uint64_t umma_desc_advance(uint64_t desc, int k) { return desc + (uint64_t)(2 * k); }

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor, K-major, SWIZZLE_128B (cute::UMMA::SmemDescriptor):
//   [0,14) start address >> 4 | [16,30) LBO >> 4 (unused for swizzled K-major, 1) |
//   [32,46) SBO >> 4 = 1024 B between 8-row groups | [46,48) version = 1 | [61,64) layout = 2
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// tcgen05 instruction descriptor (cute::UMMA::InstrDescriptor), kind::f16:
//   [4,6) D format 1 = f32 | [7,10) A format 1 = bf16 | [10,13) B format 1 = bf16 |
//   bit 15 / 16: A / B major 0 = K | [17,23) N >> 3 | [24,29) M >> 4
__device__ __forceinline__ uint32_t umma_idesc_bf16(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}


struct TcLayer {
    int N = 0, K = 0, Kp = 0;
    __nv_bfloat16* w = nullptr;  // [2][N][Kp] (owned)
    CUtensorMap mapW;     // box (64 x 256 x 1): per-layer GEMM kernel
    CUtensorMap mapW128;  // box (64 x 128 x 1)
    CUtensorMap mapW64;   // box (64 x 64 x 1): fused layer kernel, one half per CTA of a pair (multicast)
};
// weights as the fused layer kernel streams them: hidden units sorted by dependency degree (so
// that the masked matrices are block lower-triangular) and the all-zero (chunk, K block) tiles
// of every layer recorded so that their TMA loads and MMAs are skipped
struct FusedPack {
    bool ready = false;
    int uni = 0, bins = 0, D = 0, C = 0;
    std::vector<__nv_bfloat16*> w;  // per layer [2][N][Kp], permuted (owned)
    std::vector<float*> bias;       // per layer, permuted, padded (owned)
    std::vector<int*> dperm;        // per hidden layer: device copy of the degree permutation (owned; weight refresh)
    std::vector<CUtensorMap> map64; // box (64 x 64 x 1)
    uint8_t kbmask[8][128];         // [layer][chunk]: bit kb = K block kb has non-zero weights
    uint32_t* sched = nullptr;      // device: MMA issue schedule of one tile, one entry per non-zero tile (owned)
    int n_items = 0;
    double issued_macs_per_row = 0;  // MACs the schedule issues per sample row (all split terms), bench bookkeeping
};
// the pack of a CTA-pair fused kernel (fused_wide.cu, fused_dual.cu): it shares FusedPack's permuted
// planes / biases (fused.w, fused.bias) and adds its own tensor maps and issue schedule
struct WidePack {
    bool ready = false;
    int uni = 0, bins = 0, D = 0, C = 0;
    std::vector<CUtensorMap> maps;  // per layer: box (64 x 64 x 1) hidden, (64 x N_LAST/2 x 1) output layer
    uint2* sched = nullptr;         // device: one entry per non-zero (layer, chunk, K block) tile (owned)
    int n_items = 0;
    uint8_t rd_mask[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // per layer: K blocks of the A operand the layer reads
    double issued_macs_per_row = 0;  // MACs the schedule issues per sample row (all split terms)
    // holds a schedule (one that passed its dry run) for this bijector
    bool built_for(int univariate, int bins_, int D_, int C_) const {
        return ready && uni == univariate && bins == bins_ && D == D_ && C == C_;
    }
};
struct TcPack {
    std::vector<TcLayer> layers;
    std::vector<TcLayer> bwd;  // transposed weights (dgrad): N = in features, K = out features; built on first backward
    int n_terms = 3;
    int max_np = 0;  // widest padded hidden activation
    FusedPack fused;
    WidePack wide;
    WidePack dual;  // fused_dual.cu (hidden width 128 / 256, two sub-tiles in flight): same pack layout
};

inline int pad64(int v) { return (v + 63) / 64 * 64; }


// tensor map over bf16 planes [2][rows][Kp]; box = (64 x box_rows x 1), 128B swizzle
zk_status make_plane_map(CUtensorMap* map, const void* base, int64_t rows, int Kp, int box_rows);

// bf16 hi / lo split of two fp32 values, packed as (low 16 bits = first, high 16 = second).
// hi = rn_bf16(v) (one cvt.rn.bf16x2.f32 for the pair), lo = rn_bf16(v - hi): 6 instructions / pair.
__device__ __forceinline__ uint32_t pack_bf16x2_rn(float lo_half, float hi_half) {
    uint32_t d;  // cvt.rn.bf16x2.f32 d, a, b : a -> upper 16 bits, b -> lower 16 bits
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi_half), "f"(lo_half));
    return d;
}
__device__ __forceinline__ void split2_bf16(float v0, float v1, uint32_t& hi, uint32_t& lo) {
    hi = pack_bf16x2_rn(v0, v1);  // registers only (taking the address of a __nv_bfloat162 went through local memory)
    const float h0 = __uint_as_float(hi << 16), h1 = __uint_as_float(hi & 0xffff0000u);
    lo = pack_bf16x2_rn(v0 - h0, v1 - h1);
}

}  // namespace zk
