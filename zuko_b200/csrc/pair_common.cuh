// zuko_b200 — what the CTA-pair fused kernels (fused_wide.cu, fused_dual.cu) share: the layout of their
// schedule entries, the cta_group::2 forms of the tcgen05 / TMA / mbarrier instructions, the bounded
// waits with their watchdog report, the store of an A-operand lo plane fragment into its swizzled
// shared-memory layout, and the host code that fills their launch parameters.  The schedule itself is
// built and dry-run in fused_plan.cu.
#pragma once

#include <string.h>

#include "fused_common.cuh"

namespace zk {

constexpr uint32_t W_APLANE = 128 * 64 * 2;       // 16 KB: one K block (128 rows x 64 bf16) of the A lo plane
constexpr long long W_WD_CYCLES = 4000000000ll;   // watchdog: ~2 s of SM clock

// schedule entry (uint2) of a kernel with S sub-tiles per CTA (fused_wide.cu: 1, fused_dual.cu: 2):
// x = flags, y = first weight row of the chunk
//   x [2:0] A block u * (8 / S) + kb of sub-tile u (S = 2: bit 2 is the sub-tile, kb < 4) |
//     [3] first K block of its chunk | [4] last K block of its chunk |
//     [5] first read of the A block in this layer (wait a_ready) | [6] last read of the A block in this
//     layer (commit a_free) | [7] output layer | [15:8] a_ready phases (by A block) the layer consumes
//     without reading (on the sub-tile's first entry of the layer) | [18:16] layer |
//     [21:20] trailing 16-column MMA steps of the K block that are all-zero for this chunk (not issued)
constexpr uint32_t WS_FIRST = 8u, WS_LAST = 16u, WS_AWAIT = 32u, WS_AFREE = 64u, WS_OUT = 128u;

// ---------------------------------------------------------------------------
// PTX: the cta_group::2 forms
// ---------------------------------------------------------------------------
__device__ __forceinline__ void umma2_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma2_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives (once all MMAs issued so far are complete) on the mbarrier at this offset in both CTAs
__device__ __forceinline__ void umma2_commit_mc(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_dst, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// TMA load of this CTA's half of a pair's operand tile; the bytes are counted on the barrier at
// `bar_addr` (a shared::cluster address: the LEADER's barrier, cute::Sm100MmaPeerBitMask)
__device__ __forceinline__ void tma_load_3d_2sm(void* smem_dst, const CUtensorMap* map, uint32_t bar_addr,
                                                int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(bar_addr), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ uint32_t mapa_rank0(uint32_t addr) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(r) : "r"(addr));
    return r;
}
// Arrive on a barrier of the LEADER CTA.  Default semantics (.release.cta), as CUTLASS's
// ClusterBarrier::arrive(cta_id): what the arrival publishes lives in THIS CTA's tensor / shared
// memory and was completed before it (tcgen05.wait, fence.proxy.async); `.release.cluster` compiles to
// MEMBAR.ALL.GPU in front of every arrive (~2000 cycles each: profiles/r02_wide_timeline_*_v1.txt).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return done != 0;
}

// ---------------------------------------------------------------------------
// watchdog: a wait that does not end within ~2 s reports (role, what it waits for, where it is in
// the schedule) into mapped host memory and traps — a protocol bug then costs one GPU run and
// names the barrier, instead of hanging the device until the job is killed.
// ---------------------------------------------------------------------------
static __device__ __noinline__ void wd_report(uint32_t* watch, uint32_t code, uint32_t a, uint32_t b) {
    if (watch != nullptr && blockIdx.x < 2) {
        // slot per (CTA of cluster 0, warp): 8 words
        uint32_t* s = watch + 8 + ((blockIdx.x & 1) * 32 + (threadIdx.x >> 5)) * 8;
        s[0] = 0xDEAD0000u | code; s[1] = a; s[2] = b; s[3] = threadIdx.x;
        atomicAdd(watch, 1u);
        __threadfence_system();
    }
    const long long t0 = clock64();
    while (clock64() - t0 < 400000000ll) {}  // let the other roles report too
    __trap();
}
#define WD_SPIN(cond, code, a, b)                                                   \
    do {                                                                            \
        uint32_t _n = 0;                                                            \
        long long _t0 = 0;                                                          \
        while (!(cond)) {                                                           \
            if ((++_n & 1023u) == 0u) {                                             \
                const long long _t = clock64();                                     \
                if (_t0 == 0) _t0 = _t;                                             \
                else if (_t - _t0 > W_WD_CYCLES) wd_report(p.watch, (code), (a), (b)); \
            }                                                                       \
        }                                                                           \
    } while (0)

#define W_STAMP(slot)                                                                         \
    do {                                                                                      \
        if constexpr (DBG) {                                                                  \
            if (p.dbg != nullptr && blockIdx.x == 0 && stamp_on) p.dbg[(slot)] = clock64();   \
        }                                                                                     \
    } while (0)

// lo plane of 32 consecutive K elements of row r -> shared memory, K-major, 128-byte swizzle
// (the layout a TMA SWIZZLE_128B box of 64 bf16 x 128 rows has: 16-byte unit j of row r sits at
// unit j ^ (r & 7) of the row's 128 bytes; 8-row groups are 1024 bytes apart)
__device__ __forceinline__ void st_alo32(uint8_t* sAlo, int kb, int r, int half, const uint32_t* pl) {
    uint8_t* row = sAlo + (size_t)kb * W_APLANE + (size_t)(r >> 3) * 1024 + (size_t)(r & 7) * 128;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int j = half * 4 + u;
        *reinterpret_cast<uint4*>(row + (((j ^ (r & 7)) & 7) << 4)) = make_uint4(pl[4 * u], pl[4 * u + 1], pl[4 * u + 2], pl[4 * u + 3]);
    }
}

// ---------------------------------------------------------------------------
// host: launch parameters both kernels fill alike (WideParams and DualParams share these field names)
// ---------------------------------------------------------------------------
uint32_t* pair_watch_device();  // the watchdog buffer (allocated on first use) as the device sees it, or null

// Zeroes `p`, then fills in the layer's arguments, its shapes and the schedule and tensor maps of `wp`.
template <class Params>
void pair_fill_params(Params& p, const zk_mlp* m, const WidePack& wp, const FusedLayerArgs& a) {
    const TcPack* pk = (const TcPack*)m->tc;
    const int DPC = fused_dpc(a.univariate, a.bins);
    memset(&p, 0, sizeof(p));
    p.n_linear = m->n_linear;
    p.K0 = a.D + a.C;
    p.KB0 = pk->layers[0].Kp / 64;
    p.H = m->dims[1];
    p.nch_hidden = p.H / 128;
    p.D = a.D; p.C = a.C;
    p.n_last_chunks = (a.D + DPC - 1) / DPC;
    p.n_terms = pk->n_terms;
    p.M = (int)a.B;
    p.act = m->act;
    p.x = a.x; p.ldx = a.ldx; p.c = a.c; p.ldc = a.ldc;
    p.y = a.y; p.ldy = a.ldy; p.ladj = a.ladj; p.accumulate = a.accumulate;
    p.log_prob = a.log_prob; p.base_loc = a.base_loc; p.base_scale = a.base_scale;
    p.bound = a.bound;
    const float absL = fabsf(logf(a.slope));
    p.aw = 2.f / absL;
    p.ad = 1.f / absL;
    p.dbg = g_timeline;
    p.sched = wp.sched;
    p.n_items = wp.n_items;
    const bool x_ok = (a.ldx % 4 == 0) && (a.D % 4 == 0) && (((uintptr_t)a.x) % 16 == 0);
    const bool c_ok = (a.C == 0) || ((a.C % 4 == 0) && (((uintptr_t)a.c) % 16 == 0) && (a.ldc % 4 == 0));
    p.in_vec = (x_ok && c_ok) ? 1 : 0;
    for (int l = 0; l < m->n_linear; ++l) { p.mapW[l] = wp.maps[l]; p.rd_mask[l] = wp.rd_mask[l]; }
}

// Lays out the shared-memory copy of `bias_room` floats: the base table (log_prob only), the bias of the
// OUTPUT layer (47 reads per dim and thread) and as many hidden-layer biases as still fit, each 16-byte
// aligned; the others are read from global memory.  `floats`: how many floats the copy takes.
template <class Params>
zk_status pair_place_biases(Params& p, const zk_mlp* m, const FusedLayerArgs& a, uint32_t bias_room,
                            const char* what, uint32_t& floats) {
    const TcPack* pk = (const TcPack*)m->tc;
    const int L = m->n_linear;
    int off = 0;
    const int base_floats = a.log_prob ? ((3 * a.D + 3) & ~3) : 0;
    ZK_REQUIRE((uint32_t)base_floats <= bias_room, "%s: no shared memory left for the base table", what);
    bias_room -= (uint32_t)base_floats;
    auto place = [&](int l) {
        const int len = (m->dims[l + 1] + 3) & ~3;
        p.bias[l] = pk->fused.bias[l];
        p.bias_len[l] = m->dims[l + 1];
        if ((uint32_t)(off + len) <= bias_room) { p.bias_off[l] = off; off += len; }
        else p.bias_off[l] = -1;
    };
    place(L - 1);
    for (int l = 0; l < L - 1; ++l) place(l);
    for (int l = L; l < ZK_FUSED_MAX_LINEAR; ++l) { p.bias[l] = nullptr; p.bias_off[l] = -1; p.bias_len[l] = 0; }
    p.base_off = off;
    floats = (uint32_t)(off + base_floats);
    return ZK_OK;
}


}  // namespace zk
