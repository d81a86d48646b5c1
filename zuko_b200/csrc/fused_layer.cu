// zuko_b200 — ONE kernel per flow layer: conditioner (all linear layers) + bijector + ladj.
//
//   x, c  --(bf16 hi/lo split, in-kernel)-->  A operand in TENSOR MEMORY
//   for every linear layer:  tcgen05.mma  D[tmem] (+)= A[tmem] * W[smem]^T
//        W tiles are streamed from L2 by TMA, each CTA of a pair fetching half a tile and
//        multicasting it to both (cluster of 2);
//        hidden layers : epilogue (tcgen05.ld -> bias, ReLU -> bf16 hi/lo split) writes the next
//                        A operand straight back into tensor memory (tcgen05.st) — activations
//                        never touch shared memory or HBM, and the MMA reads only W from smem
//                        (with A in smem the 128-wide MMAs were shared-memory-bandwidth bound:
//                        ~108 cycles per MMA instead of 64, profiles/r01_fused_timeline_v1.txt);
//        last layer    : epilogue thread = sample row reads its D*P raw parameters from TMEM and
//                        evaluates the spline / affine bijector, the log-derivative and the
//                        per-sample sum in registers — phi never touches HBM either
//                        (SURVEY §7.2: "lane = sample row").
//   HBM traffic per sample per layer: 4 (D + C) read + 4 (D + 1) written (cfg2: 164 B instead of
//   the 9.3 kB of the unfused path).
//
// Restates for one MaskedAutoregressiveTransform layer:  flows/autoregressive.py:207-215 (meta),
// nn.py:217-218 (masked linears, mask folded into W at pack time), transforms.py:469-490,
// 554-567 (RQS) or 426-446 (affine), transforms.py:210-214 (sum over D), and on the last
// layer of a flow distributions.py:115-119 + torch normal.py:87-102 (DiagNormal log-prob).
//
// Tensor memory (512 columns x 128 lanes, lane = sample row of the tile):
//   [  0,128)  A hi : bf16 pairs, K element k in column k/2 (low half = even k)   (K <= 256)
//   [128,256)  A lo
//   [256,384)  D buffer 0 (fp32 accumulators of one <=128-column chunk)
//   [384,512)  D buffer 1
//
// Warp roles (640 threads, 1 CTA / SM, persistent over 128-row tiles, CTA pairs):
//   warp 0      W producer   (TMA multicast, 4-stage ring of 128 x 64 bf16 hi/lo tiles)
//   warp 1      MMA issuer   (one lane; M128 x N<=128 x K16, 3 MMAs per k-step: hh, hl, lh)
//   warp 2      TMEM allocator
//   warp 3      input producer (1-D TMA bulk copies of the next tile's x / c rows into smem)
//   warps 4-19  epilogue: four warp sets; hidden layers: set s owns 32 columns of a chunk;
//               last layer: set pair (chunk parity) owns the chunk, its two sets split the dims

#include <string.h>

#include <algorithm>
#include <type_traits>
#include <utility>
#include <vector>

#include "activations.cuh"
#include "fused_common.cuh"

namespace zk {

namespace {

using namespace bij;

constexpr int FM = 128;             // rows per tile
constexpr int FK = 64;              // bf16 per K block (128-byte swizzle row)
constexpr int F_MAX_WSTAGES = 8;   // the W ring is as deep as shared memory allows (see launch_fused_layer)
constexpr int F_MAXKB = 4;          // A operand: up to 4 K blocks = 256 columns
constexpr int F_EPI_WARP0 = 4;
constexpr int F_EPI_WARPS = 16;
constexpr int F_EPI_THREADS = F_EPI_WARPS * 32;  // 512
constexpr int F_THREADS = (F_EPI_WARP0 + F_EPI_WARPS) * 32;  // 640
constexpr int F_IN_MAXF = 64;       // floats per row of the staged input (D + C), TMA staging path
constexpr int F_BIAS_MAXF = 5120;   // floats of bias kept in shared memory (else read from global)
constexpr uint32_t F_PLANE = FM * FK * 2;       // 16 KB: one plane of one W tile
constexpr uint32_t F_KBLOCK = 2 * F_PLANE;      // hi + lo
constexpr uint32_t F_AUX_BYTES = 272 + 3 * 2 * FM * 4;     // 34 barrier slots + ladj partials [2][3][128]
constexpr uint32_t F_SMEM_MAX = 232448;                    // 227 KB per CTA on sm_100
constexpr uint32_t TM_ALO = 128, TM_D = 256;    // tensor-memory column map (see header)

struct FusedParams {
    CUtensorMap mapW[ZK_FUSED_MAX_LINEAR];
    const float* bias[ZK_FUSED_MAX_LINEAR];
    int bias_off[ZK_FUSED_MAX_LINEAR];  // offset of layer l's bias in the shared-memory copy
    int bias_len[ZK_FUSED_MAX_LINEAR];
    int bias_in_smem;
    uint8_t kbmask[ZK_FUSED_MAX_LINEAR][128];  // [layer][chunk]: K blocks with non-zero weights
    const uint32_t* sched;  // MMA issue schedule of one tile (device memory), see FusedPack::sched
    int n_items;
    int n_linear;
    int K0, KB0;        // real input width (D + C) and its number of 64-wide K blocks
    int H, CW;          // hidden width (multiple of 64, <= 256), hidden chunk width (128 or 64)
    int D, C;
    int n_last_chunks;  // ceil(D / DPC)
    int n_terms;        // 3 (split bf16) or 1
    int act;            // hidden activation: 1 ReLU, else ZK_ACT_* (GACT instantiation)
    int M;
    int in_tma;         // 1: x / c rows are staged through shared memory by 1-D TMA bulk copies
    int n_wstages;      // depth of the W ring (32 KB per stage)
    uint32_t in_bytes;  // bytes of one input staging buffer (0 when !in_tma)
    const float* x; int64_t ldx;
    const float* c; int64_t ldc;
    float* y; int64_t ldy;
    float* ladj; int accumulate;
    float* log_prob; const float* base_loc; const float* base_scale;
    float bound, aw, ad;
    long long* dbg;  // optional timeline buffer (clock64 stamps of CTA 0, third tile), see zk_debug_timeline
};

// timeline instrumentation: compiled in only for the DBG instantiation (zk_debug_timeline)
#define ZK_STAMP(slot)                                                                      \
    do {                                                                                    \
        if constexpr (DBG) {                                                                \
            if (p.dbg != nullptr && blockIdx.x == 0 && stamp_on) p.dbg[(slot)] = clock64(); \
        }                                                                                   \
    } while (0)

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 512;" ::: "memory"); }

template <int UNI, int KT, bool FAST, bool DBG, bool GACT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(F_THREADS, 1)
fused_layer_kernel(const __grid_constant__ FusedParams p) {
    using Cfg = LastCfg<UNI, KT>;
    constexpr int P = Cfg::P, DPC = Cfg::DPC;
    constexpr int N_LAST = (DPC * P + 15) & ~15;  // MMA N of a last-layer chunk
    static_assert(N_LAST <= 128, "a last-layer chunk must fit one accumulator buffer");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    // [W ring: n_wstages x 32 KB][input buffers: 2 x in_bytes][barriers + ladj scratch][bias copy]
    const int NW = p.n_wstages;
    uint8_t* sW = smem;
    float* s_in = (float*)(smem + (size_t)NW * F_KBLOCK);
    const uint32_t in_floats = p.in_bytes / 4;
    uint64_t* bars = (uint64_t*)(smem + (size_t)NW * F_KBLOCK + 2 * p.in_bytes);
    uint64_t* w_full = bars;                  // [8]
    uint64_t* w_empty = bars + 8;             // [8]
    uint64_t* d_full = bars + 16;             // [2]
    uint64_t* d_empty = bars + 18;            // [2]
    uint64_t* a_ready = bars + 20;            // [4]  K block kb of the A operand written
    uint64_t* a_free = bars + 24;             // [4]  every MMA of the current layer that reads K block kb of A is complete
    uint64_t* in_full = bars + 28;            // [2]  input rows of a tile landed in s_in[b]
    uint64_t* in_empty = bars + 30;           // [2]
    uint32_t* tmem_slot = (uint32_t*)(bars + 32);
    uint32_t* s_ready = tmem_slot + 1;        // number of schedule entries whose prerequisites are all met (scout -> MMA issuer)
    float* s_part = (float*)(bars + 34);      // [2][3][128] ladj partials of sets 1..3
    float* s_bias = (float*)((uint8_t*)bars + F_AUX_BYTES);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int L = p.n_linear;
    const int m_tiles = (p.M + FM - 1) / FM;
    // CTA pairs (clusters of 2) walk the tiles together: pair `cid` takes tiles 2 (cid + i ncl) + rank.
    // Both CTAs always run the same number of iterations (the W stream is shared through TMA
    // multicast); a CTA whose tile index falls off the end processes an all-masked dummy tile.
    const uint32_t rank = cluster_ctarank();
    const int cid = blockIdx.x >> 1, ncl = gridDim.x >> 1;
    const int n_iter = ((m_tiles + 1) / 2 - cid + ncl - 1) / ncl;
    const int KBH = p.H / FK;
    const int nch_hidden = p.H / p.CW;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NW; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 2); }  // empty: both CTAs
        for (int b = 0; b < 2; ++b) {
            mbar_init(&d_full[b], 1);
            mbar_init(&d_empty[b], F_EPI_THREADS);
            mbar_init(&in_full[b], 1);
            mbar_init(&in_empty[b], F_EPI_THREADS);
        }
        for (int k = 0; k < F_MAXKB; ++k) { mbar_init(&a_ready[k], F_EPI_THREADS); mbar_init(&a_free[k], 1); }
        *s_ready = 0u;
        fence_mbar_init();
    }
    if (p.bias_in_smem)
        for (int l = 0; l < L; ++l)
            for (int i = threadIdx.x; i < p.bias_len[l]; i += F_THREADS) s_bias[p.bias_off[l] + i] = p.bias[l][i];
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // the peer's barriers are initialised before any multicast / remote arrive
    tc_fence_after();
    // A 512-column allocation is the whole tensor memory, so its base is always lane 0 / column 0.
    // Using the literal keeps every tcgen05 address in uniform registers: with the address read
    // back from shared memory ptxas wrapped each UTCHMMA in an ELECT / R2UR.BROADCAST waterfall
    // loop (~110 cycles per MMA instead of 64).
    if (*tmem_slot != 0u) __trap();
    constexpr uint32_t tmem_base = 0u;

    if (warp == 0) {
        // ======================= W producer =======================
        if (lane == 0) {
            const uint32_t bytes = (p.n_terms == 3) ? F_KBLOCK : F_PLANE;
            int ws = 0;
            uint32_t wph = 0;
            for (int it = 0; it < n_iter; ++it) {
                const bool stamp_on = (it == 2);
                for (int l = 0; l < L; ++l) {
                    const bool last = (l == L - 1);
                    const int nch = last ? p.n_last_chunks : nch_hidden;
                    const int KB = (l == 0) ? p.KB0 : KBH;
                    for (int ch = 0; ch < nch; ++ch) {
                        const int n0 = last ? ch * DPC * P : ch * p.CW;
                        const uint32_t kbm = p.kbmask[l][ch] & ((1u << KB) - 1u);
                        for (int kb = 0; kb < KB; ++kb) {
                            if (!((kbm >> kb) & 1u)) continue;  // all-zero tile of the masked matrix: skipped
                            // the slot is written in BOTH CTAs: wait until both MMA issuers released it
                            if (l == 1 && ch == 1) ZK_STAMP(220 + 3 * kb);
                            mbar_wait(&w_empty[ws], wph ^ 1);
                            if (l == 1 && ch == 1) ZK_STAMP(221 + 3 * kb);
                            // this CTA fetches rows [64 rank, 64 rank + 64) of the 128-row W tile and
                            // multicasts them to the pair; the peer delivers the other half
                            uint8_t* st = sW + (size_t)ws * F_KBLOCK + rank * (F_PLANE / 2);
                            mbar_arrive_expect_tx(&w_full[ws], bytes);
                            tma_load_3d_mc(st, &p.mapW[l], &w_full[ws], kb * FK, n0 + 64 * (int)rank, 0, (uint16_t)3);
                            if (p.n_terms == 3)
                                tma_load_3d_mc(st + F_PLANE, &p.mapW[l], &w_full[ws], kb * FK, n0 + 64 * (int)rank, 1, (uint16_t)3);
                            if (l == 1 && ch == 1) ZK_STAMP(222 + 3 * kb);
                            if (++ws == NW) { ws = 0; wph ^= 1; }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ======================= MMA issuer =======================
        // The whole warp walks the tile's issue schedule (FusedPack::sched, one entry per non-zero
        // (layer, chunk, K block) tile in the order the W producer streams them); one elected lane
        // issues the MMAs and commits.  (Issuing from inside an `if (lane == 0)` region made ptxas
        // wrap every UTCHMMA in an ELECT / BRA.U.ANY waterfall loop: ~110 cycles per MMA.)
        //
        // The tensor pipe queues only ~4 MMAs (profiles/micro/mma_queue.cu: the issue loop returns
        // ~290 cycles before the last MMA completes), and this warp shares its scheduler with four
        // epilogue warps, so every instruction between the last MMA of one entry and the first of the
        // next starves the pipe — and an mbarrier probe issued behind pending tcgen05.commits costs
        // ~100 cycles by itself (profiles/micro/issuer_contention.cu).  The issuer therefore touches no
        // mbarrier at all: the scout (warp 2) waits for every prerequisite of an entry (weights landed,
        // accumulator buffer drained, A block written) and publishes the count of ready entries in
        // shared memory, which the issuer reads with one acquire load.
        const uint32_t idesc_h = umma_idesc_bf16(FM, p.CW), idesc_l = umma_idesc_bf16(FM, N_LAST);
        const int n_items = p.n_items;
        const int total = n_iter * n_items;
        int ws = 0, j = 0;
        uint32_t c = 0, seen = 0;  // c: running chunk counter (accumulator buffer = c & 1); seen: cached *s_ready
        uint32_t cur = (total > 0) ? __ldg(p.sched) : 0u;
        // entry bits: [1:0] kb, [2] first K block of its chunk, [3] last K block of its chunk,
        // [5] first use of A block kb in this layer (wait a_ready), [6] last reader of A block kb in this
        // layer (signal a_free), [7] last entry of the layer, [11:8] A blocks the layer never reads
        // (a_free at the layer's end), [15:12] a_ready phases the layer does not consume by reading
        // (set on the layer's first entry), [16] output layer
        for (int i = 0; i < total; ++i) {
            const bool stamp_on = (i / n_items == 2) && (lane == 0);
            const int jn = (j + 1 == n_items) ? 0 : j + 1;
            const uint32_t nxt = __ldg(p.sched + jn);
            const uint32_t kb = cur & 3u, buf = c & 1u;
            const uint32_t d_tmem = tmem_base + TM_D + buf * 128u;
            const uint32_t a_hi = tmem_base + kb * (uint32_t)(FK / 2), a_lo = a_hi + TM_ALO;
            const uint32_t w_addr = smem_u32(sW) + (uint32_t)ws * F_KBLOCK;
            const uint64_t dw_hi = umma_desc_k_sw128(w_addr), dw_lo = umma_desc_k_sw128(w_addr + F_PLANE);
            const uint32_t idesc = (cur & 0x10000u) ? idesc_l : idesc_h;
            const bool first = (cur & 4u) != 0;
            while (seen <= (uint32_t)i) asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(seen) : "r"(smem_u32(s_ready)) : "memory");
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
                for (int k = 0; k < FK / 16; ++k) {
                    const uint32_t acol = (uint32_t)k * 8u;  // 16 bf16 = 8 TMEM columns
                    umma_bf16_ts(d_tmem, a_hi + acol, umma_desc_advance(dw_hi, k), idesc, (!first || k > 0) ? 1u : 0u);
                    if (p.n_terms == 3) {
                        umma_bf16_ts(d_tmem, a_hi + acol, umma_desc_advance(dw_lo, k), idesc, 1u);
                        umma_bf16_ts(d_tmem, a_lo + acol, umma_desc_advance(dw_hi, k), idesc, 1u);
                    }
                }
                umma_commit_mc(&w_empty[ws], (uint16_t)3);  // releases the slot in both CTAs
                // a_free[kb] completes exactly once per layer: when the last MMA of the layer reading
                // K block kb of the A operand is done, the epilogue may overwrite that block with the
                // next layer's activations while the rest of the layer is still being multiplied
                if (cur & 64u) umma_commit(&a_free[kb]);
                if (cur & 8u) umma_commit(&d_full[buf]);
                if (cur & 128u) {  // blocks the layer does not read are released at its END: the epilogue
                                   // has consumed their previous phase by then (parity waits alias after two)
#pragma unroll
                    for (uint32_t k2 = 0; k2 < (uint32_t)F_MAXKB; ++k2)
                        if ((cur >> (8 + k2)) & 1u) umma_commit(&a_free[k2]);
                }
            }
            __syncwarp();
            if constexpr (DBG)
                if (p.dbg != nullptr && blockIdx.x == 0 && stamp_on && j < 240) p.dbg[256 + j] = clock64();
            c += (nxt >> 2) & 1u;
            cur = nxt;
            j = jn;
            if (++ws == NW) ws = 0;
        }
    } else if (warp == 2) {
        // ======================= scout =======================
        // Walks the same schedule ahead of the MMA issuer, waits for every entry's prerequisites and
        // publishes the number of entries that may be issued.
        if (lane == 0) {
            const int n_items = p.n_items;
            const int total = n_iter * n_items;
            int ws = 0, j = 0;
            uint32_t wph = 0, c = 0, a_par = 0;  // a_par: bit kb = parity of a_ready[kb]
            for (int i = 0; i < total; ++i) {
                const uint32_t it = __ldg(p.sched + j);
                if (i > 0) c += (it >> 2) & 1u;
                if (it & 4u) mbar_wait(&d_empty[c & 1u], ((c >> 1) & 1u) ^ 1u);
                if (it & 0xF000u) {  // A blocks this layer never reads: their a_ready phase is consumed here
                    for (uint32_t k2 = 0; k2 < (uint32_t)F_MAXKB; ++k2)
                        if ((it >> (12 + k2)) & 1u) { mbar_wait(&a_ready[k2], (a_par >> k2) & 1u); a_par ^= 1u << k2; }
                }
                if (it & 32u) { mbar_wait(&a_ready[it & 3u], (a_par >> (it & 3u)) & 1u); a_par ^= 1u << (it & 3u); }
                mbar_wait(&w_full[ws], wph);
                asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(smem_u32(s_ready)), "r"((uint32_t)(i + 1)) : "memory");
                if (++j == n_items) j = 0;
                if (++ws == NW) { ws = 0; wph ^= 1u; }
            }
        }
    } else if (warp == 3) {
        // ======================= input producer =======================
        if (lane == 0 && p.in_tma) {
            for (int it = 0; it < n_iter; ++it) {
                const int b = it & 1;
                const bool stamp_on = (it == 2);
                ZK_STAMP(56);
                mbar_wait(&in_empty[b], (((uint32_t)it >> 1) & 1u) ^ 1u);
                ZK_STAMP(57);
                const int t = 2 * (cid + it * ncl) + (int)rank;
                const int64_t r0 = (int64_t)t * FM;
                const int rows = (int)max((int64_t)0, min((int64_t)FM, (int64_t)p.M - r0));
                float* dst = s_in + (size_t)b * in_floats;
                const uint32_t bx = (uint32_t)rows * p.D * 4u;
                const uint32_t bc = (p.C == 0) ? 0u : ((p.ldc == 0) ? (uint32_t)p.C * 4u : (uint32_t)rows * p.C * 4u);
                if (rows == 0) {
                    mbar_arrive(&in_full[b]);  // dummy tile: nothing to copy
                } else {
                    mbar_arrive_expect_tx(&in_full[b], bx + bc);
                    bulk_g2s(dst, p.x + r0 * p.ldx, bx, &in_full[b]);
                    if (bc) bulk_g2s(dst + FM * p.D, (p.ldc == 0) ? p.c : p.c + r0 * p.ldc, bc, &in_full[b]);
                }
            }
        }
    } else if (warp >= F_EPI_WARP0) {
        // ======================= epilogue =======================
        const int s = (warp - F_EPI_WARP0) >> 2;  // warp set 0..3
        const int q = warp & 3;                   // TMEM lane quadrant
        const int r = q * 32 + lane;              // row inside the tile
        const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t chunk = 0, f_par = 0;  // f_par: bit kb = parity of a_free[kb]
        for (int tile_iter = 0; tile_iter < n_iter; ++tile_iter) {
            const int t = 2 * (cid + tile_iter * ncl) + (int)rank;  // may be >= m_tiles: dummy tile, all rows masked
            const bool stamp_on = (tile_iter == 2) && (threadIdx.x == F_EPI_WARP0 * 32);
            ZK_STAMP(48);
            const int64_t row = (int64_t)t * FM + r;
            const bool row_ok = row < p.M;
            const int ib = tile_iter & 1;
            const float* sx = s_in + (size_t)ib * in_floats;
            const float* sc = sx + FM * p.D;
            if (p.in_tma) mbar_wait(&in_full[ib], ((uint32_t)tile_iter >> 1) & 1u);
            ZK_STAMP(51);
            // ---- stage the layer-0 operand: cat(x, c) -> bf16 hi/lo pairs in TMEM; set s takes
            //      K block kb = s, s + 4, ... (one K block = 64 inputs = 32 TMEM columns) ----
            if (p.in_tma) {
                // the rows sit in shared memory (TMA): 16-byte loads, 8 lanes cover 8 consecutive rows
                const float4* sx4 = reinterpret_cast<const float4*>(sx + r * p.D);
                const float4* sc4 = reinterpret_cast<const float4*>(sc + (p.ldc == 0 ? 0 : r * p.C));
                const int d4 = row_ok ? (p.D >> 2) : 0, k4 = row_ok ? (p.K0 >> 2) : 0;  // masked rows stage zeros
                for (int kb = s; kb < p.KB0; kb += 4) {
#pragma unroll 1
                    for (int g = 0; g < 2; ++g) {  // 32 inputs = 8 float4 = 16 TMEM columns per plane
                        const int i0 = kb * 16 + g * 8;
                        uint32_t ph[16], pl[16];
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const int i = i0 + j;
                            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (i < d4) v = sx4[i];
                            else if (i < k4) v = sc4[i - (p.D >> 2)];
                            split2_bf16(v.x, v.y, ph[2 * j], pl[2 * j]);
                            split2_bf16(v.z, v.w, ph[2 * j + 1], pl[2 * j + 1]);
                        }
                        const uint32_t ta = t_lane + (uint32_t)(kb * 32 + g * 16);
                        tmem_st_x16(ta, ph);
                        tmem_st_x16(ta + TM_ALO, pl);
                    }
                }
            } else {
                const float* srcx = p.x + row * p.ldx;
                const float* srcc = (p.C == 0) ? srcx : (p.c + row * p.ldc);
                const int kx = row_ok ? p.D : 0, kc = row_ok ? p.K0 : 0;
                for (int kb = s; kb < p.KB0; kb += 4) {
#pragma unroll 1
                    for (int g = 0; g < 2; ++g) {
                        const int k0 = kb * FK + g * 32;
                        uint32_t ph[16], pl[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int k = k0 + 2 * j;
                            const float v0 = (k < kx) ? __ldg(srcx + k) : ((k < kc) ? __ldg(srcc + k - p.D) : 0.f);
                            const float v1 = (k + 1 < kx) ? __ldg(srcx + k + 1) : ((k + 1 < kc) ? __ldg(srcc + k + 1 - p.D) : 0.f);
                            split2_bf16(v0, v1, ph[j], pl[j]);
                        }
                        const uint32_t ta = t_lane + (uint32_t)(kb * 32 + g * 16);
                        tmem_st_x16(ta, ph);
                        tmem_st_x16(ta + TM_ALO, pl);
                    }
                }
            }
            ZK_STAMP(52);
            tmem_st_wait();
            tc_fence_before();
            for (int kb = 0; kb < p.KB0; ++kb) mbar_arrive(&a_ready[kb]);
            ZK_STAMP(49);

            // ---- hidden layers: D -> bias, ReLU -> hi/lo -> next A operand (tensor memory) ----
            for (int l = 0; l < L - 1; ++l) {
                const float* bias = p.bias_in_smem ? s_bias + p.bias_off[l] : p.bias[l];
                for (int ch = 0; ch < nch_hidden; ++ch, ++chunk) {
                    const uint32_t buf = chunk & 1u;
                    mbar_wait(&d_full[buf], (chunk >> 1) & 1u);
                    tc_fence_after();
                    ZK_STAMP(64 + 16 * l + 4 * ch + 0);
                    const int col0 = s * 32;              // this set's 32 columns of the chunk
                    const bool owner = col0 < p.CW;       // CW = 64: sets 2, 3 have no columns
                    // two halves of 16 columns: at most 16 raw + 32 packed registers live (the x32
                    // variant spilled the packed values to local memory under the 96-register cap)
                    uint32_t ph[16], pl[16];
                    const int nbase = ch * p.CW + col0;   // first output column = K index of the next layer
                    if (owner) {
                        const float4* b4 = reinterpret_cast<const float4*>(bias + nbase);  // 128-byte aligned
#pragma unroll
                        for (int half = 0; half < 2; ++half) {
                            uint32_t ra[16];
                            tmem_ld_x16(t_lane + TM_D + buf * 128u + (uint32_t)(col0 + 16 * half), ra);
                            tmem_ld_wait();
                            if constexpr (GACT) {  // any ZK_ACT_* (nn.py:264-265): one switch per 16 columns
                                float v[16];
#pragma unroll
                                for (int j = 0; j < 16; j += 4) {
                                    const float4 bb = b4[4 * half + (j >> 2)];
                                    v[j] = __uint_as_float(ra[j]) + bb.x; v[j + 1] = __uint_as_float(ra[j + 1]) + bb.y;
                                    v[j + 2] = __uint_as_float(ra[j + 2]) + bb.z; v[j + 3] = __uint_as_float(ra[j + 3]) + bb.w;
                                }
                                if constexpr (FAST) act_apply_n_fast<16>(v, p.act); else act_apply_n<16>(v, p.act);
#pragma unroll
                                for (int j = 0; j < 16; j += 2) split2_bf16(v[j], v[j + 1], ph[8 * half + (j >> 1)], pl[8 * half + (j >> 1)]);
                            } else {
#pragma unroll
                            for (int j = 0; j < 16; j += 4) {
                                const float4 bb = b4[4 * half + (j >> 2)];  // one broadcast 16-byte load per 4 columns
                                split2_bf16(fmaxf(__uint_as_float(ra[j]) + bb.x, 0.f), fmaxf(__uint_as_float(ra[j + 1]) + bb.y, 0.f),
                                            ph[8 * half + (j >> 1)], pl[8 * half + (j >> 1)]);
                                split2_bf16(fmaxf(__uint_as_float(ra[j + 2]) + bb.z, 0.f), fmaxf(__uint_as_float(ra[j + 3]) + bb.w, 0.f),
                                            ph[8 * half + (j >> 1) + 1], pl[8 * half + (j >> 1) + 1]);
                            }
                            }
                        }
                    }
                    if (l == 1 && ch == 1) ZK_STAMP(240);
                    tc_fence_before();
                    mbar_arrive(&d_empty[buf]);  // accumulator buffer is free again
                    if (l == 1 && ch == 1) ZK_STAMP(241);
                    ZK_STAMP(64 + 16 * l + 4 * ch + 1);
                    {   // the K blocks this chunk overwrites must have been read by every MMA of this layer
                        const int kb0 = (p.CW == 128) ? 2 * ch : ch;
                        const int kb1 = (ch == nch_hidden - 1) ? F_MAXKB : ((p.CW == 128) ? 2 * ch + 2 : ch + 1);
                        for (int kb = kb0; kb < kb1; ++kb) {  // (the last chunk also consumes the unused blocks' phases)
                            mbar_wait(&a_free[kb], (f_par >> kb) & 1u);
                            f_par ^= (1u << kb);
                        }
                        tc_fence_after();
                    }
                    ZK_STAMP(64 + 16 * l + 4 * ch + 2);
                    if (owner) {
                        const uint32_t ta = t_lane + (uint32_t)(nbase >> 1);  // K element k lives in column k / 2
                        tmem_st_x16(ta, ph);
                        tmem_st_x16(ta + TM_ALO, pl);
                        if (l == 1 && ch == 1) ZK_STAMP(242);
                        tmem_st_wait();
                    }
                    if (l == 1 && ch == 1) ZK_STAMP(243);
                    tc_fence_before();
                    if (p.CW == 128) {
                        mbar_arrive(&a_ready[ch * 2]);
                        mbar_arrive(&a_ready[ch * 2 + 1]);
                    } else {
                        mbar_arrive(&a_ready[ch]);
                    }
                    ZK_STAMP(64 + 16 * l + 4 * ch + 3);
                    if constexpr (DBG)
                        if (p.dbg != nullptr && blockIdx.x == 0 && tile_iter == 2 && threadIdx.x == F_THREADS - 32)
                            p.dbg[110 + 2 * l + ch] = clock64();  // the last epilogue warp's view of "A written"
                }
            }

            // ---- last layer: raw parameters stay in TMEM -> bijector + ladj in registers ----
            float lsum = 0.f;
            const float* bias = p.bias_in_smem ? s_bias + p.bias_off[L - 1] : p.bias[L - 1];
            for (int ch = 0; ch < p.n_last_chunks; ++ch, ++chunk) {
                const uint32_t buf = chunk & 1u;
                mbar_wait(&d_full[buf], (chunk >> 1) & 1u);
                tc_fence_after();
                if (ch < 8) ZK_STAMP(160 + 2 * ch);
                // SPC sets share a chunk (all four when it holds >= 4 dims, else the set pairs alternate
                // chunks).  Every thread first pulls the raw parameters of its dims out of tensor memory
                // and releases the accumulator buffer, THEN evaluates: the MMAs of chunk c + 2 never
                // wait for the spline evaluation of chunk c.
                constexpr int SPC = (DPC >= 4) ? 4 : 2;
                const bool mine = (SPC == 4) || ((int)buf == (s >> 1));
                const int h = (SPC == 4) ? s : (s & 1);  // which share of the chunk's dims
                const uint32_t td = t_lane + TM_D + buf * 128u;
                auto release = [&]() {
                    tc_fence_before();
                    mbar_arrive(&d_empty[buf]);
                };
                auto finish_dim = [&](int d, float yv, float lj) {
                    if (p.y) p.y[row * p.ldy + d] = yv;
                    if (p.log_prob) {
                        const float mu = p.base_loc ? p.base_loc[d] : 0.f;
                        const float sg = p.base_scale ? p.base_scale[d] : 1.f;
                        const float u = (yv - mu) / sg;
                        lj += -0.5f * u * u - logf(sg) - kHalfLog2Pi;
                    }
                    lsum += lj;
                };
                if constexpr (UNI == ZK_UNI_RQS) {
                    static_assert(DPC == SPC, "one dim per set and chunk");
                    // load the 16-column-aligned window covering the dim's P parameters
                    auto do_dim = [&](auto dloc_c) {
                        constexpr int dloc = decltype(dloc_c)::value;
                        constexpr int c_lo = dloc * P, c_hi = c_lo + P;  // columns inside the chunk
                        constexpr int w0 = c_lo & ~15;                   // window start (16-aligned)
                        constexpr int wn = ((c_hi - w0) + 15) & ~15;     // window width: 32, 48 or 64
                        static_assert(wn <= 64 && w0 + wn <= 128, "window out of range");
                        uint32_t rr[wn];
                        tmem_ld_x16(td + (uint32_t)w0, rr);
                        if constexpr (wn > 16) tmem_ld_x16(td + (uint32_t)(w0 + 16), rr + 16);
                        if constexpr (wn > 32) tmem_ld_x16(td + (uint32_t)(w0 + 32), rr + 32);
                        if constexpr (wn > 48) tmem_ld_x16(td + (uint32_t)(w0 + 48), rr + 48);
                        tmem_ld_wait();
                        release();
                        const int d = ch * DPC + dloc;
                        if (d >= p.D || !row_ok) return;
                        float pp[P];
                        const float* bd = bias + d * P;
#pragma unroll
                        for (int j = 0; j < P; ++j) pp[j] = __uint_as_float(rr[c_lo - w0 + j]) + bd[j];
                        const float xv = p.in_tma ? sx[r * p.D + d] : p.x[row * p.ldx + d];
                        float yv, lj;
                        Bin b = rqs_select<KT, FAST, false>(pp, KT, xv, p.bound, p.aw, p.ad);
                        rqs_forward_eval<FAST>(b, xv, yv, lj);
                        finish_dim(d, yv, lj);
                    };
                    if (!mine) release();
                    else if (h == 0) do_dim(std::integral_constant<int, 0>{});
                    else if (h == 1) do_dim(std::integral_constant<int, 1>{});
                    else if constexpr (SPC == 4) {
                        if (h == 2) do_dim(std::integral_constant<int, 2>{});
                        else do_dim(std::integral_constant<int, 3>{});
                    }
                } else {
                    // affine: 8 dims (16 columns: shift, scale pairs) per load; this set takes the
                    // 2 groups [2 h, 2 h + 2) of the chunk's 8 groups
                    static_assert(SPC == 4 && DPC == 64, "affine chunk layout");
                    uint32_t rr[2][16];
                    tmem_ld_x16(td + (uint32_t)((h * 2) * 16), rr[0]);
                    tmem_ld_x16(td + (uint32_t)((h * 2 + 1) * 16), rr[1]);
                    tmem_ld_wait();
                    release();
#pragma unroll
                    for (int g = 0; g < 2; ++g) {
                        const int c0 = (h * 2 + g) * 16;
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const int d = ch * DPC + (c0 >> 1) + j;
                            if (d < p.D && row_ok) {
                                const float shift = __uint_as_float(rr[g][2 * j]) + bias[2 * d];
                                const float ls = softclip<FAST>(__uint_as_float(rr[g][2 * j + 1]) + bias[2 * d + 1], p.ad);
                                const float xv = p.in_tma ? sx[r * p.D + d] : p.x[row * p.ldx + d];
                                finish_dim(d, fmaf(xv, zexp<FAST>(ls), shift), ls);
                            }
                        }
                    }
                }
                if (ch < 8) ZK_STAMP(161 + 2 * ch);
            }
            // all MMAs of this tile are complete once the last layer's a_free phases fire: A may be restaged
            for (int kb = 0; kb < F_MAXKB; ++kb) {
                mbar_wait(&a_free[kb], (f_par >> kb) & 1u);
                f_par ^= (1u << kb);
            }
            tc_fence_after();
            // ---- per-sample sum: sets 0..2 hand their partials to set 3 without waiting for it ----
            float* part = s_part + (tile_iter & 1) * (3 * FM);
            if (p.in_tma) mbar_arrive(&in_empty[ib]);  // x rows no longer needed
            if (s < 3) {
                part[s * FM + r] = lsum;
                __threadfence_block();
                asm volatile("bar.arrive 1, 512;" ::: "memory");
            } else {
                epi_bar_sync();
                if (row_ok) {
                    const float tot = lsum + part[r] + part[FM + r] + part[2 * FM + r] + (p.accumulate ? p.ladj[row] : 0.f);
                    if (p.log_prob) p.log_prob[row] = tot;
                    else if (p.ladj) p.ladj[row] = tot;
                }
            }
            ZK_STAMP(50);
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // no CTA leaves while its peer may still multicast into it
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

template <int UNI, int KT>
zk_status launch_fused_t(const FusedParams& p, bool fast, int grid, size_t smem, cudaStream_t st) {
    auto go = [&](auto kern) -> zk_status {
        ZK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F_SMEM_MAX));
        kern<<<grid, F_THREADS, smem, st>>>(p);
        return check_launch("fused_layer_kernel");
    };
    if (p.act > 1) return fast ? go(fused_layer_kernel<UNI, KT, true, false, true>) : go(fused_layer_kernel<UNI, KT, false, false, true>);
    if (p.dbg != nullptr) return fast ? go(fused_layer_kernel<UNI, KT, true, true, false>) : go(fused_layer_kernel<UNI, KT, false, true, false>);
    if (fast) return go(fused_layer_kernel<UNI, KT, true, false, false>);
    return go(fused_layer_kernel<UNI, KT, false, false, false>);
}

}  // namespace

long long* g_timeline = nullptr;

static bool fused_narrow_shape(const zk_mlp* m, int univariate, int bins, int D, int C) {
    const TcPack* pk = (const TcPack*)m->tc;
    if (!pk || m->gemm_mode == ZK_GEMM_FP32) return false;
    if (m->act < 1 || !m->plain) return false;  // plain MLPs only (residual blocks need the input of two layers back)
    if (m->n_linear < 2 || m->n_linear > ZK_FUSED_MAX_LINEAR) return false;
    const int H = m->dims[1];
    if (H % 64 != 0 || H < 64 || H > 256) return false;
    for (int i = 1; i < m->n_linear; ++i)
        if (m->dims[i] != H) return false;
    if (D + C > 256 || m->dims[0] != D + C) return false;
    if (univariate == ZK_UNI_RQS) return bins == 8 || bins == 16;
    return univariate == ZK_UNI_AFFINE;
}

int fused_layer_kind(const zk_mlp* m, int univariate, int bins, int D, int C) {
    const TcPack* pk = (const TcPack*)m->tc;  // non-null once a shape test passed
    // a pair kernel runs the layer once it takes the shape (routing knobs included) and its pack holds
    // a schedule for this bijector
    if (fused_dual_shape(m, univariate, bins, D, C) && pk->dual.built_for(univariate, bins, D, C)) return 3;
    if (fused_wide_shape(m, univariate, bins, D, C) && pk->wide.built_for(univariate, bins, D, C)) return 2;
    return fused_narrow_shape(m, univariate, bins, D, C) ? 1 : 0;
}

bool fused_layer_supported(const zk_mlp* m, int univariate, int bins, int D, int C) {
    return fused_layer_kind(m, univariate, bins, D, C) != 0;
}

namespace {
__global__ void split_permuted_kernel(const float* W, int N, int K, int Kp, const int* row_perm, const int* col_perm,
                                      __nv_bfloat16* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)N * Kp) return;
    const int n = (int)(i / Kp), k = (int)(i - (int64_t)n * Kp);
    const int sn = row_perm ? row_perm[n] : n;
    const float v = (k < K) ? W[(int64_t)sn * K + (col_perm ? col_perm[k] : k)] : 0.f;
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    out[i] = h;
    out[(int64_t)N * Kp + i] = __float2bfloat16_rn(v - __bfloat162float(h));
}
__global__ void permute_bias_kernel(const float* b, int N, const int* perm, float* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) out[i] = b[perm ? perm[i] : i];
}
}  // namespace

// Masks to the host, hidden units sorted by dependency degree, permuted bf16 hi / lo planes and
// biases on the device (shared by the narrow and the wide fused kernel).
zk_status fused_host_prepare(zk_mlp* m, const uint8_t* const* mask_dev, FusedPack& f, FusedHostPrep& hp) {
    TcPack* pk = (TcPack*)m->tc;
    const int L = m->n_linear;
    // ---- host copies of the masks (dense layers: all ones) ----
    std::vector<std::vector<uint8_t>>& Mk = hp.Mk;
    Mk.assign(L, {});
    for (int l = 0; l < L; ++l) {
        const size_t n = (size_t)m->dims[l + 1] * m->dims[l];
        Mk[l].assign(n, 1);
        if (mask_dev && mask_dev[l]) ZK_CUDA(cudaMemcpy(Mk[l].data(), mask_dev[l], n, cudaMemcpyDeviceToHost));
    }
    fused_degree_perm(m->dims.data(), L, hp.Mk, hp.perm);
    std::vector<std::vector<int>>& perm = hp.perm;
    // ---- permuted planes and biases ----
    for (auto* q : f.w) cudaFree(q);
    for (auto* q : f.bias) cudaFree(q);
    for (auto* q : f.dperm) cudaFree(q);
    f.w.clear(); f.bias.clear();
    f.dperm.assign(L - 1, nullptr);
    std::vector<int*>& dperm = f.dperm;  // kept: a weight refresh re-runs the split kernels with them
    zk_status st = ZK_OK;
    for (int l = 0; l < L - 1 && st == ZK_OK; ++l) {
        if (cudaMalloc((void**)&dperm[l], perm[l].size() * 4) != cudaSuccess ||
            cudaMemcpy(dperm[l], perm[l].data(), perm[l].size() * 4, cudaMemcpyHostToDevice) != cudaSuccess)
            st = fail(ZK_ENOMEM, "fused_host_prepare: cudaMalloc failed");
    }
    for (int l = 0; l < L && st == ZK_OK; ++l) {
        const int K = m->dims[l], N = m->dims[l + 1], Kp = pk->layers[l].Kp;
        __nv_bfloat16* w = nullptr;
        float* b = nullptr;
        if (cudaMalloc((void**)&w, (size_t)2 * N * Kp * 2) != cudaSuccess || cudaMalloc((void**)&b, ((size_t)N + 4) * 4) != cudaSuccess) {
            cudaFree(w);
            st = fail(ZK_ENOMEM, "fused_host_prepare: cudaMalloc failed");
            break;
        }
        f.w.push_back(w);
        f.bias.push_back(b);
        const int* rp = (l < L - 1) ? dperm[l] : nullptr;      // output units of hidden layers are permuted
        const int* cp = (l > 0) ? dperm[l - 1] : nullptr;       // and so are the inputs of the layer after
        split_permuted_kernel<<<(unsigned)ceil_div((int64_t)N * Kp, 256), 256, 0, 0>>>(m->w[l], N, K, Kp, rp, cp, w);
        st = check_launch("split_permuted_kernel");
        if (st != ZK_OK) break;
        cudaMemsetAsync(b, 0, ((size_t)N + 4) * 4, 0);
        permute_bias_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, 0>>>(m->b[l], N, rp, b);
        st = check_launch("permute_bias_kernel");
    }
    if (st == ZK_OK && cudaStreamSynchronize(0) != cudaSuccess) st = fail(ZK_ECUDA, "fused_host_prepare: sync failed");
    return st;
}

// The weights of `m` changed in place (same shapes, same masks): rebuild the fused kernels' permuted
// planes and biases with the permutations of the last fused_host_prepare.  Stream-ordered, no
// allocation, no host synchronisation; schedules / tensor maps depend on the masks only and stay.
zk_status fused_refresh(zk_mlp* m, cudaStream_t st) {
    TcPack* pk = (TcPack*)m->tc;
    if (!pk) return ZK_OK;
    FusedPack& f = pk->fused;
    const int L = m->n_linear;
    if ((int)f.w.size() != L || (int)f.dperm.size() != L - 1) return ZK_OK;  // no fused pack was built
    for (int l = 0; l < L; ++l) {
        const int K = m->dims[l], N = m->dims[l + 1], Kp = pk->layers[l].Kp;
        const int* rp = (l < L - 1) ? f.dperm[l] : nullptr;
        const int* cp = (l > 0) ? f.dperm[l - 1] : nullptr;
        split_permuted_kernel<<<(unsigned)ceil_div((int64_t)N * Kp, 256), 256, 0, st>>>(m->w[l], N, K, Kp, rp, cp, f.w[l]);
        ZK_TRY(check_launch("split_permuted_kernel"));
        permute_bias_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, st>>>(m->b[l], N, rp, f.bias[l]);
        ZK_TRY(check_launch("permute_bias_kernel"));
    }
    return ZK_OK;
}

zk_status fused_layer_prepare(zk_mlp* m, const uint8_t* const* mask_dev, int univariate, int bins, int D, int C) {
    TcPack* pk = (TcPack*)m->tc;
    if (fused_dual_shape(m, univariate, bins, D, C)) {  // two sub-tiles in flight (hidden width 128 / 256)
        ZK_TRY(fused_pair_prepare(m, mask_dev, univariate, bins, D, C, pk->dual, 2));
        if (pk->dual.ready) return ZK_OK;
    }
    if (fused_wide_shape(m, univariate, bins, D, C)) {  // CTA-pair kernel; hidden width 256 may fall back to the narrow one
        ZK_TRY(fused_pair_prepare(m, mask_dev, univariate, bins, D, C, pk->wide, 1));
        if (pk->wide.ready) return ZK_OK;
    }
    if (!fused_narrow_shape(m, univariate, bins, D, C)) return ZK_OK;
    FusedPack& f = pk->fused;
    const int L = m->n_linear;
    const int H = m->dims[1];
    const int CW = (H % 128 == 0) ? 128 : 64;
    const int P = fused_p(univariate, bins);
    const int DPC = fused_dpc(univariate, bins);
    FusedHostPrep hp;
    ZK_TRY(fused_host_prepare(m, mask_dev, f, hp));
    f.map64.clear();
    f.map64.resize(L);
    for (int l = 0; l < L; ++l) ZK_TRY(make_plane_map(&f.map64[l], f.w[l], m->dims[l + 1], pk->layers[l].Kp, 64));
    const FusedTileMap tm = fused_tile_map(m->dims.data(), L, hp.Mk, hp.perm, CW, univariate, bins, D);
    memset(f.kbmask, 0, sizeof(f.kbmask));
    for (int l = 0; l < L; ++l)
        for (size_t ch = 0; ch < tm.kbmask[l].size() && ch < 128; ++ch) f.kbmask[l][ch] = (uint8_t)tm.kbmask[l][ch];
    // ---- MMA issue schedule of one tile: one entry per non-zero (layer, chunk, K block) tile, in the
    //      order the W producer streams them (bit layout: see the MMA issuer in the kernel) ----
    std::vector<uint32_t> items;
    for (int l = 0; l < L; ++l) {
        const bool last = (l == L - 1);
        const int nch = std::min(128, (int)tm.kbmask[l].size());
        const int KB = (l == 0) ? pk->layers[0].Kp / 64 : H / 64;
        int last_reader[F_MAXKB];
        for (int kb = 0; kb < F_MAXKB; ++kb) last_reader[kb] = -1;
        for (int ch = 0; ch < nch; ++ch)
            for (int kb = 0; kb < KB; ++kb)
                if ((f.kbmask[l][ch] >> kb) & 1u) last_reader[kb] = ch;
        uint32_t waited = 0;
        const size_t layer_first = items.size();
        for (int ch = 0; ch < nch; ++ch) {
            const uint32_t kbm = f.kbmask[l][ch] & ((1u << KB) - 1u);
            int hi = 0;
            for (int kb = 0; kb < KB; ++kb) if ((kbm >> kb) & 1u) hi = kb;
            bool first = true;
            for (int kb = 0; kb < KB; ++kb) {
                if (!((kbm >> kb) & 1u)) continue;
                uint32_t it = (uint32_t)kb | (first ? 4u : 0u) | (kb == hi ? 8u : 0u);
                if (!((waited >> kb) & 1u)) { it |= 32u; waited |= 1u << kb; }
                if (last_reader[kb] == ch) it |= 64u;
                if (last) it |= 0x10000u;
                items.push_back(it);
                first = false;
            }
        }
        uint32_t nofree = 0, unread = 0;
        for (int kb = 0; kb < F_MAXKB; ++kb) if (last_reader[kb] < 0) nofree |= 1u << kb;
        for (int kb = 0; kb < KB; ++kb) if (!((waited >> kb) & 1u)) unread |= 1u << kb;
        items.back() |= 128u | (nofree << 8);
        items[layer_first] |= unread << 12;
    }
    cudaFree(f.sched);
    f.sched = nullptr;
    f.n_items = (int)items.size();
    {   // every entry is one (CW | N_LAST) x 64 tile of MACs per row, times the split terms
        const int N_LAST = (DPC * P + 15) & ~15;
        double macs = 0;
        for (uint32_t it : items) macs += 64.0 * ((it & 0x10000u) ? N_LAST : CW);
        f.issued_macs_per_row = macs * pk->n_terms;
    }
    if (cudaMalloc((void**)&f.sched, items.size() * 4) != cudaSuccess ||
        cudaMemcpy(f.sched, items.data(), items.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess)
        return fail(ZK_ENOMEM, "fused_layer_prepare: cudaMalloc failed");
    f.uni = univariate; f.bins = bins; f.D = D; f.C = C;
    f.ready = true;
    return ZK_OK;
}

zk_status launch_fused_layer(const zk_mlp* m, const FusedLayerArgs& a, cudaStream_t st) {
    const TcPack* pk = (const TcPack*)m->tc;
    const int kind = fused_layer_kind(m, a.univariate, a.bins, a.D, a.C);
    if (kind == 3) return launch_fused_dual(m, a, st);
    if (kind == 2) return launch_fused_wide(m, a, st);
    ZK_REQUIRE(pk && fused_narrow_shape(m, a.univariate, a.bins, a.D, a.C), "fused layer: unsupported shape");
    ZK_REQUIRE(a.B < ((int64_t)1 << 31) - FM, "fused layer: batch too large for one launch");
    if (a.B == 0) return ZK_OK;
    FusedParams p;
    int off = 0;
    for (int i = 0; i < ZK_FUSED_MAX_LINEAR; ++i) { p.bias[i] = nullptr; p.bias_off[i] = 0; p.bias_len[i] = 0; }
    const FusedPack& f = pk->fused;
    const bool packed = f.ready && f.uni == a.univariate && f.bins == a.bins && f.D == a.D && f.C == a.C;
    memset(p.kbmask, 0xff, sizeof(p.kbmask));  // unprepared handles: every tile is streamed
    ZK_REQUIRE(packed && f.sched != nullptr, "fused layer: the conditioner was not prepared for this bijector");
    memcpy(p.kbmask, f.kbmask, sizeof(p.kbmask));
    for (int i = 0; i < m->n_linear; ++i) {
        p.mapW[i] = packed ? f.map64[i] : pk->layers[i].mapW64;
        p.bias[i] = packed ? f.bias[i] : m->b[i];
        p.bias_off[i] = off;
        p.bias_len[i] = m->dims[i + 1];
        off += (m->dims[i + 1] + 3) & ~3;  // keep every layer's bias 16-byte aligned
    }
    p.bias_in_smem = (off <= F_BIAS_MAXF) ? 1 : 0;
    const uint32_t bias_bytes = p.bias_in_smem ? (uint32_t)off * 4u : 0u;
    p.n_linear = m->n_linear;
    p.K0 = a.D + a.C;
    p.KB0 = pk->layers[0].Kp / FK;
    p.H = m->dims[1];
    p.CW = (p.H % 128 == 0) ? 128 : 64;
    p.D = a.D; p.C = a.C;
    p.n_terms = pk->n_terms;
    p.act = m->act;
    p.M = (int)a.B;
    p.x = a.x; p.ldx = a.ldx; p.c = a.c; p.ldc = a.ldc;
    p.y = a.y; p.ldy = a.ldy; p.ladj = a.ladj; p.accumulate = a.accumulate;
    p.log_prob = a.log_prob; p.base_loc = a.base_loc; p.base_scale = a.base_scale;
    p.bound = a.bound;
    const float absL = fabsf(logf(a.slope));
    p.aw = 2.f / absL;
    p.ad = 1.f / absL;
    p.dbg = g_timeline;
    // the x / c rows of a tile are one contiguous block each: stage them with 1-D TMA bulk copies
    // when the 16-byte rules hold, else the epilogue threads load their rows directly
    const bool x_ok = (a.ldx == a.D) && (a.D % 4 == 0) && (((uintptr_t)a.x) % 16 == 0);
    const bool c_ok = (a.C == 0) || ((a.C % 4 == 0) && (((uintptr_t)a.c) % 16 == 0) && (a.ldc == a.C || a.ldc == 0));
    p.in_tma = (x_ok && c_ok && a.D + a.C <= F_IN_MAXF) ? 1 : 0;
    p.in_bytes = p.in_tma ? (uint32_t)FM * (uint32_t)(a.D + a.C) * 4u : 0u;
    // The W ring must cover (weight bytes per MMA time) x (TMA round trip ~4000 cycles): with 4
    // stages the MMA issuer waited ~1000 cycles per stage regardless of the MMA count per stage
    // (profiles/r01_fused_timeline_v4.txt).  Give it every byte of shared memory that is left.
    const uint32_t fixed = 1024u /*alignment slack*/ + 2u * p.in_bytes + F_AUX_BYTES + bias_bytes;
    p.n_wstages = (int)std::min<uint32_t>(F_MAX_WSTAGES, (F_SMEM_MAX - fixed) / F_KBLOCK);
    ZK_REQUIRE(p.n_wstages >= 3, "fused layer: not enough shared memory for the weight ring");
    const size_t smem = (size_t)p.n_wstages * F_KBLOCK + fixed;
    // clusters of 2 CTAs: even grid, at most one CTA per SM
    const int64_t pairs = ceil_div(ceil_div(a.B, FM), 2);
    const int grid = 2 * (int)std::min<int64_t>(pairs, sm_count() / 2);
    const bool rqs8 = a.univariate == ZK_UNI_RQS && a.bins == 8, rqs16 = a.univariate == ZK_UNI_RQS && a.bins == 16;
    p.n_last_chunks = rqs8 ? (a.D + 3) / 4 : (rqs16 ? (a.D + 1) / 2 : (a.D + 63) / 64);
    p.sched = f.sched;
    p.n_items = f.n_items;
    if (rqs8) return launch_fused_t<ZK_UNI_RQS, 8>(p, a.fast_math, grid, smem, st);
    if (rqs16) return launch_fused_t<ZK_UNI_RQS, 16>(p, a.fast_math, grid, smem, st);
    return launch_fused_t<ZK_UNI_AFFINE, 0>(p, a.fast_math, grid, smem, st);
}

}  // namespace zk
