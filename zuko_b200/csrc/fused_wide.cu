// zuko_b200 — ONE kernel per flow layer for conditioners of hidden width 384 / 512
// (BASELINE cfg3 MAF [512]^4 and cfg5 NSF [512]^3 / K16, the 8-GPU north-star config).
//
// Same contract as fused_layer.cu (flows/autoregressive.py:207-215, nn.py:217-218,
// transforms.py:469-490, 554-567, 426-446, 210-214, distributions.py:115-119): cat(x, c) -> every
// masked linear layer on tcgen05 (split bf16, fp32 accumulate) -> bijector + ladj (+ DiagNormal
// log-prob) evaluated straight from the accumulator; hidden activations and phi never reach HBM.
//
// What is different: a 512-wide activation row in bf16 hi + lo planes is 2 KB, i.e. a 128-row tile
// fills the whole tensor memory of an SM (512 columns) and leaves no room for accumulators.  So
//   * the two CTAs of a cluster form ONE MMA unit (tcgen05.mma.cta_group::2, M = 256): each CTA keeps
//     its own 128 rows, and holds only HALF of every weight tile in shared memory (the tensor core
//     reads the other half from the peer) — half the weight ring per byte of math, which frees
//   * 128 KB of shared memory for the A operand's LO plane (K-major, 128-byte swizzle, written by
//     the epilogue threads, read by the MMA through a shared-memory descriptor), while
//   * the HI plane (used by two of the three split products) stays in tensor memory [0, 256) and
//     the two 128-column accumulator buffers take [256, 512).
//   * hidden layers are updated IN PLACE: hidden units are sorted by dependency degree (pack time),
//     so the masked matrices are block lower-triangular, and chunks / K blocks are walked in
//     DESCENDING order: the chunk of the highest degrees reads every K block first, after which
//     nobody reads the top K blocks again and its own outputs (the next layer's top K blocks) can
//     overwrite them, and so on down.  The next layer starts with the K blocks that were written
//     first, so the tensor pipe does not drain at layer boundaries.  The order and every barrier
//     obligation are a table built (and dry-run for deadlocks) on the host: fused_plan.cu.
//
// Tensor memory (512 columns x 128 lanes, lane = sample row of this CTA's half tile):
//   [  0,256)  A hi : bf16 pairs, K element k in column k/2                     (K <= 512)
//   [256,384)  D buffer 0 (fp32 accumulators of one <= 128-column chunk)
//   [384,512)  D buffer 1
// Shared memory (per CTA): A lo (H / 64) x 16 KB | W ring n x 16 KB (64 rows x 64 K x hi, lo) | barriers,
//   ladj partials | bias copy.
//
// Hidden width 256 (BASELINE cfg2) runs here as well: the narrow kernel (fused_layer.cu) multicasts
// FULL weight tiles to both CTAs of a pair and reads all three split products' B operand from its own
// shared memory — 64 B/clk of operand reads plus 42 B/clk of TMA writes, against the 128 B/clk the
// shared memory delivers: its K blocks take ~1250 cycles instead of 768 (profiles/
// r01_fused_timeline_v14.txt).  The pair-MMA form halves both.
//
// Warp roles (640 threads, 1 CTA / SM, persistent over 256-row pair tiles):
//   warp 0      W producer (both CTAs: each loads its half tile; completion counted on the LEADER's barrier)
//   warp 1      MMA issuer (leader CTA only)
//   warp 2      TMEM allocator; scout (leader only: waits for every prerequisite of a schedule entry)
//   warp 3      idle
//   warps 4-19  epilogue (both CTAs; their "buffer drained" / "A block written" arrivals go to the
//               leader's barriers through the cluster shared-memory window)

#include <algorithm>

#include "activations.cuh"
#include "fused_common.cuh"
#include "pair_common.cuh"

namespace zk {

namespace {

using namespace bij;

constexpr int WM = 128;             // rows per CTA (256 per pair tile)
constexpr int WK = 64;              // bf16 per K block (128-byte swizzle row)
constexpr int W_MAXKB = 8;          // A operand: up to 8 K blocks = 512 columns
constexpr int W_EPI_WARP0 = 4;
constexpr int W_EPI_WARPS = 16;
constexpr int W_THREADS = (W_EPI_WARP0 + W_EPI_WARPS) * 32;   // 640
constexpr uint32_t W_ALO_BYTES = W_MAXKB * W_APLANE;          // 128 KB
constexpr uint32_t W_WPLANE = 64 * WK * 2;                    // 8 KB: this CTA's half of one plane of a W tile
constexpr uint32_t W_WSTAGE = 2 * W_WPLANE;                   // hi + lo
constexpr int W_MAX_WSTAGES = 8;
constexpr uint32_t W_BAR_SLOTS = 40;                          // 36 mbarriers + tmem slot / s_ready
constexpr uint32_t W_AUX_BYTES = W_BAR_SLOTS * 8 + 2 * 3 * WM * 4;  // + ladj partials [2][3][128]
constexpr uint32_t W_SMEM_MAX = 232448;                       // 227 KB per CTA on sm_100
constexpr uint32_t TMW_D = 256;                               // first accumulator column

// schedule entries: pair_common.cuh (S = 1: bits [2:0] are the K block)

struct WideParams {
    CUtensorMap mapW[ZK_FUSED_MAX_LINEAR];
    const float* bias[ZK_FUSED_MAX_LINEAR];
    int bias_off[ZK_FUSED_MAX_LINEAR];  // offset of layer l's bias in the shared-memory copy, -1: read from global
    int bias_len[ZK_FUSED_MAX_LINEAR];
    uint32_t rd_mask[ZK_FUSED_MAX_LINEAR];  // K blocks of the A operand layer l reads
    const uint2* sched;
    int n_items;
    int n_linear;
    int K0, KB0;        // real input width (D + C) and its number of 64-wide K blocks
    int H, nch_hidden;  // hidden width (384 / 512), H / 128
    int D, C;
    int n_last_chunks;  // ceil(D / DPC)
    int n_terms;        // 3 (split bf16) or 1
    int M;
    int in_vec;         // x / c rows can be read with 16-byte loads
    int n_wstages;
    int alo_blocks;     // K blocks of the A lo plane kept in shared memory: max(KB0, H / 64)
    int act;            // activation between the linear layers: 1 = ReLU, else ZK_ACT_* (GACT instantiation)
    int base_off;       // offset (floats, after the bias copy) of the base table [3][D]: loc, 1/scale, log scale + log sqrt(2 pi)
    const float* x; int64_t ldx;
    const float* c; int64_t ldc;
    float* y; int64_t ldy;
    float* ladj; int accumulate;
    float* log_prob; const float* base_loc; const float* base_scale;
    float bound, aw, ad;
    long long* dbg;   // optional timeline buffer (clock64 stamps of CTA 0), see zk_debug_timeline
    uint32_t* watch;  // watchdog report buffer (mapped host memory) or null
};

template <int UNI, int KT, bool FAST, bool DBG, bool GACT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(W_THREADS, 1)
fused_wide_kernel(const __grid_constant__ WideParams p) {
    using Cfg = LastCfg<UNI, KT>;
    constexpr int P = Cfg::P, DPC = Cfg::DPC;
    constexpr int N_LAST = (DPC * P + 15) & ~15;  // MMA N of an output-layer chunk
    constexpr int NLH = N_LAST / 2;               // rows of an output-layer W tile held by each CTA
    static_assert(N_LAST <= 128 && NLH % 8 == 0, "an output-layer chunk must fit one accumulator buffer");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int NW = p.n_wstages;
    uint8_t* sAlo = smem;
    uint8_t* sW = smem + (size_t)p.alo_blocks * W_APLANE;
    uint64_t* bars = (uint64_t*)(sW + (size_t)NW * W_WSTAGE);
    uint64_t* w_full = bars;        // [8]  (leader's copy is the one in use)
    uint64_t* w_empty = bars + 8;   // [8]  each CTA its own (multicast commit)
    uint64_t* d_full = bars + 16;   // [2]  each CTA its own (multicast commit)
    uint64_t* d_empty = bars + 18;  // [2]  leader's: 2 x 16 epilogue warps
    uint64_t* a_ready = bars + 20;  // [8]  leader's: 2 x 16 epilogue warps; K block kb of the A operand written
    uint64_t* a_free = bars + 28;   // [8]  each CTA its own: every MMA of the current layer reading K block kb is complete
    uint32_t* tmem_slot = (uint32_t*)(bars + 36);
    uint32_t* s_ready = tmem_slot + 1;  // schedule entries whose prerequisites are all met (scout -> issuer)
    float* s_part = (float*)(bars + W_BAR_SLOTS);  // [2][3][128] ladj partials of sets 0..2
    float* s_bias = (float*)((uint8_t*)bars + W_AUX_BYTES);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int L = p.n_linear;
    const uint32_t rank = cluster_ctarank();
    const int cid = blockIdx.x >> 1, ncl = gridDim.x >> 1;
    const int pair_tiles = (p.M + 2 * WM - 1) / (2 * WM);
    const int n_iter = (pair_tiles - cid + ncl - 1) / ncl;  // identical in both CTAs of the pair
    const int n_items = p.n_items;
    const int total = n_iter * n_items;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NW; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&d_full[b], 1); mbar_init(&d_empty[b], 2 * W_EPI_WARPS); }
        for (int k = 0; k < W_MAXKB; ++k) { mbar_init(&a_ready[k], 2 * W_EPI_WARPS); mbar_init(&a_free[k], 1); }
        *s_ready = 0u;
        fence_mbar_init();
    }
    for (int l = 0; l < L; ++l)
        if (p.bias_off[l] >= 0)
            for (int i = threadIdx.x; i < p.bias_len[l]; i += W_THREADS) s_bias[p.bias_off[l] + i] = p.bias[l][i];
    if (p.log_prob != nullptr)  // DiagNormal terms (torch normal.py:87-102) hoisted out of the per-dim epilogue
        for (int d = threadIdx.x; d < p.D; d += W_THREADS) {
            const float sg = p.base_scale ? p.base_scale[d] : 1.f;
            s_bias[p.base_off + d] = p.base_loc ? p.base_loc[d] : 0.f;
            s_bias[p.base_off + p.D + d] = 1.f / sg;
            s_bias[p.base_off + 2 * p.D + d] = logf(sg) + kHalfLog2Pi;
        }
    if (warp == 2) tmem_alloc2(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // both CTAs' barriers are initialised before any remote arrive / multicast commit
    tc_fence_after();
    // the whole tensor memory is allocated: base = lane 0 / column 0 (literal addresses keep every
    // tcgen05 operand in uniform registers, see fused_layer.cu)
    if (*tmem_slot != 0u) __trap();

    if (warp == 0) {
        // ======================= W producer (both CTAs) =======================
        if (lane == 0) {
            const uint32_t full0 = smem_u32(w_full) & 0xFEFFFFFFu;  // the leader CTA's w_full[0]
            const uint32_t planes = (p.n_terms == 3) ? 2u : 1u;
            int ws = 0, j = 0;
            uint32_t wph = 0;
            for (int i = 0; i < total; ++i) {
                const uint2 e = __ldg(p.sched + j);
                const int kb = (int)(e.x & 7u), l = (int)((e.x >> 16) & 7u);
                const uint32_t rows = (e.x & WS_OUT) ? (uint32_t)NLH : 64u;
                WD_SPIN(mbar_try_wait(&w_empty[ws], wph ^ 1u), 0x10, i, ws);
                // each CTA fetches rows [n0 + rows rank, + rows) — its half of the pair's N columns
                if (rank == 0) mbar_arrive_expect_tx(&w_full[ws], 2u * planes * rows * 128u);
                uint8_t* st = sW + (size_t)ws * W_WSTAGE;
                const int n0 = (int)e.y + (int)(rows * rank);
                tma_load_3d_2sm(st, &p.mapW[l], full0 + 8u * (uint32_t)ws, kb * WK, n0, 0);
                if (planes == 2u) tma_load_3d_2sm(st + W_WPLANE, &p.mapW[l], full0 + 8u * (uint32_t)ws, kb * WK, n0, 1);
                if (++j == n_items) j = 0;
                if (++ws == NW) { ws = 0; wph ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ======================= MMA issuer (leader CTA) =======================
        // One instruction drives both SMs of the pair: D rows [0,128) live in this CTA's tensor memory,
        // rows [128,256) in the peer's; each CTA supplies its own A rows and half of the B columns.
        if (rank == 0) {
            const uint32_t idesc_h = umma_idesc_bf16(2 * WM, 128), idesc_o = umma_idesc_bf16(2 * WM, N_LAST);
            int ws = 0, j = 0;
            uint32_t c = 0, seen = 0;  // c: running chunk counter (accumulator buffer = c & 1); seen: cached *s_ready
            uint32_t cur = (total > 0) ? __ldg(&p.sched[0].x) : 0u;
            for (int i = 0; i < total; ++i) {
                const bool stamp_on = DBG && (i / n_items == min(2, n_iter - 1)) && (lane == 0);
                const int jn = (j + 1 == n_items) ? 0 : j + 1;
                const uint32_t nxt = __ldg(&p.sched[jn].x);
                const uint32_t kb = cur & 7u, buf = c & 1u;
                const uint32_t d_tmem = TMW_D + buf * 128u;
                const uint32_t a_hi = kb * (uint32_t)(WK / 2);
                const uint32_t w_addr = smem_u32(sW) + (uint32_t)ws * W_WSTAGE;
                const uint64_t dw_hi = umma_desc_k_sw128(w_addr), dw_lo = umma_desc_k_sw128(w_addr + W_WPLANE);
                const uint64_t da_lo = umma_desc_k_sw128(smem_u32(sAlo) + kb * W_APLANE);
                const uint32_t idesc = (cur & WS_OUT) ? idesc_o : idesc_h;
                const bool first = (cur & WS_FIRST) != 0;
                {
                    uint32_t _n = 0;
                    long long _t0 = 0;
                    while (seen <= (uint32_t)i) {
                        asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(seen) : "r"(smem_u32(s_ready)) : "memory");
                        if ((++_n & 4095u) == 0u) {
                            const long long _t = clock64();
                            if (_t0 == 0) _t0 = _t;
                            else if (_t - _t0 > W_WD_CYCLES) wd_report(p.watch, 0x20, i, seen);
                        }
                    }
                }
                tc_fence_after();
                const int nk = 4 - (int)((cur >> 20) & 3u);
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < WK / 16; ++k) {
                        if (k >= nk) break;
                        const uint32_t acol = (uint32_t)k * 8u;  // 16 bf16 = 8 TMEM columns
                        umma2_bf16_ts(d_tmem, a_hi + acol, umma_desc_advance(dw_hi, k), idesc, (!first || k > 0) ? 1u : 0u);
                        if (p.n_terms == 3) {
                            umma2_bf16_ts(d_tmem, a_hi + acol, umma_desc_advance(dw_lo, k), idesc, 1u);
                            umma2_bf16_ss(d_tmem, umma_desc_advance(da_lo, k), umma_desc_advance(dw_hi, k), idesc, 1u);
                        }
                    }
                    umma2_commit_mc(&w_empty[ws]);             // the ring slot is free again in both CTAs
                    if (cur & WS_AFREE) umma2_commit_mc(&a_free[kb]);  // last read of A block kb in this layer
                    if (cur & WS_LAST) umma2_commit_mc(&d_full[buf]);
                }
                __syncwarp();
                if constexpr (DBG)
                    if (p.dbg != nullptr && blockIdx.x == 0 && stamp_on && j < 256) p.dbg[256 + j] = clock64();
                c += (nxt >> 3) & 1u;
                cur = nxt;
                j = jn;
                if (++ws == NW) ws = 0;
            }
        }
    } else if (warp == 2) {
        // ======================= scout (leader CTA) =======================
        if (rank == 0 && lane == 0) {
            int ws = 0, j = 0;
            uint32_t wph = 0, c = 0, a_par = 0;  // a_par: bit kb = parity of a_ready[kb]
            for (int i = 0; i < total; ++i) {
                const uint32_t it = __ldg(&p.sched[j].x);
                if (i > 0) c += (it >> 3) & 1u;
                if (it & WS_FIRST) WD_SPIN(mbar_try_wait_cluster(&d_empty[c & 1u], ((c >> 1) & 1u) ^ 1u), 0x30, i, c);
                if (it & 0xFF00u) {  // A blocks written for this layer that it never reads: consume their phase
                    for (uint32_t k2 = 0; k2 < (uint32_t)W_MAXKB; ++k2)
                        if ((it >> (8 + k2)) & 1u) {
                            WD_SPIN(mbar_try_wait_cluster(&a_ready[k2], (a_par >> k2) & 1u), 0x31, i, k2);
                            a_par ^= 1u << k2;
                        }
                }
                if (it & WS_AWAIT) {
                    const uint32_t kb = it & 7u;
                    WD_SPIN(mbar_try_wait_cluster(&a_ready[kb], (a_par >> kb) & 1u), 0x32, i, kb);
                    a_par ^= 1u << kb;
                }
                WD_SPIN(mbar_try_wait_cluster(&w_full[ws], wph), 0x33, i, ws);
                asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(smem_u32(s_ready)), "r"((uint32_t)(i + 1)) : "memory");
                if (++j == n_items) j = 0;
                if (++ws == NW) { ws = 0; wph ^= 1u; }
            }
        }
    } else if (warp >= W_EPI_WARP0) {
        // ======================= epilogue (both CTAs) =======================
        const int s = (warp - W_EPI_WARP0) >> 2;  // warp set 0..3
        const int q = warp & 3;                   // TMEM lane quadrant
        const int r = q * 32 + lane;              // row inside this CTA's half tile
        const uint32_t t_lane = ((uint32_t)(q * 32) << 16);
        const uint32_t d_empty_r = mapa_rank0(smem_u32(d_empty));  // the leader's barriers
        const uint32_t a_ready_r = mapa_rank0(smem_u32(a_ready));
        uint32_t chunk = 0, f_par = 0;  // f_par: bit kb = parity of a_free[kb]
        for (int tile_iter = 0; tile_iter < n_iter; ++tile_iter) {
            const int64_t pt = (int64_t)cid + (int64_t)tile_iter * ncl;
            const bool stamp_on = (tile_iter == min(2, n_iter - 1)) && (threadIdx.x == W_EPI_WARP0 * 32);
            W_STAMP(0);
            const int64_t row = pt * (2 * WM) + (int64_t)rank * WM + r;
            const bool row_ok = row < p.M;
            const float* xrow = p.x + (row_ok ? row : 0) * p.ldx;
            // ---- stage the layer-0 operand: cat(x, c) -> bf16 hi (tensor memory) / lo (shared memory);
            //      set s takes the 32-input half blocks hb = s, s + 4, ... ----
            {
                const float* crow = (p.C == 0) ? xrow : (p.c + (row_ok ? row : 0) * p.ldc);
                const int kx = row_ok ? p.D : 0, kc = row_ok ? p.K0 : 0;  // masked rows stage zeros
                for (int hb = s; hb < 2 * p.KB0; hb += 4) {
                    uint32_t ph[16], pl[16];
                    if (p.in_vec) {
                        const float4* x4 = reinterpret_cast<const float4*>(xrow);
                        const float4* c4 = reinterpret_cast<const float4*>(crow);
                        const int d4 = kx >> 2, k4 = kc >> 2;
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const int i4 = hb * 8 + u;
                            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (i4 < d4) v = __ldg(x4 + i4);
                            else if (i4 < k4) v = __ldg(c4 + (i4 - (p.D >> 2)));
                            split2_bf16(v.x, v.y, ph[2 * u], pl[2 * u]);
                            split2_bf16(v.z, v.w, ph[2 * u + 1], pl[2 * u + 1]);
                        }
                    } else {
#pragma unroll
                        for (int u = 0; u < 16; ++u) {
                            const int k = hb * 32 + 2 * u;
                            const float v0 = (k < kx) ? __ldg(xrow + k) : ((k < kc) ? __ldg(crow + k - p.D) : 0.f);
                            const float v1 = (k + 1 < kx) ? __ldg(xrow + k + 1) : ((k + 1 < kc) ? __ldg(crow + k + 1 - p.D) : 0.f);
                            split2_bf16(v0, v1, ph[u], pl[u]);
                        }
                    }
                    tmem_st_x16(t_lane + (uint32_t)(hb * 16), ph);
                    st_alo32(sAlo, hb >> 1, r, hb & 1, pl);
                }
            }
            tmem_st_wait();
            fence_proxy_async();  // the lo plane was written through the generic proxy, the MMA reads it through the async proxy
            tc_fence_before();
            __syncwarp();
            if (lane == 0)
                for (int kb = 0; kb < p.KB0; ++kb) mbar_arrive_cluster(a_ready_r + 8u * (uint32_t)kb);
            W_STAMP(1);

            // ---- hidden layers: D -> bias, ReLU -> hi / lo -> next A operand, in place ----
            for (int l = 0; l < L - 1; ++l) {
                const float* bias = (p.bias_off[l] >= 0) ? s_bias + p.bias_off[l] : p.bias[l];
                const uint32_t rd = p.rd_mask[l];
                for (int ch = p.nch_hidden - 1; ch >= 0; --ch, ++chunk) {
                    const uint32_t buf = chunk & 1u;
                    WD_SPIN(mbar_try_wait(&d_full[buf], (chunk >> 1) & 1u), 0x40, (uint32_t)(l * 16 + ch), chunk);
                    tc_fence_after();
                    if (l < 4) W_STAMP(8 + 8 * l + 2 * ch);
                    const int nbase = ch * 128 + s * 32;  // first output column of this thread = K index of the next layer
                    uint32_t ph[16], pl[16];
                    {
                        const float4* b4 = reinterpret_cast<const float4*>(bias + nbase);  // 128-byte aligned
#pragma unroll
                        for (int half = 0; half < 2; ++half) {
                            uint32_t ra[16];
                            tmem_ld_x16(t_lane + TMW_D + buf * 128u + (uint32_t)(s * 32 + 16 * half), ra);
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
                                const float4 bb = b4[4 * half + (j >> 2)];
                                split2_bf16(fmaxf(__uint_as_float(ra[j]) + bb.x, 0.f), fmaxf(__uint_as_float(ra[j + 1]) + bb.y, 0.f),
                                            ph[8 * half + (j >> 1)], pl[8 * half + (j >> 1)]);
                                split2_bf16(fmaxf(__uint_as_float(ra[j + 2]) + bb.z, 0.f), fmaxf(__uint_as_float(ra[j + 3]) + bb.w, 0.f),
                                            ph[8 * half + (j >> 1) + 1], pl[8 * half + (j >> 1) + 1]);
                            }
                            }
                        }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_cluster(d_empty_r + 8u * buf);  // accumulator buffer drained
                    // the K blocks this chunk overwrites must have been read by every MMA of this layer
                    for (int kb = 2 * ch; kb < 2 * ch + 2; ++kb)
                        if ((rd >> kb) & 1u) {
                            WD_SPIN(mbar_try_wait(&a_free[kb], (f_par >> kb) & 1u), 0x41, (uint32_t)(l * 16 + ch), kb);
                            f_par ^= (1u << kb);
                        }
                    tc_fence_after();
                    tmem_st_x16(t_lane + (uint32_t)(nbase >> 1), ph);  // K element k lives in column k / 2
                    st_alo32(sAlo, nbase >> 6, r, (nbase >> 5) & 1, pl);
                    tmem_st_wait();
                    fence_proxy_async();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        mbar_arrive_cluster(a_ready_r + 8u * (uint32_t)(2 * ch));
                        mbar_arrive_cluster(a_ready_r + 8u * (uint32_t)(2 * ch + 1));
                    }
                    if (l < 4) W_STAMP(8 + 8 * l + 2 * ch + 1);
                }
            }

            // ---- output layer: raw parameters stay in TMEM -> bijector + ladj in registers ----
            float lsum = 0.f;
            const float* bias = (p.bias_off[L - 1] >= 0) ? s_bias + p.bias_off[L - 1] : p.bias[L - 1];
            for (int ch = p.n_last_chunks - 1; ch >= 0; --ch, ++chunk) {
                const uint32_t buf = chunk & 1u;
                WD_SPIN(mbar_try_wait(&d_full[buf], (chunk >> 1) & 1u), 0x42, (uint32_t)ch, chunk);
                tc_fence_after();
                if (ch < 40) W_STAMP(80 + 2 * ch);
                // SPC sets share a chunk (all four when it holds >= 4 dims, else the set pairs alternate
                // chunks).  Every thread first pulls the raw parameters of its dims out of tensor memory
                // and releases the accumulator buffer, THEN evaluates.
                constexpr int SPC = (DPC >= 4) ? 4 : 2;
                const bool mine = (SPC == 4) || ((int)buf == (s >> 1));
                const int h = (SPC == 4) ? s : (s & 1);  // which share of the chunk's dims
                const uint32_t td = t_lane + TMW_D + buf * 128u;
                auto release = [&]() {  // warp-uniform call sites only
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_cluster(d_empty_r + 8u * buf);
                };
                auto finish_dim = [&](int d, float yv, float lj) {
                    if (p.y) p.y[row * p.ldy + d] = yv;
                    if (p.log_prob) {
                        const float* bt = s_bias + p.base_off + d;
                        const float u = (yv - bt[0]) * bt[p.D];
                        lj += -0.5f * u * u - bt[2 * p.D];
                    }
                    lsum += lj;
                };
                if constexpr (UNI == ZK_UNI_RQS) {
                    static_assert(DPC == SPC, "one dim per set and chunk");
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
                        const float xv = __ldg(xrow + d);
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
                    // affine: 8 dims (16 columns: shift, scale pairs) per load; set h takes the groups
                    // h and h + 4 of the chunk's 8 groups (D = 32: one group per set, all 16 warps busy)
                    static_assert(SPC == 4 && DPC == 64, "affine chunk layout");
                    const int nd = min(DPC, p.D - ch * DPC);  // dims of this chunk
                    const bool g1 = (h + 4) * 8 < nd;         // the second group holds real dims
                    uint32_t rr[2][16];
                    tmem_ld_x16(td + (uint32_t)(h * 16), rr[0]);
                    if (g1) tmem_ld_x16(td + (uint32_t)((h + 4) * 16), rr[1]);
                    tmem_ld_wait();
                    release();
                    if (row_ok) {
#pragma unroll
                        for (int g = 0; g < 2; ++g) {
                            if (g == 1 && !g1) break;
                            const int d0 = ch * DPC + (h + 4 * g) * 8;
                            float xv[8];
                            if (p.in_vec) {  // D % 4 == 0 and 16-byte aligned rows: the group's 8 x values in two loads
                                const float4 a = (d0 < p.D) ? __ldg(reinterpret_cast<const float4*>(xrow + d0)) : make_float4(0.f, 0.f, 0.f, 0.f);
                                const float4 b = (d0 + 4 < p.D) ? __ldg(reinterpret_cast<const float4*>(xrow + d0 + 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
                                xv[0] = a.x; xv[1] = a.y; xv[2] = a.z; xv[3] = a.w; xv[4] = b.x; xv[5] = b.y; xv[6] = b.z; xv[7] = b.w;
                            } else {
#pragma unroll
                                for (int j = 0; j < 8; ++j) xv[j] = (d0 + j < p.D) ? __ldg(xrow + d0 + j) : 0.f;
                            }
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const int d = d0 + j;
                                if (d < p.D) {
                                    const float shift = __uint_as_float(rr[g][2 * j]) + bias[2 * d];
                                    const float ls = softclip<FAST>(__uint_as_float(rr[g][2 * j + 1]) + bias[2 * d + 1], p.ad);
                                    finish_dim(d, fmaf(xv[j], zexp<FAST>(ls), shift), ls);
                                }
                            }
                        }
                    }
                }
                if (ch < 40) W_STAMP(81 + 2 * ch);
            }
            // the A operand may be restaged once every MMA of the output layer that reads it is complete
            {
                const uint32_t rd = p.rd_mask[L - 1];
                for (int kb = 0; kb < W_MAXKB; ++kb)
                    if ((rd >> kb) & 1u) {
                        WD_SPIN(mbar_try_wait(&a_free[kb], (f_par >> kb) & 1u), 0x43, (uint32_t)tile_iter, kb);
                        f_par ^= (1u << kb);
                    }
                tc_fence_after();
            }
            // ---- per-sample sum: sets 0..2 hand their partials to set 3 without waiting for it ----
            float* part = s_part + (tile_iter & 1) * (3 * WM);
            if (s < 3) {
                part[s * WM + r] = lsum;
                __threadfence_block();
                asm volatile("bar.arrive 1, 512;" ::: "memory");
            } else {
                asm volatile("bar.sync 1, 512;" ::: "memory");
                if (row_ok) {
                    const float tot = lsum + part[r] + part[WM + r] + part[2 * WM + r] + (p.accumulate ? p.ladj[row] : 0.f);
                    if (p.log_prob) p.log_prob[row] = tot;
                    else if (p.ladj) p.ladj[row] = tot;
                }
            }
            W_STAMP(2);
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // no CTA leaves (or frees its tensor memory) while the pair's MMAs may still touch it
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc2(0u, 512);
    }
}

template <int UNI, int KT>
zk_status launch_wide_t(const WideParams& p, bool fast, int grid, size_t smem, cudaStream_t st) {
    auto go = [&](auto kern) -> zk_status {
        ZK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)W_SMEM_MAX));
        kern<<<grid, W_THREADS, smem, st>>>(p);
        return check_launch("fused_wide_kernel");
    };
    if (p.act != 1) return fast ? go(fused_wide_kernel<UNI, KT, true, false, true>) : go(fused_wide_kernel<UNI, KT, false, false, true>);
    if (p.dbg != nullptr) return fast ? go(fused_wide_kernel<UNI, KT, true, true, false>) : go(fused_wide_kernel<UNI, KT, false, true, false>);
    if (fast) return go(fused_wide_kernel<UNI, KT, true, false, false>);
    return go(fused_wide_kernel<UNI, KT, false, false, false>);
}

}  // namespace

zk_status launch_fused_wide(const zk_mlp* m, const FusedLayerArgs& a, cudaStream_t st) {
    const TcPack* pk = (const TcPack*)m->tc;
    ZK_REQUIRE(pk && fused_wide_shape(m, a.univariate, a.bins, a.D, a.C), "fused wide layer: unsupported shape");
    const WidePack& wp = pk->wide;
    ZK_REQUIRE(wp.built_for(a.univariate, a.bins, a.D, a.C) && wp.sched,
               "fused wide layer: the conditioner was not prepared for this bijector");
    ZK_REQUIRE(a.B < ((int64_t)1 << 31) - 2 * WM, "fused wide layer: batch too large for one launch");
    if (a.B == 0) return ZK_OK;
    WideParams p;
    pair_fill_params(p, m, wp, a);
    // shared memory: A lo + aux are fixed; the weight ring gets what is left after the bias copy of
    // the OUTPUT layer and as many hidden-layer biases as still fit
    p.alo_blocks = std::max(p.KB0, p.H / WK);
    const uint32_t alo_bytes = (uint32_t)p.alo_blocks * W_APLANE;
    const uint32_t avail = W_SMEM_MAX - 1024u - alo_bytes - W_AUX_BYTES;
    p.n_wstages = (int)std::min<uint32_t>(W_MAX_WSTAGES, avail / W_WSTAGE);
    uint32_t bias_room = (avail - (uint32_t)p.n_wstages * W_WSTAGE) / 4u;  // floats
    if (bias_room < 64u && p.n_wstages > 4) { --p.n_wstages; bias_room += W_WSTAGE / 4u; }
    ZK_REQUIRE(p.n_wstages >= 3, "fused wide layer: not enough shared memory for the weight ring");
    uint32_t copy_floats = 0;
    ZK_TRY(pair_place_biases(p, m, a, bias_room, "fused wide layer", copy_floats));
    const size_t smem = 1024u + alo_bytes + (size_t)p.n_wstages * W_WSTAGE + W_AUX_BYTES + (size_t)copy_floats * 4u;
    p.watch = pair_watch_device();
    const int64_t pairs = ceil_div(a.B, 2 * WM);
    const int grid = 2 * (int)std::min<int64_t>(pairs, sm_count() / 2);
    const bool rqs8 = a.univariate == ZK_UNI_RQS && a.bins == 8, rqs16 = a.univariate == ZK_UNI_RQS && a.bins == 16;
    if (rqs8) return launch_wide_t<ZK_UNI_RQS, 8>(p, a.fast_math, grid, smem, st);
    if (rqs16) return launch_wide_t<ZK_UNI_RQS, 16>(p, a.fast_math, grid, smem, st);
    return launch_wide_t<ZK_UNI_AFFINE, 0>(p, a.fast_math, grid, smem, st);
}

}  // namespace zk
