// zuko_b200 — ONE kernel per flow layer for conditioners of hidden width 128 / 256 (BASELINE cfg2:
// NSF(16, 8, K8, [256]^3)), with TWO sample tiles in flight per CTA.
//
// Same contract and the same CTA-pair machinery as fused_wide.cu (tcgen05.mma.cta_group::2, A hi in
// tensor memory, A lo in shared memory, weights streamed as half tiles, in-place descending schedule;
// flows/autoregressive.py:207-215, nn.py:217-218, transforms.py:469-490, 554-567, 426-446, 210-214,
// distributions.py:115-119).  What is different is what the timelines of the one-tile kernels showed
// (profiles/r01_fused_timeline_v14.txt, r02_wide_timeline_cfg2.txt): with only two 128-column chunks
// per hidden layer there is nothing to hide a chunk's epilogue behind — the tensor pipe waits for the
// epilogue at every chunk, the epilogue warps wait for the tensor pipe in between, and during the
// spline evaluation of the output layer the pipe idles altogether (tensor pipe ~50 % active).
// A 256-wide activation row needs only half of the tensor / shared memory the 512-wide layout
// reserves, so each CTA keeps TWO 128-row sub-tiles resident:
//
//   tensor memory   [  0,128) A hi of sub-tile 0   [128,256) A hi of sub-tile 1
//                   [256,384) accumulator of sub-tile 0   [384,512) accumulator of sub-tile 1
//   shared memory   A lo: 2 x 4 K blocks x 16 KB | W ring | barriers, partials | bias, base table
//   epilogue warps  4..11 own sub-tile 0, 12..19 own sub-tile 1 (2 sets x 4 TMEM lane quadrants each)
//
// and the issue schedule alternates the two sub-tiles chunk by chunk: while the group of sub-tile 0
// drains and rewrites a chunk, the pipe multiplies the chunk of sub-tile 1, and the schedule simply
// wraps into the next 512-row pair tile — there is no point at which the whole CTA waits.
//
// Warp roles as in fused_wide.cu: warp 0 W producer (both CTAs), warp 1 MMA issuer and warp 2 scout
// (leader CTA), warps 4-19 epilogue.

#include <algorithm>

#include "activations.cuh"
#include "fused_common.cuh"
#include "pair_common.cuh"

namespace zk {

namespace {

using namespace bij;

constexpr int DM = 128;             // rows per CTA and sub-tile (256 per pair and sub-tile, 512 per pair tile)
constexpr int DK = 64;              // bf16 per K block
constexpr int D_MAXKB = 4;          // A operand of one sub-tile: up to 4 K blocks = 256 columns
constexpr int D_EPI_WARP0 = 4;
constexpr int D_GROUP_WARPS = 8;    // epilogue warps per sub-tile
constexpr int D_THREADS = (D_EPI_WARP0 + 2 * D_GROUP_WARPS) * 32;  // 640
constexpr uint32_t D_ALO_BYTES = 2 * D_MAXKB * W_APLANE;           // 128 KB
constexpr uint32_t D_WPLANE = 64 * DK * 2;                         // 8 KB: this CTA's half of one plane of a W tile
constexpr uint32_t D_WSTAGE = 2 * D_WPLANE;
constexpr int D_MAX_WSTAGES = 8;
constexpr uint32_t D_BAR_SLOTS = 40;                               // 36 mbarriers + tmem slot / s_ready
constexpr uint32_t D_AUX_BYTES = D_BAR_SLOTS * 8 + 2 * 2 * DM * 4; // + ladj partials [sub-tile][parity][128]
constexpr uint32_t D_SMEM_MAX = 232448;
constexpr uint32_t TMD_D = 256;                                    // first accumulator column

// schedule entries: pair_common.cuh (S = 2: bits [1:0] are the K block, bit 2 the sub-tile)
constexpr uint32_t DS_FIRST = WS_FIRST, DS_LAST = WS_LAST, DS_AWAIT = WS_AWAIT, DS_AFREE = WS_AFREE, DS_OUT = WS_OUT;

struct DualParams {
    CUtensorMap mapW[ZK_FUSED_MAX_LINEAR];
    const float* bias[ZK_FUSED_MAX_LINEAR];
    int bias_off[ZK_FUSED_MAX_LINEAR];
    int bias_len[ZK_FUSED_MAX_LINEAR];
    uint32_t rd_mask[ZK_FUSED_MAX_LINEAR];  // K blocks (of one sub-tile) layer l reads
    const uint2* sched;
    int n_items;        // entries of one pair tile (both sub-tiles)
    int n_linear;
    int K0, KB0;
    int H, nch_hidden;  // hidden width (128 / 256), H / 128
    int D, C;
    int n_last_chunks;
    int n_terms;
    int M;
    int in_vec;
    int n_wstages;
    int base_off;
    int act;            // activation between the linear layers: 1 = ReLU, else ZK_ACT_* (GACT instantiation)
    const float* x; int64_t ldx;
    const float* c; int64_t ldc;
    float* y; int64_t ldy;
    float* ladj; int accumulate;
    float* log_prob; const float* base_loc; const float* base_scale;
    float bound, aw, ad;
    long long* dbg;
    uint32_t* watch;
};

template <int UNI, int KT, bool FAST, bool DBG, bool GACT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(D_THREADS, 1)
fused_dual_kernel(const __grid_constant__ DualParams p) {
    using Cfg = LastCfg<UNI, KT>;
    constexpr int P = Cfg::P, DPC = Cfg::DPC;
    constexpr int N_LAST = (DPC * P + 15) & ~15;
    constexpr int NLH = N_LAST / 2;
    static_assert(N_LAST <= 128 && NLH % 8 == 0, "an output-layer chunk must fit one accumulator buffer");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int NW = p.n_wstages;
    uint8_t* sAlo = smem;                      // block index = 4 sub-tile + kb
    uint8_t* sW = smem + D_ALO_BYTES;
    uint64_t* bars = (uint64_t*)(sW + (size_t)NW * D_WSTAGE);
    uint64_t* w_full = bars;        // [8]  leader's
    uint64_t* w_empty = bars + 8;   // [8]  each CTA its own
    uint64_t* d_full = bars + 16;   // [2]  per sub-tile, each CTA its own
    uint64_t* d_empty = bars + 18;  // [2]  per sub-tile, leader's: 2 x 8 epilogue warps
    uint64_t* a_ready = bars + 20;  // [8]  index 4 sub-tile + kb, leader's: 2 x 8 epilogue warps
    uint64_t* a_free = bars + 28;   // [8]  index 4 sub-tile + kb, each CTA its own
    uint32_t* tmem_slot = (uint32_t*)(bars + 36);
    uint32_t* s_ready = tmem_slot + 2;  // [0] entries whose operands are ready, [1] entries whose weights landed (two scouts -> issuer)
    float* s_part = (float*)(bars + D_BAR_SLOTS);  // [2 sub-tiles][2 parities][128]
    float* s_bias = (float*)((uint8_t*)bars + D_AUX_BYTES);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int L = p.n_linear;
    const uint32_t rank = cluster_ctarank();
    const int cid = blockIdx.x >> 1, ncl = gridDim.x >> 1;
    const int pair_tiles = (p.M + 4 * DM - 1) / (4 * DM);  // 512 rows per pair tile
    const int n_iter = (pair_tiles - cid + ncl - 1) / ncl;
    const int n_items = p.n_items;
    const int total = n_iter * n_items;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NW; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&d_full[b], 1); mbar_init(&d_empty[b], 2 * D_GROUP_WARPS); }
        for (int k = 0; k < 8; ++k) { mbar_init(&a_ready[k], 2 * D_GROUP_WARPS); mbar_init(&a_free[k], 1); }
        s_ready[0] = 0u;
        s_ready[1] = 0u;
        fence_mbar_init();
    }
    for (int l = 0; l < L; ++l)
        if (p.bias_off[l] >= 0)
            for (int i = threadIdx.x; i < p.bias_len[l]; i += D_THREADS) s_bias[p.bias_off[l] + i] = p.bias[l][i];
    if (p.log_prob != nullptr)
        for (int d = threadIdx.x; d < p.D; d += D_THREADS) {
            const float sg = p.base_scale ? p.base_scale[d] : 1.f;
            s_bias[p.base_off + d] = p.base_loc ? p.base_loc[d] : 0.f;
            s_bias[p.base_off + p.D + d] = 1.f / sg;
            s_bias[p.base_off + 2 * p.D + d] = logf(sg) + kHalfLog2Pi;
        }
    if (warp == 2) tmem_alloc2(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
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
                const int kb = (int)(e.x & 3u), l = (int)((e.x >> 16) & 7u);
                const uint32_t rows = (e.x & DS_OUT) ? (uint32_t)NLH : 64u;
                WD_SPIN(mbar_try_wait(&w_empty[ws], wph ^ 1u), 0x10, i, ws);
                if (rank == 0) mbar_arrive_expect_tx(&w_full[ws], 2u * planes * rows * 128u);
                uint8_t* st = sW + (size_t)ws * D_WSTAGE;
                const int n0 = (int)e.y + (int)(rows * rank);
                tma_load_3d_2sm(st, &p.mapW[l], full0 + 8u * (uint32_t)ws, kb * DK, n0, 0);
                if (planes == 2u) tma_load_3d_2sm(st + D_WPLANE, &p.mapW[l], full0 + 8u * (uint32_t)ws, kb * DK, n0, 1);
                if constexpr (DBG)
                    if (p.dbg != nullptr && blockIdx.x == 0 && (i / n_items == min(2, n_iter - 1)) && j < 64) p.dbg[448 + j] = clock64();
                if (++j == n_items) j = 0;
                if (++ws == NW) { ws = 0; wph ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ======================= MMA issuer (leader CTA) =======================
        if (rank == 0) {
            const uint32_t idesc_h = umma_idesc_bf16(2 * DM, 128), idesc_o = umma_idesc_bf16(2 * DM, N_LAST);
            int ws = 0, j = 0;
            uint32_t seen = 0, seen_w = 0;  // cached s_ready[0] / s_ready[1]
            uint32_t cur = (total > 0) ? __ldg(&p.sched[0].x) : 0u;
            for (int i = 0; i < total; ++i) {
                const bool stamp_on = DBG && (i / n_items == min(2, n_iter - 1)) && (lane == 0);
                const int jn = (j + 1 == n_items) ? 0 : j + 1;
                const uint32_t nxt = __ldg(&p.sched[jn].x);
                const uint32_t kb = cur & 3u, u = (cur >> 2) & 1u, kb8 = 4u * u + kb;
                const uint32_t d_tmem = TMD_D + u * 128u;
                const uint32_t a_hi = u * 128u + kb * (uint32_t)(DK / 2);
                const uint32_t w_addr = smem_u32(sW) + (uint32_t)ws * D_WSTAGE;
                const uint64_t dw_hi = umma_desc_k_sw128(w_addr), dw_lo = umma_desc_k_sw128(w_addr + D_WPLANE);
                const uint64_t da_lo = umma_desc_k_sw128(smem_u32(sAlo) + kb8 * W_APLANE);
                const uint32_t idesc = (cur & DS_OUT) ? idesc_o : idesc_h;
                const bool first = (cur & DS_FIRST) != 0;
                {
                    uint32_t _n = 0;
                    long long _t0 = 0;
                    while (seen <= (uint32_t)i || seen_w <= (uint32_t)i) {
                        if (seen <= (uint32_t)i)
                            asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(seen) : "r"(smem_u32(s_ready)) : "memory");
                        if (seen_w <= (uint32_t)i)
                            asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(seen_w) : "r"(smem_u32(s_ready + 1)) : "memory");
                        if ((++_n & 4095u) == 0u) {
                            const long long _t = clock64();
                            if (_t0 == 0) _t0 = _t;
                            else if (_t - _t0 > W_WD_CYCLES) wd_report(p.watch, 0x20, i, (seen << 16) | (seen_w & 0xffffu));
                        }
                    }
                }
                tc_fence_after();
                const int nk = 4 - (int)((cur >> 20) & 3u);
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < DK / 16; ++k) {
                        if (k >= nk) break;
                        const uint32_t acol = (uint32_t)k * 8u;
                        umma2_bf16_ts(d_tmem, a_hi + acol, umma_desc_advance(dw_hi, k), idesc, (!first || k > 0) ? 1u : 0u);
                        if (p.n_terms == 3) {
                            umma2_bf16_ts(d_tmem, a_hi + acol, umma_desc_advance(dw_lo, k), idesc, 1u);
                            umma2_bf16_ss(d_tmem, umma_desc_advance(da_lo, k), umma_desc_advance(dw_hi, k), idesc, 1u);
                        }
                    }
                    umma2_commit_mc(&w_empty[ws]);
                    if (cur & DS_AFREE) umma2_commit_mc(&a_free[kb8]);
                    if (cur & DS_LAST) umma2_commit_mc(&d_full[u]);
                }
                __syncwarp();
                if constexpr (DBG)
                    if (p.dbg != nullptr && blockIdx.x == 0 && stamp_on && j < 64) p.dbg[256 + j] = clock64();
                cur = nxt;
                j = jn;
                if (++ws == NW) ws = 0;
            }
        }
    } else if (warp == 2) {
        // ======================= operand scout (leader CTA) =======================
        // A probe of an mbarrier costs ~300 cycles even when its phase completed long ago (one scout doing up
        // to three probes per entry published one entry per ~1000 cycles, less than the tensor pipe consumes;
        // DESIGN.md 5b).  So two lanes in two warps walk the schedule
        // independently, each with its own parity state: this one waits for what the EPILOGUE produces
        // (accumulator drained, A blocks written), warp 3 for what the TMA produces (weights landed);
        // the issuer reads both counters.
        if (rank == 0 && lane == 0) {
            int j = 0;
            uint32_t a_par = 0;              // bit (4 u + kb) = parity of a_ready
            uint32_t cnt[2] = {0u, 0u};      // chunks issued so far per sub-tile (its accumulator is single-buffered)
            for (int i = 0; i < total; ++i) {
                const uint32_t it = __ldg(&p.sched[j].x);
                const uint32_t u = (it >> 2) & 1u;
                if (it & DS_FIRST) {  // the k-th chunk of a sub-tile needs k drains of its accumulator
                    WD_SPIN(mbar_try_wait_cluster(&d_empty[u], (cnt[u] & 1u) ^ 1u), 0x30, i, cnt[u]);
                    ++cnt[u];
                }
                if (it & 0xFF00u) {
                    for (uint32_t k2 = 0; k2 < 8u; ++k2)
                        if ((it >> (8 + k2)) & 1u) {
                            WD_SPIN(mbar_try_wait_cluster(&a_ready[k2], (a_par >> k2) & 1u), 0x31, i, k2);
                            a_par ^= 1u << k2;
                        }
                }
                if (it & DS_AWAIT) {
                    const uint32_t kb8 = 4u * u + (it & 3u);
                    WD_SPIN(mbar_try_wait_cluster(&a_ready[kb8], (a_par >> kb8) & 1u), 0x32, i, kb8);
                    a_par ^= 1u << kb8;
                }
                asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(smem_u32(s_ready)), "r"((uint32_t)(i + 1)) : "memory");
                if constexpr (DBG)
                    if (p.dbg != nullptr && blockIdx.x == 0 && (i / n_items == min(2, n_iter - 1)) && j < 64) p.dbg[384 + j] = clock64();
                if (++j == n_items) j = 0;
            }
        }
    } else if (warp == 3) {
        // ======================= weight scout (leader CTA) =======================
        if (rank == 0 && lane == 0) {
            int ws = 0;
            uint32_t wph = 0;
            for (int i = 0; i < total; ++i) {
                WD_SPIN(mbar_try_wait_cluster(&w_full[ws], wph), 0x33, i, ws);
                asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(smem_u32(s_ready + 1)), "r"((uint32_t)(i + 1)) : "memory");
                if constexpr (DBG)
                    if (p.dbg != nullptr && blockIdx.x == 0 && (i / n_items == min(2, n_iter - 1)) && (i % n_items) < 64) p.dbg[320 + (i % n_items)] = clock64();
                if (++ws == NW) { ws = 0; wph ^= 1u; }
            }
        }
    } else if (warp >= D_EPI_WARP0) {
        // ======================= epilogue: group u = sub-tile u (both CTAs) =======================
        const int u = (warp - D_EPI_WARP0) >> 3;        // sub-tile / group
        const int s = ((warp - D_EPI_WARP0) >> 2) & 1;  // set inside the group: 64 columns of a hidden chunk
        const int q = warp & 3;                         // TMEM lane quadrant
        const int r = q * 32 + lane;
        const uint32_t t_lane = ((uint32_t)(q * 32) << 16);
        const uint32_t a_col0 = (uint32_t)u * 128u;     // this sub-tile's A hi columns
        const uint32_t d_col0 = TMD_D + (uint32_t)u * 128u;
        const uint32_t d_empty_r = mapa_rank0(smem_u32(d_empty)) + 8u * (uint32_t)u;
        const uint32_t a_ready_r = mapa_rank0(smem_u32(a_ready)) + 32u * (uint32_t)u;  // + 8 kb
        uint64_t* const my_d_full = &d_full[u];
        uint64_t* const my_a_free = &a_free[4 * u];
        uint32_t chunk = 0, f_par = 0;  // chunk: chunks of this sub-tile so far; f_par: bit kb = parity of a_free[4 u + kb]
        for (int tile_iter = 0; tile_iter < n_iter; ++tile_iter) {
            const int64_t pt = (int64_t)cid + (int64_t)tile_iter * ncl;
            const bool stamp_on = (tile_iter == min(2, n_iter - 1)) && (threadIdx.x == (D_EPI_WARP0 + 8 * u) * 32);
            const int sbase = 128 * u;  // stamp slots of this group
            W_STAMP(sbase + 0);
            const int64_t row = pt * (4 * DM) + (int64_t)u * (2 * DM) + (int64_t)rank * DM + r;
            const bool row_ok = row < p.M;
            const float* xrow = p.x + (row_ok ? row : 0) * p.ldx;
            // ---- stage the layer-0 operand of this sub-tile; set s takes the half blocks hb = s, s + 2, ... ----
            {
                const float* crow = (p.C == 0) ? xrow : (p.c + (row_ok ? row : 0) * p.ldc);
                const int kx = row_ok ? p.D : 0, kc = row_ok ? p.K0 : 0;
                for (int hb = s; hb < 2 * p.KB0; hb += 2) {
                    uint32_t ph[16], pl[16];
                    if (p.in_vec) {
                        const float4* x4 = reinterpret_cast<const float4*>(xrow);
                        const float4* c4 = reinterpret_cast<const float4*>(crow);
                        const int d4 = kx >> 2, k4 = kc >> 2;
#pragma unroll
                        for (int v = 0; v < 8; ++v) {
                            const int i4 = hb * 8 + v;
                            float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (i4 < d4) t = __ldg(x4 + i4);
                            else if (i4 < k4) t = __ldg(c4 + (i4 - (p.D >> 2)));
                            split2_bf16(t.x, t.y, ph[2 * v], pl[2 * v]);
                            split2_bf16(t.z, t.w, ph[2 * v + 1], pl[2 * v + 1]);
                        }
                    } else {
#pragma unroll
                        for (int v = 0; v < 16; ++v) {
                            const int k = hb * 32 + 2 * v;
                            const float v0 = (k < kx) ? __ldg(xrow + k) : ((k < kc) ? __ldg(crow + k - p.D) : 0.f);
                            const float v1 = (k + 1 < kx) ? __ldg(xrow + k + 1) : ((k + 1 < kc) ? __ldg(crow + k + 1 - p.D) : 0.f);
                            split2_bf16(v0, v1, ph[v], pl[v]);
                        }
                    }
                    tmem_st_x16(t_lane + a_col0 + (uint32_t)(hb * 16), ph);
                    st_alo32(sAlo, 4 * u + (hb >> 1), r, hb & 1, pl);
                }
            }
            tmem_st_wait();
            fence_proxy_async();
            tc_fence_before();
            __syncwarp();
            if (lane == 0)
                for (int kb = 0; kb < p.KB0; ++kb) mbar_arrive_cluster(a_ready_r + 8u * (uint32_t)kb);
            W_STAMP(sbase + 1);

            // ---- hidden layers: D -> bias, ReLU -> hi / lo -> next A operand, in place; set s owns 64 columns ----
            for (int l = 0; l < L - 1; ++l) {
                const float* bias = (p.bias_off[l] >= 0) ? s_bias + p.bias_off[l] : p.bias[l];
                const uint32_t rd = p.rd_mask[l];
                for (int ch = p.nch_hidden - 1; ch >= 0; --ch, ++chunk) {
                    WD_SPIN(mbar_try_wait(my_d_full, chunk & 1u), 0x40, (uint32_t)(l * 16 + ch), chunk);
                    tc_fence_after();
                    if (l < 4) W_STAMP(sbase + 8 + 8 * l + 2 * ch);
                    const int nbase = ch * 128 + s * 64;  // first output column of this thread = K index of the next layer
                    // All 64 columns of the set are pulled first and the accumulator is released BEFORE the
                    // arithmetic (ReLU only): the next chunk of this sub-tile waits for this arrive, and four
                    // load / wait / convert rounds took ~1.4 k cycles (profiles/r02_dual_timeline_recapture.txt).
                    uint32_t ph[32], pl[32];
                    if constexpr (!GACT) {
                        uint32_t ra[64];
#pragma unroll
                        for (int g = 0; g < 4; ++g) tmem_ld_x16(t_lane + d_col0 + (uint32_t)(s * 64 + 16 * g), ra + 16 * g);
                        tmem_ld_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive_cluster(d_empty_r);  // this sub-tile's accumulator is drained
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            const float4* b4 = reinterpret_cast<const float4*>(bias + nbase + 16 * g);
#pragma unroll
                            for (int j = 0; j < 16; j += 4) {
                                const float4 bb = b4[j >> 2];
                                split2_bf16(fmaxf(__uint_as_float(ra[16 * g + j]) + bb.x, 0.f), fmaxf(__uint_as_float(ra[16 * g + j + 1]) + bb.y, 0.f),
                                            ph[8 * g + (j >> 1)], pl[8 * g + (j >> 1)]);
                                split2_bf16(fmaxf(__uint_as_float(ra[16 * g + j + 2]) + bb.z, 0.f), fmaxf(__uint_as_float(ra[16 * g + j + 3]) + bb.w, 0.f),
                                            ph[8 * g + (j >> 1) + 1], pl[8 * g + (j >> 1) + 1]);
                            }
                        }
                    } else {
#pragma unroll
                        for (int g = 0; g < 4; ++g) {  // four groups of 16 columns
                            const float4* b4 = reinterpret_cast<const float4*>(bias + nbase + 16 * g);
                            uint32_t ra[16];
                            tmem_ld_x16(t_lane + d_col0 + (uint32_t)(s * 64 + 16 * g), ra);
                            tmem_ld_wait();
                            float v[16];  // any ZK_ACT_* (nn.py:264-265): one switch per 16 columns
#pragma unroll
                            for (int j = 0; j < 16; j += 4) {
                                const float4 bb = b4[j >> 2];
                                v[j] = __uint_as_float(ra[j]) + bb.x; v[j + 1] = __uint_as_float(ra[j + 1]) + bb.y;
                                v[j + 2] = __uint_as_float(ra[j + 2]) + bb.z; v[j + 3] = __uint_as_float(ra[j + 3]) + bb.w;
                            }
                            if constexpr (FAST) act_apply_n_fast<16>(v, p.act); else act_apply_n<16>(v, p.act);
#pragma unroll
                            for (int j = 0; j < 16; j += 2) split2_bf16(v[j], v[j + 1], ph[8 * g + (j >> 1)], pl[8 * g + (j >> 1)]);
                        }
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive_cluster(d_empty_r);  // this sub-tile's accumulator is drained
                    }
                    if (l < 4) W_STAMP(sbase + 100 + 2 * l + ch);
                    for (int kb = 2 * ch; kb < 2 * ch + 2; ++kb)
                        if ((rd >> kb) & 1u) {
                            WD_SPIN(mbar_try_wait(&my_a_free[kb], (f_par >> kb) & 1u), 0x41, (uint32_t)(l * 16 + ch), kb);
                            f_par ^= (1u << kb);
                        }
                    tc_fence_after();
                    tmem_st_x16(t_lane + a_col0 + (uint32_t)(nbase >> 1), ph);
                    tmem_st_x16(t_lane + a_col0 + (uint32_t)(nbase >> 1) + 16u, ph + 16);
                    st_alo32(sAlo, 4 * u + (nbase >> 6), r, 0, pl);       // the set's 64 columns are one whole K block
                    st_alo32(sAlo, 4 * u + (nbase >> 6), r, 1, pl + 16);
                    tmem_st_wait();
                    fence_proxy_async();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        mbar_arrive_cluster(a_ready_r + 8u * (uint32_t)(2 * ch));
                        mbar_arrive_cluster(a_ready_r + 8u * (uint32_t)(2 * ch + 1));
                    }
                    if (l < 4) W_STAMP(sbase + 8 + 8 * l + 2 * ch + 1);
                }
            }

            // ---- output layer: raw parameters stay in TMEM -> bijector + ladj in registers ----
            float lsum = 0.f;
            const float* bias = (p.bias_off[L - 1] >= 0) ? s_bias + p.bias_off[L - 1] : p.bias[L - 1];
            for (int ch = p.n_last_chunks - 1; ch >= 0; --ch, ++chunk) {
                WD_SPIN(mbar_try_wait(my_d_full, chunk & 1u), 0x42, (uint32_t)ch, chunk);
                tc_fence_after();
                if (ch < 20) W_STAMP(sbase + 48 + 2 * ch);
                const uint32_t td = t_lane + d_col0;
                auto release = [&]() {  // warp-uniform call sites only
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_cluster(d_empty_r);
                };
                auto finish_dim = [&](int d, float yv, float lj) {
                    if (p.y) p.y[row * p.ldy + d] = yv;
                    if (p.log_prob) {
                        const float* bt = s_bias + p.base_off + d;
                        const float uu = (yv - bt[0]) * bt[p.D];
                        lj += -0.5f * uu * uu - bt[2 * p.D];
                    }
                    lsum += lj;
                };
                if constexpr (UNI == ZK_UNI_RQS) {
                    // the set's dims of this chunk: DPC = 4 -> dims 2 s, 2 s + 1; DPC = 2 -> dim s
                    constexpr int DPS = DPC / 2;
                    static_assert(DPS == 1 || DPS == 2, "dims per set");
                    float pp[DPS][P];
                    auto pull = [&](auto dloc_c, auto slot_c) {
                        constexpr int dloc = decltype(dloc_c)::value, slot = decltype(slot_c)::value;
                        constexpr int c_lo = dloc * P, c_hi = c_lo + P;
                        constexpr int w0 = c_lo & ~15;
                        constexpr int wn = ((c_hi - w0) + 15) & ~15;
                        static_assert(wn <= 64 && w0 + wn <= 128, "window out of range");
                        uint32_t rr[wn];
                        tmem_ld_x16(td + (uint32_t)w0, rr);
                        if constexpr (wn > 16) tmem_ld_x16(td + (uint32_t)(w0 + 16), rr + 16);
                        if constexpr (wn > 32) tmem_ld_x16(td + (uint32_t)(w0 + 32), rr + 32);
                        if constexpr (wn > 48) tmem_ld_x16(td + (uint32_t)(w0 + 48), rr + 48);
                        tmem_ld_wait();
                        const int d = ch * DPC + dloc;
                        const float* bd = bias + (d < p.D ? d : 0) * P;
#pragma unroll
                        for (int j = 0; j < P; ++j) pp[slot][j] = __uint_as_float(rr[c_lo - w0 + j]) + bd[j];
                    };
                    auto eval = [&](int dloc, int slot) {
                        const int d = ch * DPC + dloc;
                        if (d >= p.D || !row_ok) return;
                        const float xv = __ldg(xrow + d);
                        float yv, lj;
                        Bin b = rqs_select<KT, FAST, false>(pp[slot], KT, xv, p.bound, p.aw, p.ad);
                        rqs_forward_eval<FAST>(b, xv, yv, lj);
                        finish_dim(d, yv, lj);
                    };
                    if constexpr (DPS == 2) {
                        if (s == 0) {
                            pull(std::integral_constant<int, 0>{}, std::integral_constant<int, 0>{});
                            pull(std::integral_constant<int, 1>{}, std::integral_constant<int, 1>{});
                        } else {
                            pull(std::integral_constant<int, 2>{}, std::integral_constant<int, 0>{});
                            pull(std::integral_constant<int, 3>{}, std::integral_constant<int, 1>{});
                        }
                        release();
                        eval(2 * s, 0);
                        eval(2 * s + 1, 1);
                    } else {
                        if (s == 0) pull(std::integral_constant<int, 0>{}, std::integral_constant<int, 0>{});
                        else pull(std::integral_constant<int, 1>{}, std::integral_constant<int, 0>{});
                        release();
                        eval(s, 0);
                    }
                } else {
                    // affine: 8 groups of 8 dims (16 columns each); set s takes the groups s, s + 2, s + 4, s + 6
                    static_assert(DPC == 64, "affine chunk layout");
                    const int nd = min(DPC, p.D - ch * DPC);
#pragma unroll 1
                    for (int gi = 0; gi < 4; ++gi) {
                        const int g = s + 2 * gi;
                        const bool live = g * 8 < nd;  // warp-uniform
                        uint32_t rr[16];
                        if (live) {
                            tmem_ld_x16(td + (uint32_t)(g * 16), rr);
                            tmem_ld_wait();
                        }
                        if (gi == 3) release();  // after the set's last read of the accumulator
                        if (!live || !row_ok) continue;
                        const int d0 = ch * DPC + g * 8;
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const int d = d0 + j;
                            if (d < p.D) {
                                const float shift = __uint_as_float(rr[2 * j]) + bias[2 * d];
                                const float ls = softclip<FAST>(__uint_as_float(rr[2 * j + 1]) + bias[2 * d + 1], p.ad);
                                finish_dim(d, fmaf(__ldg(xrow + d), zexp<FAST>(ls), shift), ls);
                            }
                        }
                    }
                }
                if (ch < 20) W_STAMP(sbase + 49 + 2 * ch);
            }
            // this sub-tile's A operand may be restaged once every MMA of the output layer that reads it is complete
            {
                const uint32_t rd = p.rd_mask[L - 1];
                for (int kb = 0; kb < D_MAXKB; ++kb)
                    if ((rd >> kb) & 1u) {
                        WD_SPIN(mbar_try_wait(&my_a_free[kb], (f_par >> kb) & 1u), 0x43, (uint32_t)tile_iter, kb);
                        f_par ^= (1u << kb);
                    }
                tc_fence_after();
            }
            // ---- per-sample sum: set 0 hands its partial to set 1 of the same group (named barrier 1 + u) ----
            float* part = s_part + (u * 2 + (tile_iter & 1)) * DM;
            if (s == 0) {
                part[r] = lsum;
                __threadfence_block();
                asm volatile("bar.arrive %0, 256;" ::"r"(1 + u) : "memory");
            } else {
                asm volatile("bar.sync %0, 256;" ::"r"(1 + u) : "memory");
                if (row_ok) {
                    const float tot = lsum + part[r] + (p.accumulate ? p.ladj[row] : 0.f);
                    if (p.log_prob) p.log_prob[row] = tot;
                    else if (p.ladj) p.ladj[row] = tot;
                }
            }
            W_STAMP(sbase + 2);
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc2(0u, 512);
    }
}

template <int UNI, int KT>
zk_status launch_dual_t(const DualParams& p, bool fast, int grid, size_t smem, cudaStream_t st) {
    auto go = [&](auto kern) -> zk_status {
        ZK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)D_SMEM_MAX));
        kern<<<grid, D_THREADS, smem, st>>>(p);
        return check_launch("fused_dual_kernel");
    };
    if (p.act != 1) return fast ? go(fused_dual_kernel<UNI, KT, true, false, true>) : go(fused_dual_kernel<UNI, KT, false, false, true>);
    if (p.dbg != nullptr) return fast ? go(fused_dual_kernel<UNI, KT, true, true, false>) : go(fused_dual_kernel<UNI, KT, false, true, false>);
    if (fast) return go(fused_dual_kernel<UNI, KT, true, false, false>);
    return go(fused_dual_kernel<UNI, KT, false, false, false>);
}

}  // namespace

zk_status launch_fused_dual(const zk_mlp* m, const FusedLayerArgs& a, cudaStream_t st) {
    const TcPack* pk = (const TcPack*)m->tc;
    ZK_REQUIRE(pk, "fused dual layer: no tensor-core pack");
    const WidePack& wp = pk->dual;
    ZK_REQUIRE(wp.built_for(a.univariate, a.bins, a.D, a.C) && wp.sched,
               "fused dual layer: the conditioner was not prepared for this bijector");
    ZK_REQUIRE(a.B < ((int64_t)1 << 31) - 4 * DM, "fused dual layer: batch too large for one launch");
    if (a.B == 0) return ZK_OK;
    DualParams p;
    pair_fill_params(p, m, wp, a);
    const uint32_t avail = D_SMEM_MAX - 1024u - D_ALO_BYTES - D_AUX_BYTES;
    p.n_wstages = (int)std::min<uint32_t>(D_MAX_WSTAGES, avail / D_WSTAGE);
    uint32_t bias_room = (avail - (uint32_t)p.n_wstages * D_WSTAGE) / 4u;
    int need_floats = a.log_prob ? ((3 * a.D + 3) & ~3) : 0;
    for (int l = 0; l < m->n_linear; ++l) need_floats += (m->dims[l + 1] + 3) & ~3;
    while ((uint32_t)need_floats > bias_room && p.n_wstages > 3) { --p.n_wstages; bias_room += D_WSTAGE / 4u; }  // biases first
    ZK_REQUIRE(p.n_wstages >= 3, "fused dual layer: not enough shared memory for the weight ring");
    uint32_t copy_floats = 0;
    ZK_TRY(pair_place_biases(p, m, a, bias_room, "fused dual layer", copy_floats));
    const size_t smem = 1024u + D_ALO_BYTES + (size_t)p.n_wstages * D_WSTAGE + D_AUX_BYTES + (size_t)copy_floats * 4u;
    p.watch = pair_watch_device();
    const int64_t pairs = ceil_div(a.B, 4 * DM);
    const int grid = 2 * (int)std::min<int64_t>(pairs, sm_count() / 2);
    const bool rqs8 = a.univariate == ZK_UNI_RQS && a.bins == 8, rqs16 = a.univariate == ZK_UNI_RQS && a.bins == 16;
    if (rqs8) return launch_dual_t<ZK_UNI_RQS, 8>(p, a.fast_math, grid, smem, st);
    if (rqs16) return launch_dual_t<ZK_UNI_RQS, 16>(p, a.fast_math, grid, smem, st);
    return launch_dual_t<ZK_UNI_AFFINE, 0>(p, a.fast_math, grid, smem, st);
}

}  // namespace zk
