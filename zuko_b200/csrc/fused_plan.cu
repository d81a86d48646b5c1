// zuko_b200 — host-side planning of the fused layer kernels (no device code): the degree permutation
// of the hidden units, the (chunk, K block) tile map all three kernels skip all-zero tiles by, and for
// the CTA-pair kernels (fused_wide.cu: S = 1 sub-tile per CTA, fused_dual.cu: S = 2) their shape test,
// the descending issue schedule, the dry run of its barrier protocol and the pack that carries it.

#include <string.h>

#include <algorithm>
#include <atomic>

#include "fused_common.cuh"
#include "pair_common.cuh"

namespace zk {

std::atomic<int> g_dual{1};           // zk_set_dual_tiles
std::atomic<int> g_wide_min_h{256};   // smallest hidden width routed to the wide kernel (zk_set_wide_min_hidden)
uint32_t* g_watch_host = nullptr;     // mapped pinned host memory the pair kernels' watchdog reports into

// Dependency degree of every hidden unit = number of network inputs it can see
// (flows/autoregressive.py:121-124 + nn.py:270-293: units of a lower order class see fewer inputs);
// sorting by degree makes the hidden -> hidden masks block lower-triangular.
void fused_degree_perm(const int* dims, int L, const std::vector<std::vector<uint8_t>>& Mk,
                       std::vector<std::vector<int>>& perm) {
    const int K0 = dims[0];
    perm.assign(L - 1, {});  // perm[l][new] = old index of hidden layer l+1's units
    // dependency sets as bit rows: dep[unit] = OR of the dep rows of the inputs it is connected to
    const int W64 = (K0 + 63) / 64;
    std::vector<uint64_t> prev, cur;
    for (int l = 0; l < L - 1; ++l) {
        const int K = dims[l], N = dims[l + 1];
        cur.assign((size_t)N * W64, 0);
        for (int n = 0; n < N; ++n) {
            uint64_t* dn = &cur[(size_t)n * W64];
            const uint8_t* mrow = &Mk[l][(size_t)n * K];
            for (int k = 0; k < K; ++k) {
                if (!mrow[k]) continue;
                if (l == 0) dn[k >> 6] |= (uint64_t)1 << (k & 63);
                else {
                    const uint64_t* dk = &prev[(size_t)k * W64];
                    for (int w = 0; w < W64; ++w) dn[w] |= dk[w];
                }
            }
        }
        std::vector<int> deg(N, 0);
        for (int n = 0; n < N; ++n)
            for (int w = 0; w < W64; ++w) deg[n] += __builtin_popcountll(cur[(size_t)n * W64 + w]);
        perm[l].resize(N);
        for (int n = 0; n < N; ++n) perm[l][n] = n;
        std::stable_sort(perm[l].begin(), perm[l].end(), [&](int a, int b) { return deg[a] < deg[b]; });
        prev.swap(cur);
    }
}

FusedTileMap fused_tile_map(const int* dims, int L, const std::vector<std::vector<uint8_t>>& Mk,
                            const std::vector<std::vector<int>>& perm, int cw, int univariate, int bins, int D) {
    const int P = fused_p(univariate, bins), DPC = fused_dpc(univariate, bins);
    FusedTileMap tm;
    tm.kbmask.resize(L);
    tm.kmax.resize(L);
    for (int l = 0; l < L; ++l) {
        const bool last = (l == L - 1);
        const int K = dims[l], N = dims[l + 1];
        const int nch = last ? (D + DPC - 1) / DPC : dims[1] / cw;
        const int rows = last ? DPC * P : cw;
        tm.kbmask[l].assign(nch, 0);
        tm.kmax[l].assign((size_t)nch * 8, 0);
        for (int ch = 0; ch < nch; ++ch) {
            const int n0 = ch * rows, n1 = std::min(N, n0 + rows);
            int* kmax = &tm.kmax[l][(size_t)ch * 8];
            uint32_t bits = 0;
            for (int n = n0; n < n1; ++n) {
                const int sn = (l < L - 1) ? perm[l][n] : n;
                const uint8_t* mrow = &Mk[l][(size_t)sn * K];
                for (int k = 0; k < K; ++k) {
                    const int sk = (l > 0) ? perm[l - 1][k] : k;
                    if (mrow[sk]) {
                        bits |= 1u << (k / 64);
                        kmax[k / 64] = std::max(kmax[k / 64], k % 64);
                    }
                }
            }
            if (bits == 0) bits = 1;  // the accumulator still has to be defined (bias-only outputs)
            tm.kbmask[l][ch] = bits;
        }
    }
    return tm;
}

// ---------------------------------------------------------------------------
// CTA-pair kernels
// ---------------------------------------------------------------------------

// Shapes the pair kernels take, routing knobs aside: all hidden widths equal, a multiple of 128 between
// half and all of one sub-tile's A operand (512 / S columns), and an input that fits that operand.
static bool pair_dims_ok(const int* dims, int L, int univariate, int bins, int D, int C, int S) {
    if (L < 2 || L > ZK_FUSED_MAX_LINEAR) return false;
    const int H = dims[1], max_k = 512 / S;
    if (H % 128 != 0 || H < max_k / 2 || H > max_k) return false;
    for (int i = 1; i < L; ++i)
        if (dims[i] != H) return false;
    if (D + C > max_k || dims[0] != D + C) return false;
    if (univariate == ZK_UNI_RQS) return bins == 8 || bins == 16;
    return univariate == ZK_UNI_AFFINE;
}

static bool pair_shape(const zk_mlp* m, int univariate, int bins, int D, int C, int S) {
    const TcPack* pk = (const TcPack*)m->tc;
    if (!pk || m->gemm_mode == ZK_GEMM_FP32) return false;
    if (!m->plain) return false;  // residual blocks need the input of two layers back, which the in-place update overwrote
    return pair_dims_ok(m->dims.data(), m->n_linear, univariate, bins, D, C, S);
}

bool fused_wide_shape(const zk_mlp* m, int univariate, int bins, int D, int C) {
    return pair_shape(m, univariate, bins, D, C, 1) && m->dims[1] >= g_wide_min_h.load();
}

bool fused_dual_shape(const zk_mlp* m, int univariate, int bins, int D, int C) {
    return g_dual.load() && pair_shape(m, univariate, bins, D, C, 2);
}

namespace {

struct PairShape {
    int S, L, nch, KB0, KBH, n_last;
};

// One agent of a dry-run interleaving: the MMA side (PAIR_MMA) or epilogue group g, run until it blocks
// (greedy) or for one step per round.
constexpr int PAIR_MMA = -1;
struct DryAgent {
    int agent;
    bool greedy;
};
using DryPolicy = std::vector<DryAgent>;

// The interleavings each kernel's schedule must survive, each agent in the listed order per round.
// S = 1: MMA side greedy, then epilogue greedy.  S = 2: MMA side greedy; both epilogue groups greedy;
// group 1 greedy; group 0 greedy (the agents not named greedy take one step per round).
const std::vector<DryPolicy>& pair_policies(int S) {
    static const std::vector<DryPolicy> one = {
        {{PAIR_MMA, true}, {0, false}},
        {{0, true}, {PAIR_MMA, false}},
    };
    static const std::vector<DryPolicy> two = {
        {{PAIR_MMA, true}, {0, false}, {1, false}},
        {{0, true}, {1, true}, {PAIR_MMA, false}},
        {{1, true}, {PAIR_MMA, false}, {0, false}},
        {{0, true}, {PAIR_MMA, false}, {1, false}},
    };
    return S == 1 ? one : two;
}

// One pair tile's work as the kernel walks it, three tiles back to back (MMA completions immediate),
// under the barrier protocol of the kernel: a schedule that can deadlock, or lets a barrier run two
// phases ahead of its waiter (parity aliasing), is rejected and the layer stays on the per-layer path.
// A blocks are numbered u * (8 / S) + kb as in the schedule; epilogue group u owns sub-tile u and
// 2 / S of the two accumulator buffers, which it takes in turn, chunk by chunk.
bool pair_dry_run(const std::vector<uint2>& items, const uint32_t* rd_mask, const PairShape& sh, const DryPolicy& policy) {
    const int n = (int)items.size();
    const int TILES = 3;
    const int NA = 8 / sh.S, NB = 2 / sh.S;  // A blocks and accumulator buffers per group
    // completed phases
    int d_full[2] = {0, 0}, d_empty[2] = {0, 0}, a_ready[8] = {0}, a_free[8] = {0};
    // phases seen by the waiter
    int d_full_seen[2] = {0, 0}, d_empty_seen[2] = {0, 0}, a_ready_seen[8] = {0}, a_free_seen[8] = {0};
    bool ok = true;
    auto complete = [&](int* done, const int* seen, int idx) {
        if (done[idx] != seen[idx]) ok = false;  // the waiter has not consumed the previous phase yet
        done[idx]++;
    };
    // ---- MMA side (scout + issuer) ----
    int mi = 0;
    int chunks[2] = {0, 0};  // chunks started per group
    auto mma_step = [&]() -> bool {
        if (mi >= TILES * n) return false;
        const uint32_t it = items[mi % n].x;
        const int a = (int)(it & 7u), g = a / NA;
        const int k = (it & WS_FIRST) ? chunks[g] : chunks[g] - 1;  // the group's chunk this entry belongs to
        const int buf = g * NB + k % NB;
        // the k-th chunk of a group is the (k / NB)-th use of its buffer: it needs k / NB drains
        if ((it & WS_FIRST) && d_empty[buf] < k / NB) return false;
        for (int k2 = 0; k2 < 8; ++k2)
            if (((it >> (8 + k2)) & 1u) && a_ready[k2] <= a_ready_seen[k2]) return false;
        if ((it & WS_AWAIT) && a_ready[a] <= a_ready_seen[a]) return false;
        // all prerequisites met: consume and issue (MMAs complete in order, at once)
        if (it & WS_FIRST) { d_empty_seen[buf] = k / NB; ++chunks[g]; }
        for (int k2 = 0; k2 < 8; ++k2)
            if ((it >> (8 + k2)) & 1u) a_ready_seen[k2]++;
        if (it & WS_AWAIT) a_ready_seen[a]++;
        if (it & WS_AFREE) complete(a_free, a_free_seen, a);
        if (it & WS_LAST) complete(d_full, d_full_seen, buf);
        ++mi;
        return true;
    };
    // ---- epilogue groups: a flat list of steps each ----
    enum { STAGE, WAIT_FULL, DRAIN, WAIT_FREE, WRITE };
    struct Step { int kind, a, b; };  // WAIT_FULL(buf, phases), DRAIN(buf), WAIT_FREE(A block), WRITE(first of two A blocks)
    std::vector<Step> steps[2];
    for (int g = 0; g < sh.S; ++g) {
        const int a0 = g * NA;
        int k = 0;
        auto chunk = [&](std::vector<Step>& s) {
            const int buf = g * NB + k % NB;
            s.push_back({WAIT_FULL, buf, k / NB + 1});
            s.push_back({DRAIN, buf, 0});
            ++k;
        };
        for (int t = 0; t < TILES; ++t) {
            steps[g].push_back({STAGE, a0, 0});
            for (int l = 0; l < sh.L - 1; ++l)
                for (int ch = sh.nch - 1; ch >= 0; --ch) {
                    chunk(steps[g]);
                    for (int kb = 2 * ch; kb < 2 * ch + 2; ++kb)
                        if ((rd_mask[l] >> kb) & 1u) steps[g].push_back({WAIT_FREE, a0 + kb, 0});
                    steps[g].push_back({WRITE, a0 + 2 * ch, 0});
                }
            for (int ch = sh.n_last - 1; ch >= 0; --ch) chunk(steps[g]);
            for (int kb = 0; kb < NA; ++kb)
                if ((rd_mask[sh.L - 1] >> kb) & 1u) steps[g].push_back({WAIT_FREE, a0 + kb, 0});
        }
    }
    size_t ei[2] = {0, 0};
    auto epi_step = [&](int g) -> bool {
        if (ei[g] >= steps[g].size()) return false;
        const Step& s = steps[g][ei[g]];
        switch (s.kind) {
            case STAGE:
                for (int kb = 0; kb < sh.KB0; ++kb) complete(a_ready, a_ready_seen, s.a + kb);
                break;
            case WAIT_FULL:
                if (d_full[s.a] < s.b) return false;
                d_full_seen[s.a] = s.b;
                break;
            case DRAIN: complete(d_empty, d_empty_seen, s.a); break;
            case WAIT_FREE:
                if (a_free[s.a] <= a_free_seen[s.a]) return false;
                a_free_seen[s.a]++;
                break;
            case WRITE:
                complete(a_ready, a_ready_seen, s.a);
                complete(a_ready, a_ready_seen, s.a + 1);
                break;
        }
        ++ei[g];
        return true;
    };
    // d_empty bookkeeping: the scout's parity wait for the k-th use passes on phase k - 1 ... the
    // "seen" counter above is set when it passes, so `complete` flags a drain that outruns it by two.
    for (;;) {
        bool progress = false;
        for (const DryAgent& ag : policy) {
            auto step = [&] { return ag.agent == PAIR_MMA ? mma_step() : epi_step(ag.agent); };
            if (ag.greedy) {
                while (step()) progress = true;
            } else if (step()) {
                progress = true;
            }
        }
        if (!progress) break;
    }
    bool drained = true;
    for (int g = 0; g < sh.S; ++g) drained = drained && ei[g] == steps[g].size();
    return ok && mi == TILES * n && drained;
}

// The issue schedule of one pair tile (entry layout: pair_common.cuh): per layer, chunks and K blocks in
// DESCENDING order (see fused_wide.cu), the S sub-tiles alternating chunk by chunk.  Returns false when
// the dry run rejects the schedule (the layer then stays on the per-layer path).
bool pair_build_schedule(const int* dims, int L, const std::vector<std::vector<uint8_t>>& Mk,
                         const std::vector<std::vector<int>>& perm, int univariate, int bins, int D, int S,
                         std::vector<uint2>& items, uint32_t* rd_mask /*[8]*/) {
    const int H = dims[1];
    const int P = fused_p(univariate, bins), DPC = fused_dpc(univariate, bins);
    const int NA = 8 / S;
    PairShape sh;
    sh.S = S; sh.L = L; sh.nch = H / 128; sh.KB0 = pad64(dims[0]) / 64; sh.KBH = H / 64;
    sh.n_last = (D + DPC - 1) / DPC;
    const FusedTileMap tm = fused_tile_map(dims, L, Mk, perm, 128, univariate, bins, D);
    items.clear();
    for (int l = 0; l < 8; ++l) rd_mask[l] = 0u;
    uint32_t written = (1u << sh.KB0) - 1u;  // per sub-tile: A blocks with a pending a_ready phase when the layer starts
    for (int l = 0; l < L; ++l) {
        const bool last = (l == L - 1);
        const std::vector<uint32_t>& kbmask = tm.kbmask[l];
        const int nch = (int)kbmask.size();
        const int KB = (l == 0) ? sh.KB0 : sh.KBH;
        uint32_t rd = 0;
        for (int ch = 0; ch < nch; ++ch) rd |= kbmask[ch] & ((1u << KB) - 1u);
        rd_mask[l] = rd;
        int last_reader[8];
        for (int kb = 0; kb < 8; ++kb) last_reader[kb] = -1;
        for (int ch = nch - 1; ch >= 0; --ch)  // issue order: the last reader is the lowest chunk
            for (int kb = 0; kb < KB; ++kb)
                if ((kbmask[ch] >> kb) & 1u) last_reader[kb] = ch;
        uint32_t waited[2] = {0u, 0u};
        size_t layer_first[2] = {(size_t)-1, (size_t)-1};
        for (int ch = nch - 1; ch >= 0; --ch) {
            const uint32_t kbm = kbmask[ch] & ((1u << KB) - 1u);
            int lo = 0;
            for (int kb = KB - 1; kb >= 0; --kb) if ((kbm >> kb) & 1u) lo = kb;
            for (int u = 0; u < S; ++u) {
                bool first = true;
                for (int kb = KB - 1; kb >= 0; --kb) {
                    if (!((kbm >> kb) & 1u)) continue;
                    uint32_t it = (uint32_t)(u * NA + kb) | (first ? WS_FIRST : 0u) | (kb == lo ? WS_LAST : 0u) | ((uint32_t)l << 16);
                    if (!((waited[u] >> kb) & 1u)) { it |= WS_AWAIT; waited[u] |= 1u << kb; }
                    if (last_reader[kb] == ch) it |= WS_AFREE;
                    if (last) it |= WS_OUT;
                    it |= (uint32_t)(3 - tm.kmax[l][(size_t)ch * 8 + kb] / 16) << 20;  // trailing all-zero 16-column steps of the block are not issued
                    if (layer_first[u] == (size_t)-1) layer_first[u] = items.size();
                    items.push_back(make_uint2(it, (uint32_t)(last ? ch * DPC * P : ch * 128)));
                    first = false;
                }
            }
        }
        for (int u = 0; u < S; ++u) items[layer_first[u]].x |= ((written & ~rd) << (u * NA)) << 8;  // written for this layer but never read by it
        written = last ? 0u : ((1u << sh.KBH) - 1u);
    }
    for (const DryPolicy& policy : pair_policies(S))
        if (!pair_dry_run(items, rd_mask, sh, policy)) return false;
    return true;
}

}  // namespace

int pair_schedule_host(int S, int n_linear, const int* dims, const uint8_t* const* masks_host, int univariate, int bins,
                       int D, int C, uint32_t* out_items, int max_items, uint32_t* out_rd_mask, int* out_perm) {
    if (!pair_dims_ok(dims, n_linear, univariate, bins, D, C, S)) return -1;
    std::vector<std::vector<uint8_t>> Mk(n_linear);
    for (int l = 0; l < n_linear; ++l) {
        const size_t n = (size_t)dims[l + 1] * dims[l];
        Mk[l].assign(n, 1);
        if (masks_host && masks_host[l]) memcpy(Mk[l].data(), masks_host[l], n);
    }
    std::vector<std::vector<int>> perm;
    fused_degree_perm(dims, n_linear, Mk, perm);
    std::vector<uint2> items;
    uint32_t rd[8];
    if (!pair_build_schedule(dims, n_linear, Mk, perm, univariate, bins, D, S, items, rd)) return -2;
    if ((int)items.size() > max_items) return -3;
    for (size_t i = 0; i < items.size(); ++i) { out_items[2 * i] = items[i].x; out_items[2 * i + 1] = items[i].y; }
    if (out_rd_mask) for (int l = 0; l < 8; ++l) out_rd_mask[l] = rd[l];
    if (out_perm) {
        size_t o = 0;
        for (int l = 0; l < n_linear - 1; ++l)
            for (int v : perm[l]) out_perm[o++] = v;
    }
    return (int)items.size();
}

zk_status fused_pair_prepare(zk_mlp* m, const uint8_t* const* mask_dev, int univariate, int bins, int D, int C,
                             WidePack& wp, int S) {
    TcPack* pk = (TcPack*)m->tc;
    wp.ready = false;
    const int L = m->n_linear;
    const int P = fused_p(univariate, bins), DPC = fused_dpc(univariate, bins);
    const int N_LAST = (DPC * P + 15) & ~15;
    FusedHostPrep hp;
    ZK_TRY(fused_host_prepare(m, mask_dev, pk->fused, hp));
    wp.maps.assign(L, CUtensorMap{});
    for (int l = 0; l < L; ++l)
        ZK_TRY(make_plane_map(&wp.maps[l], pk->fused.w[l], m->dims[l + 1], pk->layers[l].Kp, (l == L - 1) ? N_LAST / 2 : 64));
    std::vector<uint2> items;
    uint32_t rdm[8];
    if (!pair_build_schedule(m->dims.data(), L, hp.Mk, hp.perm, univariate, bins, D, S, items, rdm)) return ZK_OK;  // per-layer path
    for (int l = 0; l < 8; ++l) wp.rd_mask[l] = (uint8_t)rdm[l];
    {
        double macs = 0;
        for (const uint2& it : items) macs += 16.0 * (4 - (int)((it.x >> 20) & 3u)) * ((it.x & WS_OUT) ? N_LAST : 128);
        wp.issued_macs_per_row = macs / S * pk->n_terms;  // the schedule covers S sub-tiles
    }
    cudaFree(wp.sched);
    wp.sched = nullptr;
    wp.n_items = (int)items.size();
    if (cudaMalloc((void**)&wp.sched, items.size() * sizeof(uint2)) != cudaSuccess ||
        cudaMemcpy(wp.sched, items.data(), items.size() * sizeof(uint2), cudaMemcpyHostToDevice) != cudaSuccess)
        return fail(ZK_ENOMEM, "fused_pair_prepare: cudaMalloc failed");
    wp.uni = univariate; wp.bins = bins; wp.D = D; wp.C = C;
    wp.ready = true;
    return ZK_OK;
}

uint32_t* pair_watch_device() {
    if (g_watch_host == nullptr) {
        uint32_t* h = nullptr;
        if (cudaHostAlloc((void**)&h, W_WATCH_WORDS * 4, cudaHostAllocMapped) == cudaSuccess) {
            memset(h, 0, W_WATCH_WORDS * 4);
            g_watch_host = h;
        } else {
            cudaGetLastError();
        }
    }
    void* d = nullptr;
    if (g_watch_host != nullptr && cudaHostGetDevicePointer(&d, g_watch_host, 0) != cudaSuccess) {
        cudaGetLastError();
        d = nullptr;
    }
    return (uint32_t*)d;
}

}  // namespace zk
