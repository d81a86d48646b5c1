// zuko_b200 — fully fused flow-layer kernel (conditioner + bijector + ladj): interface.
#pragma once

#include <atomic>

#include "mlp.cuh"

#define ZK_FUSED_MAX_LINEAR 6

namespace zk {

struct FusedLayerArgs {
    int univariate = ZK_UNI_RQS;
    int bins = 8;
    int D = 0, C = 0;
    float bound = 5.f, slope = 1e-3f;
    const float* x = nullptr; int64_t ldx = 0;
    const float* c = nullptr; int64_t ldc = 0;
    int64_t B = 0;
    float* y = nullptr; int64_t ldy = 0;  // may be null (log_prob only)
    float* ladj = nullptr; int accumulate = 0;
    float* log_prob = nullptr; const float* base_loc = nullptr; const float* base_scale = nullptr;
    bool fast_math = true;
};

// true when the autoregressive layer (conditioner `m`, univariate, D, C) can run as ONE kernel
bool fused_layer_supported(const zk_mlp* m, int univariate, int bins, int D, int C);
// which kernel: 0 none, 1 one CTA per tile (fused_layer.cu), 2 CTA pairs (fused_wide.cu), 3 CTA pairs with two sub-tiles (fused_dual.cu)
int fused_layer_kind(const zk_mlp* m, int univariate, int bins, int D, int C);
// Builds the fused kernel's weight pack for this conditioner (degree-sorted hidden units, zero-tile
// map); `mask_dev` are the DEVICE mask pointers of zk_mlp_desc (may be null = dense).  No-op when
// the shape is not supported by the fused kernel.
zk_status fused_layer_prepare(zk_mlp* m, const uint8_t* const* mask_dev, int univariate, int bins, int D, int C);
// ---- CTA-pair variants on cta_group::2, planned in fused_plan.cu: wide (fused_wide.cu, hidden width
// 256 - 512) and dual-tile (fused_dual.cu, hidden width 128 / 256, two sub-tiles in flight per CTA) ----
// shape tests only (and the routing knobs g_wide_min_h / g_dual); the layer runs fused once
// fused_pair_prepare built a schedule that passed its dry run
bool fused_wide_shape(const zk_mlp* m, int univariate, int bins, int D, int C);
bool fused_dual_shape(const zk_mlp* m, int univariate, int bins, int D, int C);
zk_status launch_fused_wide(const zk_mlp* m, const FusedLayerArgs& a, cudaStream_t stream);
zk_status launch_fused_dual(const zk_mlp* m, const FusedLayerArgs& a, cudaStream_t stream);
// Host-only entry behind zk_debug_wide_schedule (S = 1) / zk_debug_dual_schedule (S = 2): the schedule of
// one pair tile from masks on the HOST, no CUDA call.  Entries, or -1 unsupported shape, -2 rejected by
// the dry run, -3 more than max_items.
int pair_schedule_host(int S, int n_linear, const int* dims, const uint8_t* const* masks_host, int univariate, int bins,
                       int D, int C, uint32_t* out_items, int max_items, uint32_t* out_rd_mask, int* out_perm);
extern std::atomic<int> g_dual;
extern std::atomic<int> g_wide_min_h;
constexpr int W_WATCH_WORDS = 1024;
extern uint32_t* g_watch_host;  // watchdog report buffer of the pair kernels (W_WATCH_WORDS, pinned host memory) or null
zk_status fused_refresh(zk_mlp* m, cudaStream_t stream);  // weights changed in place: re-split into the fused packs
extern long long* g_timeline;  // device buffer of >= 256 stamps, or null (zk_debug_timeline)
zk_status launch_fused_layer(const zk_mlp* m, const FusedLayerArgs& a, cudaStream_t stream);

}  // namespace zk
