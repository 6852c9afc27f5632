// libmxprune, second translation unit: the kernels of round 2 (cost-follows-k attention epilogue, the fused
// predictor + attention kernel) and their launchers.  Split from mxprune.cu so that the two halves compile in parallel.
#include <cuda_runtime.h>
#include <stdint.h>

#include "mxprune.h"
#include "mxprune_host.cuh"
#include "mxprune_device.cuh"
#include "mxprune_attend.cuh"
#include "mxprune_attend_sparse.cuh"
#include "mxprune_fused.cuh"
#include "mxprune_fused_launch.cuh"

namespace mxp {

// k_attend_sparse with output element type OT (== p.out_dt); grid and dyn from attend_sparse_try
template <int OT>
static int launch_attend_sparse_ot(const AttnParams& p, int top_k, dim3 grid, size_t dyn, cudaStream_t st) {
    MXP_ENSURE_DYN_SMEM((k_attend_sparse<true, OT>), 160 * 1024);
    MXP_ENSURE_DYN_SMEM((k_attend_sparse<false, OT>), 160 * 1024);
    if (p.bf16) k_attend_sparse<true, OT><<<grid, K2P_T, dyn, st>>>(p, top_k);
    else k_attend_sparse<false, OT><<<grid, K2P_T, dyn, st>>>(p, top_k);
    return check_launch("k_attend_sparse");
}

int attend_sparse_try(const AttnParams& p, int top_k, cudaStream_t st, int* rc_out) {
    const OpsLayout O = ops_layout(p.Nq, p.Nk, p.hd);
    // domain: one key block, no additive bias, a uniform row population of at most 35 % of the keys, and the row
    // lists + operands of two CTAs resident per SM
    if (g_fused_path.load() == 0 || !O.single || p.key_bias || top_k < 1 || top_k * 100 > 35 * p.Nk) return 1;
    const K2sSmem L = k2s_smem_layout(O, top_k);
    if (L.total > SMEM_2CTA) return 1;
    auto run = [&]() -> int {
        const int heads = p.B * p.H;
        int splits = (148 * 2 + heads - 1) / heads;
        if (splits > O.q_tiles) splits = O.q_tiles;
        if (splits < 1) splits = 1;
        dim3 grid((unsigned)heads, (unsigned)splits);
        // residency bounded by the 512 TMEM columns of an SM (see launch_attend)
        const int max_ctas = 512 / k2p_tmem_cols(O);
        size_t dyn = L.total;
        const size_t floor_bytes = SMEM_PER_SM / (size_t)(max_ctas + 1) + 1024;
        if (dyn < floor_bytes) dyn = floor_bytes;
        if (p.out_dt == DT_BF16) return launch_attend_sparse_ot<DT_BF16>(p, top_k, grid, dyn, st);
        if (p.out_dt == DT_F16) return launch_attend_sparse_ot<DT_F16>(p, top_k, grid, dyn, st);
        return launch_attend_sparse_ot<DT_F32>(p, top_k, grid, dyn, st);
    };
    *rc_out = run();
    return 0;
}


// ---- the fused kernel --------------------------------------------------------------------------------
FusedSlotLayout fused_slot_layout(int Nq, int Nk, int hd) {
    const OpsLayout O = ops_layout(Nq, Nk, hd);
    auto a256 = [](size_t x) { return (x + 255) & ~(size_t)255; };
    FusedSlotLayout S;
    S.k = a256(O.q_head_bytes);
    S.v = S.k + a256(O.k_head_bytes);
    S.mask = S.v + a256(O.v_head_bytes);
    S.bytes = S.mask + a256((size_t)Nq * O.nw * 4);
    return S;
}

size_t fused_workspace_bytes(int Nq, int Nk, int hd) {
    if (Nk > 256 || hd < 32 || (hd & 7)) return 0;
    return (size_t)2 * 160 * fused_slot_layout(Nq, Nk, hd).bytes;       // two groups per SM, up to 160 SMs
}

constexpr int FUSED_MIN_HEADS = 64;       // default policy: fewer heads take the three kernels (see fused_try)
static std::atomic<unsigned long long*> g_fused_timing{nullptr};
static std::atomic<int> g_fused_pingpong{1};
void fused_set_pingpong(int on) { g_fused_pingpong = on; }
void fused_set_timing_buffer(unsigned long long* buf) { g_fused_timing = buf; }

// head_dim 64 (DeiT / ViT heads) has its own instantiations with the staging geometry folded at compile time; they are
// compiled in their own translation unit (mxprune_fused64.cu)
extern template int launch_fused_hd<8, 0, 64>(const FusedParams&, const FusedMaps&, int, cudaStream_t);
extern template int launch_fused_hd<7, 13, 64>(const FusedParams&, const FusedMaps&, int, cudaStream_t);
extern template int launch_fused_hd<7, 14, 64>(const FusedParams&, const FusedMaps&, int, cudaStream_t);
extern template int launch_fused_hd<7, 0, 64>(const FusedParams&, const FusedMaps&, int, cudaStream_t);
template <int NC, int HG>
static int launch_fused_one(const FusedParams& p, const FusedMaps& maps, int grid, cudaStream_t st) {
#ifndef MXP_FUSED_NO_HD64
    if (p.hd == 64 && p.sparse) return launch_fused_hd<NC, HG, 64>(p, maps, grid, st);
#endif
    return launch_fused_hd<NC, HG, 0>(p, maps, grid, st);
}

int launch_fused_16(int dt, int nc, int hg, const FusedParams& p, const FusedMaps& maps, int grid, cudaStream_t st);

int fused_try(const FusedArgs& a, cudaStream_t st, int* rc_out) {
    // domain: the exponent-sign predictor on the tensor-core paths, one key block of 129..256 keys, a real selection
    // (top_k < Nk), no key bias, enough heads to give every group of half the chip one
    if (g_fused_path.load() == 0 || g_attn_path.load() != 0 || g_predict_path.load() != 0) return 1;
    if (a.Nk > 256 || a.Nk <= 128 || a.hd < 32 || (a.hd & 7) || a.top_k >= a.Nk) return 1;
    const int heads = a.B * a.H;
    if (heads < (g_fused_path.load() == 2 ? 2 : FUSED_MIN_HEADS)) return 1;
    // between one head per SM (both groups of a CTA share a head: 28 us per call at 96 - 144 heads against 31 - 32 us for the
    // three kernels) and ~1.7 heads per SM every group holds a whole head for ~50 us while the three kernels spread the
    // same heads over tiles and row splits (192 heads: 53 vs 47 us; 288 heads: 53 vs 58 us - tools/ab_small_heads.py)
    if (g_fused_path.load() != 2 && heads > sm_count() && heads < (sm_count() * 27) / 16) return 1;
    const int nc = a.Nk <= 224 ? 7 : 8;
    const int nb = (a.hd + 31) / 32;
    const int G = fused_G(a.hd, nc), ring = fused_ring(a.hd, nc);
    const K1cSmem L1 = k1c_smem_layout(a.hd, nc, ring, G);
    if (L1.total > FUSED_GROUP_SMEM - 256) return 1;
    const OpsLayout O = ops_layout(a.Nq, a.Nk, a.hd);
    const bool sparse = a.top_k * 100 <= 35 * a.Nk && k2s_smem_layout(O, a.top_k).total <= FUSED_GROUP_SMEM - 256;
    // measured on B200 (tools/ab_fused.py): with the cost-follows-k epilogue the fused launch beats the three kernels
    // (DeiT-base layer 0.504 vs 0.521 ms); with the dense epilogue it does not (DiT-XL/2 1.01 vs 0.95 ms) - both phases
    // are then issue-bound and gain nothing from sharing an SM.  Path 2 forces it (tests, A/B).
    if (!sparse && g_fused_path.load() != 2) return 1;
    // measured as well (tools/sweep_c5.py, tools/ab_fused.py): with 64-row steps (G = 1: three MX blocks per row, or a
    // predictor operand that leaves no room for 128-row slots) phase 1 needs twice the steps and the fused launch loses
    // to the three kernels (256 tokens x head_dim 72, top_k 26: 0.94 vs 0.76 ms; PixArt's 77: 1.00 vs 0.84 ms)
    if (G != 2 && g_fused_path.load() != 2) return 1;
    if (!sparse && k2_smem_layout(O).total > FUSED_GROUP_SMEM - 256) return 1;
    const FusedSlotLayout S = fused_slot_layout(a.Nq, a.Nk, a.hd);
    int grid = sm_count();
    if (grid > 160) grid = 160;
    // up to one CTA per head: with heads <= SMs every CTA's two groups share one head (one query tile each - the kernel's
    // shared-round rule), with up to twice that every group gets its own head on as many SMs as there are
    if (grid > heads) grid = heads;
    if (!a.slots || a.slots_bytes < (size_t)2 * grid * S.bytes) return 1;
    FusedMaps maps;
    if (!make_view_maps(a.q, a.B, a.H, a.Nq, a.hd, &maps.q_main, &maps.q_tail, a.dt) ||
        !make_view_maps(a.k, a.B, a.H, a.Nk, a.hd, &maps.k_main, &maps.k_tail, a.dt) ||
        !make_view_maps(a.v, a.B, a.H, a.Nk, a.hd, &maps.v_main, &maps.v_tail, a.dt)) {
        if (a.dt == DT_F32) return 1;
        *rc_out = fail(MXP_E_UNSUPPORTED, "16-bit q/k/v: the views cannot be described by a TMA tensor map");
        return 0;
    }
    FusedParams p{};
    p.B = a.B; p.H = a.H; p.Nq = a.Nq; p.Nk = a.Nk; p.hd = a.hd; p.top_k = a.top_k; p.bf16 = a.bf16; p.flush = a.flush;
    p.scale = a.scale;
    p.out = a.out; p.o_sB = a.o_sB; p.o_sH = a.o_sH; p.o_sN = a.o_sN; p.out16 = a.out_dt != DT_F32;
    p.mask_out = a.mask_out;
    p.slots = a.slots; p.slot_bytes = S.bytes; p.slot_k = S.k; p.slot_v = S.v; p.slot_mask = S.mask;
    p.ring = ring; p.G = G; p.sparse = sparse ? 1 : 0;
    p.timing = g_fused_timing.load();
    p.pingpong = (g_fused_pingpong.load() && sparse) ? 1 : 0;   // the phase-1 token pays when phase 2 is the latency-bound one
    const int hg = nc == 8 ? 0 : (a.Nk > 192 && a.Nk <= 208) ? 13 : a.Nk > 208 ? 14 : 0;
    if (a.dt != DT_F32) *rc_out = launch_fused_16(a.dt, nc, hg, p, maps, grid, st);      // mxprune_fused16.cu
    else if (nc == 8) *rc_out = launch_fused_one<8, 0>(p, maps, grid, st);
    else if (a.Nk > 192 && a.Nk <= 208) *rc_out = launch_fused_one<7, 13>(p, maps, grid, st);
    else if (a.Nk > 208) *rc_out = launch_fused_one<7, 14>(p, maps, grid, st);
    else *rc_out = launch_fused_one<7, 0>(p, maps, grid, st);
    return 0;
}

}  // namespace mxp
