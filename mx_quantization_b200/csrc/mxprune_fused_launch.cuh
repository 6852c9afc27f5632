// Launcher template of the fused kernel, shared by the translation units that instantiate it
// (mxprune_fused.cu: any head_dim; mxprune_fused64.cu: the head_dim 64 specialisations).
#pragma once
#include "mxprune_host.cuh"
#include "mxprune_fused.cuh"

namespace mxp {

// DT: element type of q / k / v (DT_*); KMAX: register bound of the cost-follows-k epilogue (attend_sparse_head)
template <int NC, int HG, int HD, int DT, int KMAX>
int launch_fused_k(const FusedParams& p, const FusedMaps& maps, int grid, cudaStream_t st) {
    const size_t dyn = 2 * FUSED_GROUP_SMEM;
    if (p.bf16) {
        MXP_ENSURE_DYN_SMEM((k_fused_pruned_attention<NC, HG, true, HD, DT, KMAX>), (int)dyn);
        k_fused_pruned_attention<NC, HG, true, HD, DT, KMAX><<<grid, FUSED_T, dyn, st>>>(p, maps);
    } else {
        MXP_ENSURE_DYN_SMEM((k_fused_pruned_attention<NC, HG, false, HD, DT, KMAX>), (int)dyn);
        k_fused_pruned_attention<NC, HG, false, HD, DT, KMAX><<<grid, FUSED_T, dyn, st>>>(p, maps);
    }
    return check_launch("k_fused_pruned_attention");
}

// rows of up to 2 * K2S_KMAX kept keys take the sparse epilogue's register path, longer ones its list path
template <int NC, int HG, int HD, int DT = DT_F32>
int launch_fused_hd(const FusedParams& p, const FusedMaps& maps, int grid, cudaStream_t st) {
    if (p.sparse && p.top_k <= 2 * K2S_KMAX) return launch_fused_k<NC, HG, HD, DT, K2S_KMAX>(p, maps, grid, st);
    return launch_fused_k<NC, HG, HD, DT, 0>(p, maps, grid, st);
}

}  // namespace mxp
