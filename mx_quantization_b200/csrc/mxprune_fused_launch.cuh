// Launcher template of the fused kernel, shared by the translation units that instantiate it
// (mxprune_fused.cu: any head_dim; mxprune_fused64.cu: the head_dim 64 specialisations).
#pragma once
#include "mxprune_host.cuh"
#include "mxprune_fused.cuh"

namespace mxp {

// DT: element type of q / k / v (DT_*)
template <int NC, int HG, int HD, int DT = DT_F32>
int launch_fused_hd(const FusedParams& p, const FusedMaps& maps, int grid, cudaStream_t st) {
    const size_t dyn = 2 * FUSED_GROUP_SMEM;
    if (p.bf16) {
        MXP_ENSURE_DYN_SMEM((k_fused_pruned_attention<NC, HG, true, HD, DT>), (int)dyn);
        k_fused_pruned_attention<NC, HG, true, HD, DT><<<grid, FUSED_T, dyn, st>>>(p, maps);
    } else {
        MXP_ENSURE_DYN_SMEM((k_fused_pruned_attention<NC, HG, false, HD, DT>), (int)dyn);
        k_fused_pruned_attention<NC, HG, false, HD, DT><<<grid, FUSED_T, dyn, st>>>(p, maps);
    }
    return check_launch("k_fused_pruned_attention");
}

}  // namespace mxp
