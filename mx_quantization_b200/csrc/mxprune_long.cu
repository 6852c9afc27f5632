// libmxprune, fourth translation unit: the long-sequence (Nk > 256) exact-attention kernel with two lanes per query
// row and a pipelined key-block stream (mxprune_attend_long.cuh), and its launcher.
#include <cuda_runtime.h>
#include <stdint.h>

#include "mxprune.h"
#include "mxprune_host.cuh"
#include "mxprune_device.cuh"
#include "mxprune_attend.cuh"
#include "mxprune_attend_long.cuh"

namespace mxp {

// k_attend_long_pair with output element type OT (== p.out_dt); grid and dyn from launch_attend_long_pair
template <int OT>
static int launch_attend_long_pair_ot(const AttnParams& p, dim3 grid, size_t dyn, cudaStream_t st) {
    MXP_ENSURE_DYN_SMEM((k_attend_long_pair<true, OT>), (int)(SMEM_PER_SM - 2048));
    MXP_ENSURE_DYN_SMEM((k_attend_long_pair<false, OT>), (int)(SMEM_PER_SM - 2048));
    if (p.key_bias) {
        MXP_ENSURE_DYN_SMEM((k_attend_long_pair<true, OT, true>), (int)(SMEM_PER_SM - 2048));
        MXP_ENSURE_DYN_SMEM((k_attend_long_pair<false, OT, true>), (int)(SMEM_PER_SM - 2048));
        if (p.bf16) k_attend_long_pair<true, OT, true><<<grid, K2P_T, dyn, st>>>(p);
        else k_attend_long_pair<false, OT, true><<<grid, K2P_T, dyn, st>>>(p);
    } else if (p.bf16) {
        k_attend_long_pair<true, OT><<<grid, K2P_T, dyn, st>>>(p);
    } else {
        k_attend_long_pair<false, OT><<<grid, K2P_T, dyn, st>>>(p);
    }
    return check_launch("k_attend_long_pair");
}

int launch_attend_long_pair(const AttnParams& p, cudaStream_t st) {
    const OpsLayout O = ops_layout(p.Nq, p.Nk, p.hd);
    const KLPSmem L = klp_smem_layout(O);
    // pass 1 uses V buffer 0 as its second K buffer; with key blocks of 128 rows both blocks are 256 hdp bytes and the
    // layout is at most 160 KiB (hd = 128), so these hold for every supported head_dim
    if (O.k_blk_bytes != O.v_blk_bytes || L.total > SMEM_PER_SM - 2048)
        return fail(MXP_E_UNSUPPORTED, "head_dim %d: the long-sequence attention kernel needs K / V blocks of equal size "
                    "(%zu / %zu bytes) and %zu bytes of shared memory", p.hd, O.k_blk_bytes, O.v_blk_bytes, L.total);
    // one CTA per query tile (a CTA holds nothing across tiles); 256 TMEM columns per CTA: at most two CTAs per SM,
    // which the dynamic shared-memory request enforces (see launch_attend)
    dim3 grid((unsigned)((size_t)p.B * p.H * O.q_tiles));
    size_t dyn = L.total;
    const size_t floor_bytes = SMEM_PER_SM / 3 + 1024;
    if (dyn < floor_bytes) dyn = floor_bytes;
    if (p.out_dt == DT_BF16) return launch_attend_long_pair_ot<DT_BF16>(p, grid, dyn, st);
    if (p.out_dt == DT_F16) return launch_attend_long_pair_ot<DT_F16>(p, grid, dyn, st);
    return launch_attend_long_pair_ot<DT_F32>(p, grid, dyn, st);
}

}  // namespace mxp
