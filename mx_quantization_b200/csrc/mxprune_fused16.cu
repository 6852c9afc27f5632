// libmxprune: the fused kernel for bf16 / fp16 q, k, v (include/mxprune.h, *_dt entry points).  The same kernel as
// mxprune_fused.cu with a 16-bit element type for the TMA staging and, when asked, the output store; in its own
// translation unit so that it compiles in parallel.  head_dim is a run-time value except for DeiT-shaped heads
// (head_dim 64, 193 - 208 keys, cost-follows-k epilogue), which keep their compile-time instantiation.
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

template <int DT>
static int launch_fused_16_dt(int nc, int hg, const FusedParams& p, const FusedMaps& maps, int grid, cudaStream_t st) {
    if (nc == 8) return launch_fused_hd<8, 0, 0, DT>(p, maps, grid, st);
    if (hg == 13) {
        if (p.hd == 64 && p.sparse) return launch_fused_hd<7, 13, 64, DT>(p, maps, grid, st);
        return launch_fused_hd<7, 13, 0, DT>(p, maps, grid, st);
    }
    if (hg == 14) return launch_fused_hd<7, 14, 0, DT>(p, maps, grid, st);
    return launch_fused_hd<7, 0, 0, DT>(p, maps, grid, st);
}

int launch_fused_16(int dt, int nc, int hg, const FusedParams& p, const FusedMaps& maps, int grid, cudaStream_t st) {
    return dt == DT_BF16 ? launch_fused_16_dt<DT_BF16>(nc, hg, p, maps, grid, st)
                         : launch_fused_16_dt<DT_F16>(nc, hg, p, maps, grid, st);
}

}  // namespace mxp
