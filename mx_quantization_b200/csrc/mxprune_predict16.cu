// libmxprune: the tensor-core predictor k_predict_topk_tc for bf16 / fp16 q and k (include/mxprune.h, *_dt entry
// points), with the instantiation policy of the fp32 calls (launch_predict_topk_tc_dt, mxprune_predict_tc.cuh).  Its own
// translation unit so that it compiles in parallel with mxprune.cu.
#include <cuda_runtime.h>
#include <stdint.h>

#include "mxprune.h"
#include "mxprune_host.cuh"
#include "mxprune_device.cuh"
#include "mxprune_predict_tc.cuh"

namespace mxp {

int launch_predict_topk_tc_16(const PredParams& p, const K1cMaps& maps, const K1cSmem& L, size_t dyn, dim3 grid, int nc,
                              cudaStream_t st) {
    return p.dt == DT_BF16 ? launch_predict_topk_tc_dt<DT_BF16>(p, maps, L, dyn, grid, nc, st)
                           : launch_predict_topk_tc_dt<DT_F16>(p, maps, L, dyn, grid, nc, st);
}

}  // namespace mxp
