// maz_infer_wide.cu -- the wide instance (48 < KA <= 128) of the two-tiles-in-flight kernel (infer_twin.cuh), launched by
// maz_infer_recurrent (maz_infer.cu).  It has a translation unit of its own: ptxas of CUDA 12.9 crashes (segmentation fault) when one
// module holds both instances of that kernel, whose epilogue functions they share.
#include <cuda_runtime.h>

#define MAZ_FUSED_NO_KERNEL
#include "../../include/maz_infer.h"
#include "umma.cuh"
#include "infer_fused.cuh"
#include "infer_twin.cuh"

namespace maz {
namespace twin {

const void *wide_kernel() { return (const void *)k_recurrent_inference_twin<true>; }

cudaError_t launch_wide(const cudaLaunchConfig_t &cfg, const maz_infer_desc &d)
{
    return cudaLaunchKernelEx(&cfg, k_recurrent_inference_twin<true>, d);
}

}  // namespace twin
}  // namespace maz
