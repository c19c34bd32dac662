// Translation unit of the batched_kernel instantiations for fp32-stored Hessians (TA = float, batched.cuh): the launch
// tables launch_batched<GEN, float> that batched.cu dispatches to.  A separate unit only so that the two sets of 30 kernels
// compile in parallel; the fp64 instantiations stay in batched.cu.
#include "batched.cuh"

namespace ccqp {

template cudaError_t launch_batched<false, float>(const BatchedCtx&, int, bool, int, cudaStream_t);
template cudaError_t launch_batched<true, float>(const BatchedCtx&, int, bool, int, cudaStream_t);

}  // namespace ccqp
