// Translation unit of the dense_kernel / dense_kernel_emu instantiations that run fp32-stored dense Hessians.
//
// The reference's only use of A is A.dot(v) (solvers.py:133): for a float32 A NumPy widens every entry exactly and runs
// the product in fp64.  These kernels do the same on the device -- A is streamed as fp32 (half the HBM bytes of the fp64
// kernels) and every entry is widened in a register in front of its fma -- with the fp64 loop's lane mapping, FMA chains
// and reduction order (dense.cuh dot_seg_aligned / dot_seg_generic for const float*), so a solve returns the same bits as
// the fp64 solve of the widened matrix.  The SAME solver programs (dense.cuh) are compiled a second time here, CSR phase
// compiled out, inside their own namespace (every `ccqp::` entity of the headers becomes `ccqp_f32::`), like csr.cu: the
// fp64 kernels keep their own translation unit and code (the schedule of the dense loop depends on everything inlined
// next to it).  capi.cu routes every launch of a handle that holds an fp32 matrix through f32_variant_launch(), and
// ccqp_debug_solve_emulated() through f32_variant_launch_emu(); the context struct is the same plain-data struct in both
// namespaces.
#define CCQP_DENSE_ONLY 1
#define CCQP_A_F32 1
#define ccqp ccqp_f32
#include "dense.cuh"
#undef ccqp
#include "internal.h"

namespace ccqp_f32 {

template <int OP>
static cudaError_t launch(const DenseCtx& c, int grid, size_t smem, bool cooperative, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(dense_kernel<OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDenseSmemLimit);
    if (e != cudaSuccess) return e;
    DenseCtx cc = c;
    void* args[] = {&cc};
    if (cooperative) return cudaLaunchCooperativeKernel((const void*)dense_kernel<OP>, dim3(grid), dim3(kDenseThreads), args, smem, stream);
    return cudaLaunchKernel((const void*)dense_kernel<OP>, dim3(grid), dim3(kDenseThreads), args, smem, stream);
}

template <int OP>
static cudaError_t launch_emu(const DenseCtx* d_ctxs, int world, int G, size_t smem, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(dense_kernel_emu<OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDenseSmemLimit);
    if (e != cudaSuccess) return e;
    void* args[] = {(void*)&d_ctxs, (void*)&G};
    return cudaLaunchCooperativeKernel((const void*)dense_kernel_emu<OP>, dim3(world * G), dim3(kDenseThreads), args, smem, stream);
}

}  // namespace ccqp_f32

namespace ccqp {

size_t f32_variant_ctx_bytes() { return sizeof(ccqp_f32::DenseCtx); }

cudaError_t f32_variant_launch(int op, const void* ctx, int grid, size_t smem, bool cooperative, cudaStream_t stream) {
    const ccqp_f32::DenseCtx& c = *static_cast<const ccqp_f32::DenseCtx*>(ctx);
    using namespace ccqp_f32;
    switch (op) {
        case OP_PGD: return launch<OP_PGD>(c, grid, smem, cooperative, stream);
        case OP_APGD: return launch<OP_APGD>(c, grid, smem, cooperative, stream);
        case OP_APGD_AR: return launch<OP_APGD_AR>(c, grid, smem, cooperative, stream);
        case OP_BBPGD: return launch<OP_BBPGD>(c, grid, smem, cooperative, stream);
        case OP_BBPGDF: return launch<OP_BBPGDF>(c, grid, smem, cooperative, stream);
        case OP_SPG: return launch<OP_SPG>(c, grid, smem, cooperative, stream);
        case OP_MPRGP: return launch<OP_MPRGP>(c, grid, smem, cooperative, stream);
        case OP_GEMV: return launch<OP_GEMV>(c, grid, smem, cooperative, stream);
        case OP_PROJECT: return launch<OP_PROJECT>(c, grid, smem, cooperative, stream);
        case OP_NORMAL: return launch<OP_NORMAL>(c, grid, smem, cooperative, stream);
        case OP_PROJGRAD: return launch<OP_PROJGRAD>(c, grid, smem, cooperative, stream);
    }
    return cudaErrorInvalidValue;
}

cudaError_t f32_variant_launch_emu(int solver, const void* d_ctxs, int world, int G, size_t smem, cudaStream_t stream) {
    const ccqp_f32::DenseCtx* d = static_cast<const ccqp_f32::DenseCtx*>(d_ctxs);
    using namespace ccqp_f32;
    switch (solver) {
        case CCQP_SOLVER_PGD: return launch_emu<OP_PGD>(d, world, G, smem, stream);
        case CCQP_SOLVER_APGD: return launch_emu<OP_APGD>(d, world, G, smem, stream);
        case CCQP_SOLVER_APGD_AR: return launch_emu<OP_APGD_AR>(d, world, G, smem, stream);
        case CCQP_SOLVER_BBPGD: return launch_emu<OP_BBPGD>(d, world, G, smem, stream);
        case CCQP_SOLVER_BBPGDF: return launch_emu<OP_BBPGDF>(d, world, G, smem, stream);
        case CCQP_SOLVER_SPG: return launch_emu<OP_SPG>(d, world, G, smem, stream);
        case CCQP_SOLVER_MPRGP: return launch_emu<OP_MPRGP>(d, world, G, smem, stream);
    }
    return cudaErrorInvalidValue;
}

}  // namespace ccqp
