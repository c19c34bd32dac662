// The launch table of one compilation of the dense.cuh solver programs.  dense_f64.cu, dense_f32.cu, csr.cu and emu.cu each
// include this after dense.cuh while their namespace rename is active, so everything here lands in that unit's namespace;
// the unit then defines its KernelBuild (internal.h) as describe<KernelBuild>(...).  capi.cu launches only through those
// descriptors.
#pragma once
#include "../../include/ccqp_b200.h"

#ifndef CCQP_DENSE_KERNELS
#define CCQP_DENSE_KERNELS 1    // dense_kernel<OP>: the solves and test hooks of a handle
#endif
#ifndef CCQP_EMU_KERNELS
#define CCQP_EMU_KERNELS 0      // dense_kernel_emu<OP>: the ranks of an emulated box in one launch (ccqp_debug_solve_emulated)
#endif

namespace ccqp {

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute of each kernel instantiation: the caller asks for
// it once per device (set_smem_limit)
inline cudaError_t allow_dense_smem(const void* kernel, bool set_smem_limit) {
    return set_smem_limit ? cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDenseSmemLimit) : cudaSuccess;
}

#if CCQP_DENSE_KERNELS
template <int OP>
cudaError_t launch(const DenseCtx& c, int grid, size_t smem, bool cooperative, bool set_smem_limit, cudaStream_t stream) {
    const void* kernel = (const void*)dense_kernel<OP>;
    if (cudaError_t e = allow_dense_smem(kernel, set_smem_limit)) return e;
    void* args[] = {const_cast<DenseCtx*>(&c)};
    if (cooperative) return cudaLaunchCooperativeKernel(kernel, dim3(grid), dim3(kDenseThreads), args, smem, stream);
    return cudaLaunchKernel(kernel, dim3(grid), dim3(kDenseThreads), args, smem, stream);
}

// `op` is a DenseOp; `ctx` points at a DenseCtx
cudaError_t launch_op(int op, const void* ctx, int grid, size_t smem, bool cooperative, bool set_smem_limit, cudaStream_t stream) {
    const DenseCtx& c = *static_cast<const DenseCtx*>(ctx);
    switch (op) {
#ifndef CCQP_SWEEP_BUILD    // tuning build (tools/sweep_gemv.py): only the mat-vec hook is compiled
        case OP_PGD: return launch<OP_PGD>(c, grid, smem, cooperative, set_smem_limit, stream);
        case OP_APGD: return launch<OP_APGD>(c, grid, smem, cooperative, set_smem_limit, stream);
        case OP_APGD_AR: return launch<OP_APGD_AR>(c, grid, smem, cooperative, set_smem_limit, stream);
        case OP_BBPGD: return launch<OP_BBPGD>(c, grid, smem, cooperative, set_smem_limit, stream);
        case OP_BBPGDF: return launch<OP_BBPGDF>(c, grid, smem, cooperative, set_smem_limit, stream);
        case OP_SPG: return launch<OP_SPG>(c, grid, smem, cooperative, set_smem_limit, stream);
        case OP_MPRGP: return launch<OP_MPRGP>(c, grid, smem, cooperative, set_smem_limit, stream);
        case OP_PROJECT: return launch<OP_PROJECT>(c, grid, smem, cooperative, set_smem_limit, stream);
        case OP_NORMAL: return launch<OP_NORMAL>(c, grid, smem, cooperative, set_smem_limit, stream);
        case OP_PROJGRAD: return launch<OP_PROJGRAD>(c, grid, smem, cooperative, set_smem_limit, stream);
#endif
        case OP_GEMV: return launch<OP_GEMV>(c, grid, smem, cooperative, set_smem_limit, stream);
    }
    return cudaErrorNotSupported;
}
#else
constexpr decltype(nullptr) launch_op = nullptr;           // no dense_kernel in this build
#endif

#if CCQP_EMU_KERNELS
// one cooperative launch of world * G CTAs; d_ctxs: the ranks' contexts in device memory
template <int OP>
cudaError_t launch_emu(const DenseCtx* d_ctxs, int world, int G, size_t smem, bool set_smem_limit, cudaStream_t stream) {
    const void* kernel = (const void*)dense_kernel_emu<OP>;
    if (cudaError_t e = allow_dense_smem(kernel, set_smem_limit)) return e;
    void* args[] = {(void*)&d_ctxs, (void*)&G};
    return cudaLaunchCooperativeKernel(kernel, dim3(world * G), dim3(kDenseThreads), args, smem, stream);
}

// `solver` is a ccqp_solver; `d_ctxs` points at world DenseCtx in device memory
cudaError_t launch_emu_solver(int solver, const void* d_ctxs, int world, int G, size_t smem, bool set_smem_limit, cudaStream_t stream) {
    [[maybe_unused]] const DenseCtx* d = static_cast<const DenseCtx*>(d_ctxs);   // (a tuning build has no cases)
    switch (solver) {
#ifndef CCQP_SWEEP_BUILD
        case CCQP_SOLVER_PGD: return launch_emu<OP_PGD>(d, world, G, smem, set_smem_limit, stream);
        case CCQP_SOLVER_APGD: return launch_emu<OP_APGD>(d, world, G, smem, set_smem_limit, stream);
        case CCQP_SOLVER_APGD_AR: return launch_emu<OP_APGD_AR>(d, world, G, smem, set_smem_limit, stream);
        case CCQP_SOLVER_BBPGD: return launch_emu<OP_BBPGD>(d, world, G, smem, set_smem_limit, stream);
        case CCQP_SOLVER_BBPGDF: return launch_emu<OP_BBPGDF>(d, world, G, smem, set_smem_limit, stream);
        case CCQP_SOLVER_SPG: return launch_emu<OP_SPG>(d, world, G, smem, set_smem_limit, stream);
        case CCQP_SOLVER_MPRGP: return launch_emu<OP_MPRGP>(d, world, G, smem, set_smem_limit, stream);
#endif
    }
    return cudaErrorNotSupported;
}
#else
constexpr decltype(nullptr) launch_emu_solver = nullptr;   // no dense_kernel_emu in this build
#endif

// this build's entry of the launch table (KernelBuild is internal.h's, which cannot be named inside the rename)
template <class KernelBuild>
constexpr KernelBuild describe(const char* unit, int index) {
    return KernelBuild{unit, index, kDenseThreads, sizeof(DenseCtx), CCQP_DENSE_ONLY ? 0 : kCsrRowsMax,
                       launch_op, launch_emu_solver};
}

}  // namespace ccqp
