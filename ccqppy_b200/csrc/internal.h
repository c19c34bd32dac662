// Entry points between the translation units of libccqp_b200.so: capi.cu (C-ABI, host code), batched.cu + batched_sym.cu
// (batched kernels), upload.cu (host -> device matrix copies), and the four compilations of the dense solver kernels, one
// unit each because each sees dense.cuh with different macros: dense_f64.cu (fp64 Hessians), dense_f32.cu (fp32-stored
// Hessians), csr.cu (CSR Hessians), emu.cu (emulated ranks, a test vehicle).  The rest are separate units only so that
// they compile in parallel.
#pragma once
#include <cuda_runtime.h>

#include <functional>
#include <string>

#include "../../include/ccqp_b200.h"

namespace ccqp {

struct DenseCtx;

// batched.cu (+ batched_sym.cu: the kernels behind `symmetric`) -- returns a ccqp_status; `alloc(bytes)` returns a device workspace of at least that size
int batched_solve_entry(cudaStream_t stream, int sm_count, int solver, const ccqp_params& prm, long long batch, long long n,
                        const double* A, const double* b, const double* x0, const double* lb, const double* ub,
                        const double* uniforms, long long n_uniforms, double* x_out, int memtype, ccqp_result* results,
                        ccqp_result* summary, cudaEvent_t ev0, cudaEvent_t ev1, int* launches, std::string& err,
                        const std::function<void*(size_t)>& alloc, bool symmetric = false);

// the same with a projection table (any block kinds) instead of a Box per problem: the block structure is shared by all
// problems of the batch; per_problem = false: ONE host parameter array `params` for all of them, true: params is
// [batch][n_params] in `memtype` memory, row i for problem i
int batched_solve_table_entry(cudaStream_t stream, int sm_count, int solver, const ccqp_params& prm, long long batch, long long n,
                              const double* A, const double* b, const double* x0, const ccqp_block* blocks, long long n_blocks,
                              const double* params, long long n_params, bool per_problem, const double* uniforms,
                              long long n_uniforms, double* x_out, int memtype, ccqp_result* results, ccqp_result* summary,
                              cudaEvent_t ev0, cudaEvent_t ev1, int* launches, std::string& err,
                              const std::function<void*(size_t)>& alloc);

// upload.cu -- host -> device copy of a square matrix; a symmetric one crosses PCIe as its upper block triangle (checked on the host
// while the copies run) and is mirrored on the device: the device copy is bit-identical to a full upload either way
cudaError_t upload_square_matrix(cudaStream_t stream, double* dst, long long ldd, const double* A, long long n, long long lda,
                                 bool declared_symmetric, bool* used_mirror, long long* bytes);
cudaError_t mirror_lower(cudaStream_t stream, double* dst, long long n, long long ldd);
bool host_matrix_mirrors(const double* A, long long n, long long lda, int threads);
int upload_block_rows();

// One compilation of the dense.cuh solver programs (kernel_build.cuh).  `ctx` points at a DenseCtx, `d_ctxs` at world of
// them in device memory; `op` is a DenseOp, `solver` a ccqp_solver; set_smem_limit: first launch of that kernel on this
// device, raise its dynamic shared-memory limit first.
struct KernelBuild {
    const char* unit;           // translation unit, for error messages
    int index;                  // 0 .. kNumBuilds - 1
    int threads;                // kDenseThreads of that build
    size_t ctx_bytes;           // sizeof(DenseCtx) as that build sees it
    int csr_rows_max;           // CSR tiling of that build (0: no CSR phase)
    cudaError_t (*launch)(int op, const void* ctx, int grid, size_t smem, bool cooperative, bool set_smem_limit,
                          cudaStream_t stream);                         // null: no dense_kernel
    cudaError_t (*launch_emu)(int solver, const void* d_ctxs, int world, int G, size_t smem, bool set_smem_limit,
                              cudaStream_t stream);                     // null: no dense_kernel_emu
};
constexpr int kNumBuilds = 4;
extern const KernelBuild kBuildF64, kBuildF32, kBuildCsr, kBuildEmu;

}  // namespace ccqp
