// Entry points between the translation units of libccqp_b200.so (the kernels are split over several .cu files
// only so that they compile in parallel): capi.cu (C-ABI, dense kernels), batched.cu (batched kernels),
// emu.cu (emulated-ranks instantiations of the dense kernels, a test vehicle), csr.cu (CSR Hessians),
// dense_f32.cu (fp32-stored dense Hessians).
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

// the same with ONE projection table (any block kinds) shared by all problems of the batch instead of a Box per problem
int batched_solve_table_entry(cudaStream_t stream, int sm_count, int solver, const ccqp_params& prm, long long batch, long long n,
                              const double* A, const double* b, const double* x0, const ccqp_block* blocks, long long n_blocks,
                              const double* params, long long n_params, const double* uniforms, long long n_uniforms, double* x_out,
                              int memtype, ccqp_result* results, ccqp_result* summary, cudaEvent_t ev0, cudaEvent_t ev1, int* launches,
                              std::string& err, const std::function<void*(size_t)>& alloc);

// upload.cu -- host -> device copy of a square matrix; a symmetric one crosses PCIe as its upper block triangle (checked on the host
// while the copies run) and is mirrored on the device: the device copy is bit-identical to a full upload either way
cudaError_t upload_square_matrix(cudaStream_t stream, double* dst, long long ldd, const double* A, long long n, long long lda,
                                 bool declared_symmetric, bool* used_mirror, long long* bytes);
cudaError_t mirror_lower(cudaStream_t stream, double* dst, long long n, long long ldd);
bool host_matrix_mirrors(const double* A, long long n, long long lda, int threads);
int upload_block_rows();

// emu.cu -- one cooperative launch of dense_kernel_emu<solver> over world * G CTAs
cudaError_t launch_dense_emu(int solver, const DenseCtx* d_ctxs, int world, int G, size_t smem, cudaStream_t stream);

// csr.cu -- the solver kernels compiled for CSR Hessians (many warps per SM, dense mat-vec loop compiled out); `ctx` points
// at a DenseCtx, `op` is a DenseOp.  csr_variant_smem(): dynamic shared memory of that build's CSR tiling.
int csr_variant_threads();
size_t csr_variant_smem();
int csr_variant_rows_max();
size_t csr_variant_ctx_bytes();
cudaError_t csr_variant_launch(int op, const void* ctx, int grid, size_t smem, bool cooperative, cudaStream_t stream);

// dense_f32.cu -- the dense solver kernels compiled for an fp32-stored Hessian (widened in registers); `ctx` points at a
// DenseCtx (`d_ctxs`: world of them in device memory), `op` is a DenseOp, `solver` a ccqp_solver
size_t f32_variant_ctx_bytes();
cudaError_t f32_variant_launch(int op, const void* ctx, int grid, size_t smem, bool cooperative, cudaStream_t stream);
cudaError_t f32_variant_launch_emu(int solver, const void* d_ctxs, int world, int G, size_t smem, cudaStream_t stream);

}  // namespace ccqp
