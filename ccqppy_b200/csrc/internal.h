// Entry points between the translation units of libccqp_b200.so: capi.cu (C-ABI, host code), batched.cu (fp64 batched kernels
// and the host side of every batched call) + batched_f32.cu (the same kernels for fp32 A) + batched_sym.cu (batched kernels
// for symmetric Hessians, fp64 and fp32 A), upload.cu (host -> device matrix copies), and the four compilations of the dense solver kernels, one
// unit each because each sees dense.cuh with different macros: dense_f64.cu (fp64 Hessians), dense_f32.cu (fp32-stored
// Hessians), csr.cu (CSR Hessians), emu.cu (emulated ranks, a test vehicle).  The rest are separate units only so that
// they compile in parallel.
#pragma once
#include <cuda_runtime.h>

#include <string>

#include "../../include/ccqp_b200.h"

namespace ccqp {

struct DenseCtx;

// A device buffer that only grows: the handle's workspaces (capi.cu, batched.cu).
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// capi.cu -- the one check of a block table (ccqp_set_projection, batched tables): the blocks tile [0, n) in order from 0,
// every dim > 0, every kind a ccqp_block_kind, param_off >= 0 and param_off + block_param_count() <= n_params, all of it
// without overflow for any 64-bit input (n itself stays <= LLONG_MAX / 2).  Returns n, or -1 for a malformed table.
long long block_table_unknowns(const ccqp_block* blocks, long long n_blocks, long long n_params);
long long block_param_count(int kind, long long dim);      // parameters a block takes from params[param_off ..]

// One batched call: problem i is solve(A[i], b[i], x0[i], op_i) for i < batch, each of n <= 128 unknowns.
enum class BatchedSet {
    kBox,           // Box per problem: lb[i] / ub[i] (ccqp_solve_batched, ccqp_solve_batched_sym)
    kTable,         // one block table for every problem, parameters one host array (ccqp_solve_batched_table)
    kTables,        // one block structure, row i of block_params [batch][n_params] for problem i (ccqp_solve_batched_tables)
};
// capi.cu fills it by aggregate initialisation in this field order: a field is never moved, only appended.
struct BatchedRequest {
    int solver;
    const ccqp_params* params;
    long long batch, n;
    const double* A;                // [batch][n][n]
    const double* b;                // [batch][n]
    const double* x0;               // [batch][n] or null
    const double* uniforms;         // SPG: [batch][n_uniforms]
    long long n_uniforms;
    double* x_out;                  // [batch][n]
    int memtype;                    // where every array above, lb / ub and kTables' block_params live
    ccqp_result* results;           // [batch] or null
    ccqp_result* summary;           // or null
    BatchedSet set;
    // kBox
    const double* lb;               // [batch][n]
    const double* ub;
    bool symmetric;                 // the caller declares every A[i] symmetric: where batched_sym_supported() (batched.cuh)
                                    // only the upper block triangle is read, otherwise the general kernels run
    // kTable / kTables
    const ccqp_block* blocks;
    long long n_blocks;
    const double* block_params;
    long long n_params;
    // the _f32 entry points: A is null and this is the [batch][n][n] Hessian, stored as fp32 (widened exactly in registers)
    const float* A32;
};

// batched.cu (+ batched_sym.cu: the kernels behind `symmetric`) -- the request's arguments are checked for null and
// size already; returns a ccqp_status, adds the kernels it launched to `launches` and, for CCQP_ERR_CUDA, names the failed
// call in `err`.  `ws` is the device workspace, grown as needed.
int batched_solve(const BatchedRequest& r, cudaStream_t stream, int sm_count, cudaEvent_t ev0, cudaEvent_t ev1, DevBuf& ws,
                  long long& launches, std::string& err);

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
