// Translation unit of the batched solver kernels (batched.cuh); see internal.h.
#include "batched.cuh"
#include "internal.h"

namespace ccqp {

int batched_solve_entry(cudaStream_t stream, int sm_count, int solver, const ccqp_params& prm, long long batch, long long n,
                        const double* A, const double* b, const double* x0, const double* lb, const double* ub,
                        const double* uniforms, long long n_uniforms, double* x_out, int memtype, ccqp_result* results,
                        ccqp_result* summary, cudaEvent_t ev0, cudaEvent_t ev1, int* launches, std::string& err,
                        const std::function<void*(size_t)>& alloc, bool symmetric) {
    return batched_solve(stream, sm_count, nullptr, symmetric, solver, prm, batch, n, A, b, x0, lb, ub, uniforms, n_uniforms, x_out,
                         memtype, results, summary, ev0, ev1, launches, err, alloc);
}

// The same validation as ccqp_set_projection (capi.cu), for a table of n <= 128 unknowns, and its per-element expansion: the
// kind and norm block of every element, and where in a parameter row its lower bound, upper bound and block parameter sit.
// The values themselves are read by the kernel, from the row of the problem being solved.
static int batched_table_layout(const ccqp_block* blocks, long long n_blocks, long long n, long long n_params, BatchedTable& tab) {
    tab.ekind.assign(kBNMax, (uint8_t)kIdentity);
    tab.eoff.assign(kBNMax, 0); tab.edim.assign(kBNMax, 0); tab.enk.assign(kBNMax, 0);
    tab.eidx.assign(4 * n, -1);
    auto ilo = [&](long long i) -> int& { return tab.eidx[4 * i]; };
    auto ihi = [&](long long i) -> int& { return tab.eidx[4 * i + 1]; };
    auto ipar = [&](long long i) -> int& { return tab.eidx[4 * i + 2]; };
    long long at = 0;
    for (long long k = 0; k < n_blocks; ++k) {
        const ccqp_block& bl = blocks[k];
        if (bl.offset != at || bl.dim <= 0 || bl.kind < 0 || bl.kind > CCQP_BLOCK_SOC || bl.param_off < 0 || at + bl.dim > n)
            return CCQP_ERR_INVALID_ARG;
        const long long need = (bl.kind == CCQP_BLOCK_IDENTITY) ? 0 : (bl.kind == CCQP_BLOCK_BOX) ? 2 * bl.dim
                               : (bl.kind == CCQP_BLOCK_LOWER || bl.kind == CCQP_BLOCK_UPPER) ? bl.dim : 1;
        if (bl.param_off + need > n_params || bl.param_off + need > INT_MAX) return CCQP_ERR_INVALID_ARG;
        const int p = (int)bl.param_off;
        for (long long j = 0; j < bl.dim; ++j) {
            const long long i = at + j;
            switch (bl.kind) {
                case CCQP_BLOCK_IDENTITY: break;
                case CCQP_BLOCK_LOWER: ilo(i) = p + (int)j; tab.ekind[i] = kLower; break;
                case CCQP_BLOCK_UPPER: ihi(i) = p + (int)j; tab.ekind[i] = kUpper; break;
                case CCQP_BLOCK_BOX: ilo(i) = p + (int)j; ihi(i) = p + (int)(bl.dim + j); tab.ekind[i] = kBox; break;
                default:
                    tab.ekind[i] = kElemNorm; tab.eoff[i] = (int)at; tab.edim[i] = (int)bl.dim; tab.enk[i] = bl.kind; ipar(i) = p;
                    tab.has_norm = 1;
            }
        }
        at += bl.dim;
    }
    return at == n ? CCQP_OK : CCQP_ERR_INVALID_ARG;
}

int batched_solve_table_entry(cudaStream_t stream, int sm_count, int solver, const ccqp_params& prm, long long batch, long long n,
                              const double* A, const double* b, const double* x0, const ccqp_block* blocks, long long n_blocks,
                              const double* params, long long n_params, bool per_problem, const double* uniforms,
                              long long n_uniforms, double* x_out, int memtype, ccqp_result* results, ccqp_result* summary,
                              cudaEvent_t ev0, cudaEvent_t ev1, int* launches, std::string& err,
                              const std::function<void*(size_t)>& alloc) {
    if (n > kBNMax) return CCQP_ERR_UNSUPPORTED;
    BatchedTable tab;
    const int st = batched_table_layout(blocks, n_blocks, n, n_params, tab);
    if (st != CCQP_OK) return st;
    tab.params = params; tab.n_params = n_params; tab.per_problem = per_problem;
    return batched_solve(stream, sm_count, &tab, false, solver, prm, batch, n, A, b, x0, nullptr, nullptr, uniforms, n_uniforms, x_out,
                         memtype, results, summary, ev0, ev1, launches, err, alloc);
}

}  // namespace ccqp
