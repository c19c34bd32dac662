// Translation unit of the fp64 batched solver kernels (batched.cuh; the fp32 ones: batched_f32.cu) and of the host side of
// every batched call: a BatchedRequest (internal.h) becomes one kernel context and one persistent launch.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "batched.cuh"
#include "internal.h"

namespace ccqp {

cudaError_t launch_persistent(const void* kern, int threads, size_t dyn, const BatchedCtx& c, int sm_count, cudaStream_t stream) {
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    cudaError_t e = dyn ? cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn) : cudaSuccess;
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, dyn);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    if (const char* v = getenv("CCQP_BATCHED_CTAS_PER_SM")) per_sm = std::max(1, std::min(per_sm, atoi(v)));   // tuning hook
    long long grid = (long long)sm_count * per_sm;
    if (grid > c.batch) grid = c.batch;
    void* args[] = {const_cast<BatchedCtx*>(&c)};
    const cudaError_t launched = cudaLaunchKernel(kern, dim3((unsigned)grid), dim3(threads), args, dyn, stream);
    const cudaError_t last = cudaGetLastError();        // clears the launch error, as after a <<< >>> launch
    return launched != cudaSuccess ? launched : last;
}

namespace {

// Smallest double q >= 0 with pred(sqrt(q)) false ... expressed through the bit pattern: for
// non-negative doubles the IEEE ordering equals the ordering of the bit patterns, and sqrt is
// monotone and correctly rounded on both host and device, so the reference's test on sqrt(q)
// is equivalent to a comparison of q with a threshold found by bisection.
double sqrt_threshold(double tol, bool strict) {
    // strict:  returns thr with  (q <  thr) <=> (sqrt(q) <  tol)
    // !strict: returns thr with  (q <= thr) <=> (sqrt(q) <= tol)
    if (tol != tol) return NAN;                                   // every comparison is false
    auto holds = [&](unsigned long long bits) {
        double q; std::memcpy(&q, &bits, 8);
        const double r = std::sqrt(q);
        return strict ? (r < tol) : (r <= tol);
    };
    const unsigned long long inf_bits = 0x7ff0000000000000ULL;
    if (!holds(0)) return strict ? 0.0 : -1.0;                    // never true for q >= 0
    if (holds(inf_bits)) return strict ? NAN : INFINITY;          // tol = +inf (strict: inf < inf is false, handled below)
    unsigned long long lo = 0, hi = inf_bits;                     // holds(lo), !holds(hi)
    while (hi - lo > 1) {
        const unsigned long long mid = lo + (hi - lo) / 2;
        if (holds(mid)) lo = mid; else hi = mid;
    }
    double out;
    const unsigned long long pick = strict ? hi : lo;
    std::memcpy(&out, &pick, 8);
    return out;
}

// The block structure of a table per element: its kind and norm block, and where in a parameter row its lower bound, upper
// bound and block parameter sit.  The values themselves are read by the kernel, from the row of the problem being solved.
struct BatchedTable {
    std::vector<uint8_t> ekind;
    std::vector<int> eoff, edim, enk;
    std::vector<int> eidx;          // [n][4]: lower bound / upper bound / block parameter index into a row, -1: none
    int has_norm = 0;
};

// false: the table is malformed for this call (block_table_unknowns, it covers [0, n), every index fits an int)
bool expand_table(const BatchedRequest& r, BatchedTable& tab) {
    if (block_table_unknowns(r.blocks, r.n_blocks, r.n_params) != r.n) return false;
    tab.ekind.assign(kBNMax, (uint8_t)kIdentity);
    tab.eoff.assign(kBNMax, 0); tab.edim.assign(kBNMax, 0); tab.enk.assign(kBNMax, 0);
    tab.eidx.assign(4 * r.n, -1);
    for (long long k = 0; k < r.n_blocks; ++k) {
        const ccqp_block& bl = r.blocks[k];
        if (bl.param_off + block_param_count(bl.kind, bl.dim) > INT_MAX) return false;
        const int p = (int)bl.param_off;
        for (long long j = 0; j < bl.dim; ++j) {
            const long long i = bl.offset + j;
            int* e = &tab.eidx[4 * i];
            switch (bl.kind) {
                case CCQP_BLOCK_IDENTITY: break;
                case CCQP_BLOCK_LOWER: e[0] = p + (int)j; tab.ekind[i] = kLower; break;
                case CCQP_BLOCK_UPPER: e[1] = p + (int)j; tab.ekind[i] = kUpper; break;
                case CCQP_BLOCK_BOX: e[0] = p + (int)j; e[1] = p + (int)(bl.dim + j); tab.ekind[i] = kBox; break;
                default:
                    tab.ekind[i] = kElemNorm; tab.eoff[i] = (int)bl.offset; tab.edim[i] = (int)bl.dim; tab.enk[i] = bl.kind;
                    e[2] = p;
                    tab.has_norm = 1;
            }
        }
    }
    return true;
}

}  // namespace

int batched_solve(const BatchedRequest& r, cudaStream_t stream, int sm_count, cudaEvent_t ev0, cudaEvent_t ev1, DevBuf& ws,
                  long long& launches, std::string& err) {
#define BCU(call)                                                                                  \
    do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { err = std::string(#call) + ": " + cudaGetErrorString(e__); return CCQP_ERR_CUDA; } } while (0)
    const long long batch = r.batch, n = r.n, n_uniforms = r.n_uniforms;
    const int solver = r.solver;
    const ccqp_params& prm = *r.params;
    const bool table = r.set != BatchedSet::kBox, per_problem = r.set == BatchedSet::kTables;
    if (n > kBNMax) return CCQP_ERR_UNSUPPORTED;
    BatchedTable tab;
    if (table && !expand_table(r, tab)) return CCQP_ERR_INVALID_ARG;
    if (table && solver == CCQP_SOLVER_MPRGP) return CCQP_ERR_UNSUPPORTED;     // batched MPRGP: Box per problem only
    if (batch >= (1LL << 31) - 1024) return CCQP_ERR_INVALID_ARG;
    const bool host = r.memtype == CCQP_MEM_HOST;
    if (solver == CCQP_SOLVER_SPG && (n_uniforms < 0 || (n_uniforms > 0 && !r.uniforms))) return CCQP_ERR_INVALID_ARG;
    if (solver < 0 || solver > CCQP_SOLVER_MPRGP) return CCQP_ERR_INVALID_ARG;
    // A is fp64, or fp32 for the _f32 entry points (r.A32): the kernels widen it in registers, nothing else changes
    const bool f32 = r.A32 != nullptr;
    const void* A = f32 ? static_cast<const void*>(r.A32) : static_cast<const void*>(r.A);
    const long long esz = f32 ? 4 : 8;
    const size_t szA = (size_t)batch * n * n * esz, szV = (size_t)batch * n * 8;
    const size_t szU = (solver == CCQP_SOLVER_SPG) ? (size_t)batch * n_uniforms * 8 : 0;
    const size_t szO = (size_t)batch * sizeof(BatchedOut);
    auto al = [](size_t v) { return (v + 255) / 256 * 256; };
    // parameter rows of a general table: a shared row and the rows of a host array are copied with an even pitch, so that
    // every row starts 16-byte aligned and its bulk copy (rounded up to 16 bytes) stays inside the copy
    const long long np = table ? std::max(r.n_params, 0LL) : 0, ppitch = np + (np & 1);
    const size_t szP = !table ? 0 : !per_problem ? (size_t)ppitch * 8 : host ? (size_t)batch * ppitch * 8 : 0;
    size_t total = 256 + al(szO) + 8 * al((size_t)kBNMax * 8) + al(szP);
    if (host) total += al(szA) + 4 * al(szV) + al(szV) + al(szU);
    unsigned char* wsp = static_cast<unsigned char*>(ws.ensure(total) == cudaSuccess ? ws.p : nullptr);
    if (!wsp) { err = "workspace allocation failed"; return CCQP_ERR_CUDA; }
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char* p = wsp + off; off += al(bytes); return p; };
    unsigned* counter = reinterpret_cast<unsigned*>(take(256));
    BatchedOut* dout = reinterpret_cast<BatchedOut*>(take(szO));
    BatchedCtx c;
    std::memset(&c, 0, sizeof(c));
    if (host) {
        void* dA = take(szA);
        double* db = reinterpret_cast<double*>(take(szV));
        double* dlb = reinterpret_cast<double*>(take(szV));
        double* dub = reinterpret_cast<double*>(take(szV));
        double* dx0 = reinterpret_cast<double*>(take(szV));
        double* dxo = reinterpret_cast<double*>(take(szV));
        double* du = szU ? reinterpret_cast<double*>(take(szU)) : nullptr;
        BCU(cudaMemcpyAsync(dA, A, szA, cudaMemcpyHostToDevice, stream));
        BCU(cudaMemcpyAsync(db, r.b, szV, cudaMemcpyHostToDevice, stream));
        if (!table) BCU(cudaMemcpyAsync(dlb, r.lb, szV, cudaMemcpyHostToDevice, stream));
        if (!table) BCU(cudaMemcpyAsync(dub, r.ub, szV, cudaMemcpyHostToDevice, stream));
        if (r.x0) BCU(cudaMemcpyAsync(dx0, r.x0, szV, cudaMemcpyHostToDevice, stream));
        if (du) BCU(cudaMemcpyAsync(du, r.uniforms, szU, cudaMemcpyHostToDevice, stream));
        c.A = dA; c.b = db; c.lb = dlb; c.ub = dub; c.x0 = r.x0 ? dx0 : nullptr; c.uniforms = du; c.x_out = dxo;
    } else {
        c.A = A; c.b = r.b; c.lb = r.lb; c.ub = r.ub; c.x0 = r.x0; c.uniforms = (solver == CCQP_SOLVER_SPG) ? r.uniforms : nullptr;
        c.x_out = r.x_out;
    }
    c.bound_stride = n;
    if (table) {    // the block structure: five small per-element arrays, uploaded once per call
        auto up = [&](const void* src, size_t bytes) -> void* {
            void* d = take(bytes);
            return cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, stream) == cudaSuccess ? d : nullptr;
        };
        c.ekind = static_cast<const uint8_t*>(up(tab.ekind.data(), (size_t)n));
        c.eoff = static_cast<const int*>(up(tab.eoff.data(), (size_t)n * 4));
        c.edim = static_cast<const int*>(up(tab.edim.data(), (size_t)n * 4));
        c.enk = static_cast<const int*>(up(tab.enk.data(), (size_t)n * 4));
        c.eidx = static_cast<const int4*>(up(tab.eidx.data(), (size_t)n * 16));
        if (!c.ekind || !c.eoff || !c.edim || !c.enk || !c.eidx) { err = "table upload failed"; return CCQP_ERR_CUDA; }
        c.has_norm = tab.has_norm;
        c.lb = c.ub = nullptr;
        // the parameter rows: one shared row (stride 0), a host array copied with an even pitch, or a device array in place
        if (np > 0 && (!per_problem || host)) {
            double* dp = reinterpret_cast<double*>(take(szP));
            const long long rows = per_problem ? batch : 1;
            if (ppitch == np) BCU(cudaMemcpyAsync(dp, r.block_params, (size_t)rows * np * 8, cudaMemcpyHostToDevice, stream));
            else BCU(cudaMemcpy2DAsync(dp, (size_t)ppitch * 8, r.block_params, (size_t)np * 8, (size_t)np * 8, (size_t)rows,
                                       cudaMemcpyHostToDevice, stream));
            c.params = dp;
            c.param_stride = per_problem ? ppitch : 0;
        } else {
            c.params = np > 0 ? r.block_params : nullptr;
            c.param_stride = np;
        }
    }
    c.n_uniforms = (solver == CCQP_SOLVER_SPG) ? n_uniforms : 0;
    c.out = dout; c.counter = counter;
    c.batch = (int)batch; c.n = (int)n;
    // an fp32 A with n % 4 != 0 (rows not 16-byte multiples) or a base off a 16-byte boundary takes the per-element global
    // loads: no copy is ever rounded up past the end of [batch][n][n]
    c.tma_ok = ((n * esz) % 16 == 0 && (reinterpret_cast<uintptr_t>(c.A) & 15) == 0) ? 1 : 0;
    c.vec_ok = (!f32 && n % 4 == 0 && (reinterpret_cast<uintptr_t>(c.A) & 31) == 0) ? 1 : 0;
    c.pf_ok = ((n * n * esz) % 16 == 0 && (reinterpret_cast<uintptr_t>(c.A) & 15) == 0) ? 1 : 0;
    c.vtma_ok = (n % 2 == 0 && ((reinterpret_cast<uintptr_t>(c.b) | reinterpret_cast<uintptr_t>(c.lb) | reinterpret_cast<uintptr_t>(c.ub)) & 15) == 0) ? 1 : 0;
    if (table) {    // a parameter row is staged with b when every row is 16-byte aligned and fits vstage[1..2] (2 N doubles)
        const long long N = n <= kBN ? kBN : kBNMax;
        const bool rows_ok = np == 0 || (c.param_stride % 2 == 0 && (reinterpret_cast<uintptr_t>(c.params) & 15) == 0 && ppitch <= 2 * N);
        c.vtma_ok = (c.vtma_ok && rows_ok) ? 1 : 0;
        c.prow_bytes = c.vtma_ok ? (int)(ppitch * 8) : 0;
    }
    c.tol = prm.tol; c.max_mv = prm.max_mv; c.step = prm.step_size;
    c.tau = prm.tau; c.sig1 = prm.sigma1; c.sig2 = prm.sigma2; c.m = prm.m;
    c.thr_lt = sqrt_threshold(prm.tol, true);
    c.thr_le = sqrt_threshold(prm.tol, false);
    c.max_mv_i = (prm.max_mv != prm.max_mv || prm.max_mv >= 2147483000.0) ? INT_MAX
                 : (prm.max_mv <= -2147483000.0 ? INT_MIN : (int)std::ceil(prm.max_mv));
    BCU(cudaMemsetAsync(counter, 0, 256, stream));
    BCU(cudaEventRecord(ev0, stream));
    const bool wreg = prm.m == kBWinReg;
    const bool use_sym = r.symmetric && !table && batched_sym_supported(solver, n);
    auto launch = [&](auto elem) {
        using TA = decltype(elem);
        return use_sym ? launch_batched_sym<TA>(c, solver, wreg, sm_count, stream)
               : table ? launch_batched<true, TA>(c, solver, wreg, sm_count, stream)
                       : launch_batched<false, TA>(c, solver, wreg, sm_count, stream);
    };
    BCU(f32 ? launch(float{}) : launch(double{}));
    launches += 1;
    BCU(cudaEventRecord(ev1, stream));
    if (host) BCU(cudaMemcpyAsync(r.x_out, c.x_out, szV, cudaMemcpyDeviceToHost, stream));
    std::vector<BatchedOut> hout((size_t)batch);
    BCU(cudaMemcpyAsync(hout.data(), dout, szO, cudaMemcpyDeviceToHost, stream));
    BCU(cudaStreamSynchronize(stream));
    float ms = 0.f;
    BCU(cudaEventElapsedTime(&ms, ev0, ev1));
    long long tot_mv = 0, tot_gemv = 0, tot_it = 0, tot_dr = 0, nconv = 0;
    int first_status = 0;
    double hbmA = (double)esz * n * n;          // bytes of A[i] the kernel reads
    if (use_sym) { hbmA = 0; for (long long i = 0; i < n; ++i) hbmA += (double)esz * (double)(n - 8 * (i / 8)); }
    if (per_problem) hbmA += 8.0 * (double)np;  // the problem's parameter row
    for (long long i = 0; i < batch; ++i) {
        const BatchedOut& o = hout[(size_t)i];
        if (r.results) {
            ccqp_result& res = r.results[i];
            std::memset(&res, 0, sizeof(res));
            res.residual = o.residual; res.mv_count = o.mv; res.gemv_count = o.gemv; res.iterations = o.iters;
            res.uniforms_used = o.draws; res.converged = o.converged; res.status = o.status;
            res.hbm_bytes = hbmA + 8.0 * n * (r.x0 ? 5 : 4);
        }
        tot_mv += o.mv; tot_gemv += o.gemv; tot_it += o.iters; tot_dr += o.draws; nconv += o.converged;
        if (o.status && !first_status) first_status = o.status;
    }
    if (ccqp_result* summary = r.summary) {
        std::memset(summary, 0, sizeof(*summary));
        summary->gpu_seconds = ms * 1e-3;
        summary->mv_count = tot_mv; summary->gemv_count = tot_gemv; summary->iterations = tot_it;
        summary->uniforms_used = tot_dr; summary->converged = (nconv == batch) ? 1 : 0;
        summary->status = first_status;
        summary->hbm_bytes = (double)batch * (hbmA + 8.0 * n * (r.x0 ? 5 : 4)) + 8.0 * (double)tot_dr;
        summary->kernel_launches = 1;
        summary->residual = NAN;
    }
    return CCQP_OK;
#undef BCU
}

}  // namespace ccqp
