// C-ABI of the B200-native CCQP hot path (see include/ccqp_b200.h for the contract).
// Host-side code only marshals: it uploads/borrows the Hessian shard, turns the block table into
// the device projection tables, launches ONE persistent cooperative kernel per solve and copies
// the result record back.  No algorithm runs on the CPU here.
#include "../../include/ccqp_b200.h"

#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

#include "dense.cuh"        // DenseCtx, DenseOut and the tiling constants; the kernels are launched through KernelBuild (internal.h)
#include "internal.h"
#include "microbench.cuh"

using namespace ccqp;

struct ccqp_handle {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string last_error;
    // matrix shard: doubles, or floats when a_f32 (ccqp_set_matrix_f32); lda counts entries
    const void* dA = nullptr;
    bool a_f32 = false;
    DevBuf a_own;
    // operator-form (CSR) alternative to dA
    const long long* d_ptr = nullptr;
    const int* d_idx = nullptr;
    const double* d_val = nullptr;
    DevBuf ptr_own, idx_own, val_own, tile_row;   // tile_row: see csr_tile_rows_kernel
    long long nnz = 0;
    bool have_matrix() const { return dA != nullptr || d_val != nullptr; }
    bool upload_mirrored = false;       // the last host matrix was symmetric and crossed PCIe as its upper block triangle
    bool mirror_pending = false;        // ... and the blocks below its block diagonal have not been filled in yet (upload.cu)
    long long upload_bytes = 0;         // bytes of the last host -> device matrix copy
    long long n = 0, lda = 0, row0 = 0, nrows = 0;
    // projection
    bool have_proj = false;
    long long proj_n = 0;
    DevBuf lo, hi, ekind, bkind, boff, bdim, bpar, small_ids, big_ids;
    int nblk = 0, nsmall = 0, nbig = 0, has_cone_ref = 0;
    // workspaces
    DevBuf work, partials, flags, out_dev, uniforms, batched_ws, dbg;
    void* out_host = nullptr;   // pinned
    long long npad = 0;
    long long launches = 0;
    // a solve enqueued by ccqp_solve_async() and not yet collected by ccqp_solve_wait()
    bool pending = false, pending_dbg = false;
    int pending_solver = 0;
    long long pending_launches0 = 0;
    // row-sharded multi-GPU solves: peers' symmetric buffers mapped through CUDA IPC
    int world = 1, rank = 0;
    char* peer_base[kMaxWorld] = {nullptr};
    bool comm_ready = false;
    bool comm_prepared = false;     // ccqp_comm_prepare() ran since the last sharded solve (stale packets would match)
    bool emulated = false;          // rank of an emulated box (ccqp_debug_emulate_ranks): peers live on the same device
    DevBuf emu_ctx;                 // rank 0 of an emulated box: the ranks' kernel contexts
    // cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute of each kernel instantiation: one bit per
    // instantiation (smem_bit), one mask per KernelBuild, kept per handle (a handle owns exactly one device)
    unsigned smem_attr_mask[kNumBuilds] = {};
};

namespace {

// csr_tile_row[g] = the row that contains stored entry g * kCsrTile (the last row whose pointer is <= that entry;
// nrows when the entry lies beyond the end of the stream): which rows a tile of the entry stream touches, without a
// search inside the mat-vec.  One thread per tile boundary, once per matrix.
__global__ void csr_tile_rows_kernel(const long long* __restrict__ ptr, int nrows, int* __restrict__ tile_row, int count) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= count) return;
    const long long nnz = ptr[nrows], E = (long long)g * kCsrTile;
    if (E >= nnz) { tile_row[g] = nrows; return; }
    int lo = 0, hi = nrows;                                    // first r with ptr[r] > E
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (ptr[mid] > E) hi = mid; else lo = mid + 1; }
    tile_row[g] = lo - 1;
}

const char* kStatusText[] = {
    "ok", "invalid argument", "no CUDA device (this library has no CPU path)", "CUDA runtime error",
    "unsupported request", "matrix or projection not set",
    "Cone normal not implemented, yet.", "SPG consumed all supplied uniform samples",
    "Range exceeds valid bounds", "device barrier timed out", "multi-GPU exchange error"};

#define CU(h, call)                                                                  \
    do {                                                                             \
        cudaError_t e__ = (call);                                                    \
        if (e__ != cudaSuccess) {                                                    \
            (h)->last_error = std::string(#call) + ": " + cudaGetErrorString(e__);   \
            return CCQP_ERR_CUDA;                                                    \
        }                                                                            \
    } while (0)

long long round_up(long long v, long long m) { return (v + m - 1) / m * m; }

ccqp_status copy_in(ccqp_handle* h, double* dst, const double* src, long long count, int memtype) {
    CU(h, cudaMemcpyAsync(dst, src, (size_t)count * 8,
                          memtype == CCQP_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
    return CCQP_OK;
}
ccqp_status copy_out(ccqp_handle* h, double* dst, const double* src, long long count, int memtype) {
    CU(h, cudaMemcpyAsync(dst, src, (size_t)count * 8,
                          memtype == CCQP_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
    return CCQP_OK;
}

// slots of the work buffer (each npad doubles)
enum { W_B = 0, W_X0, W_XOUT, W_HIN, W_HOUT, W_YTMP, W_VEC0, W_COUNT = W_VEC0 + kNumVec };

// The work buffer has the layout of the multi-GPU symmetric buffer (common.cuh kSym*Off): flags,
// scalar exchange slots, then the work vectors.  Single GPU: a private allocation.  Sharded: the
// allocation exported to the peers, fixed at ccqp_comm_export() time.
size_t work_bytes(long long npad) { return kSymVecOff + (size_t)W_COUNT * npad * 8; }

ccqp_status ensure_work(ccqp_handle* h) {
    const long long npad = round_up(h->n, 64) + 64;
    if (npad != h->npad || !h->work.p) {
        if (h->world > 1) { h->last_error = "problem size differs from the one given to ccqp_comm_export"; return CCQP_ERR_COMM; }
        CU(h, h->work.ensure(work_bytes(npad)));
        h->npad = npad;
    }
    CU(h, h->partials.ensure((size_t)2 * h->sm_count * kMaxRed * 8));
    CU(h, h->flags.ensure(kSyncBytes));
    CU(h, h->out_dev.ensure(sizeof(DenseOut)));
    if (!h->out_host) CU(h, cudaMallocHost(&h->out_host, 4096));
    return CCQP_OK;
}

struct Tiling { int grid, CW, SW, np, nseg, rows_max, accum; size_t smem; };

// The compilation of the solver kernels that runs a handle's launches (the only place that knows the rule).  The ranks
// of an emulated box run in one launch of dense_kernel_emu: emu.cu's (fp64, dense and CSR phase at the product's CTA
// width) or dense_f32.cu's.
const KernelBuild& build_for(const ccqp_handle* h) {
    if (h->emulated) return h->a_f32 ? kBuildF32 : kBuildEmu;
    return h->d_val ? kBuildCsr : h->a_f32 ? kBuildF32 : kBuildF64;
}

// The kernels take DenseCtx as plain bytes: a build that sees another DenseCtx must not be launched
static_assert(sizeof(DenseCtx) % 8 == 0, "DenseCtx");
bool same_headers(ccqp_handle* h, const KernelBuild& b) {
    if (b.ctx_bytes == sizeof(DenseCtx)) return true;
    h->last_error = std::string(b.unit) + " was built from different headers";
    return false;
}

// the bit of a kernel in smem_attr_mask[build]: dense_kernel<op> (OP_PROJGRAD -> bit 10), dense_kernel_emu<solver> from bit 16
constexpr unsigned smem_bit(int op) { return 1u << (op < 100 ? op : 7 + (op - 100)); }
constexpr unsigned emu_smem_bit(int solver) { return 1u << (16 + solver); }

// the hooks that never touch the matrix (projection-only use): one row per CTA, one 128-column panel
Tiling projection_tiling(const ccqp_handle* h) {
    Tiling t;
    t.grid = (int)std::max<long long>(1, std::min<long long>(h->sm_count, h->n));
    t.CW = 128; t.SW = 128; t.np = 1; t.nseg = 1; t.rows_max = 1; t.accum = 0;
    t.smem = dense_smem_bytes(128, 1, 1);
    return t;
}

// Tuning overrides from the environment are accepted only when they are usable (a bad value is ignored, not obeyed)
int env_int(const char* name, int fallback, bool (*ok)(int)) {
    const char* e = getenv(name);
    if (!e || !*e) return fallback;
    char* end = nullptr;
    const long v = strtol(e, &end, 10);
    if (end == e || *end != 0 || v < INT_MIN || v > INT_MAX || !ok((int)v)) {
        fprintf(stderr, "[ccqp] ignoring %s=%s (not a usable value)\n", name, e);
        return fallback;
    }
    return (int)v;
}
bool ok_mult128(int v) { return v >= 128 && v % 128 == 0 && v <= 16384; }
bool ok_csr_group(int v) { return v == 1 || v == 2 || v == 4 || v == 8 || v == 16 || v == 32; }
bool ok_bool(int v) { return v == 0 || v == 1; }

Tiling choose_tiling(const ccqp_handle* h) {
    Tiling t;
    const long long n = h->n, nrows = h->nrows;
    // One CTA per SM, but never more CTAs than there is work for: a CTA should own at least 8K matrix entries
    // (16K stored entries of a CSR matrix); tiny problems (the reference's own 3x3 tests) then run in ONE CTA,
    // whose syncs are plain __syncthreads() (grid_xsync).
    // Sharded solves: every rank must launch the SAME grid, because the elementwise reductions that every rank
    // repeats on the full vectors are summed CTA by CTA (a different grid = a different summation order = scalars
    // that differ in the last bit across ranks = ranks that may take different branches).  So the grid is derived
    // from n and world only (the even split), never from this rank's own row count or nnz; a rank whose
    // block-aligned shard has fewer rows than CTAs simply has some CTAs without rows (they still take part in
    // the syncs and the elementwise passes).  All ranks of a box have the same SM count.
    const bool sharded = h->world > 1;
    const long long rows_ref = sharded ? std::max<long long>(1, n / h->world) : nrows;
    const long long work = h->d_val ? (sharded ? rows_ref : h->nnz / 16384) : (rows_ref * n) / 8192;
    t.grid = (int)std::max(1LL, std::min<long long>(std::min<long long>(h->sm_count, rows_ref), std::max(1LL, work)));
    t.accum = 0;
    if (h->d_val) {     // CSR: the two panel buffers together are the ring of TMA stages of the entry stream
        // (the psum region holds the row-pointer windows, whose size follows the CTA width of the build that runs them)
        t.CW = kCsrCW; t.SW = kCsrCW; t.np = 1; t.nseg = 1; t.rows_max = build_for(h).csr_rows_max;
        t.smem = dense_smem_bytes(t.CW, t.rows_max, t.nseg);
        return t;
    }
    t.rows_max = (int)((nrows + t.grid - 1) / t.grid) + 1;
    const int cw_cap = (int)round_up(n, 128);
    t.CW = std::min(8192, cw_cap);
    t.SW = std::min(2048, t.CW);
    // tuning overrides (multiples of 128; SW must divide CW)
    t.CW = std::min(env_int("CCQP_CW", t.CW, ok_mult128), cw_cap);
    t.SW = std::min(env_int("CCQP_SW", t.SW, ok_mult128), t.CW);
    if (t.CW % t.SW != 0) t.SW = t.CW;
    const int sw0 = t.SW;
    auto layout = [&]() {
        t.np = (int)((n + t.CW - 1) / t.CW);
        const int spp_full = t.CW / t.SW;
        const int last = (int)(n - (long long)(t.np - 1) * t.CW);
        t.nseg = t.accum ? spp_full : (t.np - 1) * spp_full + (last + t.SW - 1) / t.SW;
        t.smem = dense_smem_bytes(t.CW, t.rows_max, t.nseg);
    };
    for (;;) {
        layout();
        // fewer, wider segments when a CTA owns many rows of a very wide matrix; only while 2 SW still divides CW: the
        // psum slot of (panel p, segment s) is p * (CW / SW) + s, so a width that does not divide CW would give a full
        // panel more segments than slots and its last segment would land in the next panel's first slot
        if (t.smem <= kDenseSmemTarget || t.CW % (2 * t.SW) != 0) break;
        t.SW *= 2;
    }
    if (t.smem > kDenseSmemTarget) {
        // very wide matrices (n beyond ~100k on one GPU): one partial sum per (row, segment of the whole row) no
        // longer fits; keep one slot per (row, segment of a PANEL) and add the panels up in panel order instead
        t.accum = 1;
        t.SW = sw0;
        layout();
    }
    return t;
}

void fill_ctx(ccqp_handle* h, DenseCtx& c, const Tiling& t) {
    std::memset(&c, 0, sizeof(c));
    double* w = reinterpret_cast<double*>(h->work.as<char>() + kSymVecOff);
    c.A = h->dA; c.lda = h->lda; c.n = (int)h->n; c.row0 = (int)h->row0; c.nrows = (int)h->nrows;
    // 4 entries per vector load: 32-byte (fp64) / 16-byte (fp32) aligned rows; a contiguous widened copy of an fp32 matrix
    // takes the same loop as the fp32 original
    c.aligned = ((reinterpret_cast<uintptr_t>(h->dA) & (h->a_f32 ? 15 : 31)) == 0 && (h->lda % 4) == 0) ? 1 : 0;
    c.csr_ptr = h->d_ptr; c.csr_idx = h->d_idx; c.csr_val = h->d_val;
    {
        const double mean = h->d_val ? (double)h->nnz / (double)std::max<long long>(h->nrows, 1) : 0.0;
        // lanes that sum one row out of the shared-memory products: about 8-16 entries per lane
        // (a tile of 4096 entries should hold about as many rows as there are groups: one pass over the rows)
        const double per_tile = build_for(h).threads * mean / kCsrTile;   // lanes per row of a tile
        c.csr_group = per_tile >= 32 ? 32 : per_tile >= 16 ? 16 : per_tile >= 8 ? 8 : per_tile >= 4 ? 4 : per_tile >= 2 ? 2 : 1;
        c.csr_group = env_int("CCQP_CSR_GROUP", c.csr_group, ok_csr_group);
        c.csr_l1 = env_int("CCQP_CSR_L1", 1, ok_bool);
        c.csr_tma = ((reinterpret_cast<uintptr_t>(h->d_val) & 15) == 0 && (reinterpret_cast<uintptr_t>(h->d_idx) & 15) == 0) ? 1 : 0;
        c.csr_tma = std::min(c.csr_tma, env_int("CCQP_CSR_TMA", 1, ok_bool));
        c.csr_tile_row = h->tile_row.as<int>();
    }
    c.b = w + W_B * h->npad; c.x0 = w + W_X0 * h->npad; c.x_out = w + W_XOUT * h->npad;
    c.hook_in = w + W_HIN * h->npad; c.hook_out = w + W_HOUT * h->npad;
    c.ytmp = w + W_YTMP * h->npad;
    for (int i = 0; i < kNumVec; ++i) c.vec[i] = w + (W_VEC0 + i) * h->npad;
    c.T.n = (int)h->n;
    c.T.lo = h->lo.as<double>(); c.T.hi = h->hi.as<double>(); c.T.ekind = h->ekind.as<uint8_t>();
    c.T.nblk = h->nblk; c.T.bkind = h->bkind.as<int>(); c.T.boff = h->boff.as<int>();
    c.T.bdim = h->bdim.as<int>(); c.T.bpar = h->bpar.as<double>();
    c.T.nsmall = h->nsmall; c.T.small_ids = h->small_ids.as<int>();
    c.T.nbig = h->nbig; c.T.big_ids = h->big_ids.as<int>();
    c.T.has_cone_ref = h->has_cone_ref;
    c.T.all_elementwise = (h->nsmall + h->nbig) == 0;
    c.T.e0 = 0; c.T.e1 = (int)h->n;   // every rank repeats the elementwise work on the full vectors
    c.gs.partials = h->partials.as<unsigned long long>();
    c.gs.arrive = reinterpret_cast<unsigned*>(h->flags.as<char>() + kSyncArriveOff);
    c.gs.abort = reinterpret_cast<unsigned*>(h->flags.as<char>() + kSyncAbortOff);
    c.gs.go = reinterpret_cast<unsigned*>(h->flags.as<char>() + kSyncGoOff);
    c.gs.result = reinterpret_cast<unsigned long long*>(h->flags.as<char>() + kSyncResultOff);
    c.gs.closerless = env_int("CCQP_SYNC_CLOSERLESS", 1, ok_bool);
    c.x.world = h->world; c.x.rank = h->rank;
    for (int s = 0; s < kMaxWorld; ++s) c.x.base[s] = (s < h->world) ? h->peer_base[s] : nullptr;
    if (h->world == 1) c.x.base[0] = h->work.as<char>();
    c.out = h->out_dev.as<DenseOut>();
    c.CW = t.CW; c.SW = t.SW; c.np = t.np; c.nseg = t.nseg; c.rows_max = t.rows_max; c.psum_accum = t.accum;
    const double entry_bytes = h->a_f32 ? 4.0 : 8.0;
    c.evict_first = ((double)h->nrows * (double)h->n * entry_bytes > 96.0 * 1024 * 1024) ? 1 : 0;
    c.evict_first = env_int("CCQP_EVICT_FIRST", c.evict_first, ok_bool);
    {   // a shard larger than L2: keep a fixed slice of it resident (same tasks every mat-vec), stream the rest evict-first
        const double shard = (double)h->nrows * (double)h->n * entry_bytes;
        const int mb = env_int("CCQP_L2_RESIDENT_MB", 64, [](int v) { return v >= 0 && v <= 120; });
        const double f = shard > 0 ? (double)mb * 1024.0 * 1024.0 / shard : 0.0;
        c.resident_256 = (int)std::min(256.0, std::floor(f * 256.0 + 0.5));
    }
}

// the device copy of a symmetric host matrix is completed by its first user (upload.cu)
ccqp_status finish_matrix(ccqp_handle* h) {
    if (h->mirror_pending) {
        h->mirror_pending = false;
        CU(h, mirror_lower(h->stream, h->a_own.as<double>(), h->n, h->lda));
        h->launches += 1;
    }
    return CCQP_OK;
}

ccqp_status launch_dense(ccqp_handle* h, int op, DenseCtx& c, const Tiling& t, bool cooperative) {
    if (ccqp_status fs = finish_matrix(h)) return fs;
    if (t.smem > kDenseSmemLimit) {
        h->last_error = "dense tiling needs more shared memory than one SM has";
        return CCQP_ERR_UNSUPPORTED;
    }
    const KernelBuild* b = &build_for(h);
    if (!b->launch) {       // emu.cu has no dense_kernel: the hooks of an emulated fp64 rank run the product's build, which has no CSR phase
        if (c.csr_val) {
            h->last_error = "the unit-test hooks of an emulated rank do not take a CSR matrix";
            return CCQP_ERR_UNSUPPORTED;
        }
        b = &kBuildF64;
    }
    if (!same_headers(h, *b)) return CCQP_ERR_CUDA;
    if (cooperative) CU(h, cudaMemsetAsync(h->flags.p, 0, kSyncBytes, h->stream));   // barrier counters
    unsigned& mask = h->smem_attr_mask[b->index];
    CU(h, b->launch(op, &c, t.grid, t.smem, cooperative, !(mask & smem_bit(op)), h->stream));
    mask |= smem_bit(op);
    h->launches += 1;
    return CCQP_OK;
}

ccqp_status launch_by_solver(ccqp_handle* h, int solver, DenseCtx& c, const Tiling& t) {
    constexpr int kSolverOp[] = {OP_PGD, OP_APGD, OP_APGD_AR, OP_BBPGD, OP_BBPGDF, OP_SPG, OP_MPRGP};   // by ccqp_solver
    if (solver < CCQP_SOLVER_PGD || solver > CCQP_SOLVER_MPRGP) return CCQP_ERR_INVALID_ARG;
    return launch_dense(h, kSolverOp[solver], c, t, true);
}

bool params_ok(const ccqp_params* p, int solver) {
    if (!p) return false;
    if (solver == CCQP_SOLVER_SPG && (p->m < 1 || p->m > kMaxWindow)) return false;
    return true;
}

}  // namespace

long long ccqp::block_param_count(int kind, long long dim) {
    return kind == CCQP_BLOCK_IDENTITY ? 0 : kind == CCQP_BLOCK_BOX ? 2 * dim
           : (kind == CCQP_BLOCK_LOWER || kind == CCQP_BLOCK_UPPER) ? dim : 1;
}

long long ccqp::block_table_unknowns(const ccqp_block* blocks, long long n_blocks, long long n_params) {
    long long n = 0;
    for (long long k = 0; k < n_blocks; ++k) {
        const ccqp_block& b = blocks[k];
        // written so that nothing overflows: n stays <= LLONG_MAX / 2 (so does 2 dim), and param_off <= n_params is
        // tested before n_params - param_off is formed
        if (b.offset != n || b.dim <= 0 || b.dim > LLONG_MAX / 2 - n || b.kind < 0 || b.kind > CCQP_BLOCK_SOC ||
            b.param_off < 0 || b.param_off > n_params || block_param_count(b.kind, b.dim) > n_params - b.param_off)
            return -1;
        n += b.dim;
    }
    return n;
}

extern "C" {

int ccqp_abi_version(void) { return CCQP_ABI_VERSION; }

const char* ccqp_status_string(int status) {
    if (status < 0 || status > 10) return "unknown status";
    return kStatusText[status];
}

const char* ccqp_last_error(const ccqp_handle* h) { return h ? h->last_error.c_str() : ""; }

ccqp_status ccqp_create(ccqp_handle** out, int device) {
    if (!out) return CCQP_ERR_INVALID_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return CCQP_ERR_NO_DEVICE;
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) return CCQP_ERR_NO_DEVICE; }
    if (device >= count) return CCQP_ERR_INVALID_ARG;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return CCQP_ERR_NO_DEVICE;
    if (prop.major != 10) return CCQP_ERR_NO_DEVICE;   // kernels are built for sm_100a only
    ccqp_handle* h = new ccqp_handle();
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&h->ev0) != cudaSuccess || cudaEventCreate(&h->ev1) != cudaSuccess) {
        delete h;
        return CCQP_ERR_CUDA;
    }
    h->own_stream = true;
    *out = h;
    return CCQP_OK;
}

ccqp_status ccqp_destroy(ccqp_handle* h) {
    if (!h) return CCQP_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->world > 1 && !h->emulated) ccqp_comm_detach(h);
    DevBuf* bufs[] = {&h->a_own, &h->lo, &h->hi, &h->ekind, &h->bkind, &h->boff, &h->bdim, &h->bpar, &h->small_ids,
                      &h->big_ids, &h->work, &h->partials, &h->flags, &h->out_dev, &h->uniforms,
                      &h->batched_ws, &h->dbg, &h->ptr_own, &h->idx_own, &h->val_own, &h->emu_ctx, &h->tile_row};
    for (DevBuf* b : bufs) b->release();
    if (h->out_host) cudaFreeHost(h->out_host);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return CCQP_OK;
}

ccqp_status ccqp_set_stream(ccqp_handle* h, void* cuda_stream) {
    if (!h) return CCQP_ERR_INVALID_ARG;
    if (h->own_stream && h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); }
    h->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    h->own_stream = false;
    return CCQP_OK;
}

ccqp_status ccqp_get_info(const ccqp_handle* h, int32_t* sm_count, int32_t* dense_grid, int32_t* dense_threads,
                          int64_t* dense_smem_bytes) {
    if (!h) return CCQP_ERR_INVALID_ARG;
    if (sm_count) *sm_count = h->sm_count;
    if (dense_threads) *dense_threads = kDenseThreads;
    if (h->have_matrix()) {
        Tiling t = choose_tiling(h);
        if (dense_grid) *dense_grid = t.grid;
        if (dense_smem_bytes) *dense_smem_bytes = (int64_t)t.smem;
    } else {
        if (dense_grid) *dense_grid = h->sm_count;
        if (dense_smem_bytes) *dense_smem_bytes = 0;
    }
    return CCQP_OK;
}

// A dense shard of `elem`-byte entries (8: fp64, 4: fp32), borrowed in place from device memory or copied from the host
// into rows padded to a multiple of 4 entries (32- / 16-byte aligned rows for the 256- / 128-bit loads)
static ccqp_status set_matrix_dense(ccqp_handle* h, const void* A, int elem, int64_t n, int64_t lda, int64_t row_begin,
                                    int64_t n_rows, int memtype, bool declared_symmetric) {
    if (!h || !A || n <= 0 || n >= (1LL << 31) - 256 || lda < n || row_begin < 0 || n_rows <= 0 || row_begin + n_rows > n)
        return CCQP_ERR_INVALID_ARG;
    CU(h, cudaSetDevice(h->device));
    h->n = n; h->row0 = row_begin; h->nrows = n_rows;
    h->d_ptr = nullptr; h->d_idx = nullptr; h->d_val = nullptr; h->nnz = 0;
    h->mirror_pending = false; h->upload_mirrored = false;
    if (memtype == CCQP_MEM_DEVICE) {
        h->dA = A; h->lda = lda;
        h->upload_bytes = 0;
    } else {
        const long long ldd = round_up(n, 4);
        CU(h, h->a_own.ensure((size_t)n_rows * ldd * elem + 64));
        if (elem == 8 && row_begin == 0 && n_rows == n) {    // a whole fp64 matrix: half of the PCIe traffic if it turns out to be symmetric (upload.cu)
            CU(h, upload_square_matrix(h->stream, h->a_own.as<double>(), ldd, static_cast<const double*>(A), n, lda, declared_symmetric,
                                       &h->upload_mirrored, &h->upload_bytes));
            h->mirror_pending = h->upload_mirrored;
        } else {
            CU(h, cudaMemcpy2DAsync(h->a_own.p, (size_t)ldd * elem, A, (size_t)lda * elem, (size_t)n * elem, (size_t)n_rows,
                                    cudaMemcpyHostToDevice, h->stream));
            h->upload_bytes = n_rows * n * elem;
        }
        h->dA = h->a_own.p; h->lda = ldd;
    }
    h->a_f32 = elem == 4;
    return CCQP_OK;
}

ccqp_status ccqp_set_matrix(ccqp_handle* h, const double* A, int64_t n, int64_t lda, int64_t row_begin, int64_t n_rows,
                            int memtype) {
    return set_matrix_dense(h, A, 8, n, lda, row_begin, n_rows, memtype, false);
}

ccqp_status ccqp_set_matrix_symmetric(ccqp_handle* h, const double* A, int64_t n, int64_t lda, int memtype) {
    return set_matrix_dense(h, A, 8, n, lda, 0, n, memtype, true);
}

ccqp_status ccqp_set_matrix_f32(ccqp_handle* h, const float* A, int64_t n, int64_t lda, int64_t row_begin, int64_t n_rows,
                                int memtype) {
    return set_matrix_dense(h, A, 4, n, lda, row_begin, n_rows, memtype, false);
}

ccqp_status ccqp_get_upload_info(ccqp_handle* h, int64_t* bytes, int32_t* mirrored) {
    if (!h) return CCQP_ERR_INVALID_ARG;
    if (bytes) *bytes = h->upload_bytes;
    if (mirrored) *mirrored = h->upload_mirrored ? 1 : 0;
    return CCQP_OK;
}

int32_t ccqp_host_matrix_is_block_symmetric(const double* A, int64_t n, int64_t lda, int32_t threads) {
    if (!A || n <= 0 || lda < n) return -1;
    return host_matrix_mirrors(A, n, lda, threads) ? 1 : 0;
}

int32_t ccqp_upload_block_rows(void) { return upload_block_rows(); }

ccqp_status ccqp_set_matrix_csr(ccqp_handle* h, const int64_t* indptr, const int32_t* indices, const double* values,
                                int64_t n, int64_t nnz, int64_t row_begin, int64_t n_rows, int memtype) {
    if (!h || !indptr || n <= 0 || n >= (1LL << 31) - 256 || nnz < 0 || (nnz > 0 && (!indices || !values)) || row_begin < 0 ||
        n_rows <= 0 || row_begin + n_rows > n)
        return CCQP_ERR_INVALID_ARG;
    CU(h, cudaSetDevice(h->device));
    h->n = n; h->row0 = row_begin; h->nrows = n_rows; h->nnz = nnz;
    h->dA = nullptr; h->lda = 0; h->a_f32 = false;
    h->mirror_pending = false; h->upload_mirrored = false; h->upload_bytes = 0;
    if (memtype == CCQP_MEM_DEVICE) {
        h->d_ptr = reinterpret_cast<const long long*>(indptr); h->d_idx = indices; h->d_val = values;
    } else {
        if (indptr[0] != 0 || indptr[n_rows] != nnz) return CCQP_ERR_INVALID_ARG;
        for (int64_t r = 0; r < n_rows; ++r) if (indptr[r + 1] < indptr[r]) return CCQP_ERR_INVALID_ARG;
        for (int64_t q = 0; q < nnz; ++q) if (indices[q] < 0 || indices[q] >= n) return CCQP_ERR_INVALID_ARG;
        CU(h, h->ptr_own.ensure((size_t)(n_rows + 1) * 8));
        CU(h, h->idx_own.ensure((size_t)std::max<int64_t>(nnz, 1) * 4));
        CU(h, h->val_own.ensure((size_t)std::max<int64_t>(nnz, 1) * 8));
        CU(h, cudaMemcpyAsync(h->ptr_own.p, indptr, (size_t)(n_rows + 1) * 8, cudaMemcpyHostToDevice, h->stream));
        if (nnz) {
            CU(h, cudaMemcpyAsync(h->idx_own.p, indices, (size_t)nnz * 4, cudaMemcpyHostToDevice, h->stream));
            CU(h, cudaMemcpyAsync(h->val_own.p, values, (size_t)nnz * 8, cudaMemcpyHostToDevice, h->stream));
        }
        CU(h, cudaStreamSynchronize(h->stream));       // pageable host arrays may go away
        h->d_ptr = h->ptr_own.as<long long>(); h->d_idx = h->idx_own.as<int>(); h->d_val = h->val_own.as<double>();
    }
    const int count = (int)((nnz + kCsrTile - 1) / kCsrTile) + 1;
    CU(h, h->tile_row.ensure((size_t)count * 4));
    csr_tile_rows_kernel<<<(count + 255) / 256, 256, 0, h->stream>>>(h->d_ptr, (int)n_rows, h->tile_row.as<int>(), count);
    CU(h, cudaGetLastError());
    h->launches += 1;
    return CCQP_OK;
}

ccqp_status ccqp_set_projection(ccqp_handle* h, const ccqp_block* blocks, int64_t n_blocks, const double* params,
                                int64_t n_params) {
    if (!h || !blocks || n_blocks <= 0 || (n_params > 0 && !params)) return CCQP_ERR_INVALID_ARG;
    CU(h, cudaSetDevice(h->device));
    const long long n = block_table_unknowns(blocks, n_blocks, n_params);
    if (n < 0 || n >= (1LL << 31) - 256) return CCQP_ERR_INVALID_ARG;
    const long long npad = round_up(n, 64) + 64;
    const double inf = std::numeric_limits<double>::infinity();
    std::vector<double> lo(npad, -inf), hi(npad, inf), bpar(n_blocks, 0.0);
    std::vector<uint8_t> ek(npad, (uint8_t)kIdentity);
    std::vector<int> bkind(n_blocks), boff(n_blocks), bdim(n_blocks), small_ids, big_ids;
    int has_cone = 0;
    for (int64_t k = 0; k < n_blocks; ++k) {
        const ccqp_block& b = blocks[k];
        bkind[k] = b.kind; boff[k] = (int)b.offset; bdim[k] = (int)b.dim;
        const double* p = params ? params + b.param_off : nullptr;
        switch (b.kind) {
            case CCQP_BLOCK_IDENTITY: break;
            case CCQP_BLOCK_LOWER:
                for (long long j = 0; j < b.dim; ++j) { lo[b.offset + j] = p[j]; ek[b.offset + j] = kLower; }
                break;
            case CCQP_BLOCK_UPPER:
                for (long long j = 0; j < b.dim; ++j) { hi[b.offset + j] = p[j]; ek[b.offset + j] = kUpper; }
                break;
            case CCQP_BLOCK_BOX:
                for (long long j = 0; j < b.dim; ++j) { lo[b.offset + j] = p[j]; hi[b.offset + j] = p[b.dim + j]; ek[b.offset + j] = kBox; }
                break;
            default:
                bpar[k] = p[0];
                for (long long j = 0; j < b.dim; ++j) ek[b.offset + j] = kElemNorm;
                (b.dim <= kSmallDim ? small_ids : big_ids).push_back((int)k);
                if (b.kind == CCQP_BLOCK_CONE_REF) has_cone = 1;
        }
    }
    auto up = [&](DevBuf& d, const void* src, size_t bytes) -> cudaError_t {
        cudaError_t e = d.ensure(bytes ? bytes : 8);
        if (e != cudaSuccess || !bytes) return e;
        return cudaMemcpyAsync(d.p, src, bytes, cudaMemcpyHostToDevice, h->stream);
    };
    CU(h, up(h->lo, lo.data(), npad * 8));
    CU(h, up(h->hi, hi.data(), npad * 8));
    CU(h, up(h->ekind, ek.data(), npad));
    CU(h, up(h->bkind, bkind.data(), n_blocks * 4));
    CU(h, up(h->boff, boff.data(), n_blocks * 4));
    CU(h, up(h->bdim, bdim.data(), n_blocks * 4));
    CU(h, up(h->bpar, bpar.data(), n_blocks * 8));
    CU(h, up(h->small_ids, small_ids.data(), small_ids.size() * 4));
    CU(h, up(h->big_ids, big_ids.data(), big_ids.size() * 4));
    CU(h, cudaStreamSynchronize(h->stream));   // the host vectors die here
    h->nblk = (int)n_blocks; h->nsmall = (int)small_ids.size(); h->nbig = (int)big_ids.size();
    h->has_cone_ref = has_cone; h->proj_n = n; h->have_proj = true;
    return CCQP_OK;
}

}  // extern "C"

namespace {
// Everything of a dense solve up to (not including) the kernel launch: argument checks, work buffers, input
// copies on `stream`, the kernel context.  Shared by ccqp_solve_async() and ccqp_debug_solve_emulated().
ccqp_status prepare_dense_solve(ccqp_handle* h, cudaStream_t stream, int solver, const ccqp_params* params, const double* b,
                                const double* x0, const double* uniforms, int64_t n_uniforms, int memtype, bool zero_work,
                                DenseCtx& c, Tiling& t) {
    if (!h || !b || !params_ok(params, solver) || solver < 0 || solver > CCQP_SOLVER_MPRGP) return CCQP_ERR_INVALID_ARG;
    if (h->pending) return CCQP_ERR_NOT_READY;          // one solve in flight per handle
    if (!h->have_matrix() || !h->have_proj) return CCQP_ERR_NOT_READY;
    if (h->proj_n != h->n) return CCQP_ERR_INVALID_ARG;
    if (solver == CCQP_SOLVER_SPG && (n_uniforms < 0 || (n_uniforms > 0 && !uniforms))) return CCQP_ERR_INVALID_ARG;
    CU(h, cudaSetDevice(h->device));
    ccqp_status st = ensure_work(h);
    if (st != CCQP_OK) return st;
    const long long n = h->n, npad = h->npad;
    double* w = reinterpret_cast<double*>(h->work.as<char>() + kSymVecOff);
    // zero everything (vector tails must be zero), then fill.  Real sharded solves: ccqp_comm_prepare() did it
    // before the host-side barrier, because peers write into this buffer as soon as they start.
    if (zero_work) CU(h, cudaMemsetAsync(h->work.p, 0, work_bytes(npad), stream));
    else if (!x0) CU(h, cudaMemsetAsync(w + W_X0 * npad, 0, (size_t)npad * 8, stream));
    const cudaMemcpyKind kind = memtype == CCQP_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    CU(h, cudaMemcpyAsync(w + W_B * npad, b, (size_t)n * 8, kind, stream));
    if (x0) CU(h, cudaMemcpyAsync(w + W_X0 * npad, x0, (size_t)n * 8, kind, stream));
    t = choose_tiling(h);
    fill_ctx(h, c, t);
    c.tol = params->tol; c.max_mv = params->max_mv; c.step = params->step_size;
    c.tau = params->tau; c.sig1 = params->sigma1; c.sig2 = params->sigma2; c.m = params->m;
    if (solver == CCQP_SOLVER_SPG) {
        if (memtype == CCQP_MEM_DEVICE) c.uniforms = uniforms;
        else {
            CU(h, h->uniforms.ensure((size_t)std::max<int64_t>(n_uniforms, 1) * 8));
            if (n_uniforms) CU(h, cudaMemcpyAsync(h->uniforms.p, uniforms, (size_t)n_uniforms * 8, cudaMemcpyHostToDevice, stream));
            c.uniforms = h->uniforms.as<double>();
        }
        c.n_uniforms = n_uniforms;
    }
    return CCQP_OK;
}

void fill_result(const ccqp_handle* h, const DenseOut* o, float ms, long long launches, ccqp_result* result) {
    const long long n = h->n;
    std::memset(result, 0, sizeof(*result));
    result->residual = o->residual;
    result->gpu_seconds = ms * 1e-3;
    result->mv_count = o->mv;
    result->gemv_count = o->gemv;
    result->iterations = o->iters;
    result->uniforms_used = o->draws;
    result->converged = o->converged;
    result->status = o->status;
    // per mat-vec: CSR 12 bytes per stored entry + row pointers, dense 8 (fp32 Hessian: 4) bytes per entry, + v and y
    const double entry_bytes = h->a_f32 ? 4.0 : 8.0;
    result->hbm_bytes = h->d_val ? (double)o->gemv * (12.0 * (double)h->nnz + 8.0 * (double)(h->nrows + 1) + 8.0 * (double)n + 8.0 * (double)h->nrows)
                                 : (double)o->gemv * (entry_bytes * (double)h->nrows * (double)n + 8.0 * (double)n + 8.0 * (double)h->nrows);
    result->kernel_launches = launches;
}
}  // namespace

extern "C" {

ccqp_status ccqp_solve_async(ccqp_handle* h, int solver, const ccqp_params* params, const double* b, const double* x0,
                             const double* uniforms, int64_t n_uniforms, double* x_out, int memtype) {
    if (!h || !x_out) return CCQP_ERR_INVALID_ARG;
    h->last_error.clear();
    if (h->emulated) { h->last_error = "handles of an emulated box solve through ccqp_debug_solve_emulated()"; return CCQP_ERR_UNSUPPORTED; }
    const bool sharded = h->world > 1;
    if (!sharded && h->have_matrix() && (h->row0 != 0 || h->nrows != h->n)) return CCQP_ERR_UNSUPPORTED;   // a shard needs ccqp_comm_attach
    if (sharded && !h->comm_ready) return CCQP_ERR_NOT_READY;
    // the exchange buffer (work vectors, {data, epoch} packet slots) must have been cleared by ccqp_comm_prepare() and
    // a host barrier since the previous solve: packet epochs restart at 1 with every launch, so stale packets would match
    if (sharded && !h->comm_prepared) { h->last_error = "ccqp_comm_prepare() must be called (and the ranks synchronised) before every sharded solve"; return CCQP_ERR_NOT_READY; }
    DenseCtx c;
    Tiling t;
    ccqp_status st = prepare_dense_solve(h, h->stream, solver, params, b, x0, uniforms, n_uniforms, memtype, !sharded, c, t);
    if (st != CCQP_OK) return st;
    h->comm_prepared = false;
    const bool dbg_timing = getenv("CCQP_DEBUG_TIMING") != nullptr;
    if (dbg_timing) {
        CU(h, h->dbg.ensure(kDbgSlots * kDbgIters * 8));
        CU(h, cudaMemsetAsync(h->dbg.p, 0, kDbgSlots * kDbgIters * 8, h->stream));
        c.dbg = h->dbg.as<long long>();
    }
    if ((st = finish_matrix(h)) != CCQP_OK) return st;      // after this solve's own host -> device copies, outside the timed region
    const long long launches0 = h->launches;
    CU(h, cudaEventRecord(h->ev0, h->stream));
    if ((st = launch_by_solver(h, solver, c, t)) != CCQP_OK) return st;
    CU(h, cudaEventRecord(h->ev1, h->stream));
    CU(h, cudaMemcpyAsync(h->out_host, h->out_dev.p, sizeof(DenseOut), cudaMemcpyDeviceToHost, h->stream));
    if ((st = copy_out(h, x_out, c.x_out, h->n, memtype)) != CCQP_OK) return st;
    h->pending = true; h->pending_solver = solver; h->pending_launches0 = launches0; h->pending_dbg = dbg_timing;
    return CCQP_OK;
}

ccqp_status ccqp_solve_wait(ccqp_handle* h, ccqp_result* result) {
    if (!h || !result) return CCQP_ERR_INVALID_ARG;
    if (!h->pending) return CCQP_ERR_NOT_READY;
    h->pending = false;
    CU(h, cudaSetDevice(h->device));
    const int solver = h->pending_solver;
    const long long launches0 = h->pending_launches0;
    const bool dbg_timing = h->pending_dbg;
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) {
        h->last_error = std::string("solver kernel: ") + cudaGetErrorString(e);
        return e == cudaErrorLaunchFailure ? CCQP_ERR_DEVICE_TIMEOUT : CCQP_ERR_CUDA;
    }
    float ms = 0.f;
    CU(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    if (dbg_timing && h->rank == 0) {      // mean time between consecutive stamps of CTA 0 over the recorded iterations, us
        std::vector<long long> t(kDbgSlots * kDbgIters);
        CU(h, cudaMemcpy(t.data(), h->dbg.p, t.size() * 8, cudaMemcpyDeviceToHost));
        double acc[kDbgSlots] = {0};
        int cnt = 0, used = 0;
        for (int it = 1; it + 1 < kDbgIters; ++it) {
            const long long* r = &t[it * kDbgSlots];
            const long long* nx = &t[(it + 1) * kDbgSlots];
            if (!r[0] || !nx[0]) continue;
            int last = 0;
            for (int s = 1; s < kDbgSlots; ++s) if (r[s]) { acc[last] += (r[s] - r[last]) * 1e-3; last = s; }
            acc[last] += (nx[0] - r[last]) * 1e-3;
            used = std::max(used, last + 1);
            ++cnt;
        }
        if (cnt) {
            fprintf(stderr, "[ccqp timing] world %d solver %d, us per phase (mean of %d iterations):", h->world, solver, cnt);
            for (int s = 0; s < used; ++s) fprintf(stderr, " %.1f", acc[s] / cnt);
            fprintf(stderr, "\n");
        }
    }
    const DenseOut* o = reinterpret_cast<const DenseOut*>(h->out_host);
    fill_result(h, o, ms, h->launches - launches0, result);
    return (ccqp_status)o->status;
}

ccqp_status ccqp_solve(ccqp_handle* h, int solver, const ccqp_params* params, const double* b, const double* x0,
                       const double* uniforms, int64_t n_uniforms, double* x_out, int memtype, ccqp_result* result) {
    if (!result) return CCQP_ERR_INVALID_ARG;
    const ccqp_status st = ccqp_solve_async(h, solver, params, b, x0, uniforms, n_uniforms, x_out, memtype);
    if (st != CCQP_OK) return st;
    return ccqp_solve_wait(h, result);
}

static ccqp_status run_hook(ccqp_handle* h, int op, const double* in, double* out, long long n_in, long long n_out,
                            int memtype) {
    if (!h || !in || !out) return CCQP_ERR_INVALID_ARG;
    CU(h, cudaSetDevice(h->device));
    if (op == OP_GEMV) { if (!h->have_matrix()) return CCQP_ERR_NOT_READY; }
    else {
        if (!h->have_proj) return CCQP_ERR_NOT_READY;
        if (!h->have_matrix()) { h->n = h->proj_n; h->row0 = 0; h->nrows = h->proj_n; }   // projection-only use
        else if (h->proj_n != h->n) return CCQP_ERR_INVALID_ARG;
    }
    ccqp_status st = ensure_work(h);
    if (st != CCQP_OK) return st;
    if (h->world > 1) return CCQP_ERR_UNSUPPORTED;   // hooks are single-GPU
    const long long npad = h->npad;
    double* w = reinterpret_cast<double*>(h->work.as<char>() + kSymVecOff);
    CU(h, cudaMemsetAsync(w + W_HIN * npad, 0, (size_t)2 * npad * 8, h->stream));
    if ((st = copy_in(h, w + W_HIN * npad, in, n_in, memtype)) != CCQP_OK) return st;
    const Tiling t = h->have_matrix() ? choose_tiling(h) : projection_tiling(h);
    DenseCtx c;
    fill_ctx(h, c, t);
    if ((st = launch_dense(h, op, c, t, false)) != CCQP_OK) return st;
    if ((st = copy_out(h, out, c.hook_out, n_out, memtype)) != CCQP_OK) return st;
    CU(h, cudaStreamSynchronize(h->stream));
    return CCQP_OK;
}

ccqp_status ccqp_gemv(ccqp_handle* h, const double* v, double* y, int memtype) {
    if (!h) return CCQP_ERR_INVALID_ARG;
    return run_hook(h, OP_GEMV, v, y, h->n, h->nrows, memtype);
}
ccqp_status ccqp_gemv_timed(ccqp_handle* h, const double* v_dev, double* y_dev, int repeats, double* seconds) {
    if (!h || !v_dev || !y_dev || repeats <= 0 || !seconds) return CCQP_ERR_INVALID_ARG;
    if (!h->have_matrix()) return CCQP_ERR_NOT_READY;
    CU(h, cudaSetDevice(h->device));
    ccqp_status st = ensure_work(h);
    if (st != CCQP_OK) return st;
    const Tiling t = choose_tiling(h);
    DenseCtx c;
    fill_ctx(h, c, t);
    c.hook_in = v_dev; c.hook_out = y_dev;
    if ((st = launch_dense(h, OP_GEMV, c, t, false)) != CCQP_OK) return st;   // warm-up
    CU(h, cudaEventRecord(h->ev0, h->stream));
    for (int i = 0; i < repeats; ++i)
        if ((st = launch_dense(h, OP_GEMV, c, t, false)) != CCQP_OK) return st;
    CU(h, cudaEventRecord(h->ev1, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    float ms = 0.f;
    CU(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    *seconds = ms * 1e-3 / repeats;
    return CCQP_OK;
}
ccqp_status ccqp_project(ccqp_handle* h, const double* x, double* out, int memtype) {
    if (!h) return CCQP_ERR_INVALID_ARG;
    return run_hook(h, OP_PROJECT, x, out, h->proj_n, h->proj_n, memtype);
}
ccqp_status ccqp_normal(ccqp_handle* h, const double* x, double* out, int memtype) {
    if (!h) return CCQP_ERR_INVALID_ARG;
    if (h->has_cone_ref) return CCQP_ERR_NORMAL_NOT_IMPLEMENTED;
    return run_hook(h, OP_NORMAL, x, out, h->proj_n, h->proj_n, memtype);
}

ccqp_status ccqp_projected_gradient(ccqp_handle* h, const double* x, const double* g, double* free_out, double* chopped_out,
                                    int memtype) {
    if (!h || !x || !g || !free_out || !chopped_out) return CCQP_ERR_INVALID_ARG;
    if (!h->have_proj) return CCQP_ERR_NOT_READY;
    if (h->nsmall + h->nbig > 0) return h->has_cone_ref ? CCQP_ERR_NORMAL_NOT_IMPLEMENTED : CCQP_ERR_UNSUPPORTED;   // Sphere / Cone / SOC leaves
    if (h->world > 1) return CCQP_ERR_UNSUPPORTED;
    CU(h, cudaSetDevice(h->device));
    if (!h->have_matrix()) { h->n = h->proj_n; h->row0 = 0; h->nrows = h->proj_n; }
    else if (h->proj_n != h->n) return CCQP_ERR_INVALID_ARG;
    ccqp_status st = ensure_work(h);
    if (st != CCQP_OK) return st;
    const long long n = h->proj_n, npad = h->npad;
    double* w = reinterpret_cast<double*>(h->work.as<char>() + kSymVecOff);
    CU(h, cudaMemsetAsync(w + W_HIN * npad, 0, (size_t)2 * npad * 8, h->stream));
    CU(h, cudaMemsetAsync(w + W_VEC0 * npad, 0, (size_t)3 * npad * 8, h->stream));
    if ((st = copy_in(h, w + W_HIN * npad, x, n, memtype)) != CCQP_OK) return st;
    if ((st = copy_in(h, w + W_VEC0 * npad, g, n, memtype)) != CCQP_OK) return st;
    const Tiling t = projection_tiling(h);
    DenseCtx c;
    fill_ctx(h, c, t);
    c.csr_val = nullptr;              // the hooks never touch the matrix
    if ((st = launch_dense(h, OP_NORMAL, c, t, false)) != CCQP_OK) return st;
    if ((st = launch_dense(h, OP_PROJGRAD, c, t, false)) != CCQP_OK) return st;
    if ((st = copy_out(h, free_out, c.vec[1], n, memtype)) != CCQP_OK) return st;
    if ((st = copy_out(h, chopped_out, c.vec[2], n, memtype)) != CCQP_OK) return st;
    CU(h, cudaStreamSynchronize(h->stream));
    return CCQP_OK;
}

// Every batched call: the checks of its arguments, then batched.cu.
static ccqp_status solve_batched(ccqp_handle* h, const BatchedRequest& r) {
    const bool box = r.set == BatchedSet::kBox;
    if (!h || !params_ok(r.params, r.solver) || r.batch <= 0 || r.n <= 0 || !(r.A || r.A32) || !r.b || !r.x_out ||
        (box ? (!r.lb || !r.ub)
             : (!r.blocks || r.n_blocks <= 0 || (r.n_params > 0 && !r.block_params) || (r.set == BatchedSet::kTables && r.n_params < 0))))
        return CCQP_ERR_INVALID_ARG;
    CU(h, cudaSetDevice(h->device));
    return (ccqp_status)batched_solve(r, h->stream, h->sm_count, h->ev0, h->ev1, h->batched_ws, h->launches, h->last_error);
}

ccqp_status ccqp_solve_batched(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch, int64_t n,
                               const double* A, const double* b, const double* x0, const double* lb, const double* ub,
                               const double* uniforms, int64_t n_uniforms, double* x_out, int memtype,
                               ccqp_result* results, ccqp_result* summary) {
    return solve_batched(h, {solver, params, batch, n, A, b, x0, uniforms, n_uniforms, x_out, memtype, results, summary,
                             BatchedSet::kBox, lb, ub, false});
}

ccqp_status ccqp_solve_batched_sym(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch, int64_t n,
                                   const double* A, const double* b, const double* x0, const double* lb, const double* ub,
                                   const double* uniforms, int64_t n_uniforms, double* x_out, int memtype,
                                   ccqp_result* results, ccqp_result* summary) {
    return solve_batched(h, {solver, params, batch, n, A, b, x0, uniforms, n_uniforms, x_out, memtype, results, summary,
                             BatchedSet::kBox, lb, ub, true});
}

ccqp_status ccqp_solve_batched_table(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch, int64_t n,
                                     const double* A, const double* b, const double* x0, const ccqp_block* blocks, int64_t n_blocks,
                                     const double* block_params, int64_t n_params, const double* uniforms, int64_t n_uniforms,
                                     double* x_out, int memtype, ccqp_result* results, ccqp_result* summary) {
    return solve_batched(h, {solver, params, batch, n, A, b, x0, uniforms, n_uniforms, x_out, memtype, results, summary,
                             BatchedSet::kTable, nullptr, nullptr, false, blocks, n_blocks, block_params, n_params});
}

ccqp_status ccqp_solve_batched_tables(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch, int64_t n,
                                      const double* A, const double* b, const double* x0, const ccqp_block* blocks, int64_t n_blocks,
                                      const double* block_params, int64_t n_params, const double* uniforms, int64_t n_uniforms,
                                      double* x_out, int memtype, ccqp_result* results, ccqp_result* summary) {
    return solve_batched(h, {solver, params, batch, n, A, b, x0, uniforms, n_uniforms, x_out, memtype, results, summary,
                             BatchedSet::kTables, nullptr, nullptr, false, blocks, n_blocks, block_params, n_params});
}

// The fp32 twins: the same requests with A32 in place of A
ccqp_status ccqp_solve_batched_f32(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch, int64_t n,
                                   const float* A, const double* b, const double* x0, const double* lb, const double* ub,
                                   const double* uniforms, int64_t n_uniforms, double* x_out, int memtype,
                                   ccqp_result* results, ccqp_result* summary) {
    return solve_batched(h, {solver, params, batch, n, nullptr, b, x0, uniforms, n_uniforms, x_out, memtype, results, summary,
                             BatchedSet::kBox, lb, ub, false, nullptr, 0, nullptr, 0, A});
}

ccqp_status ccqp_solve_batched_sym_f32(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch, int64_t n,
                                       const float* A, const double* b, const double* x0, const double* lb, const double* ub,
                                       const double* uniforms, int64_t n_uniforms, double* x_out, int memtype,
                                       ccqp_result* results, ccqp_result* summary) {
    return solve_batched(h, {solver, params, batch, n, nullptr, b, x0, uniforms, n_uniforms, x_out, memtype, results, summary,
                             BatchedSet::kBox, lb, ub, true, nullptr, 0, nullptr, 0, A});
}

ccqp_status ccqp_solve_batched_table_f32(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch, int64_t n,
                                         const float* A, const double* b, const double* x0, const ccqp_block* blocks,
                                         int64_t n_blocks, const double* block_params, int64_t n_params, const double* uniforms,
                                         int64_t n_uniforms, double* x_out, int memtype, ccqp_result* results,
                                         ccqp_result* summary) {
    return solve_batched(h, {solver, params, batch, n, nullptr, b, x0, uniforms, n_uniforms, x_out, memtype, results, summary,
                             BatchedSet::kTable, nullptr, nullptr, false, blocks, n_blocks, block_params, n_params, A});
}

ccqp_status ccqp_solve_batched_tables_f32(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch, int64_t n,
                                          const float* A, const double* b, const double* x0, const ccqp_block* blocks,
                                          int64_t n_blocks, const double* block_params, int64_t n_params, const double* uniforms,
                                          int64_t n_uniforms, double* x_out, int memtype, ccqp_result* results,
                                          ccqp_result* summary) {
    return solve_batched(h, {solver, params, batch, n, nullptr, b, x0, uniforms, n_uniforms, x_out, memtype, results, summary,
                             BatchedSet::kTables, nullptr, nullptr, false, blocks, n_blocks, block_params, n_params, A});
}

namespace {
__global__ void div3_kernel(const double* a0, const double* a1, const double* a2, const double* b, double* q0, double* q1,
                            double* q2, long long count) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x)
        div3_same_divisor(a0[i], a1[i], a2[i], b[i], q0[i], q1[i], q2[i]);
}
}  // namespace

ccqp_status ccqp_debug_divide(ccqp_handle* h, const double* a0, const double* a1, const double* a2, const double* b,
                            double* q0, double* q1, double* q2, int64_t count) {
    if (!h || !a0 || !a1 || !a2 || !b || !q0 || !q1 || !q2 || count <= 0) return CCQP_ERR_INVALID_ARG;
    CU(h, cudaSetDevice(h->device));
    div3_kernel<<<h->sm_count * 4, 256, 0, h->stream>>>(a0, a1, a2, b, q0, q1, q2, count);
    CU(h, cudaGetLastError());
    CU(h, cudaStreamSynchronize(h->stream));
    h->launches += 1;
    return CCQP_OK;
}

ccqp_status ccqp_fp64_peak(ccqp_handle* h, int blocks_per_sm, int threads_per_block, double* tflops) {
    if (!h || !tflops || blocks_per_sm < 1 || blocks_per_sm > 32 || threads_per_block < 32 || threads_per_block > 256 ||
        threads_per_block % 32 != 0)
        return CCQP_ERR_INVALID_ARG;
    CU(h, cudaSetDevice(h->device));
    CU(h, h->out_dev.ensure(4096));
    const int grid = h->sm_count * blocks_per_sm;
    int iters = 1 << 12;
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {          // rep 0 is the warm-up; the best of the rest counts
        CU(h, cudaEventRecord(h->ev0, h->stream));
        fp64_peak_kernel<<<grid, threads_per_block, 0, h->stream>>>(h->out_dev.as<double>(), iters, 0.999999, 1e-7);
        CU(h, cudaGetLastError());
        CU(h, cudaEventRecord(h->ev1, h->stream));
        CU(h, cudaStreamSynchronize(h->stream));
        float ms = 0.f;
        CU(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        h->launches += 1;
        const double flops = 2.0 * kPeakFmaPerIter * (double)iters * (double)grid * threads_per_block;
        if (rep == 0) { if (ms < 20.f) iters = (int)std::min(1.0e6, iters * 20.0 / std::max(ms, 0.05f)); continue; }
        best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    *tflops = best;
    return CCQP_OK;
}

ccqp_status ccqp_microbench(ccqp_handle* h, double* cycles_per_op, int32_t n_out) {
    if (!h || !cycles_per_op || n_out < PROBE_COUNT) return CCQP_ERR_INVALID_ARG;
    CU(h, cudaSetDevice(h->device));
    CU(h, h->out_dev.ensure(4096));
    long long* dcyc = reinterpret_cast<long long*>(h->out_dev.as<char>() + 1024);
    double* sink = reinterpret_cast<double*>(h->out_dev.as<char>() + 2048);
    const int reps = 2048;
    long long cyc[PROBE_COUNT];
    for (int rep = 0; rep < 2; ++rep) {
        probe_kernel<<<1, 64, 0, h->stream>>>(dcyc, sink, reps, 0.75, 0.999999);
        CU(h, cudaGetLastError());
        CU(h, cudaMemcpyAsync(cyc, dcyc, sizeof(cyc), cudaMemcpyDeviceToHost, h->stream));
        CU(h, cudaStreamSynchronize(h->stream));
        h->launches += 1;
    }
    for (int k = 0; k < PROBE_COUNT; ++k) cycles_per_op[k] = (double)cyc[k] / reps;
    cycles_per_op[PROBE_DFMA_X8_REUSE] /= 8; cycles_per_op[PROBE_DFMA_X8_2RF] /= 8; cycles_per_op[PROBE_DFMA_MATVEC64] /= 64;   // per DFMA
    return CCQP_OK;
}

ccqp_status ccqp_debug_emulate_ranks(ccqp_handle* const* hs, int world, int64_t n) {
    if (!hs || world < 2 || world > kMaxWorld || n <= 0) return CCQP_ERR_INVALID_ARG;
    for (int r = 0; r < world; ++r)
        if (!hs[r] || hs[r]->device != hs[0]->device || (hs[r]->world > 1 && !hs[r]->emulated)) return CCQP_ERR_INVALID_ARG;
    ccqp_handle* h0 = hs[0];
    CU(h0, cudaSetDevice(h0->device));
    cudaDeviceProp prop;
    CU(h0, cudaGetDeviceProperties(&prop, h0->device));
    if (prop.multiProcessorCount / world < 1) return CCQP_ERR_UNSUPPORTED;
    const long long npad = round_up(n, 64) + 64;
    for (int r = 0; r < world; ++r) {
        ccqp_handle* h = hs[r];
        CU(h, cudaStreamSynchronize(h->stream));
        h->work.release();
        CU(h, h->work.ensure(work_bytes(npad)));
        h->npad = npad; h->n = n;
        h->world = world; h->rank = r; h->emulated = true; h->comm_ready = true; h->comm_prepared = false;
        h->sm_count = prop.multiProcessorCount / world;     // all ranks' CTAs must be co-resident in ONE cooperative launch
    }
    for (int r = 0; r < world; ++r)
        for (int s = 0; s < kMaxWorld; ++s) hs[r]->peer_base[s] = s < world ? hs[s]->work.as<char>() : nullptr;
    return CCQP_OK;
}

ccqp_status ccqp_debug_solve_emulated(ccqp_handle* const* hs, int world, int solver, const ccqp_params* params, const double* b,
                                      const double* x0, const double* uniforms, int64_t n_uniforms, double* x_out, int memtype,
                                      ccqp_result* results) {
    if (!hs || !x_out || !results || world < 2 || world > kMaxWorld) return CCQP_ERR_INVALID_ARG;
    for (int r = 0; r < world; ++r)
        if (!hs[r] || !hs[r]->emulated || hs[r]->world != world || hs[r]->rank != r) return CCQP_ERR_INVALID_ARG;
    ccqp_handle* h0 = hs[0];
    h0->last_error.clear();
    for (int r = 1; r < world; ++r)
        if (hs[r]->a_f32 != h0->a_f32) { h0->last_error = "ranks disagree on the matrix type (fp32 / fp64)"; return CCQP_ERR_INVALID_ARG; }
    const KernelBuild& build = build_for(h0);
    if (!same_headers(h0, build)) return CCQP_ERR_CUDA;
    cudaStream_t stream = h0->stream;
    std::vector<DenseCtx> ctxs((size_t)world);
    size_t smem = 0;
    int G = 0;
    for (int r = 0; r < world; ++r) {
        CU(hs[r], cudaStreamSynchronize(hs[r]->stream));          // set_matrix / set_projection copies of this rank
        Tiling t;
        const ccqp_status st = prepare_dense_solve(hs[r], stream, solver, params, b, x0, uniforms, n_uniforms, memtype, true, ctxs[r], t);
        if (st != CCQP_OK) { h0->last_error = hs[r]->last_error; return st; }
        if (r > 0 && t.grid != G) { h0->last_error = "ranks disagree on the grid"; return CCQP_ERR_COMM; }
        G = t.grid;
        smem = std::max(smem, t.smem);
        CU(hs[r], cudaMemsetAsync(hs[r]->flags.p, 0, kSyncBytes, stream));
    }
    if (smem > kDenseSmemLimit) return CCQP_ERR_UNSUPPORTED;
    CU(h0, h0->emu_ctx.ensure(sizeof(DenseCtx) * world));
    CU(h0, cudaMemcpyAsync(h0->emu_ctx.p, ctxs.data(), sizeof(DenseCtx) * world, cudaMemcpyHostToDevice, stream));
    CU(h0, cudaEventRecord(h0->ev0, stream));
    unsigned& mask = h0->smem_attr_mask[build.index];
    CU(h0, build.launch_emu(solver, h0->emu_ctx.p, world, G, smem, !(mask & emu_smem_bit(solver)), stream));
    mask |= emu_smem_bit(solver);
    CU(h0, cudaEventRecord(h0->ev1, stream));
    h0->launches += 1;
    std::vector<DenseOut> outs((size_t)world);
    const cudaMemcpyKind kind = memtype == CCQP_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    for (int r = 0; r < world; ++r) {
        CU(h0, cudaMemcpyAsync(&outs[r], hs[r]->out_dev.p, sizeof(DenseOut), cudaMemcpyDeviceToHost, stream));
        CU(h0, cudaMemcpyAsync(x_out + (size_t)r * hs[r]->n, ctxs[r].x_out, (size_t)hs[r]->n * 8, kind, stream));
    }
    cudaError_t e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) {
        h0->last_error = std::string("emulated solver kernel: ") + cudaGetErrorString(e);
        return e == cudaErrorLaunchFailure ? CCQP_ERR_DEVICE_TIMEOUT : CCQP_ERR_CUDA;
    }
    float ms = 0.f;
    CU(h0, cudaEventElapsedTime(&ms, h0->ev0, h0->ev1));
    for (int r = 0; r < world; ++r) fill_result(hs[r], &outs[r], ms, 1, &results[r]);
    return (ccqp_status)outs[0].status;
}

struct CommDesc {                 // CCQP_COMM_DESC_BYTES = 128
    cudaIpcMemHandle_t handle;    // 64 bytes
    unsigned long long bytes;
    long long n;
    int device, rank, world, abi;
    char pad[128 - 64 - 8 - 8 - 16];
};
static_assert(sizeof(CommDesc) == CCQP_COMM_DESC_BYTES, "descriptor size");

ccqp_status ccqp_comm_export(ccqp_handle* h, int rank, int world, int64_t n, void* desc) {
    if (!h || !desc || world < 2 || world > kMaxWorld || rank < 0 || rank >= world || n <= 0) return CCQP_ERR_INVALID_ARG;
    CU(h, cudaSetDevice(h->device));
    if (h->comm_ready) ccqp_comm_detach(h);
    const long long npad = round_up(n, 64) + 64;
    h->work.release();                                    // a fresh allocation: the IPC handle names its base
    CU(h, h->work.ensure(work_bytes(npad)));
    h->npad = npad; h->n = n;
    CU(h, cudaMemset(h->work.p, 0, work_bytes(npad)));
    CommDesc d;
    std::memset(&d, 0, sizeof(d));
    CU(h, cudaIpcGetMemHandle(&d.handle, h->work.p));
    d.bytes = work_bytes(npad); d.n = n; d.device = h->device; d.rank = rank; d.world = world; d.abi = CCQP_ABI_VERSION;
    std::memcpy(desc, &d, sizeof(d));
    h->world = world; h->rank = rank; h->comm_ready = false;
    return CCQP_OK;
}

ccqp_status ccqp_comm_attach(ccqp_handle* h, const void* all_descs) {
    if (!h || !all_descs || h->world < 2) return CCQP_ERR_INVALID_ARG;
    CU(h, cudaSetDevice(h->device));
    const CommDesc* d = static_cast<const CommDesc*>(all_descs);
    for (int s = 0; s < h->world; ++s) {
        if (d[s].rank != s || d[s].world != h->world || d[s].n != h->n || d[s].abi != CCQP_ABI_VERSION ||
            d[s].bytes != work_bytes(h->npad)) { h->last_error = "inconsistent exchange descriptors"; return CCQP_ERR_COMM; }
        if (s == h->rank) { h->peer_base[s] = h->work.as<char>(); continue; }
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, d[s].handle, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            h->last_error = std::string("cudaIpcOpenMemHandle(rank ") + std::to_string(s) + "): " + cudaGetErrorString(e);
            return CCQP_ERR_COMM;
        }
        h->peer_base[s] = static_cast<char*>(p);
    }
    h->comm_ready = true;
    return CCQP_OK;
}

ccqp_status ccqp_comm_prepare(ccqp_handle* h) {
    if (!h || h->world < 2 || !h->comm_ready) return CCQP_ERR_NOT_READY;
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaMemsetAsync(h->work.p, 0, work_bytes(h->npad), h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    h->comm_prepared = true;
    return CCQP_OK;
}

ccqp_status ccqp_comm_detach(ccqp_handle* h) {
    if (!h) return CCQP_ERR_INVALID_ARG;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    for (int s = 0; s < h->world; ++s)
        if (s != h->rank && h->peer_base[s]) cudaIpcCloseMemHandle(h->peer_base[s]);
    for (int s = 0; s < kMaxWorld; ++s) h->peer_base[s] = nullptr;
    h->world = 1; h->rank = 0; h->comm_ready = false; h->comm_prepared = false;
    return CCQP_OK;
}

}  // extern "C"
