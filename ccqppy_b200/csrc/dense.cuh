// Dense CCQP solvers as ONE persistent cooperative kernel per solve (sm_100a).
//
// Layout of a solve on the device
//   * grid = one CTA per SM (kDenseThreads threads), launched cooperatively; CTA c owns a
//     contiguous band of rows of the (row-shard of the) Hessian A for every mat-vec of the solve.
//   * the solver loop of the reference (solvers.py) runs entirely inside the kernel: phases are
//     separated by a grid barrier; scalar control flow (step lengths, stopping tests, branch
//     choices) is evaluated redundantly and bit-identically by every thread from
//     deterministically reduced partial sums, so all CTAs take the same branches with no host
//     round trip.
//   * mat-vec phase (gemv_phase): the input vector is staged into shared memory in column panels
//     by the TMA engine (cp.async.bulk + mbarrier, double buffered); A is streamed exactly once
//     with 256-bit read-only loads (16 in flight per lane), FMA-accumulated per lane and reduced
//     with warp shuffles; work inside a CTA is split into (row, column-segment) tasks so that all
//     warps stay busy even when a CTA owns only a few rows (the 8-GPU row shard).  The epilogue
//     functor of each solver fuses "+ b", the vector updates and the row-local dot products.
//   * elementwise phases (projection, axpy, residual terms, masks) run over the grid with the
//     functor-based project_pass of proj.cuh.
//
// Algorithmic bytes per mat-vec: 8 * n_rows * n (A) + 8 n (v) + 8 n_rows (y)   (SURVEY 8d).
// fp32 build (CCQP_A_F32, dense_f32.cu): A is stored as fp32 and widened in registers, 4 * n_rows * n for A.
#pragma once
#include "proj.cuh"

namespace ccqp {

// 256 threads x 16 loads in flight per lane (128 KB in flight per SM), not 512 x 4: the mat-vec loop is
// inlined into solver programs that keep 50-70 registers of their own state live across it, and at
// 128 registers per thread (512 threads) the loop of the larger programs spilled and streamed at
// 4.3 TB/s (MPRGP) instead of 6.5; with 255 registers per thread every program runs the same loop.
// In isolation 512 x 4 is 3 % faster (profiles/r01_gemv_sweep.log), inside the solvers it is not.
#ifndef CCQP_DENSE_THREADS
#define CCQP_DENSE_THREADS 256
#endif
#ifndef CCQP_UNROLL
#define CCQP_UNROLL 16
#endif
#ifndef CCQP_DENSE_LDS
#define CCQP_DENSE_LDS 0      // 1: the dense loop reads the staged vector panel with explicit ld.shared (A/B build, profiles/README.md)
#endif
#ifndef CCQP_CSR_ONLY
#define CCQP_CSR_ONLY 0       // 1: the dense mat-vec loop is compiled out (csr.cu: the many-warps build of the solver programs)
#endif
#ifndef CCQP_DENSE_ONLY
#define CCQP_DENSE_ONLY 0     // 1: the CSR mat-vec phase is compiled out (dense_f64.cu: the product's dense kernels carry no CSR code --
#endif                        //    the register allocation and the schedule of the dense loop depend on everything inlined next to it)
#ifndef CCQP_A_F32
#define CCQP_A_F32 0          // 1: the dense Hessian is stored as fp32 and widened to fp64 in registers (dense_f32.cu)
#endif
#ifndef CCQP_UNROLL_F32
#define CCQP_UNROLL_F32 32    // fp32 build: 128-bit loads in flight per lane (32 x 16 bytes = the fp64 loop's 16 x 32)
#endif
constexpr int kDenseThreads = CCQP_DENSE_THREADS;
constexpr int kDenseWarps = kDenseThreads / 32;
constexpr int kUnroll = CCQP_UNROLL;  // 256-bit loads in flight per lane
constexpr int kUnrollF32 = CCQP_UNROLL_F32;
#if CCQP_A_F32
using AElem = float;                  // what DenseCtx::A points at
#else
using AElem = double;
#endif
constexpr int kMaxWindow = 64;        // SPG non-monotone window

enum DenseOp : int {
    OP_PGD = 0, OP_APGD = 1, OP_APGD_AR = 2, OP_BBPGD = 3, OP_BBPGDF = 4, OP_SPG = 5, OP_MPRGP = 6,
    OP_GEMV = 100, OP_PROJECT = 101, OP_NORMAL = 102, OP_PROJGRAD = 103
};

struct DenseOut {          // written by CTA 0 / thread 0
    double residual;
    long long mv, gemv, iters, draws;
    int converged, status;
};

constexpr int kNumVec = 12;

struct DenseCtx {
    // Hessian row shard: AElem (fp64, or fp32 in the fp32 build) entries; lda counts entries
    const void* A;
    long long lda;
    int n;              // columns = unknowns
    int row0, nrows;    // rows [row0, row0+nrows) live on this device
    int aligned;        // vector path usable (fp64: A base and lda*8 multiples of 32 bytes; fp32: base 16-byte aligned, lda % 4 == 0)
    // operator-form Hessian (CSR) instead of the dense rows: csr_val != nullptr
    const long long* csr_ptr;   // [nrows + 1], relative to this shard (csr_ptr[0] = 0)
    const int* csr_idx;         // [nnz] column indices
    const double* csr_val;      // [nnz]
    int csr_group;              // lanes that share one row: 2, 4, 8, 16 or 32 (from the mean row length)
    int csr_l1;                 // gather v through L1 (see ld_ca)
    int csr_tma;                // values and column ids are 16-byte aligned: tiles can be moved by bulk copies
    const int* csr_tile_row;    // [ceil(nnz / 4096) + 1]: the row that contains entry g * 4096 (nrows beyond the end)
    const double* b;    // [npad]
    const double* x0;   // [npad] (zeros if the caller passed none)
    ProjTable T;
    double* vec[kNumVec];   // work vectors, [npad] each, zero tails
    GridSyncCtx gs;         // arrive / go words, partials [2][grid][kMaxRed], results
    const double* uniforms;
    long long n_uniforms;
    double tol, max_mv, step, tau, sig1, sig2;
    int m;
    double* x_out;      // [npad]
    DenseOut* out;
    // mat-vec tiling
    int CW;             // panel width (columns staged in shared memory at a time), multiple of 128
    int SW;             // task segment width, multiple of 128, divides CW
    int np;             // number of panels
    int nseg;           // total segments per row
    int rows_max;       // max rows owned by one CTA
    int evict_first;    // stream A with L2 evict-first
    int resident_256;   // ... except the first resident_256/256 of every CTA's (row, segment) tasks, which keep the normal policy
                        // and so stay in L2 from one mat-vec to the next (a fixed ~70 MB slice of A never touches HBM again)
    int psum_accum;     // nseg counts the segments of ONE panel; the panels' partial sums are added up in panel order
    // test hooks
    const double* hook_in;
    double* hook_out;
    double* ytmp;       // [nrows] CSR phase: row sums of this rank's rows, handed from the tile loop to the epilogue pass
    long long* dbg;     // phase time stamps of CTA 0 (tuning aid, CCQP_DEBUG_TIMING=1); null = off
    // row-sharded multi-GPU solves (world == 1: unused)
    XComm x;
};

// shared memory carve-up (dynamic)
struct DenseSmem {
    double* vbuf[2];
    double* psum;
    double* scratch;        // kMaxRed*32 doubles
    uint64_t* mbar;         // kNumMbar
    unsigned long long* ascratch;   // 32
};

constexpr int kNumMbar = 8;
constexpr size_t kDenseSmemLimit = 220 * 1024;    // cudaFuncAttributeMaxDynamicSharedMemorySize of the dense kernels
constexpr size_t kDenseSmemTarget = 200 * 1024;   // what the tiling aims to stay under

__host__ __device__ inline size_t dense_smem_bytes(int CW, int rows_max, int nseg) {
    size_t s = 0;
    s += 2 * (size_t)CW * 8;
    s += (size_t)rows_max * nseg * 8;
    s += kMaxRed * 32 * 8;
    s += 32 * 8;
    s += kNumMbar * 8;
    return s + 128;
}

struct Kst {                // per-thread kernel state
    unsigned epoch, xepoch; // grid_xsync counts (identical in every thread of every CTA of every rank)
    DenseSmem sm;
    int bid, nblk;          // this CTA's index in / the size of the rank's grid (blockIdx.x / gridDim.x unless ranks are emulated)
    int gtid, gstride;
    int r0, r1;             // rows of this CTA (global indices)
    unsigned parbits;       // mbarrier phase parities, bit i = barrier i (dense: 2 panel buffers; CSR: 4 column-id + 4 value stages)
    int yq;                 // next buffer of the mat-vec output pool
    long long mv, gemv, iters, draws;
};

// ------------------------------------------------------------------------------------------
// reductions across the grid (the barrier also orders all prior global writes)
// ------------------------------------------------------------------------------------------
// Barrier between phases: the whole grid, and every rank of a sharded solve (common.cuh grid_xsync).
// kCross: the sync closes a mat-vec phase, whose output rows other ranks are about to read.
template <bool kCross>
__device__ __forceinline__ void barrier_only(Kst& k, const DenseCtx& c) {
    unsigned long long none[1] = {0};
    grid_xsync<0, false>(c.gs, c.x, k.epoch, k.xepoch, kCross, none, reinterpret_cast<unsigned long long*>(k.sm.scratch), k.bid, k.nblk);
}

// store into a vector that a later mat-vec reads in full: the owning rank also writes the entry
// into every peer's copy of the vector (same offset in the peer's symmetric buffer, over NVLink)
__device__ __forceinline__ void pub_store(const DenseCtx& c, double* vec, int i, double v) {
    vec[i] = v;
    if (c.x.world > 1) {
        const size_t off = reinterpret_cast<char*>(vec + i) - c.x.base[c.x.rank];
#pragma unroll 1
        for (int s = 0; s < c.x.world; ++s)
            if (s != c.x.rank) *reinterpret_cast<double*>(c.x.base[s] + off) = v;
    }
}

// Sum of K per-thread values over the grid (and over all ranks), fused with the phase barrier.
// Order: lanes -> warps -> CTAs (strided over 32 lanes, then a shuffle tree) -> ranks in rank
// order; fixed for a given launch shape, identical on every rank.
// kCross = true: the values are partial sums over this rank's ROWS (mat-vec epilogue) and the sync
// closes the mat-vec phase; kCross = false: every rank summed the full-length vectors itself.
template <int K, bool kCross>
__device__ __forceinline__ void reduce_sync(Kst& k, const DenseCtx& c, double (&a)[K]) {
    cta_sum<K>(a, k.sm.scratch);
    unsigned long long v[K];
#pragma unroll
    for (int j = 0; j < K; ++j) v[j] = (unsigned long long)__double_as_longlong(a[j]);
    grid_xsync<K, false>(c.gs, c.x, k.epoch, k.xepoch, kCross, v, reinterpret_cast<unsigned long long*>(k.sm.scratch), k.bid, k.nblk);
#pragma unroll
    for (int j = 0; j < K; ++j) a[j] = __longlong_as_double((long long)v[j]);
}

// bitwise AND of a 64-bit mask over the grid (and over all ranks)
__device__ __forceinline__ unsigned long long and_sync(Kst& k, const DenseCtx& c, unsigned long long m) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    m = warp_and64(m);
    if (lane == 0) k.sm.ascratch[warp] = m;
    __syncthreads();
    unsigned long long v[1] = {~0ull};
    for (int w = 0; w < kDenseWarps; ++w) v[0] &= k.sm.ascratch[w];      // every thread: a one-CTA solve returns these as they are
    grid_xsync<1, true>(c.gs, c.x, k.epoch, k.xepoch, false, v, reinterpret_cast<unsigned long long*>(k.sm.scratch), k.bid, k.nblk);
    return v[0];
}

// ------------------------------------------------------------------------------------------
// mat-vec phase
// ------------------------------------------------------------------------------------------
// A is read as fp64 (256-bit loads of four doubles) or, in the fp32 build (dense_f32.cu), as fp32 (128-bit loads of four
// floats, one chunk of 128 columns = 512 bytes per warp), with the same lane -> column mapping, FMA chains and reductions:
// every fp32 entry is widened exactly in a register before its fma, so the result is bit-identical to the fp64 loop on
// the widened matrix.  kUnrollF32 loads in flight per lane keep the fp64 loop's 512 bytes per lane.
template <class T> constexpr int kUnrollOf = sizeof(T) == 8 ? kUnroll : kUnrollF32;
static_assert(kUnroll >= 1 && kUnroll <= 32 && kUnrollF32 >= 1 && kUnrollF32 <= 32,
              "the remainder chain of dot_seg_aligned (16/8/4/2/1) covers at most 31 chunks");

// U consecutive 128-column chunks: all U vector loads of the lane are issued before the first FMA.
// The fp32 loop reads the vector panel with explicit ld.shared: with plain loads the compiler hoisted the 32 vector reads
// of a batch next to the A loads, and APGD / APGD-AR / BBPGD / BBPGDf spilled (72-184 bytes, ptxas -v).
template <bool kEF, int U, class T>
__device__ __forceinline__ void dot_chunks(const T* ap, const double* vp, double& a0, double& a1, double& a2, double& a3) {
    constexpr bool kLds = CCQP_DENSE_LDS || sizeof(T) == 4;
    T r[U][4];
#pragma unroll
    for (int u = 0; u < U; ++u) ldg_vec4_stream<kEF>(ap + (size_t)u * 128, r[u]);
    const uint32_t vp32 = smem_u32(vp);       // kLds: explicit LDS.128 pairs instead of the generic LD.E.128 the compiler emits for vp
#pragma unroll
    for (int u = 0; u < U; ++u) {
        double4 v;
        if constexpr (kLds) {
            asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(vp32 + (uint32_t)u * 1024u));
            asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v.z), "=d"(v.w) : "r"(vp32 + (uint32_t)u * 1024u + 16u));
        } else {
            v = *reinterpret_cast<const double4*>(vp + (size_t)u * 128);
        }
        a0 = fma((double)r[u][0], v.x, a0);
        a1 = fma((double)r[u][1], v.y, a1);
        a2 = fma((double)r[u][2], v.z, a2);
        a3 = fma((double)r[u][3], v.w, a3);
    }
}

// One (row, segment) task of a warp: lanes own 4 consecutive columns of every 128-column chunk.
// Chunks are consumed in order (kUnrollOf<T> at a time, then 16/8/4/2/1 for the remainder), so the
// summation order does not depend on the blocking.
template <bool kEF, class T>
__device__ __forceinline__ double dot_seg_aligned(const T* __restrict__ arow, const double* vs, int ncol, int lane) {
    constexpr int kU = kUnrollOf<T>;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    const int nchunk = ncol >> 7;
    const T* ap = arow + lane * 4;
    const double* vp = vs + lane * 4;
    int c = 0;
    for (; c + kU <= nchunk; c += kU) dot_chunks<kEF, kU>(ap + (size_t)c * 128, vp + (size_t)c * 128, a0, a1, a2, a3);
    if (kU > 16 && c + 16 <= nchunk) { dot_chunks<kEF, 16>(ap + (size_t)c * 128, vp + (size_t)c * 128, a0, a1, a2, a3); c += 16; }
    if (kU > 8 && c + 8 <= nchunk) { dot_chunks<kEF, 8>(ap + (size_t)c * 128, vp + (size_t)c * 128, a0, a1, a2, a3); c += 8; }
    if (kU > 4 && c + 4 <= nchunk) { dot_chunks<kEF, 4>(ap + (size_t)c * 128, vp + (size_t)c * 128, a0, a1, a2, a3); c += 4; }
    if (kU > 2 && c + 2 <= nchunk) { dot_chunks<kEF, 2>(ap + (size_t)c * 128, vp + (size_t)c * 128, a0, a1, a2, a3); c += 2; }
    if (c < nchunk) { dot_chunks<kEF, 1>(ap + (size_t)c * 128, vp + (size_t)c * 128, a0, a1, a2, a3); c += 1; }
    const int col = (nchunk << 7) + lane * 4;
    if (col < ncol) {
        a0 = fma((double)ldg_stream(arow + col), vs[col], a0);
        if (col + 1 < ncol) a1 = fma((double)ldg_stream(arow + col + 1), vs[col + 1], a1);
        if (col + 2 < ncol) a2 = fma((double)ldg_stream(arow + col + 2), vs[col + 2], a2);
        if (col + 3 < ncol) a3 = fma((double)ldg_stream(arow + col + 3), vs[col + 3], a3);
    }
    return (a0 + a1) + (a2 + a3);
}

// any alignment / any lda: scalar loads, lanes contiguous
template <class T>
__device__ __forceinline__ double dot_seg_generic(const T* __restrict__ arow, const double* vs, int ncol, int lane) {
    double a0 = 0.0, a1 = 0.0;
    int c = lane;
    for (; c + 32 < ncol; c += 64) {
        const double x0 = ldg_stream(arow + c), x1 = ldg_stream(arow + c + 32);
        a0 = fma(x0, vs[c], a0);
        a1 = fma(x1, vs[c + 32], a1);
    }
    if (c < ncol) a0 = fma((double)ldg_stream(arow + c), vs[c], a0);
    return a0 + a1;
}

// CSR mat-vec phase (operator-form A: contact-style Hessians D^T M^-1 D are sparse).
//
// The stored entries are treated as ONE stream, independent of the row structure ("CSR-stream"):
//   * CTAs own nnz-balanced, row-aligned ranges of the stream (dense_body: a binary search in the row
//     pointers for bid * nnz / G), so a few long rows cannot unbalance the grid;
//   * the stream is cut into tiles of kCsrTile = 4096 entries at GLOBAL multiples of 4096, and the TMA engine
//     copies a tile's values (32 KB) and column ids (16 KB) into a ring of kCsrStages shared-memory stages with
//     two bulk copies and one mbarrier per tile (cp.async.bulk with an L2 evict-first hint, SASS UBLKCP/SYNCS):
//     up to 3 x 48 KB per SM are in flight with no register cost, independent of what the warps are doing, and
//     the stream does not push the vectors (the gather targets) out of L2;
//   * csr_tile_row[g] (computed once per matrix, ccqp_set_matrix_csr) names the row that contains entry g * 4096,
//     so the rows a tile touches are known without a search: their row pointers are fetched with one coalesced
//     load into a shared-memory window while the gather is in flight;
//   * consuming a tile: every thread takes 16 entries, lane-consecutive (entry u*256 + tid), gathers v through
//     L1 (ld.global.ca is legal here: the phase starts behind the sync's acquire and nobody writes v during it;
//     for banded rows a warp-level gather covers 32 consecutive columns = 8 full sectors), multiplies and writes
//     the products IN PLACE over the values; after ONE barrier per tile groups of csr_group lanes sum the rows
//     that end inside the tile straight from shared memory (stride csr_group, then a shuffle tree).  A row that
//     continues into the next tile leaves its partial sum in a carry slot.  The steps are software-pipelined: the
//     gather of tile t+1 is issued BEFORE the rows of tile t are summed and consumed after, so the L2 latency of
//     the gather hides behind the row sums.  The barrier that ends step t also proves that everybody is done with
//     tile t, whose stage thread 0 then refills with tile t + kCsrStages.
//   Summation order per row: tile by tile, inside a tile lane by lane + fixed tree; tile boundaries do not depend
//   on the launch shape.  The stream's final tile, if its length is not a multiple of 4 entries (bulk copies move
//   multiples of 16 bytes), is read with ordinary loads.
// Algorithmic HBM bytes per mat-vec: 12 per stored entry + 8 (rows + 1) + the vectors.
constexpr int kCsrTile = 4096;                       // independent of the launch shape (csr_tile_row is built for it)
constexpr int kCsrE = kCsrTile / kDenseThreads;      // entries per thread per tile: 16 at 256 threads, 4 at 1024
static_assert(kCsrE * kDenseThreads == kCsrTile && kCsrE >= 1, "threads per CTA must divide the CSR tile");
constexpr int kCsrStages = 4;                        // stages of the value ring and of the column-id ring
constexpr int kCsrDesc = 8;                          // tile descriptors alive at a time (written 4 tiles ahead, read until the rows are summed)
constexpr int kCsrStageBytes = kCsrTile * 12;         // values, then column ids
constexpr int kCsrCW = kCsrStages * kCsrStageBytes / 16;   // "panel width" that makes the two panel buffers hold the ring
constexpr int kCsrWin = kDenseThreads + 1;            // row pointers of a tile kept in shared memory
constexpr int kCsrRowsMax = 2 * kCsrWin + 8;          // "rows_max" that makes the psum region hold two such windows

__device__ __forceinline__ void bulk_g2s_evict_first(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(pol) : "memory");
}

template <class Epi>
__device__ __forceinline__ void gemv_phase_csr(Kst& k, const DenseCtx& c, const double* v, Epi epi) {
    const int tid = threadIdx.x;
    // register copies of what the phase reads from the context: in the outlined form (gemv_phase_csr_outlined) `c` is a
    // reference into parameter memory, and every shared-memory access below is a compiler barrier for such loads
    const long long* const csr_ptr = c.csr_ptr;
    const int* const csr_idx = c.csr_idx;
    const double* const csr_val = c.csr_val;
    const int* const csr_tile_row = c.csr_tile_row;
    double* const ytmp = c.ytmp;
    const int row0 = c.row0, csr_l1 = c.csr_l1, csr_tma = c.csr_tma, shard_rows = c.nrows;
    const int G = c.csr_group, glane = tid & (G - 1), gid = tid / G, ngroups = kDenseThreads / G;
    const int warp_gid0 = (tid & ~31) / G;                           // first group of this warp
    const int cr0 = k.r0 - row0, cr1 = k.r1 - row0;               // this CTA's rows, relative to the shard
    // every shared-memory array of the phase is addressed explicitly (SharedArr: ld.shared / st.shared whatever the compiler
    // still knows about the pointers kept in Kst)
    const SharedArr<double> carry_slot(k.sm.scratch);                 // [2], by tile parity
    const SharedArr<int4> dsc(k.sm.scratch + 4);                      // [kCsrDesc][2]: per-tile descriptors, written by thread 0
    const SharedArr<int> win(k.sm.psum);                              // [2][kCsrWin], by tile parity: tile-relative row pointers
    unsigned char* ring = reinterpret_cast<unsigned char*>(k.sm.vbuf[0]);
    double* const val_ring = reinterpret_cast<double*>(ring);                                     // [kCsrStages][kCsrTile] values -> products
    int* const idx_ring = reinterpret_cast<int*>(ring + (size_t)kCsrStages * kCsrTile * 8);       // [kCsrStages][kCsrTile] column ids
    const SharedArr<double> val_sh(val_ring);
    const SharedArr<int> idx_sh(idx_ring);
    uint64_t* const ibar = k.sm.mbar;                                 // column-id stages
    uint64_t* const vbar = k.sm.mbar + kCsrStages;                    // value stages
    unsigned parbits = k.parbits;                                     // a register copy for the phase (Kst may live in local memory)
    const long long P0 = cr1 > cr0 ? csr_ptr[cr0] : 0, P1 = cr1 > cr0 ? csr_ptr[cr1] : 0;
    if (P1 > P0) {                                                    // CTA-uniform
        const long long g0 = P0 / kCsrTile;
        const int nt = (int)((P1 - 1) / kCsrTile - g0) + 1;
        // Thread 0 describes a tile ONCE for everybody when it starts the copy of the tile's column ids: {first row (open since
        // the previous tile, or the CTA's first), rows, this CTA's entry range [lo, hi) inside the tile}, {entries, slow path}.
        // All positions inside a tile are 32-bit and tile-relative from here on: the 64-bit row pointers are touched once per row.
        const long long nnz = csr_ptr[shard_rows];
        auto tile_cnt = [&](int t) { const long long T = (g0 + t) * kCsrTile; return (int)(nnz - T < kCsrTile ? nnz - T : kCsrTile); };
        auto tile_slow = [&](int cnt) { return ((cnt & 3) || !csr_tma) ? 1 : 0; };   // ragged final tile of the stream / unaligned arrays
        // thread 0 issues the tiles in order; the two csr_tile_row entries a descriptor needs are fetched one issue ahead
        // (tr_a = csr_tile_row[g0 + t], tr_b = csr_tile_row[g0 + t + 1] for the NEXT tile t to be issued), so that the thread
        // everybody waits for at the step's barrier never sits on an L2 round trip of its own
        int tr_a = 0, tr_b = 0;
        if (tid == 0) { tr_a = csr_tile_row[g0]; tr_b = csr_tile_row[g0 + 1]; }
        auto issue_idx = [&](int t) {                                 // thread 0 only, t = 0, 1, 2, ... in order
            const long long T = (g0 + t) * kCsrTile;
            const int cnt = tile_cnt(t), slow = tile_slow(cnt);
            int r_cur = t == 0 ? cr0 : tr_a, r_last = tr_b;
            tr_a = tr_b;
            if (t + 1 < nt) tr_b = csr_tile_row[g0 + t + 2];        // consumed by the next issue, a step from now
            if (r_last > cr1 - 1 || T + cnt >= P1) r_last = cr1 - 1;
            const int lo = (int)((T > P0 ? T : P0) - T), hi = (int)((T + cnt < P1 ? T + cnt : P1) - T);
            dsc[2 * (t % kCsrDesc)] = make_int4(r_cur, r_last - r_cur + 1, lo, hi);
            dsc[2 * (t % kCsrDesc) + 1] = make_int4(cnt, slow, 0, 0);
            if (slow) return;
            const int st = t % kCsrStages;
            mbar_expect_tx(&ibar[st], (uint32_t)cnt * 4u);
            bulk_g2s_evict_first(idx_ring + (size_t)st * kCsrTile, csr_idx + T, (uint32_t)cnt * 4u, &ibar[st]);
        };
        auto issue_val = [&](int t) {                                 // thread 0 only
            const int cnt = tile_cnt(t);
            if (tile_slow(cnt)) return;
            const int st = t % kCsrStages;
            mbar_expect_tx(&vbar[st], (uint32_t)cnt * 8u);
            bulk_g2s_evict_first(val_ring + (size_t)st * kCsrTile, csr_val + (g0 + t) * kCsrTile, (uint32_t)cnt * 8u, &vbar[st]);
        };
        if (tid == 0) {
            carry_slot[0] = 0.0;
            fence_proxy_async();
            for (int t = 0; t < nt && t < kCsrStages; ++t) { issue_idx(t); issue_val(t); }
        }
        __syncthreads();                                              // descriptors of the first tiles are visible
        struct Tile { int r_cur, nrows, lo, hi, cnt, slow; };
        auto describe = [&](int t) {
            const int4 d0 = dsc[2 * (t % kCsrDesc)], d1 = dsc[2 * (t % kCsrDesc) + 1];
            Tile d; d.r_cur = d0.x; d.nrows = d0.y; d.lo = d0.z; d.hi = d0.w; d.cnt = d1.x; d.slow = d1.y;
            return d;
        };
        // pointer of row r as a position inside the tile that starts at T, clamped to [lo, hi + 1] (hi + 1 = "beyond this CTA's part")
        auto rel = [&](long long p, long long T, const Tile& d) { p -= T; return p < d.lo ? d.lo : (p > d.hi ? d.hi + 1 : (int)p); };
        // G(t): the gather of tile t leaves (kCsrE loads per thread, results in registers) + the tile's row pointers
        auto gather_issue = [&](int t, double (&x)[kCsrE], long long& wv) {
            const Tile d = describe(t);
            const int st = t % kCsrStages;
            if (tid <= d.nrows && tid < kCsrWin) wv = csr_ptr[d.r_cur + tid];     // consumed a step later (finish_products)
            if (d.slow) return;
            const SharedArr<int> idx = idx_sh + st * kCsrTile;
            mbar_wait(&ibar[st], (parbits >> st) & 1u);
            parbits ^= 1u << st;
            int j[kCsrE];
            if (d.cnt == kCsrTile) {
#pragma unroll
                for (int u = 0; u < kCsrE; ++u) j[u] = idx[u * kDenseThreads + tid];
            } else {
#pragma unroll
                for (int u = 0; u < kCsrE; ++u) { const int q = u * kDenseThreads + tid; j[u] = q < d.cnt ? idx[q] : 0; }
            }
#pragma unroll
            for (int u = 0; u < kCsrE; ++u) x[u] = csr_l1 ? ld_ca(v + j[u]) : ld_cg(v + j[u]);
        };
        // F(t): products of tile t in place over its values (the gather left two steps ago), row-pointer window of the tile
        auto finish_products = [&](int t, const double (&x)[kCsrE], long long wv) {
            const Tile d = describe(t);
            const int st = t % kCsrStages;
            const SharedArr<double> prod = val_sh + st * kCsrTile;
            if (tid <= d.nrows && tid < kCsrWin) win[(t & 1) * kCsrWin + tid] = rel(wv, (g0 + t) * kCsrTile, d);
            if (d.slow) {
                const long long T = (g0 + t) * kCsrTile;
                for (int q = tid; q < d.cnt; q += kDenseThreads) {
                    const double xv = csr_l1 ? ld_ca(v + __ldg(csr_idx + T + q)) : ld_cg(v + __ldg(csr_idx + T + q));
                    prod[q] = ldg_stream(csr_val + T + q) * xv;
                }
                return;
            }
            mbar_wait(&vbar[st], (parbits >> (kCsrStages + st)) & 1u);
            parbits ^= 1u << (kCsrStages + st);
            if (d.cnt == kCsrTile) {
#pragma unroll
                for (int u = 0; u < kCsrE; ++u) prod[u * kDenseThreads + tid] *= x[u];
            } else {
#pragma unroll
                for (int u = 0; u < kCsrE; ++u) { const int q = u * kDenseThreads + tid; if (q < d.cnt) prod[q] *= x[u]; }
            }
        };
        // R(t): the rows of tile t, summed from the products in shared memory
        auto row_sums = [&](int t) {
            const Tile cur = describe(t);
            const SharedArr<int> pw = win + (t & 1) * kCsrWin;
            const SharedArr<double> prod = val_sh + (t % kCsrStages) * kCsrTile;
            const double carry_in = carry_slot[t & 1];
            for (int kk = 0; kk * ngroups < cur.nrows; ++kk) {        // CTA-uniform trip count
                if (warp_gid0 + kk * ngroups >= cur.nrows) continue;  // warp-uniform: nothing for this warp in this pass
                const int i = gid + kk * ngroups, r = cur.r_cur + i;
                const bool active = i < cur.nrows;
                int p0 = cur.hi, p1 = cur.hi;
                if (active) {
                    if (i + 1 < kDenseThreads) { p0 = pw[i]; p1 = pw[i + 1]; }      // the window holds the pointers of rows 0 .. threads-1
                                                                                       // (slot i is filled by thread i); beyond it: global loads
                    else { const long long T = (g0 + t) * kCsrTile; p0 = rel(csr_ptr[r], T, cur); p1 = rel(csr_ptr[r + 1], T, cur); }
                }
                const bool complete = active && p1 <= cur.hi;         // the row ends inside this CTA's part of the tile
                const int hi = p1 < cur.hi ? p1 : cur.hi;
                // lane glane takes entries start + glane, + G, + 2G, ...: even ones into a0, odd ones into a1, eight loads in
                // flight at a time (the warps that sum rows are the critical path of the step: everybody else waits for them)
                double a0 = 0.0, a1 = 0.0;
                for (int q = (p0 < cur.hi ? p0 : cur.hi) + glane; q < hi; q += 8 * G) {
                    double pv[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) pv[u] = (q + u * G < hi) ? prod[q + u * G] : 0.0;
#pragma unroll
                    for (int u = 0; u < 8; u += 2) { a0 += pv[u]; a1 += pv[u + 1]; }
                }
                double acc = a0 + a1;
                for (int o = G >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                if (glane == 0 && active) {
                    if (i == 0) acc = carry_in + acc;                 // earlier tiles' part of the row first
                    if (complete) ytmp[r] = acc;                    // the epilogue runs after the tile loop, all rows side by side
                    else carry_slot[(t + 1) & 1] = acc;               // the one row that continues into the next tile (the last one)
                }
            }
        };
        // Software pipeline, two tiles deep: in step t the gather of tile t+2 LEAVES, the rows of tile t are summed, the
        // products of tile t+1 (whose gather left a whole step ago) are formed, and ONE barrier closes the step: no step waits
        // for memory.  The column ids of a tile are consumed two steps before its values, so they travel in separate rings
        // (4 stages each): ids of tile t+4 and values of tile t+3 are requested at the top of step t.
        double xa[kCsrE], xb[kCsrE];
        long long wa = 0, wb = 0;
        gather_issue(0, xa, wa);
        if (nt > 1) gather_issue(1, xb, wb);
        finish_products(0, xa, wa);
        __syncthreads();
        auto step = [&](int t, double (&x_even)[kCsrE], long long& w_even, double (&x_odd)[kCsrE], long long& w_odd) {
            // tiles t and t+2 share (x_even, w_even); tile t+1 uses (x_odd, w_odd)
            if (tid == 0) {               // everybody is behind the barrier that ended step t-1 (t = 0: the prologue's)
                const bool i4 = t + kCsrStages < nt, v3 = t >= 1 && t - 1 + kCsrStages < nt;
                if (i4 || v3) fence_proxy_async();
                if (i4) issue_idx(t + kCsrStages);                    // id stage of tile t: read in step t-2
                if (v3) issue_val(t - 1 + kCsrStages);                // value stage of tile t-1: summed in step t-1
            }
            if (t + 2 < nt) gather_issue(t + 2, x_even, w_even);
            row_sums(t);
            if (t + 1 < nt) finish_products(t + 1, x_odd, w_odd);
            __syncthreads();          // products + row-pointer window of tile t+1 and the carry of tile t are visible;
                                      // everybody has finished tile t
        };
        for (int t = 0; t < nt; t += 2) {
            step(t, xa, wa, xb, wb);
            if (t + 1 < nt) step(t + 1, xb, wb, xa, wa);
        }
        // epilogue pass: one row per thread at a time, so the loads an epilogue does (e.g. SPG's d_r for d.Ad) overlap across
        // rows instead of stalling the tile loop once per tile (the last step's barrier made the row sums visible to the CTA)
        for (int r = cr0 + tid; r < cr1; r += kDenseThreads) epi(row0 + r, ld_cg(ytmp + r));
    } else {
        for (int r = cr0 + tid; r < cr1; r += kDenseThreads) epi(row0 + r, 0.0);     // a range of empty rows
    }
    k.parbits = parbits;
    k.gemv += 1;
    __syncthreads();
}

// The CSR phase as a function of its own: for a solver program whose live state does not fit next to the tile loop's
// registers (MPRGP: the inlined phase spilled inside the loop) the call gives the loop its own register allocation; the
// caller's state is saved once around the call instead of being spilled and reloaded in every step.
template <class Epi>
__device__ __noinline__ void gemv_phase_csr_outlined(Kst& k, const DenseCtx& c, const double* v, Epi epi) {
    gemv_phase_csr(k, c, v, epi);
}

// y_row = sum_j A[row][j] v[j] for the rows of this CTA; epi(row, y_row) is called once per row.
// v: full-length global vector (npad entries, zero tail), complete before the phase starts.
template <bool kOutlineCsr = false, class Epi>
__device__ __forceinline__ void gemv_phase(Kst& k, const DenseCtx& c, const double* v, Epi epi) {
    if constexpr (!CCQP_DENSE_ONLY) {
        if (CCQP_CSR_ONLY || c.csr_val) {
            if constexpr (kOutlineCsr && CCQP_CSR_ONLY) gemv_phase_csr_outlined(k, c, v, epi);
            else gemv_phase_csr(k, c, v, epi);
            return;
        }
    }
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = c.n, CW = c.CW, SW = c.SW, np = c.np, nseg = c.nseg;
    const int nrows_cta = k.r1 - k.r0;
    const int spp_full = CW / SW;

    auto panel_cols = [&](int p) { return min(CW, n - p * CW); };
    auto issue = [&](int p, int buf) {
        const uint32_t bytes = (uint32_t)(((panel_cols(p) + 1) & ~1) * 8);
        mbar_expect_tx(&k.sm.mbar[buf], bytes);
        bulk_g2s(k.sm.vbuf[buf], v + (size_t)p * CW, bytes, &k.sm.mbar[buf]);
    };
    if (tid == 0) {
        fence_proxy_async();
        issue(0, 0);
        if (np > 1) issue(1, 1);
    }
    for (int p = 0; p < np; ++p) {
        const int buf = p & 1;
        mbar_wait(&k.sm.mbar[buf], (k.parbits >> buf) & 1u);
        k.parbits ^= 1u << buf;
        const int pc = panel_cols(p);
        const int spp = (pc + SW - 1) / SW;
        const int ntask = nrows_cta * spp;
        const double* vb = k.sm.vbuf[buf];
        const int t_res = c.evict_first ? (int)(((long long)ntask * c.resident_256) >> 8) : ntask;   // tasks [0, t_res) stay in L2
        for (int t = warp; t < ntask; t += kDenseWarps) {
            const int row = t / spp, seg = t - row * spp;
            const int col0 = seg * SW;
            const int ncol = min(SW, pc - col0);
            const AElem* arow = static_cast<const AElem*>(c.A) + (size_t)(k.r0 - c.row0 + row) * c.lda + (size_t)p * CW + col0;
            double acc;
            if (c.aligned) acc = t >= t_res ? dot_seg_aligned<true>(arow, vb + col0, ncol, lane)
                                            : dot_seg_aligned<false>(arow, vb + col0, ncol, lane);
            else acc = dot_seg_generic(arow, vb + col0, ncol, lane);
            acc = warp_sum(acc);
            if (lane == 0) {
                if (!c.psum_accum) k.sm.psum[(size_t)row * nseg + p * spp_full + seg] = acc;
                else { double* q = k.sm.psum + (size_t)row * nseg + seg; *q = (p == 0) ? acc : *q + acc; }   // (row, seg) tasks of
            }                                                           // different panels are separated by the barrier below
        }
        __syncthreads();   // every warp is done with vbuf[buf]; psum of this panel is visible
        if (tid == 0 && p + 2 < np) { fence_proxy_async(); issue(p + 2, buf); }
    }
    k.gemv += 1;
    for (int r = tid; r < nrows_cta; r += kDenseThreads) {
        const double* ps = k.sm.psum + (size_t)r * nseg;
        double s = ps[0];
        for (int q = 1; q < nseg; ++q) s += ps[q];
        epi(k.r0 + r, s);
    }
    __syncthreads();       // psum is free again
}

// ------------------------------------------------------------------------------------------
// small helpers for the solver programs
// ------------------------------------------------------------------------------------------
// Sharded solves ("replicated vectors, sharded matrix").  Every rank keeps ALL vectors in full and
// repeats the (tiny) elementwise work; only the mat-vec is split by rows.  The rows a rank computes
// are written into every peer's copy of the output vector from inside the mat-vec epilogue
// (pub_store: the all-gather, fused), and the sync that closes the mat-vec phase is the only
// cross-GPU sync of an iteration (it also carries the row-local partial sums: the all-reduce).
// Mat-vec outputs land in a rotating pool of three buffers: a fast rank may already be writing the
// output of phase q+1 into a slow rank's memory while that rank still reads the output of phase q
// (or q-1, e.g. BBPGD's previous gradient), so a buffer is reused only every third output; values
// that must live longer are copied to a rank-local vector by the elementwise pass that reads them.
#define CCQP_ELEMS(i) for (int i = k.gtid; i < c.n; i += k.gstride)

constexpr int kPool = 3;                    // vec[kNumVec - 3 ..] are the mat-vec output pool
__device__ __forceinline__ double* next_y(Kst& k, const DenseCtx& c) {
    double* y = c.vec[kNumVec - kPool + k.yq];
    k.yq = (k.yq + 1 == kPool) ? 0 : k.yq + 1;
    return y;
}

__device__ __forceinline__ void swap_ptr(double*& a, double*& b) { double* t = a; a = b; b = t; }

// residual probe of solvers.py:137-139: sum over i of (cs * (x_i - P(x - gd*g)_i))^2
// (the reference scales the vector first and then takes the 2-norm)
template <class XF, class GF>
__device__ __forceinline__ double residual_partial(Kst& k, const DenseCtx& c, double cs, XF xf, GF gf) {
    double acc = 0.0;
    project_pass(c.T, k.gtid, k.gstride, k.sm.scratch,
                 [&](int i) { return xf(i) - kGd * gf(i); },
                 [&](int i, double, double p) { const double d = cs * (xf(i) - p); acc = fma(d, d, acc); });
    return acc;
}

__device__ __forceinline__ void finish(Kst& k, const DenseCtx& c, const double* xsol, double res, int status) {
    CCQP_ELEMS(i) c.x_out[i] = ld_cg(xsol + i);   // every rank holds the full solution
    if (k.bid == 0 && threadIdx.x == 0) {
        DenseOut o;
        o.residual = res;
        o.mv = k.mv; o.gemv = k.gemv; o.iters = k.iters; o.draws = k.draws;
        o.converged = ((double)k.mv < c.max_mv) ? 1 : 0;
        o.status = status;
        *c.out = o;
    }
}

constexpr int kDbgSlots = 8, kDbgIters = 64;
__device__ __forceinline__ void dbg_stamp(const DenseCtx& c, long long it, int slot) {
    if (c.dbg && blockIdx.x == 0 && threadIdx.x == 0 && it < kDbgIters) {   // (the launch's first CTA = rank 0's CTA 0)
        long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        c.dbg[it * kDbgSlots + slot] = t;
    }
}

__device__ __forceinline__ bool hit_max(const Kst& k, const DenseCtx& c) { return (double)k.mv >= c.max_mv; }

// ------------------------------------------------------------------------------------------
// PGD / BBPGD / BBPGDf                          solvers.py:114-170, 606-669, 741-819
// ------------------------------------------------------------------------------------------
template <int MODE>
__device__ void solve_pgd_family(Kst& k, const DenseCtx& c) {
    double *x = c.vec[0], *xm = c.vec[1], *xmin = c.vec[2], *gmin = c.vec[3];
    const double cs = 1.0 / (3 * (double)c.n * kGd);
    const double* b = c.b;
    CCQP_ELEMS(i) { const double v = c.x0[i]; x[i] = v; xm[i] = v; if (MODE == OP_BBPGDF) { xmin[i] = v; gmin[i] = v; } }
    barrier_only<false>(k, c);
    double* gm = next_y(k, c);
    gemv_phase(k, c, xm, [&](int r, double s) { pub_store(c, gm, r, s + b[r]); });
    k.mv = 1;
    barrier_only<true>(k, c);
    double a1[1] = {residual_partial(k, c, cs, [&](int i) { return ld_cg(xm + i); }, [&](int i) { return ld_cg(gm + i); })};
    reduce_sync<1, false>(k, c, a1);
    double res = sqrt(a1[0]);
    double resmin = INFINITY;
    const double* xsol = x;
    if (res >= c.tol) {
        double step = c.step;
        if (MODE != OP_PGD) {   // alpha0 = g.g / g.Ag, product not counted (:635, :775)
            double a2[2] = {0.0, 0.0};
            gemv_phase(k, c, gm, [&](int r, double s) { const double gr = ld_cg(gm + r); a2[0] = fma(gr, s, a2[0]); a2[1] = fma(gr, gr, a2[1]); });
            reduce_sync<2, true>(k, c, a2);
            step = a2[1] / a2[0];
        }
        for (;;) {
            project_pass(c.T, k.gtid, k.gstride, k.sm.scratch,
                         [&](int i) { return ld_cg(xm + i) - step * ld_cg(gm + i); },
                         [&](int i, double, double p) { x[i] = p; });
            barrier_only<false>(k, c);
            double* g = next_y(k, c);
            gemv_phase(k, c, x, [&](int r, double s) { pub_store(c, g, r, s + b[r]); });
            k.mv += 1;
            barrier_only<true>(k, c);
            xsol = x;
            if (hit_max(k, c)) break;
            double a3[3] = {0.0, 0.0, 0.0};
            project_pass(c.T, k.gtid, k.gstride, k.sm.scratch,
                         [&](int i) { return ld_cg(x + i) - kGd * ld_cg(g + i); },
                         [&](int i, double, double p) {
                             const double xi = ld_cg(x + i);
                             const double d = cs * (xi - p);
                             a3[0] = fma(d, d, a3[0]);
                             if (MODE != OP_PGD) {
                                 const double s = xi - ld_cg(xm + i), y = ld_cg(g + i) - ld_cg(gm + i);
                                 a3[1] = fma(s, s, a3[1]);
                                 a3[2] = fma(s, y, a3[2]);
                             }
                         });
            reduce_sync<3, false>(k, c, a3);
            res = sqrt(a3[0]);
            k.iters += 1;
            if (res < c.tol) break;
            if (MODE == OP_BBPGDF) {   // :793-800
                if (res < resmin) {
                    resmin = res;
                    CCQP_ELEMS(i) { xmin[i] = ld_cg(x + i); gmin[i] = ld_cg(g + i); }
                }
                if (step < 10 * kEps) {   // stagnation: x replaced (g is not), BB sums redone
                    barrier_only<false>(k, c);
                    project_pass(c.T, k.gtid, k.gstride, k.sm.scratch,
                                 [&](int i) { return ld_cg(xmin + i) - kGd * ld_cg(gmin + i); },
                                 [&](int i, double, double p) { x[i] = p; });
                    barrier_only<false>(k, c);
                    double a2[2] = {0.0, 0.0};
                    CCQP_ELEMS(i) {
                        const double s = ld_cg(x + i) - ld_cg(xm + i), y = ld_cg(g + i) - ld_cg(gm + i);
                        a2[0] = fma(s, s, a2[0]);
                        a2[1] = fma(s, y, a2[1]);
                    }
                    reduce_sync<2, false>(k, c, a2);
                    a3[1] = a2[0]; a3[2] = a2[1];
                }
            }
            if (MODE != OP_PGD) step = a3[1] / (a3[2] + 10 * kEps);
            swap_ptr(x, xm);
            gm = g;
        }
    }
    barrier_only<false>(k, c);
    finish(k, c, xsol, res, 0);
}

// ------------------------------------------------------------------------------------------
// SPG-QP                                                           solvers.py:906-975
// ------------------------------------------------------------------------------------------
static __device__ void solve_spg(Kst& k, const DenseCtx& c) {
    double *x = c.vec[0], *g = c.vec[1], *d = c.vec[2];
    const double* b = c.b;
    CCQP_ELEMS(i) x[i] = c.x0[i];
    barrier_only<false>(k, c);
    double a2[2] = {0.0, 0.0};
    double* g0 = next_y(k, c);
    gemv_phase(k, c, x, [&](int r, double s) {
        const double gr = s + b[r];
        pub_store(c, g0, r, gr);
        a2[0] = fma(gr, ld_cg(x + r), a2[0]);   // f0 = g.x (:923, kept as written)
        a2[1] = fma(gr, gr, a2[1]);
    });
    reduce_sync<2, true>(k, c, a2);
    double f = a2[0];
    const double gg = a2[1];
    CCQP_ELEMS(i) g[i] = ld_cg(g0 + i);         // g lives for the whole solve: rank-local copy
    double a1[1] = {0.0};
    gemv_phase(k, c, g0, [&](int r, double s) { a1[0] = fma(ld_cg(g0 + r), s, a1[0]); });
    reduce_sync<1, true>(k, c, a1);
    double alpha = gg / a1[0];
    k.mv = 2;
    double window[kMaxWindow];
    int wcount = 1, whead = 0;          // ring buffer = deque(maxlen=m)
    window[0] = f;
    double dd_rep = NAN;                 // residual reported = sqrt(d.d) of the last completed test
    double bk = 0.0;                     // pending update x += bk d, g += bk Ad (applied lazily)
    const double* Ad = c.vec[3];         // all zeros; multiplied by bk == 0 in the first pass
    int status = 0;
    double u_next = c.n_uniforms > 0 ? c.uniforms[0] : 0.0;   // the sample of iteration k+1 is fetched during iteration k
    for (;;) {
        dbg_stamp(c, k.iters, 0);
        double s2[2] = {0.0, 0.0};       // d.d, d.g
        project_pass(c.T, k.gtid, k.gstride, k.sm.scratch,
                     [&](int i) {
                         const double xi = fma(bk, ld_cg(d + i), ld_cg(x + i));
                         const double gi = fma(bk, ld_cg(Ad + i), ld_cg(g + i));
                         return xi - alpha * gi;
                     },
                     [&](int i, double, double p) {
                         // x += bk*d ; g += bk*Ad  (:961-962) fused with d = P(x - alpha g) - x (:937)
                         const double xi = fma(bk, ld_cg(d + i), ld_cg(x + i));
                         const double gi = fma(bk, ld_cg(Ad + i), ld_cg(g + i));
                         const double di = p - xi;
                         x[i] = xi; g[i] = gi; d[i] = di;
                         s2[0] = fma(di, di, s2[0]);
                         s2[1] = fma(di, gi, s2[1]);
                     });
        bk = 0.0;
        dbg_stamp(c, k.iters, 1);
        reduce_sync<2, false>(k, c, s2);
        dbg_stamp(c, k.iters, 2);
        double s1[1] = {0.0};
        double* Adn = next_y(k, c);
        gemv_phase(k, c, d, [&](int r, double s) { pub_store(c, Adn, r, s); s1[0] = fma(ld_cg(d + r), s, s1[0]); });
        Ad = Adn;
        k.mv += 1;
        dbg_stamp(c, k.iters, 3);
        reduce_sync<1, true>(k, c, s1);
        dbg_stamp(c, k.iters, 4);
        if (hit_max(k, c)) break;
        const double dd = s2[0], dg = s2[1], dAd = s1[0];
        dd_rep = dd;
        if (sqrt(dd) <= c.tol) break;
        double fmax = window[0];
        for (int j = 1; j < wcount; ++j) fmax = fmax > window[j] ? fmax : window[j];
        const double xi = (fmax - f) / dAd;
        const double beta = -dg / dAd;
        const double bhat = c.tau * beta + sqrt((c.tau * c.tau) * (beta * beta) + 2 * xi);
        // Python's min(bhat, sig2): sig2 only if sig2 < bhat, so a NaN bhat is kept
        const double hi = (c.sig2 < bhat) ? c.sig2 : bhat;
        if (hi != hi) { status = 8; break; }                       // CCQP_ERR_RANGE
        if (k.draws >= c.n_uniforms) { status = 7; break; }        // CCQP_ERR_UNIFORMS_EXHAUSTED
        const double u = u_next;
        k.draws += 1;
        u_next = k.draws < c.n_uniforms ? c.uniforms[k.draws] : 0.0;
        bk = c.sig1 + (hi - c.sig1) * u;
        f += bk * bk * dg + 0.5 * (bk * bk) * dAd;                  // :963 as written
        if (wcount < c.m) { window[wcount++] = f; }
        else { window[whead] = f; whead = (whead + 1) % c.m; }
        alpha = dd / dAd;
        k.iters += 1;
    }
    barrier_only<false>(k, c);
    finish(k, c, x, sqrt(dd_rep), status);
}

// ------------------------------------------------------------------------------------------
// APGD and its anti-relaxation variant              solvers.py:242-343, 415-533
// ------------------------------------------------------------------------------------------
template <bool AR>
__device__ void solve_apgd(Kst& k, const DenseCtx& c) {
    double *x = c.vec[0], *xp = c.vec[1], *y = c.vec[2], *yn = c.vec[3], *g = c.vec[4];
    double *xhat = c.vec[5], *v0 = c.vec[6];
    const double* b = c.b;
    const double cs = 1.0 / (3 * (double)c.n * kGd);
    double a1[1] = {0.0};
    CCQP_ELEMS(i) {
        const double v = c.x0[i];
        x[i] = v; xp[i] = v; y[i] = v;
        if (AR) xhat[i] = 1.0;
        const double dv = v - 1.0;
        v0[i] = dv;
        a1[0] = fma(dv, dv, a1[0]);
    }
    reduce_sync<1, false>(k, c, a1);
    const double dn2 = a1[0];
    a1[0] = 0.0;
    gemv_phase(k, c, v0, [&](int, double s) { a1[0] = fma(s, s, a1[0]); });
    reduce_sync<1, true>(k, c, a1);
    double L = sqrt(a1[0]) / sqrt(dn2);
    double t = 1.0 / L;
    k.mv = 1;
    double theta = 1.0, res = NAN, resmin = INFINITY;
    const double* Axp = v0;              // set by the first inner mat-vec
    for (;;) {
        double r12[2] = {0.0, 0.0};
        double* gy = next_y(k, c);
        gemv_phase(k, c, y, [&](int r, double s) {
            const double yr = ld_cg(y + r), br = b[r];
            pub_store(c, gy, r, s + br);
            r12[0] = fma(yr, s, r12[0]);
            r12[1] = fma(yr, br, r12[1]);
        });
        k.mv += 1;
        reduce_sync<2, true>(k, c, r12);
        if (hit_max(k, c)) break;
        const double rt1 = r12[0] * 0.5, rt2 = r12[1];
        // g is read again by the backtracking steps and the restart test: rank-local copy
        project_pass(c.T, k.gtid, k.gstride, k.sm.scratch,
                     [&](int i) { return ld_cg(y + i) - t * ld_cg(gy + i); },
                     [&](int i, double, double p) { g[i] = ld_cg(gy + i); xp[i] = p; });
        barrier_only<false>(k, c);
        for (;;) {   // Lipschitz backtracking :288-310
            double q[4] = {0.0, 0.0, 0.0, 0.0};
            double* ax = next_y(k, c);
            gemv_phase(k, c, xp, [&](int r, double s) {
                pub_store(c, ax, r, s);
                const double xr = ld_cg(xp + r), df = xr - ld_cg(y + r);
                q[0] = fma(xr, s, q[0]);
                q[1] = fma(xr, b[r], q[1]);
                q[2] = fma(ld_cg(g + r), df, q[2]);
                q[3] = fma(df, df, q[3]);
            });
            Axp = ax;
            k.mv += 1;
            reduce_sync<4, true>(k, c, q);
            if (hit_max(k, c)) break;   // leaves the inner loop only (:292-293)
            const double lt1 = q[0] * 0.5, lt2 = q[1], rt3 = q[2], rt4 = 0.5 * L * q[3];
            if ((lt1 + lt2) <= (rt1 + rt2 + rt3 + rt4)) break;
            L *= 2;
            t = 1.0 / L;
            project_pass(c.T, k.gtid, k.gstride, k.sm.scratch,
                         [&](int i) { return ld_cg(y + i) - t * ld_cg(g + i); },
                         [&](int i, double, double p) { xp[i] = p; });
            barrier_only<false>(k, c);
        }
        double theta_n = 0.5 * (-theta * theta + theta * sqrt(4 + theta * theta));
        const double beta = theta * (1 - theta) / (theta * theta + theta_n);
        double r2[2] = {0.0, 0.0};
        project_pass(c.T, k.gtid, k.gstride, k.sm.scratch,
                     [&](int i) { return ld_cg(xp + i) - kGd * (ld_cg(Axp + i) + b[i]); },
                     [&](int i, double, double p) {
                         const double xpi = ld_cg(xp + i), xi = ld_cg(x + i);
                         const double dr = cs * (xpi - p);
                         r2[0] = fma(dr, dr, r2[0]);
                         if (AR) r2[1] = fma(ld_cg(g + i), xpi - xi, r2[1]);
                         yn[i] = (1 + beta) * xpi - beta * xi;
                     });
        reduce_sync<2, false>(k, c, r2);
        res = sqrt(r2[0]);
        k.iters += 1;
        if (AR && res < resmin) {
            resmin = res;
            CCQP_ELEMS(i) xhat[i] = ld_cg(xp + i);
        }
        if (res < c.tol) break;
        if (AR && r2[1] > 0) {   // :510-512
            CCQP_ELEMS(i) yn[i] = ld_cg(xp + i);
            theta_n = 1;
            barrier_only<false>(k, c);
        }
        L *= 0.9;
        t = 1.0 / L;
        swap_ptr(y, yn);
        swap_ptr(x, xp);   // afterwards xp names the previous x (what :336 returns on the mv limit)
        theta = theta_n;
    }
    barrier_only<false>(k, c);
    finish(k, c, AR ? xhat : xp, res, 0);
}

// ------------------------------------------------------------------------------------------
// MPRGP with BB / expansion steps                                 solvers.py:1048-1200
// ------------------------------------------------------------------------------------------
// Feasibility bisection (:1112-1118) in one pass: bit j of the result is set iff
// all(isclose(yf, P(yf))) holds for yf = x - (af * 2^-j) p.  Halving is exact in fp64, so the
// step lengths tested are bit-identical to the reference's alpha_f *= 0.5 sequence.
static __device__ unsigned long long bisect_mask(Kst& k, const DenseCtx& c, const double* x, const double* p, double af) {
    unsigned long long m = ~0ull;
    const ProjTable& T = c.T;
    CCQP_ELEMS(i) {
        const int kd = T.ekind[i];
        if (kd == kElemNorm || kd == kIdentity) continue;
        const double xi = ld_cg(x + i), pi = ld_cg(p + i), lo = T.lo[i], hi = T.hi[i];
        double a = af;
        for (int j = 0; j < 64; ++j, a *= 0.5) {
            const double yf = xi - a * pi;
            if (!is_close(yf, clamp_elem(kd, yf, lo, hi))) m &= ~(1ull << j);
        }
    }
    // small norm blocks (Sphere / Cone / SOC with <= 8 entries, the friction-style case): one thread per
    // block keeps x and p of the block in registers and tests all 64 step lengths itself
    for (int sidx = k.gtid; sidx < T.nsmall; sidx += k.gstride) {
        const int bl = T.small_ids[sidx];
        const int off = T.boff[bl], dim = T.bdim[bl];
        double xb[kSmallDim], pb[kSmallDim];
#pragma unroll
        for (int j = 0; j < kSmallDim; ++j) if (j < dim) { xb[j] = ld_cg(x + off + j); pb[j] = ld_cg(p + off + j); }
        NormRule R;
        R.kind = T.bkind[bl]; R.par = T.bpar[bl];
        const int nsq = (R.kind == kSoc) ? dim - 1 : dim;
        double a = af;
        for (int step = 0; step < 64; ++step, a *= 0.5) {
            double t[kSmallDim];
            double ss = 0.0;
#pragma unroll
            for (int j = 0; j < kSmallDim; ++j) {
                if (j < dim) {
                    t[j] = xb[j] - a * pb[j];
                    if (j < nsq) ss = (j == 0) ? t[j] * t[j] : fma(t[j], t[j], ss);     // same chain as project_pass
                }
            }
            R.r = sqrt(ss);
            R.last = 0.0;
#pragma unroll
            for (int j = 0; j < kSmallDim; ++j) if (j == dim - 1) R.last = t[j];
            R.finish();
            bool ok = true;
#pragma unroll
            for (int j = 0; j < kSmallDim; ++j) if (j < dim && !is_close(t[j], R.apply(t[j], j == dim - 1))) ok = false;
            if (!ok) m &= ~(1ull << step);
        }
    }
    if (T.nbig > 0) {   // one CTA per large norm block: one projection pass per step length (rare)
        double a = af;
        for (int j = 0; j < 64; ++j, a *= 0.5) {
            bool ok = true;
            project_pass<false, false>(T, k.gtid, k.gstride, k.sm.scratch,
                                       [&](int i) { return ld_cg(x + i) - a * ld_cg(p + i); },
                                       [&](int, double t, double pr) { if (!is_close(t, pr)) ok = false; });
            if (!ok) m &= ~(1ull << j);
        }
    }
    return and_sync(k, c, m);
}

// y = epi(r, (A vin)_r) for this rank's rows, complete in `dst` on every rank when the call
// returns.  Sharded solves go through the output pool and copy (see the top of this section);
// a single GPU writes dst directly.  Ends with a barrier.
template <bool kOutlineCsr = false, class Epi>
__device__ __forceinline__ void gemv_into(Kst& k, const DenseCtx& c, const double* vin, double* dst, Epi epi) {
    double* y = (c.x.world > 1) ? next_y(k, c) : dst;
    gemv_phase<kOutlineCsr>(k, c, vin, [&](int r, double s) { pub_store(c, y, r, epi(r, s)); });
    barrier_only<true>(k, c);
    if (y != dst) {
        CCQP_ELEMS(i) dst[i] = ld_cg(y + i);
        barrier_only<false>(k, c);
    }
}

static __device__ void solve_mprgp(Kst& k, const DenseCtx& c) {
    double *xk = c.vec[0], *xn = c.vec[1], *gk = c.vec[2], *gn = c.vec[3], *p = c.vec[4], *Ap = c.vec[5];
    double *nv = c.vec[6], *w = c.vec[7], *dl = c.vec[8];
    const double* b = c.b;
    const double cs = 1.0 / (3 * (double)c.n * kGd);
    int status = 0;
    project_pass(c.T, k.gtid, k.gstride, k.sm.scratch, [&](int i) { return c.x0[i]; },
                 [&](int i, double, double pr) { xk[i] = pr; xn[i] = pr; });
    barrier_only<false>(k, c);
    gemv_into<true>(k, c, xk, gk, [&](int r, double s) { return s + b[r]; });
    k.mv = 1;
    CCQP_ELEMS(i) gn[i] = ld_cg(gk + i);
    double a1[1] = {residual_partial(k, c, cs, [&](int i) { return ld_cg(xk + i); }, [&](int i) { return ld_cg(gk + i); })};
    reduce_sync<1, false>(k, c, a1);
    double res = sqrt(a1[0]);
    if (res >= c.tol) {
        double a2[2] = {0.0, 0.0};
        gemv_phase<true>(k, c, gk, [&](int r, double s) { const double gr = ld_cg(gk + r); a2[0] = fma(gr, s, a2[0]); a2[1] = fma(gr, gr, a2[1]); });
        k.mv += 1;                                   // counted (:1077-1078)
        reduce_sync<2, true>(k, c, a2);
        double abb = a2[1] / a2[0];
        bool abb_lazy = false;                       // true: abb = BB(xk - xn) still to be evaluated
        project_pass(c.T, k.gtid, k.gstride, k.sm.scratch, [&](int i) { return ld_cg(xk + i); },
                     [&](int i, double t, double pr) { p[i] = is_close(t, pr) ? ld_cg(gk + i) : 0.0; });
        barrier_only<false>(k, c);
        for (;;) {
            dbg_stamp(c, k.iters, 0);
            gemv_into<true>(k, c, xk, gk, [&](int r, double s) { return s + b[r]; });
            k.mv += 1;
            dbg_stamp(c, k.iters, 1);
            if (hit_max(k, c)) break;
            // delta = isclose(xk, P(xk)); psi = delta*gk   (:1093-1094)
            double q3[3] = {0.0, 0.0, 0.0};          // psi.psi, psi.p, #(!delta)
            project_pass(c.T, k.gtid, k.gstride, k.sm.scratch, [&](int i) { return ld_cg(xk + i); },
                         [&](int i, double t, double pr) {
                             const bool cl = is_close(t, pr);
                             const double psi = cl ? ld_cg(gk + i) : 0.0;
                             q3[0] = fma(psi, psi, q3[0]);
                             q3[1] = fma(psi, ld_cg(p + i), q3[1]);
                             if (!cl) q3[2] += 1.0;
                             dl[i] = cl ? 1.0 : 0.0;
                         });
            reduce_sync<3, false>(k, c, q3);
            dbg_stamp(c, k.iters, 2);
            if (c.T.has_cone_ref) { status = 6; break; }   // normal_vector raises (:1095, ss:465)
            double betbet = 0.0;
            if (q3[2] > 0.0) {
                // rare: some entries of xk are not (close to) feasible; the chopped gradient
                // needs normal_vector(xk) and the GLOBAL n.g (:1095-1097)
                normal_pass(c.T, k.gtid, k.gstride, k.sm.scratch, [&](int i) { return ld_cg(xk + i); }, nv);
                barrier_only<false>(k, c);
                double s1[1] = {0.0};
                CCQP_ELEMS(i) s1[0] = fma(ld_cg(nv + i), ld_cg(gk + i), s1[0]);
                reduce_sync<1, false>(k, c, s1);
                const double mng = s1[0] < 0.0 ? s1[0] : 0.0;    // np.min([0, n.g])
                double s2[1] = {0.0};
                CCQP_ELEMS(i) {
                    const double bv = (1.0 - ld_cg(dl + i)) * (ld_cg(gk + i) - mng * ld_cg(nv + i));
                    s2[0] = fma(bv, bv, s2[0]);
                }
                reduce_sync<1, false>(k, c, s2);
                betbet = s2[0];
            }
            if (betbet < q3[0]) {
                double s1[1] = {0.0};
                {
                    double* y = (c.x.world > 1) ? next_y(k, c) : Ap;
                    gemv_phase<true>(k, c, p, [&](int r, double s) { pub_store(c, y, r, s); s1[0] = fma(ld_cg(p + r), s, s1[0]); });
                    k.mv += 1;
                    reduce_sync<1, true>(k, c, s1);
                    if (y != Ap) {
                        CCQP_ELEMS(i) Ap[i] = ld_cg(y + i);
                        barrier_only<false>(k, c);
                    }
                }
                dbg_stamp(c, k.iters, 3);
                if (hit_max(k, c)) break;
                const double pAp = s1[0];
                const double acg = q3[1] / pAp;
                double af = acg + 10 * kEps;
                for (int pass = 0;; ++pass) {         // :1112-1118
                    const unsigned long long m = bisect_mask(k, c, xk, p, af);
                    if (m) { const int j = __ffsll((long long)m) - 1; for (int q = 0; q < j; ++q) af *= 0.5; break; }
                    for (int q = 0; q < 64; ++q) af *= 0.5;
                    if (pass >= 20) break;            // af == 0 by now; the reference would spin forever
                }
                dbg_stamp(c, k.iters, 4);
                if (acg <= af) {
                    // conjugate-gradient step :1121-1135
                    project_pass(c.T, k.gtid, k.gstride, k.sm.scratch,
                                 [&](int i) { return ld_cg(xk + i) - acg * ld_cg(p + i); },
                                 [&](int i, double yv, double pr) {
                                     const double api = ld_cg(Ap + i);
                                     const double gni = ld_cg(gk + i) - acg * api;
                                     xn[i] = yv;
                                     gn[i] = gni;
                                     const double psy = is_close(yv, pr) ? gni : 0.0;
                                     const double bet = psy * api / pAp;          // elementwise "beta" (:1134)
                                     p[i] = psy - bet * ld_cg(p + i);
                                 });
                    abb_lazy = true;
                    barrier_only<false>(k, c);
                } else {
                    // expansion step with a BB step length :1136-1163
                    double s2[2] = {0.0, 0.0};
                    CCQP_ELEMS(i) {
                        const double xi = ld_cg(xk + i), gi = ld_cg(gk + i);
                        const double xh = xi - af * ld_cg(p + i), gh = gi - af * ld_cg(Ap + i);
                        const double sx = xh - xi, sg = gh - gi;
                        s2[0] = fma(sx, sx, s2[0]);
                        s2[1] = fma(sx, sg, s2[1]);
                    }
                    reduce_sync<2, false>(k, c, s2);
                    const double a = s2[0] / (s2[1] + 10 * kEps);
                    project_pass(c.T, k.gtid, k.gstride, k.sm.scratch,
                                 [&](int i) {
                                     const double xh = ld_cg(xk + i) - af * ld_cg(p + i);
                                     const double gh = ld_cg(gk + i) - af * ld_cg(Ap + i);
                                     return xh - a * gh;
                                 },
                                 [&](int i, double, double pr) { xn[i] = pr; });
                    barrier_only<false>(k, c);
                    dbg_stamp(c, k.iters, 5);
                    gemv_into<true>(k, c, xn, gn, [&](int r, double s) { return s + b[r]; });
                    k.mv += 1;
                    dbg_stamp(c, k.iters, 6);
                    if (hit_max(k, c)) break;
                    project_pass(c.T, k.gtid, k.gstride, k.sm.scratch, [&](int i) { return ld_cg(xn + i); },
                                 [&](int i, double t, double pr) { p[i] = is_close(t, pr) ? ld_cg(gn + i) : 0.0; });
                    abb_lazy = true;
                    barrier_only<false>(k, c);
                }
            } else {
                // proportioning step :1164-1182
                if (abb_lazy) {   // alpha_bb of the previous iteration, evaluated only when needed
                    double s1[1] = {0.0};
                    CCQP_ELEMS(i) { const double dv = ld_cg(xk + i) - ld_cg(xn + i); w[i] = dv; s1[0] = fma(dv, dv, s1[0]); }
                    reduce_sync<1, false>(k, c, s1);
                    double s2[1] = {0.0};
                    gemv_phase<true>(k, c, w, [&](int r, double s) { s2[0] = fma(ld_cg(w + r), s, s2[0]); });
                    reduce_sync<1, true>(k, c, s2);
                    abb = s1[0] / (s2[0] + 10 * kEps);
                }
                project_pass(c.T, k.gtid, k.gstride, k.sm.scratch,
                             [&](int i) { return ld_cg(xk + i) - abb * ld_cg(gk + i); },
                             [&](int i, double, double pr) { xn[i] = pr; });
                abb_lazy = true;
                k.mv += 1;            // gk = A xk + b is re-evaluated by the reference (:1174); same value
                barrier_only<false>(k, c);
                if (hit_max(k, c)) break;
                project_pass(c.T, k.gtid, k.gstride, k.sm.scratch, [&](int i) { return ld_cg(xn + i); },
                             [&](int i, double t, double pr) { p[i] = is_close(t, pr) ? ld_cg(gn + i) : 0.0; });   // stale gn (:1181)
                barrier_only<false>(k, c);
            }
            double r1[1] = {residual_partial(k, c, cs, [&](int i) { return ld_cg(xn + i); }, [&](int i) { return ld_cg(gn + i); })};
            reduce_sync<1, false>(k, c, r1);
            res = sqrt(r1[0]);
            k.iters += 1;
            if (res < c.tol) break;
            swap_ptr(xk, xn);
            swap_ptr(gk, gn);
        }
    }
    barrier_only<false>(k, c);
    finish(k, c, xn, res, status);
}

// ------------------------------------------------------------------------------------------
// kernel
// ------------------------------------------------------------------------------------------
template <int OP>
__device__ __forceinline__ void dense_body(const DenseCtx& c, const int bid, const int nblk) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Kst k;
    {
        unsigned char* q = smem_raw;
        k.sm.vbuf[0] = reinterpret_cast<double*>(q); q += (size_t)c.CW * 8;
        k.sm.vbuf[1] = reinterpret_cast<double*>(q); q += (size_t)c.CW * 8;
        k.sm.psum = reinterpret_cast<double*>(q); q += (size_t)c.rows_max * c.nseg * 8;
        k.sm.scratch = reinterpret_cast<double*>(q); q += kMaxRed * 32 * 8;
        k.sm.ascratch = reinterpret_cast<unsigned long long*>(q); q += 32 * 8;
        k.sm.mbar = reinterpret_cast<uint64_t*>(q);
    }
    k.epoch = 0;
    k.xepoch = 0;
    k.bid = bid;
    k.nblk = nblk;
    k.gtid = bid * kDenseThreads + threadIdx.x;
    k.gstride = nblk * kDenseThreads;
    k.r0 = c.row0 + (int)(((long long)c.nrows * bid) / nblk);
    k.r1 = c.row0 + (int)(((long long)c.nrows * (bid + 1)) / nblk);
    if (!CCQP_DENSE_ONLY && c.csr_val) {    // CSR: nnz-balanced, row-aligned split (first row whose start is at or beyond bid * nnz / G)
        const long long nnz = c.csr_ptr[c.nrows];
        auto first_row_at = [&](long long target) {
            int lo = 0, hi = c.nrows;                                 // smallest r in [0, nrows] with csr_ptr[r] >= target
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (c.csr_ptr[mid] >= target) hi = mid; else lo = mid + 1; }
            return lo;
        };
        k.r0 = c.row0 + (bid == 0 ? 0 : first_row_at(nnz / nblk * bid + nnz % nblk * bid / nblk));
        k.r1 = c.row0 + (bid == nblk - 1 ? c.nrows : first_row_at(nnz / nblk * (bid + 1) + nnz % nblk * (bid + 1) / nblk));
    }
    k.parbits = 0u;
    k.mv = k.gemv = k.iters = k.draws = 0;
    k.yq = 0;
    if (threadIdx.x == 0) {
        for (int i = 0; i < kNumMbar; ++i) mbar_init(&k.sm.mbar[i], 1);
        mbar_fence_init();
    }
    __syncthreads();

    if constexpr (OP == OP_PGD || OP == OP_BBPGD || OP == OP_BBPGDF) solve_pgd_family<OP>(k, c);
    else if constexpr (OP == OP_SPG) solve_spg(k, c);
    else if constexpr (OP == OP_APGD) solve_apgd<false>(k, c);
    else if constexpr (OP == OP_APGD_AR) solve_apgd<true>(k, c);
    else if constexpr (OP == OP_MPRGP) solve_mprgp(k, c);
    else if constexpr (OP == OP_GEMV) {
        gemv_phase(k, c, c.hook_in, [&](int r, double s) { c.hook_out[r - c.row0] = s; });
    } else if constexpr (OP == OP_PROJECT) {
        project_pass(c.T, k.gtid, k.gstride, k.sm.scratch, [&](int i) { return c.hook_in[i]; },
                     [&](int i, double, double p) { c.hook_out[i] = p; });
    } else if constexpr (OP == OP_NORMAL) {
        normal_pass(c.T, k.gtid, k.gstride, k.sm.scratch, [&](int i) { return c.hook_in[i]; }, c.hook_out);
    } else if constexpr (OP == OP_PROJGRAD) {
        // projected_gradient(x, g) of the elementwise kinds (solution_spaces.py:162-184, 238-260, 324-347, per leaf of a
        // DisjointProjOp :527-538): hook_in = x, vec[0] = g, hook_out = normal_vector(x) (an OP_NORMAL launch before this
        // one); vec[1] = free gradient, vec[2] = chopped gradient.  Box's activity test is the reference's, as written (:339-340).
        const double *g = c.vec[0], *nv = c.hook_out;
        double *fr = c.vec[1], *ch = c.vec[2];
        CCQP_ELEMS(i) {
            const int kd = c.T.ekind[i];
            const double x = c.hook_in[i], gi = g[i], lo = c.T.lo[i], hi = c.T.hi[i];
            bool act = false;
            if (kd == kLower) act = is_close(x, lo);
            else if (kd == kUpper) act = is_close(x, hi);
            else if (kd == kBox) act = is_close(x, hi) || x > hi || is_close(x, (lo != 0.0) ? lo : (x < hi ? 1.0 : 0.0));
            const double t = nv[i] * gi;
            const double m = (t < 0.0 || t != t) ? t : 0.0;              // np.min((normal*g, 0)) keeps a NaN
            fr[i] = act ? 0.0 : gi;
            ch[i] = act ? gi - m * nv[i] : 0.0;
        }
    }
}

template <int OP>
__global__ void __launch_bounds__(kDenseThreads, 1) dense_kernel(const DenseCtx c) {
    dense_body<OP>(c, (int)blockIdx.x, (int)gridDim.x);
}

// Test vehicle for the multi-GPU exchange protocol on ONE GPU: `world` ranks inside a single cooperative launch.
// CTAs [r*G, (r+1)*G) play rank r with rank r's context (its row shard, its work buffer, its sync words); the
// "peer" buffers are the other ranks' buffers in the same device memory, so pub_store / grid_xsync execute exactly
// the code of a real sharded solve (LL packets included), only the stores do not cross NVLink.  (Ranks as separate
// launches on one GPU would deadlock: nothing guarantees that kernels that wait on one another run concurrently.)
template <int OP>
__global__ void __launch_bounds__(kDenseThreads, 1) dense_kernel_emu(const DenseCtx* __restrict__ ctxs, const int G) {
    __shared__ DenseCtx c;
    {
        const int* src = reinterpret_cast<const int*>(ctxs + blockIdx.x / G);
        int* dst = reinterpret_cast<int*>(&c);
        for (int i = threadIdx.x; i < (int)(sizeof(DenseCtx) / sizeof(int)); i += kDenseThreads) dst[i] = src[i];
    }
    __syncthreads();
    dense_body<OP>(c, (int)blockIdx.x % G, G);
}

}  // namespace ccqp
