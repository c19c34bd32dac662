// Batched mode: thousands of small independent QPs (n <= 128), one CTA per problem at a time, the whole solver loop of the
// reference inside one persistent kernel (no host round trips).  Problem i is
//     CCQPSolverX(tol,max_mv).solve(A[i], b[i], x0[i], BoxProjOp(n, lb[i], ub[i]))          (ccqp_solve_batched)
// or  CCQPSolverX(tol,max_mv).solve(A[i], b[i], x0[i], op)  with ONE operator of any kind    (ccqp_solve_batched_table)
// or  CCQPSolverX(tol,max_mv).solve(A[i], b[i], x0[i], op_i), op_i one block structure with its own parameters
//                                                                                         (ccqp_solve_batched_tables)
// (solvers.py:94/220/393/583/719/878/1026 with solution_spaces.py:77-560).
//
// Data path per problem (n = 64: 32 KB of A, 2 KB of vectors in, 512 B out):
//   * A lives in REGISTERS for the whole solve.  n <= 64: 64 threads, thread t = 8*rb + cb keeps the 8 x 8 sub-block
//     A[8rb .. 8rb+7][8cb .. 8cb+7] (64 doubles = 128 registers), 6 CTAs per SM.  64 < n <= 128: 256 threads, a 16 x 16 grid
//     of the same 8 x 8 sub-blocks, one CTA per SM (struct BL<NT>).  The problem AFTER the current one travels into a padded
//     shared-memory tile by TMA row copies (cp.async.bulk + one mbarrier; its b / lb / ub rows -- general table: b and its
//     parameter row -- ride on the same mbarrier) while the current one iterates; the register fill from the tile is
//     conflict-free LDS.128.  The work queue is two problems deep, so neither the atomic that hands out problems nor any global load sits on a problem's dependent chain.
//   * mat-vec: the input vector is published through a double-buffered, bank-padded shared array (one barrier); a thread reads
//     only its 8-entry slice (4 LDS.128), does 64 DFMAs (8 rows x 8 columns, 8 independent chains) and the lanes of a row
//     block combine their partial rows with a 3-stage exchange butterfly (7 SHFL.64 + 7 DADD) after which the thread holds y
//     of the unknown it owns.
//     Why not "thread t keeps row t" (the first version of this kernel): every thread then reads all 64 entries of x per
//     mat-vec, and a warp-wide LDS.128 occupies the shared-memory crossbar for 4 cycles (512 bytes delivered) whether or
//     not the lanes read the same address: 256 crossbar cycles per mat-vec per problem against 64 cycles of FP64 pipe.  ncu
//     showed exactly that (shared-memory wavefronts 59 %, FP64 pipe 32 %; profiles/r01_ncu_full_first.csv).  The 8 x 8
//     blocking needs 32 crossbar cycles for x plus 28 for the shuffles.  (A 4 x 16 blocking, 2-stage butterfly but 8 LDS.128
//     per thread, measured slower and was removed in round 2.)
//   * dot products: K <= 4 sums are reduced together with an exchange butterfly (6 SHFL.64 + 6 DADD for K = 3 instead of
//     15 + 15), then the warps swap through shared memory (one barrier).  CCQP_BATCHED_DMMA=1 runs the 32-lane sums on the
//     FP64 tensor path instead (measured equal, DESIGN.md 2.2).
//   * stopping tests compare the SQUARED residual with a host-computed threshold that is exactly equivalent to the
//     reference's sqrt(.) < tol (sqrt is monotone), so no sqrt is on the per-iteration critical path; the reported
//     residual is computed once at the end.
//   * everything else (projection, axpy, step lengths) is per-thread register arithmetic, with the reference's rounding
//     (compiled with -fmad=false; explicit fma() only in the sums).
//   Problems are handed out through an atomic counter (iteration counts differ per problem); results do not depend on the
//   schedule.
//
// Bounds: HBM bytes/problem = 8 n^2 + 32 n (+8 n for x0, + uniforms read by SPG);
//         fp64 flops/problem = 2 n^2 * (mat-vecs executed).
#pragma once
#include <algorithm>
#include <climits>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <functional>
#include <string>
#include <vector>

#include "proj.cuh"
#include "../../include/ccqp_b200.h"

#ifndef CCQP_BATCHED_STAGE
#define CCQP_BATCHED_STAGE 1    // 1: A reaches the registers through a TMA-filled shared tile (next problem in flight
#endif                          //    during the solve); 0: straight from L2 (bulk L2 prefetch of the next problem)
namespace ccqp {

// Launch shape and layout of one problem.
//   NT = 64 threads, n <= 64 (the benchmark configuration): thread t = 8 rb + cb keeps the 8 x 8 sub-block (row block rb, column
//   block cb) of A in registers and owns unknown t.
//   NT = 256 threads, n <= 128: thread t = 16 rb + cb, a 16 x 16 grid of 8 x 8 sub-blocks.  The 16 lanes of a row block end the
//   mat-vec with 8 row sums, so TWO neighbouring lanes hold (and redundantly update) the same unknown 8 rb + (cb >> 1); the even
//   lane of the pair is its owner: it publishes the entry, feeds the reductions and writes the result.
template <int NT>
struct BL {
    static_assert(NT == 64 || NT == 256, "threads per problem");
    static constexpr int N = NT == 64 ? 64 : 128;      // max unknowns per problem
    static constexpr int NB = N / 8;                   // column blocks = lanes that share a row block
    static constexpr int SH = NT == 64 ? 0 : 1;        // log2 of the lanes that hold one unknown
    static constexpr int WARPS = NT / 32;
    static constexpr int SLICE = 8 + 2;                // pitch of one 8-entry slice of the mat-vec input: consecutive slices start 16
                                                       // bytes further into the 128-byte bank window (conflict-free LDS.128)
    static constexpr int XS = NB * SLICE;
    static constexpr int PITCH = N + 2;                // tile row pitch (doubles): conflict-free LDS.128 register fill
    static constexpr uint32_t XS_BYTES = XS * 8, RED_BYTES = WARPS * 32;
};
constexpr int kBN = 64;                 // the small layout's limit
constexpr int kBNMax = 128;             // largest n of the batched mode
constexpr int kBRows = 8, kBCols = 8;   // sub-block of A held by one thread
constexpr int kBWindow = 64;            // SPG window limit (generic path)
constexpr int kBWinReg = 5;             // SPG window kept in registers when m == kBWinReg (the reference default)

struct BatchedOut {
    double residual;
    int mv, gemv, iters, draws;
    int converged, status;
};

struct BatchedCtx {
    const double* A;        // [batch][n][n]
    const double* b;        // [batch][n]
    const double* x0;       // [batch][n] or null
    const double* lb;       // [batch][n] (Box per problem; unused by the general table)
    const double* ub;
    long long bound_stride; // n
    // general projection table (ccqp_solve_batched_table / _tables): the block structure is shared by all problems of the
    // batch, problem i takes its parameters from the row params + i * param_stride; null ekind = Box per problem
    const uint8_t* ekind;   // [n] kIdentity / kLower / kUpper / kBox / kElemNorm
    const int* eoff;        // [n] first element of the norm block the element belongs to
    const int* edim;        // [n] its dimension
    const int* enk;         // [n] its kind (kSphere / kConeRef / kSoc)
    const int4* eidx;       // [n] where the element's lower bound / upper bound / block parameter (radius / aspect ratio)
                            // sit in a parameter row (x / y / z); -1: none (-inf / +inf / unused)
    int has_norm;           // some element belongs to a norm block
    const double* uniforms; // [batch][n_uniforms]
    long long n_uniforms;
    double* x_out;          // [batch][n]
    BatchedOut* out;        // [batch]
    unsigned* counter;      // work queue head
    int batch, n;
    int tma_ok;             // rows of A can be moved with 16-byte bulk copies (8n % 16 == 0, 16-byte aligned base)
    int vec_ok;             // rows of A can be read with 256-bit loads (n % 4 == 0, 32-byte aligned base)
    int pf_ok;              // whole problems can be bulk-prefetched into L2 (16-byte granularity)
    int vtma_ok;            // b / lb / ub rows (general table: b and parameter rows) can be moved with 16-byte bulk copies
                            // (n even, 16-byte aligned bases; general table: see prow_bytes)
    double tol, max_mv, step, tau, sig1, sig2;
    double thr_lt;          // q <  thr_lt  <=>  sqrt(q) <  tol      (solvers.py:156 etc.)
    double thr_le;          // q <= thr_le  <=>  sqrt(q) <= tol      (SPG, solvers.py:949)
    int max_mv_i;           // mv >= max_mv_i  <=>  (double)mv >= max_mv
    int m;
    // general table: parameter rows (param_stride 0: one row shared by the whole batch)
    const double* params;
    long long param_stride;
    int prow_bytes;         // bytes of a parameter row the bulk copy moves when vtma_ok: a multiple of 16, <= 16 N (the
                            // vstage[1..2] area); 0: no parameters
};

template <bool GEN, int NT>
struct BatchedSmem {
#if CCQP_BATCHED_STAGE
    double tile[BL<NT>::N * BL<NT>::PITCH];   // the NEXT problem's A, landed by TMA while the current one iterates
    double vstage[3][BL<NT>::N];              // ... and its b / lower / upper bounds (general table: b / parameter row
                                              // of up to 2 N entries in vstage[1..2]) on the same mbarrier
#endif
    double xs[2][BL<NT>::XS];                 // mat-vec input, double buffered
    double red[2][BL<NT>::WARPS][4];          // [parity][warp][slot]
    double pj[GEN ? 2 : 1][GEN ? BL<NT>::N : 2];   // general table: the vector being projected, for the members of norm blocks
#if CCQP_BATCHED_STAGE
    uint64_t mbar;
#endif
    int next;               // the problem after the next one (fetched during the solve of the current one)
    int first;              // prologue: this CTA's first problem
};

// Shared-memory accesses of the solver loop go through 32-bit shared-space addresses computed once
// per thread: with generic pointers the compiler re-derives the shared window base (S2UR
// SR_CgaCtaId + ULEA, a scoreboard stall) in front of every access of the loop.
struct BShared {
    uint32_t xs_wr;     // where the owner of an unknown publishes its entry (buffer 0)
    uint32_t xs_rd;     // this thread's 8-entry slice (buffer 0)
    uint32_t red;       // red[0][0][0]
};

__device__ __forceinline__ void sts_f64(uint32_t addr, double v) {
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}
__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void lds_f64x2(uint32_t addr, double& x, double& y) {
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(x), "=d"(y) : "r"(addr) : "memory");
}

__device__ __forceinline__ double shfl_xor_f64(double v, int mask) { return __shfl_xor_sync(0xffffffffu, v, mask); }

// Sum K (<= 4) values over the 64 threads; result in every thread; ONE __syncthreads.
// Exchange butterfly: after the first stages each lane carries ONE of the K sums, so the tree
// costs max(K,2)+3 shuffles and adds instead of 5K.  Fixed order => deterministic.
#ifndef CCQP_BATCHED_DMMA
#define CCQP_BATCHED_DMMA 0     // 1: the 32-lane sums of cta64_sum run on the FP64 tensor path (2 DMMA.8x8x4 + 1 DADD per sum)
#endif
// D(8x8) = A(8x4) B(4x8) + C, FP64 (SASS DMMA.8x8x4): lane l holds A[l/4][l%4], B[l%4][l/4], C/D[l/4][2(l%4)], [2(l%4)+1]
__device__ __forceinline__ void dmma884_ones(double& d0, double& d1, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%4,%5};"
                 : "=d"(d0), "=d"(d1) : "d"(1.0), "d"(b), "d"(0.0), "d"(0.0));
}

// Cross-warp part of bsum: the warps' partial sums (red[parity][warp][slot]) are added in warp order
template <int K, int NT>
__device__ __forceinline__ void bsum_collect(double (&a)[K], uint32_t base) {
    if constexpr (NT == 64) {
        if constexpr (K == 1) {
            a[0] = lds_f64(base) + lds_f64(base + 32);
        } else {
            double p0, p1, q0, q1;
            lds_f64x2(base, p0, p1);
            lds_f64x2(base + 32, q0, q1);
            a[0] = p0 + q0; a[1] = p1 + q1;
            if constexpr (K == 3) a[2] = lds_f64(base + 16) + lds_f64(base + 48);
            if constexpr (K == 4) {
                lds_f64x2(base + 16, p0, p1);
                lds_f64x2(base + 48, q0, q1);
                a[2] = p0 + q0; a[3] = p1 + q1;
            }
        }
    } else {
        double v[BL<NT>::WARPS][4];
#pragma unroll
        for (int w = 0; w < BL<NT>::WARPS; ++w) {
            lds_f64x2(base + w * 32, v[w][0], v[w][1]);
            if constexpr (K > 2) lds_f64x2(base + w * 32 + 16, v[w][2], v[w][3]);
        }
#pragma unroll
        for (int j = 0; j < K; ++j) {
            double t = v[0][j];
#pragma unroll
            for (int w = 1; w < BL<NT>::WARPS; ++w) t += v[w][j];
            a[j] = t;
        }
    }
}

template <int K, int NT>
__device__ __forceinline__ void bsum(double (&a)[K], const BShared& sh, int& parity, bool own) {
    static_assert(K >= 1 && K <= 4, "K");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if constexpr (BL<NT>::SH != 0) {        // an unknown held by two lanes counts once
#pragma unroll
        for (int j = 0; j < K; ++j) a[j] = own ? a[j] : 0.0;
    }
#if CCQP_BATCHED_DMMA
    // With A = ones the first product leaves the sums of the 8 quads of lanes (a lane receives the two quads of ITS octet
    // l%4), one add makes the octet sums, and the second product adds the four octets: the warp total in every lane.
    // K independent chains, 2 DMMA + 1 DADD deep, against 5 dependent SHFL.64 + DADD stages; fixed order => deterministic.
    {
        double p[K], e0, e1;
#pragma unroll
        for (int j = 0; j < K; ++j) { dmma884_ones(e0, e1, a[j]); p[j] = e0 + e1; }
#pragma unroll
        for (int j = 0; j < K; ++j) { dmma884_ones(e0, e1, p[j]); p[j] = e0; }
        const uint32_t base = sh.red + (uint32_t)parity * BL<NT>::RED_BYTES;
        if (lane < K) {
            double v = p[0];
#pragma unroll
            for (int j = 1; j < K; ++j) v = (lane == j) ? p[j] : v;
            sts_f64(base + (uint32_t)(warp * 4 + lane) * 8u, v);
        }
        __syncthreads();
        bsum_collect<K, NT>(a, base);
        parity ^= 1;
        return;
    }
#endif
    double v;
    int slot;            // which of the K sums this lane ends up carrying (lanes 0..3 are used)
    if constexpr (K == 1) {
        v = a[0] + shfl_xor_f64(a[0], 1);
        v += shfl_xor_f64(v, 2);
        slot = 0;
    } else if constexpr (K == 2) {
        const bool odd = lane & 1;
        const double keep = odd ? a[1] : a[0], send = odd ? a[0] : a[1];
        v = keep + shfl_xor_f64(send, 1);
        v += shfl_xor_f64(v, 2);
        slot = lane & 1;
    } else {
        const bool odd = lane & 1;
        const double a3 = (K == 4) ? a[K - 1] : 0.0;
        double k0 = odd ? a[2] : a[0], k1 = odd ? a3 : a[1];
        const double s0 = odd ? a[0] : a[2], s1 = odd ? a[1] : a3;
        k0 += shfl_xor_f64(s0, 1);
        if (K == 4) k1 += shfl_xor_f64(s1, 1);
        else { const double r = shfl_xor_f64(s1, 1); k1 = odd ? 0.0 : k1 + r; }   // slot 3 unused for K == 3
        const bool up = lane & 2;
        const double keep = up ? k1 : k0, send = up ? k0 : k1;
        v = keep + shfl_xor_f64(send, 2);
        slot = 2 * (lane & 1) + ((lane >> 1) & 1);
    }
    v += shfl_xor_f64(v, 4);
    v += shfl_xor_f64(v, 8);
    v += shfl_xor_f64(v, 16);
    const uint32_t base = sh.red + (uint32_t)parity * BL<NT>::RED_BYTES;      // red[parity]: WARPS x 4 slots x 8 bytes
    if (lane < 4 && slot < K) sts_f64(base + (uint32_t)(warp * 4 + slot) * 8u, v);
    __syncthreads();
    bsum_collect<K, NT>(a, base);
    parity ^= 1;
}

// bitwise AND of a 64-bit mask over the threads of the CTA (MPRGP's bisection); ONE __syncthreads
template <int NT>
__device__ __forceinline__ unsigned long long band(unsigned long long m, const BShared& sh, int& parity) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    m = warp_and64(m);
    const uint32_t base = sh.red + (uint32_t)parity * BL<NT>::RED_BYTES;
    if (lane == 0) sts_f64(base + (uint32_t)warp * 32u, __longlong_as_double((long long)m));
    __syncthreads();
    unsigned long long r = ~0ull;
#pragma unroll
    for (int w = 0; w < BL<NT>::WARPS; ++w) r &= (unsigned long long)__double_as_longlong(lds_f64(base + w * 32));
    parity ^= 1;
    return r;
}

__device__ __forceinline__ double clampd(double t, double lo, double hi) { return t < lo ? lo : (t > hi ? hi : t); }

// Publish v (this thread's unknown, as the mat-vec input) and return (A v) for that unknown.
// Thread t = NB*rb + cb holds the 8 x 8 sub-block (row block rb, column block cb).  With key = cb >> SH (3 bits), register row
// i holds row 8*rb + (i ^ key) of A (the fill permutes the rows), so that in the exchange butterfly below the partial sums a
// lane keeps and the ones it sends sit in FIXED registers: no per-lane selects.  Stage h = 4, 2, 1 (lane distance h << SH): a
// lane keeps the rows whose bit h agrees with its own key and receives the partner's partial sums of exactly those rows; after
// the last stage the lane holds row 0 ^ key = key complete over its half of the column blocks, and (NT = 256) one more add with
// the neighbouring lane completes it: the thread holds y for the unknown 8*rb + key it owns.
// `act` is false for the padding (unknown index >= n): it is published as an exact zero whatever v is, so a
// non-finite step length cannot leak NaNs into the active rows through the zero columns of A.
template <int NT>
__device__ __forceinline__ double matvec(const double (&a)[kBRows][kBCols], const BShared& sh, int& xpar, bool act,
                                         double v) {
    constexpr int SH = BL<NT>::SH;
    const uint32_t boff = (uint32_t)xpar * BL<NT>::XS_BYTES;
    if (SH == 0 || !(threadIdx.x & 1)) sts_f64(sh.xs_wr + boff, act ? v : 0.0);
    __syncthreads();
    const uint32_t xp = sh.xs_rd + boff;
    xpar ^= 1;
    double x[kBCols];
#pragma unroll
    for (int j = 0; j < kBCols; j += 2) lds_f64x2(xp + j * 8, x[j], x[j + 1]);
    double s[kBRows];
#pragma unroll
    for (int r = 0; r < kBRows; ++r) s[r] = a[r][0] * x[0];         // one chain per row
#pragma unroll
    for (int j = 1; j < kBCols; ++j)
#pragma unroll
        for (int r = 0; r < kBRows; ++r) s[r] = fma(a[r][j], x[j], s[r]);
#pragma unroll
    for (int h = kBRows / 2; h >= 1; h >>= 1)
#pragma unroll
        for (int i = 0; i < h; ++i) s[i] += shfl_xor_f64(s[i + h], h << SH);
    if constexpr (SH != 0) s[0] += shfl_xor_f64(s[0], 1);
    return s[0];
}

struct BState {                 // per-thread view of one problem (thread t <-> unknown t)
    double b, lo, hi, x0;       // general table: a member of a norm block has no bounds, its `lo` is the block's parameter
    double cs;                  // 1/(3 n gd)
    bool act;                   // the unknown exists (index < n)
    bool own;                   // ... and this thread is the lane that owns it (NT = 64: the same thing)
    int u;                      // index of the unknown
    // general table only
    int kind;                   // element kind
    int boff, bdim, bnk;        // norm block of this element (its parameter: lo)
    uint32_t pj;                // shared address of pj[0][0]
};

// P(t)_own for the general table.  Elementwise kinds: compare/select as in proj.cuh.  Members of a norm block (Sphere /
// reference Cone / SOC of any dimension <= n): the vector goes through shared memory, every member reads its block and
// forms the norm with the sequential FMA chain of project_pass (proj.cuh), then applies the block's rule to its own entry.
// Every thread of the CTA must call it (one barrier when the table has norm blocks).
template <int NT>
__device__ __forceinline__ double project_general(const BState& s, bool has_norm, int& ppar, double t) {
    double p = clamp_elem(s.kind, t, s.lo, s.hi);
    if (has_norm) {
        const uint32_t base = s.pj + (uint32_t)ppar * (BL<NT>::N * 8u);
        sts_f64(base + (uint32_t)s.u * 8u, t);        // (NT = 256: both lanes of an unknown store the same value)
        __syncthreads();
        if (s.kind == kElemNorm) {
            NormRule R;
            R.kind = s.bnk; R.par = s.lo;
            const int nsq = (s.bnk == kSoc) ? s.bdim - 1 : s.bdim;
            double ss = 0.0, last = 0.0;
            for (int j = 0; j < s.bdim; ++j) {
                const double tj = lds_f64(base + (uint32_t)(s.boff + j) * 8u);
                if (j < nsq) ss = (j == 0) ? tj * tj : fma(tj, tj, ss);
                last = tj;
            }
            R.r = sqrt(ss); R.last = last;
            R.finish();
            p = R.apply(t, s.u == s.boff + s.bdim - 1);
        }
        ppar ^= 1;
    }
    return p;
}

// SPG's deque(maxlen=m) (solvers.py:931).  Only max() over the contents is ever taken (:953), so the
// order of the entries is irrelevant: for the reference default m = 5 the window is a 5-register
// shift register padded with -inf (max ignores the padding; 4 moves + 4 compares per iteration);
// any other m uses a ring buffer in local memory.
template <bool REG>
struct SpgWindow {
    double w[REG ? kBWinReg : kBWindow];
    int count, head;
    __device__ __forceinline__ void init(double f) {
        if constexpr (REG) {
#pragma unroll
            for (int j = 0; j < kBWinReg - 1; ++j) w[j] = -INFINITY;
            w[kBWinReg - 1] = f;
        } else { w[0] = f; count = 1; head = 0; }
    }
    __device__ __forceinline__ double max() const {
        if constexpr (REG) {
            double fmax = w[0];
#pragma unroll
            for (int j = 1; j < kBWinReg; ++j) fmax = fmax > w[j] ? fmax : w[j];
            return fmax;
        } else {
            double fmax = w[0];
            for (int j = 1; j < count; ++j) fmax = fmax > w[j] ? fmax : w[j];
            return fmax;
        }
    }
    __device__ __forceinline__ void push(double f, int m) {
        if constexpr (REG) {
#pragma unroll
            for (int j = 0; j < kBWinReg - 1; ++j) w[j] = w[j + 1];
            w[kBWinReg - 1] = f;
        } else {
            if (count < m) { w[count] = f; count++; }
            else { w[head] = f; head = (head + 1 == m) ? 0 : head + 1; }
        }
    }
};

template <int SOLVER, bool WREG, bool GEN, int NT>
__device__ __forceinline__ void solve_one(const BatchedCtx& c, const double (&a)[kBRows][kBCols], const BShared& sm,
                                          const BState& s, const double* uni, int& par, int& xpar, double& xsol,
                                          BatchedOut& o) {
    int mv = 0, gemv = 0, iters = 0, draws = 0, status = 0;
    double res = NAN;
    const int maxmv = c.max_mv_i;
    int ppar = 0;
    // the projection: Box per problem (solution_spaces.py:363-366), or the batch's general table
    auto P = [&](double t) { if constexpr (GEN) return project_general<NT>(s, c.has_norm != 0, ppar, t); else return clampd(t, s.lo, s.hi); };
    auto resid2 = [&](double x, double g) { const double d = s.cs * (x - P(x - kGd * g)); return d * d; };

    if constexpr (SOLVER == CCQP_SOLVER_PGD || SOLVER == CCQP_SOLVER_BBPGD || SOLVER == CCQP_SOLVER_BBPGDF) {
        // solvers.py:114-170, 606-669, 741-819
        double x = s.x0, xm = s.x0, g, gm, xmin = s.x0, gmin = s.x0, resmin = INFINITY;
        gm = matvec<NT>(a, sm, xpar, s.act, xm) + s.b; gemv++; mv = 1;
        double r1[1] = {resid2(xm, gm)};
        bsum<1, NT>(r1, sm, par, s.own);
        double res2 = r1[0];
        if (!(res2 < c.thr_lt)) {
            double step = c.step;
            if (SOLVER != CCQP_SOLVER_PGD) {
                const double ag = matvec<NT>(a, sm, xpar, s.act, gm); gemv++;          // not counted (:635)
                double q[2] = {gm * gm, gm * ag};
                bsum<2, NT>(q, sm, par, s.own);
                step = q[0] / q[1];
            }
            for (;;) {
                x = P(xm - step * gm);
                g = matvec<NT>(a, sm, xpar, s.act, x) + s.b; gemv++; mv++;
                if (mv >= maxmv) break;
                const double sx = x - xm, sy = g - gm;
                double q[3] = {resid2(x, g), sx * sx, sx * sy};
                if (SOLVER == CCQP_SOLVER_PGD) { double q1[1] = {q[0]}; bsum<1, NT>(q1, sm, par, s.own); q[0] = q1[0]; }
                else bsum<3, NT>(q, sm, par, s.own);
                res2 = q[0];
                iters++;
                if (res2 < c.thr_lt) break;
                if (SOLVER == CCQP_SOLVER_BBPGDF) {                   // :793-800
                    res = sqrt(res2);
                    if (res < resmin) { resmin = res; xmin = x; gmin = g; }
                    if (step < 10 * kEps) {
                        x = P(xmin - kGd * gmin);
                        const double sx2 = x - xm;
                        double q2[2] = {sx2 * sx2, sx2 * sy};
                        bsum<2, NT>(q2, sm, par, s.own);
                        q[1] = q2[0]; q[2] = q2[1];
                    }
                }
                if (SOLVER != CCQP_SOLVER_PGD) step = q[1] / (q[2] + 10 * kEps);
                xm = x; gm = g;
            }
        }
        res = sqrt(res2);
        xsol = x;
    } else if constexpr (SOLVER == CCQP_SOLVER_SPG) {
        // solvers.py:906-975
        double x = s.x0;
        double g = matvec<NT>(a, sm, xpar, s.act, x) + s.b; gemv++;
        const double ag = matvec<NT>(a, sm, xpar, s.act, g); gemv++;
        double q0[3] = {g * x, g * g, g * ag};
        bsum<3, NT>(q0, sm, par, s.own);
        double f = q0[0];
        double alpha = q0[1] / q0[2];
        mv = 2;
        SpgWindow<WREG> win;
        win.init(f);
        double dd_rep = NAN;
        // the stream of uniforms lives in global memory: the sample of iteration k+1 is fetched while iteration k runs
        // (an L2 round trip per iteration would otherwise sit on the dependent chain)
        double u_next = (c.n_uniforms > 0) ? __ldg(uni) : 0.0;
        for (;;) {
            const double d = P(x - alpha * g) - x;
            const double ad = matvec<NT>(a, sm, xpar, s.act, d); gemv++; mv++;
            if (mv >= maxmv) break;
            double q[3] = {d * d, d * ad, d * g};
            bsum<3, NT>(q, sm, par, s.own);
            const double dd = q[0], dAd = q[1], dg = q[2];
            dd_rep = dd;
            if (dd <= c.thr_le) break;                                // sqrt(dd) <= tol (:949)
            const double fmax = win.max();
            double xi, beta, alpha_next;                              // (fmax - f)/dAd, -dg/dAd, dd/dAd (:954,:955,:966)
            div3_same_divisor(fmax - f, -dg, dd, dAd, xi, beta, alpha_next);
            const double bhat = c.tau * beta + sqrt((c.tau * c.tau) * (beta * beta) + 2 * xi);
            const double hi = (c.sig2 < bhat) ? c.sig2 : bhat;        // Python min(bhat, sig2)
            if (hi != hi) { status = CCQP_ERR_RANGE; break; }
            if (draws >= c.n_uniforms) { status = CCQP_ERR_UNIFORMS_EXHAUSTED; break; }
            const double bk = c.sig1 + (hi - c.sig1) * u_next;
            draws++;
            u_next = (draws < c.n_uniforms) ? __ldg(uni + draws) : 0.0;
            x += bk * d;
            g += bk * ad;
            f += bk * bk * dg + 0.5 * (bk * bk) * dAd;                // :963 as written
            win.push(f, c.m);
            alpha = alpha_next;
            iters++;
        }
        res = sqrt(dd_rep);
        xsol = x;
    } else if constexpr (SOLVER == CCQP_SOLVER_APGD || SOLVER == CCQP_SOLVER_APGD_AR) {
        // solvers.py:242-343, 415-533
        constexpr bool AR = SOLVER == CCQP_SOLVER_APGD_AR;
        double x = s.x0, y = s.x0, xp = s.x0, xhat = 1.0, axp = 0.0;
        const double d0 = s.act ? (s.x0 - 1.0) : 0.0;
        const double ad0 = matvec<NT>(a, sm, xpar, s.act, d0); gemv++; mv = 1;
        double q0[2] = {ad0 * ad0, d0 * d0};
        bsum<2, NT>(q0, sm, par, s.own);
        double L = sqrt(q0[0]) / sqrt(q0[1]);
        double t = 1.0 / L, theta = 1.0, resmin = INFINITY, res2 = NAN;
        for (;;) {
            const double ay = matvec<NT>(a, sm, xpar, s.act, y); gemv++; mv++;
            if (mv >= maxmv) break;
            const double g = ay + s.b;
            xp = P(y - t * g);
            bool have12 = false;
            double rt1 = 0.0, rt2 = 0.0;
            for (;;) {
                axp = matvec<NT>(a, sm, xpar, s.act, xp); gemv++; mv++;
                const bool lim = mv >= maxmv;
                const double df = xp - y;
                double qa[4] = {xp * axp, xp * s.b, g * df, df * df};
                bsum<4, NT>(qa, sm, par, s.own);
                if (!have12) {       // the two outer sums (:285-286) ride along with the first inner reduction
                    double qb[2] = {y * ay, y * s.b};
                    bsum<2, NT>(qb, sm, par, s.own);
                    rt1 = qb[0] * 0.5; rt2 = qb[1];
                    have12 = true;
                }
                if (lim) break;      // leaves the inner loop only (:292-293)
                if ((qa[0] * 0.5 + qa[1]) <= (rt1 + rt2 + qa[2] + 0.5 * L * qa[3])) break;
                L *= 2;
                t = 1.0 / L;
                xp = P(y - t * g);
            }
            double theta_n = 0.5 * (-theta * theta + theta * sqrt(4 + theta * theta));
            const double beta = theta * (1 - theta) / (theta * theta + theta_n);
            double yn = (1 + beta) * xp - beta * x;
            double q[2] = {resid2(xp, axp + s.b), AR ? g * (xp - x) : 0.0};
            if (AR) bsum<2, NT>(q, sm, par, s.own);
            else { double q1[1] = {q[0]}; bsum<1, NT>(q1, sm, par, s.own); q[0] = q1[0]; }
            res2 = q[0];
            iters++;
            if (AR) { res = sqrt(res2); if (res < resmin) { resmin = res; xhat = xp; } }
            if (res2 < c.thr_lt) break;
            if (AR && q[1] > 0) { yn = xp; theta_n = 1; }
            L *= 0.9;
            t = 1.0 / L;
            y = yn;
            { const double tmp = x; x = xp; xp = tmp; }   // buffer swap (:332-334)
            theta = theta_n;
        }
        res = sqrt(res2);
        xsol = AR ? xhat : xp;
    } else if constexpr (SOLVER == CCQP_SOLVER_MPRGP) {
        // solvers.py:1048-1200 with the Box operator of solution_spaces.py:280-366; statement by statement the
        // dense program (dense.cuh solve_mprgp) with one unknown per thread
        auto feas = [&](double v) { return is_close(v, clampd(v, s.lo, s.hi)); };
        double xk = clampd(s.x0, s.lo, s.hi), xn = xk;
        double gk = matvec<NT>(a, sm, xpar, s.act, xk) + s.b, gn = gk; gemv++; mv = 1;
        double r1[1] = {resid2(xk, gk)};
        bsum<1, NT>(r1, sm, par, s.own);
        double res2 = r1[0];
        if (!(res2 < c.thr_lt)) {
            const double ag = matvec<NT>(a, sm, xpar, s.act, gk); gemv++; mv++;       // counted (:1077-1078)
            double q2[2] = {gk * ag, gk * gk};
            bsum<2, NT>(q2, sm, par, s.own);
            double abb = q2[1] / q2[0];
            bool abb_lazy = false;                      // true: abb = BB(xk - xn) still to be evaluated
            double p = feas(xk) ? gk : 0.0, Ap = 0.0;
            for (;;) {
                gk = matvec<NT>(a, sm, xpar, s.act, xk) + s.b; gemv++; mv++;
                if (mv >= maxmv) break;
                const bool cl = feas(xk);                                          // delta (:1093)
                const double psi = cl ? gk : 0.0;
                double q3[3] = {psi * psi, psi * p, (cl || !s.act) ? 0.0 : 1.0};
                bsum<3, NT>(q3, sm, par, s.own);
                double betbet = 0.0;
                if (q3[2] > 0.0) {
                    // some entry is not (close to) feasible: normal_vector of the Box (:306-322) and the GLOBAL n.g
                    const double px = clampd(xk, s.lo, s.hi), dx = xk - px;
                    double d1[1] = {dx * dx};
                    bsum<1, NT>(d1, sm, par, s.own);
                    double nv = 0.0;
                    if (s.act && is_close(sqrt(d1[0]), 0.0)) nv = is_close(px, s.hi) ? 1.0 : (is_close(px, s.lo) ? -1.0 : 0.0);
                    double s1[1] = {nv * gk};
                    bsum<1, NT>(s1, sm, par, s.own);
                    const double mng = s1[0] < 0.0 ? s1[0] : 0.0;                  // np.min([0, n.g])
                    const double bv = ((cl || !s.act) ? 0.0 : 1.0) * (gk - mng * nv);
                    double s2[1] = {bv * bv};
                    bsum<1, NT>(s2, sm, par, s.own);
                    betbet = s2[0];
                }
                if (betbet < q3[0]) {
                    Ap = matvec<NT>(a, sm, xpar, s.act, p); gemv++; mv++;
                    double s1[1] = {p * Ap};
                    bsum<1, NT>(s1, sm, par, s.own);
                    if (mv >= maxmv) break;
                    const double pAp = s1[0];
                    const double acg = q3[1] / pAp;
                    double af = acg + 10 * kEps;
                    for (int pass = 0;; ++pass) {                                  // feasibility bisection :1112-1118
                        unsigned long long m = ~0ull;
                        if (s.act) {
                            double al = af;
                            for (int j = 0; j < 64; ++j, al *= 0.5) if (!feas(xk - al * p)) m &= ~(1ull << j);
                        }
                        m = band<NT>(m, sm, par);
                        if (m) { const int j = __ffsll((long long)m) - 1; for (int q = 0; q < j; ++q) af *= 0.5; break; }
                        for (int q = 0; q < 64; ++q) af *= 0.5;
                        if (pass >= 20) break;
                    }
                    if (acg <= af) {                                               // conjugate-gradient step :1121-1135
                        const double yv = xk - acg * p;
                        const double gni = gk - acg * Ap;
                        xn = yv; gn = gni;
                        const double psy = feas(yv) ? gni : 0.0;
                        const double bet = psy * Ap / pAp;                         // elementwise "beta" (:1134)
                        p = psy - bet * p;
                        abb_lazy = true;
                    } else {                                                       // expansion step :1136-1163
                        const double xh = xk - af * p, gh = gk - af * Ap;
                        const double sx = xh - xk, sg = gh - gk;
                        double s2[2] = {sx * sx, sx * sg};
                        bsum<2, NT>(s2, sm, par, s.own);
                        const double al = s2[0] / (s2[1] + 10 * kEps);
                        xn = clampd(xh - al * gh, s.lo, s.hi);
                        gn = matvec<NT>(a, sm, xpar, s.act, xn) + s.b; gemv++; mv++;
                        if (mv >= maxmv) break;
                        p = feas(xn) ? gn : 0.0;
                        abb_lazy = true;
                    }
                } else {                                                           // proportioning step :1164-1182
                    if (abb_lazy) {
                        const double w = xk - xn;
                        const double Aw = matvec<NT>(a, sm, xpar, s.act, w); gemv++;  // not counted (:1129,:1163,:1172)
                        double s2[2] = {w * w, w * Aw};
                        bsum<2, NT>(s2, sm, par, s.own);
                        abb = s2[0] / (s2[1] + 10 * kEps);
                    }
                    xn = clampd(xk - abb * gk, s.lo, s.hi);
                    abb_lazy = true;
                    mv++;                    // gk = A xk + b is re-evaluated by the reference (:1174); same value
                    if (mv >= maxmv) break;
                    p = feas(xn) ? gn : 0.0;                                       // stale gn (:1181)
                }
                double r2[1] = {resid2(xn, gn)};
                bsum<1, NT>(r2, sm, par, s.own);
                res2 = r2[0];
                iters++;
                if (res2 < c.thr_lt) break;
                { const double t = xk; xk = xn; xn = t; }
                { const double t = gk; gk = gn; gn = t; }
            }
        }
        res = sqrt(res2);
        xsol = xn;
    }
    o.residual = res;
    o.mv = mv; o.gemv = gemv; o.iters = iters; o.draws = draws;
    o.converged = (mv < maxmv && status == 0) ? 1 : 0;   // a problem that stopped on an error is not a converged one
    o.status = status;
}

#ifndef CCQP_BATCHED_CTAS
#define CCQP_BATCHED_CTAS 6     // resident CTAs per SM the register budget is cut for (6 -> 168 registers)
#endif
constexpr int batched_min_ctas(int solver) {
    return (solver == CCQP_SOLVER_PGD || solver == CCQP_SOLVER_BBPGD || solver == CCQP_SOLVER_SPG) ? CCQP_BATCHED_CTAS : 5;
}

extern __shared__ __align__(16) unsigned char batched_dyn_smem[];       // NT = 256: the 141 KB of BatchedSmem are dynamic

template <int SOLVER, bool WREG, bool GEN, int NT>
__global__ void __launch_bounds__(NT, NT == 64 ? (GEN ? 5 : batched_min_ctas(SOLVER)) : 1) batched_kernel(const BatchedCtx c) {
    using L = BL<NT>;
    BatchedSmem<GEN, NT>* smp;
    if constexpr (NT == 64) { __shared__ __align__(16) BatchedSmem<GEN, 64> sm_static; smp = &sm_static; }
    else smp = reinterpret_cast<BatchedSmem<GEN, NT>*>(batched_dyn_smem);
    BatchedSmem<GEN, NT>& sm = *smp;
    const int t = threadIdx.x, n = c.n;
    const int cb = t & (L::NB - 1), key = cb >> L::SH, row0 = kBRows * (t / L::NB), col0 = kBCols * cb;
    const int u = row0 + key;               // the unknown this thread holds (NT = 64: u == t)
    const bool primary = L::SH == 0 || !(t & 1);
    int par = 0, xpar = 0;
    BShared sh;
    sh.xs_wr = smem_u32(&sm.xs[0][u + 2 * (u / kBCols)]);
    sh.xs_rd = smem_u32(&sm.xs[0][L::SLICE * cb]);
    sh.red = smem_u32(&sm.red[0][0][0]);
    const size_t prob_elems = (size_t)n * n;

    auto prefetch_l2 = [&](int prob) {      // the whole next problem, one instruction (TMA engine)
        if (c.pf_ok && t == 0)
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(c.A + (size_t)prob * prob_elems),
                         "r"((unsigned)(prob_elems * 8)) : "memory");
    };
#if CCQP_BATCHED_STAGE
    const bool staged = c.tma_ok != 0;
    const bool vstaged = staged && c.vtma_ok != 0;
    unsigned phase = 0;
    if (t == 0) { mbar_init(&sm.mbar, 1); mbar_fence_init(); }
    auto issue_load = [&](int prob) {       // one 8n-byte bulk copy per row into the padded tile (+ 3 for the vectors), one mbarrier
        if constexpr (GEN) {
            // b into vstage[0], the problem's parameter row into vstage[1..2].  bb / pb are the one definition of what is
            // copied: thread 0 announces exactly bb + pb bytes besides A, and a copy is issued iff its size is non-zero
            // (announced bytes that never arrive would leave mbar_wait spinning forever).
            const uint32_t bb = vstaged ? (uint32_t)(n * 8) : 0u, pb = vstaged ? (uint32_t)c.prow_bytes : 0u;
            if (t == 0) mbar_expect_tx(&sm.mbar, (uint32_t)(prob_elems * 8) + bb + pb);
            if (t < n) bulk_g2s(sm.tile + t * L::PITCH, c.A + (size_t)prob * prob_elems + (size_t)t * n, (uint32_t)(n * 8), &sm.mbar);
            if (bb != 0u && t == NT - 1) bulk_g2s(sm.vstage[0], c.b + (size_t)prob * n, bb, &sm.mbar);
            if (pb != 0u && t == NT - 2) bulk_g2s(sm.vstage[1], c.params + (size_t)prob * c.param_stride, pb, &sm.mbar);
        } else {
            if (t == 0) mbar_expect_tx(&sm.mbar, (uint32_t)(prob_elems * 8) + (vstaged ? 3u * (uint32_t)(n * 8) : 0u));
            if (t < n) bulk_g2s(sm.tile + t * L::PITCH, c.A + (size_t)prob * prob_elems + (size_t)t * n, (uint32_t)(n * 8), &sm.mbar);
            if (vstaged && t >= NT - 3) {   // three otherwise idle-ish threads (the mbarrier's expect_tx is program-ordered only in thread 0,
                const int w = t - (NT - 3); // but a complete_tx that arrives first just drives the pending count negative: legal)
                const double* src = w == 0 ? c.b + (size_t)prob * n : (w == 1 ? c.lb : c.ub) + (size_t)prob * c.bound_stride;
                bulk_g2s(sm.vstage[w], src, (uint32_t)(n * 8), &sm.mbar);
            }
        }
    };
#else
    const bool staged = false, vstaged = false;
#endif
    // Work queue, two problems deep: `cur` is being solved, `nxt` is known (its A is in flight), and the index after that is
    // fetched by thread 0 at the start of a solve and published at its end -- the atomic's round trip hides behind the solve.
    if (t == 0) { sm.first = (int)atomicAdd(c.counter, 1u); sm.next = (int)atomicAdd(c.counter, 1u); }
    __syncthreads();
    int cur = sm.first;
#if CCQP_BATCHED_STAGE
    if (staged && cur < c.batch) { fence_proxy_async(); issue_load(cur); }
#endif
    while (cur < c.batch) {
        // ---- register fill: this thread's sub-block; register row r <- row row0 + (r ^ key) (see matvec)
        double a[kBRows][kBCols];
        const double* Ap = c.A + (size_t)cur * prob_elems;
        BState s;
        s.u = u;
        s.act = u < n;
        s.own = s.act && primary;
        const size_t vo = (size_t)cur * n + u;
        const size_t bo = (size_t)cur * c.bound_stride + u;
        if (staged) {
#if CCQP_BATCHED_STAGE
            mbar_wait(&sm.mbar, phase);
            phase ^= 1u;
            const uint32_t tb = smem_u32(sm.tile);
#pragma unroll
            for (int r = 0; r < kBRows; ++r) {
                const int row = row0 + (r ^ key);
#pragma unroll
                for (int j = 0; j < kBCols; j += 2) {
                    if (row < n && col0 + j < n) lds_f64x2(tb + (uint32_t)(row * L::PITCH + col0 + j) * 8u, a[r][j], a[r][j + 1]);
                    else { a[r][j] = 0.0; a[r][j + 1] = 0.0; }
                }
            }
            if (vstaged) {
                s.b = s.act ? sm.vstage[0][u] : 0.0;
                if constexpr (!GEN) {
                    s.lo = s.act ? sm.vstage[1][u] : 0.0;
                    s.hi = s.act ? sm.vstage[2][u] : 0.0;
                }
            }
#endif
        } else if (c.vec_ok) {
#pragma unroll
            for (int r = 0; r < kBRows; ++r) {
#pragma unroll
                for (int j = 0; j < kBCols; j += 4) {
                    const int row = row0 + (r ^ key);
                    if (row < n && col0 + j < n) {
                        double v[4];
                        ldg_vec4_stream<false>(Ap + (size_t)row * n + col0 + j, v);
                        a[r][j] = v[0]; a[r][j + 1] = v[1]; a[r][j + 2] = v[2]; a[r][j + 3] = v[3];
                    } else { a[r][j] = 0.0; a[r][j + 1] = 0.0; a[r][j + 2] = 0.0; a[r][j + 3] = 0.0; }
                }
            }
        } else {
#pragma unroll
            for (int r = 0; r < kBRows; ++r)
#pragma unroll
                for (int j = 0; j < kBCols; ++j)
                    a[r][j] = (row0 + (r ^ key) < n && col0 + j < n) ? ldg_stream(Ap + (size_t)(row0 + (r ^ key)) * n + col0 + j) : 0.0;
        }
        if (!vstaged) {
            s.b = s.act ? c.b[vo] : 0.0;
            if constexpr (!GEN) {
                s.lo = s.act ? c.lb[bo] : 0.0;
                s.hi = s.act ? c.ub[bo] : 0.0;
            }
        }
        if constexpr (GEN) {
            s.kind = s.act ? c.ekind[u] : kIdentity;
            s.boff = s.act ? c.eoff[u] : 0; s.bdim = s.act ? c.edim[u] : 0; s.bnk = s.act ? c.enk[u] : 0;
            // this problem's bounds / block parameter: its parameter row (staged next to b, or in global memory) at the
            // element's indices
            const int4 e = s.act ? __ldg(c.eidx + u) : make_int4(-1, -1, -1, -1);
            const double* prow = c.params + (size_t)cur * c.param_stride;
            auto prm = [&](int k, double none) {
                if (k < 0) return none;
#if CCQP_BATCHED_STAGE
                if (vstaged) return lds_f64(smem_u32(&sm.vstage[1][0]) + (uint32_t)k * 8u);   // the row runs on into vstage[2]
#endif
                return __ldg(prow + k);
            };
            const bool nb = s.kind == kElemNorm;
            s.lo = prm(nb ? e.z : e.x, nb ? 0.0 : -INFINITY);
            s.hi = prm(e.y, INFINITY);
            s.pj = smem_u32(&sm.pj[0][0]);
        }
        s.x0 = (s.act && c.x0) ? c.x0[vo] : 0.0;
        s.cs = 1.0 / (3 * (double)n * kGd);
        __syncthreads();                       // everyone has read its part of the tile / the staged vectors; sm.next (written by
        const int nxt = sm.next;               // thread 0 at the end of the previous solve) is visible
        unsigned after = 0;
        if (nxt < c.batch) {                   // the next problem travels while this one iterates
#if CCQP_BATCHED_STAGE
            if (staged) { fence_proxy_async(); issue_load(nxt); } else
#endif
            prefetch_l2(nxt);
            if (c.x0 && s.own) asm volatile("prefetch.global.L2 [%0];" ::"l"(c.x0 + (size_t)nxt * n + u));
            if (t == 0) after = atomicAdd(c.counter, 1u);     // consumed at the end of the solve
        } else if (t == 0) after = (unsigned)c.batch;

        double xsol = 0.0;
        BatchedOut o;
        solve_one<SOLVER, WREG, GEN, NT>(c, a, sh, s, c.uniforms ? c.uniforms + (size_t)cur * c.n_uniforms : nullptr, par, xpar,
                                     xsol, o);
        if (s.own) c.x_out[vo] = xsol;
        if (t == 0) { c.out[cur] = o; sm.next = (int)after; }   // everybody read the old value right after the barrier above
        cur = nxt;
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
// Smallest double q >= 0 with pred(sqrt(q)) false ... expressed through the bit pattern: for
// non-negative doubles the IEEE ordering equals the ordering of the bit patterns, and sqrt is
// monotone and correctly rounded on both host and device, so the reference's test on sqrt(q)
// is equivalent to a comparison of q with a threshold found by bisection.
inline double sqrt_threshold(double tol, bool strict) {
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

#ifndef CCQP_BATCHED_DEVICE_ONLY        // batched_sym.cu shares the context / helpers above, not the launchers below
template <int SOLVER, bool WREG, bool GEN, int NT>
inline cudaError_t launch_batched_nt(const BatchedCtx& c, int sm_count, cudaStream_t stream) {
    int per_sm = 0;
    const size_t dyn = NT == 64 ? 0 : sizeof(BatchedSmem<GEN, NT>);
    auto kern = batched_kernel<SOLVER, WREG, GEN, NT>;
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    cudaError_t e = dyn ? cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn) : cudaSuccess;
    if (e != cudaSuccess) return e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, NT, dyn);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    if (const char* e = getenv("CCQP_BATCHED_CTAS_PER_SM")) per_sm = std::max(1, std::min(per_sm, atoi(e)));   // tuning hook
    long long grid = (long long)sm_count * per_sm;
    if (grid > c.batch) grid = c.batch;
    kern<<<(unsigned)grid, NT, dyn, stream>>>(c);
    return cudaGetLastError();
}
// n <= 64: 64 threads per problem, A in 128 registers per thread, up to 6 problems per SM; 64 < n <= 128: 256 threads, one per SM
template <int SOLVER, bool WREG, bool GEN = false>
inline cudaError_t launch_batched(const BatchedCtx& c, int sm_count, cudaStream_t stream) {
    return c.n <= kBN ? launch_batched_nt<SOLVER, WREG, GEN, 64>(c, sm_count, stream)
                      : launch_batched_nt<SOLVER, WREG, GEN, 256>(c, sm_count, stream);
}

// The block structure of a general table, per element, on the HOST (batched.cu batched_table_layout), and where its
// parameters are: one row shared by every problem (ccqp_solve_batched_table, a host array) or one row per problem
// (ccqp_solve_batched_tables, [batch][n_params] where A lives)
struct BatchedTable {
    std::vector<uint8_t> ekind;
    std::vector<int> eoff, edim, enk;
    std::vector<int> eidx;          // [n][4]: lower bound / upper bound / block parameter index into a row, -1: none
    int has_norm = 0;
    const double* params = nullptr;
    long long n_params = 0;
    bool per_problem = false;
};

// batched_sym.cu: the one-warp-per-problem kernels for symmetric Hessians (n <= 64; PGD / BBPGD / BBPGDf / SPG, Box per problem)
bool batched_sym_supported(int solver, long long n);
cudaError_t launch_batched_sym(const BatchedCtx& c, int solver, bool wreg, int sm_count, cudaStream_t stream);

// Returns a ccqp_status.  `alloc(bytes)` returns a device workspace of at least that size.
// tab != nullptr: the general table replaces the per-problem Box (lb / ub are ignored).
// sym: the caller declares every A[i] symmetric (ccqp_solve_batched_sym); where batched_sym_supported() the upper block triangle
// alone is read, otherwise the general kernels run (same answer for a symmetric A).
inline int batched_solve(cudaStream_t stream, int sm_count, const BatchedTable* tab, bool sym, int solver, const ccqp_params& prm,
                         long long batch, long long n, const double* A, const double* b, const double* x0,
                         const double* lb, const double* ub, const double* uniforms, long long n_uniforms, double* x_out,
                         int memtype, ccqp_result* results, ccqp_result* summary, cudaEvent_t ev0, cudaEvent_t ev1,
                         int* launches, std::string& err, const std::function<void*(size_t)>& alloc) {
#define BCU(call)                                                                                  \
    do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { err = std::string(#call) + ": " + cudaGetErrorString(e__); return CCQP_ERR_CUDA; } } while (0)
    if (n > kBNMax) return CCQP_ERR_UNSUPPORTED;
    if (tab && solver == CCQP_SOLVER_MPRGP) return CCQP_ERR_UNSUPPORTED;     // batched MPRGP: Box per problem only
    if (batch >= (1LL << 31) - 1024) return CCQP_ERR_INVALID_ARG;
    const bool host = memtype == CCQP_MEM_HOST;
    if (solver == CCQP_SOLVER_SPG && (n_uniforms < 0 || (n_uniforms > 0 && !uniforms))) return CCQP_ERR_INVALID_ARG;
    const size_t szA = (size_t)batch * n * n * 8, szV = (size_t)batch * n * 8;
    const size_t szU = (solver == CCQP_SOLVER_SPG) ? (size_t)batch * n_uniforms * 8 : 0;
    const size_t szO = (size_t)batch * sizeof(BatchedOut);
    auto al = [](size_t v) { return (v + 255) / 256 * 256; };
    // parameter rows of a general table: a shared row and the rows of a host array are copied with an even pitch, so that
    // every row starts 16-byte aligned and its bulk copy (rounded up to 16 bytes) stays inside the copy
    const long long np = tab ? std::max(tab->n_params, 0LL) : 0, ppitch = np + (np & 1);
    const size_t szP = !tab ? 0 : !tab->per_problem ? (size_t)ppitch * 8 : host ? (size_t)batch * ppitch * 8 : 0;
    size_t total = 256 + al(szO) + 8 * al((size_t)kBNMax * 8) + al(szP);
    if (host) total += al(szA) + 4 * al(szV) + al(szV) + al(szU);
    unsigned char* ws = static_cast<unsigned char*>(alloc(total));
    if (!ws) { err = "workspace allocation failed"; return CCQP_ERR_CUDA; }
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char* p = ws + off; off += al(bytes); return p; };
    unsigned* counter = reinterpret_cast<unsigned*>(take(256));
    BatchedOut* dout = reinterpret_cast<BatchedOut*>(take(szO));
    BatchedCtx c;
    std::memset(&c, 0, sizeof(c));
    if (host) {
        double* dA = reinterpret_cast<double*>(take(szA));
        double* db = reinterpret_cast<double*>(take(szV));
        double* dlb = reinterpret_cast<double*>(take(szV));
        double* dub = reinterpret_cast<double*>(take(szV));
        double* dx0 = reinterpret_cast<double*>(take(szV));
        double* dxo = reinterpret_cast<double*>(take(szV));
        double* du = szU ? reinterpret_cast<double*>(take(szU)) : nullptr;
        BCU(cudaMemcpyAsync(dA, A, szA, cudaMemcpyHostToDevice, stream));
        BCU(cudaMemcpyAsync(db, b, szV, cudaMemcpyHostToDevice, stream));
        if (!tab) BCU(cudaMemcpyAsync(dlb, lb, szV, cudaMemcpyHostToDevice, stream));
        if (!tab) BCU(cudaMemcpyAsync(dub, ub, szV, cudaMemcpyHostToDevice, stream));
        if (x0) BCU(cudaMemcpyAsync(dx0, x0, szV, cudaMemcpyHostToDevice, stream));
        if (du) BCU(cudaMemcpyAsync(du, uniforms, szU, cudaMemcpyHostToDevice, stream));
        c.A = dA; c.b = db; c.lb = dlb; c.ub = dub; c.x0 = x0 ? dx0 : nullptr; c.uniforms = du; c.x_out = dxo;
    } else {
        c.A = A; c.b = b; c.lb = lb; c.ub = ub; c.x0 = x0; c.uniforms = (solver == CCQP_SOLVER_SPG) ? uniforms : nullptr;
        c.x_out = x_out;
    }
    c.bound_stride = n;
    if (tab) {        // the block structure: five small per-element arrays, uploaded once per call
        auto up = [&](const void* src, size_t bytes) -> void* {
            void* d = take(bytes);
            return cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, stream) == cudaSuccess ? d : nullptr;
        };
        c.ekind = static_cast<const uint8_t*>(up(tab->ekind.data(), (size_t)n));
        c.eoff = static_cast<const int*>(up(tab->eoff.data(), (size_t)n * 4));
        c.edim = static_cast<const int*>(up(tab->edim.data(), (size_t)n * 4));
        c.enk = static_cast<const int*>(up(tab->enk.data(), (size_t)n * 4));
        c.eidx = static_cast<const int4*>(up(tab->eidx.data(), (size_t)n * 16));
        if (!c.ekind || !c.eoff || !c.edim || !c.enk || !c.eidx) { err = "table upload failed"; return CCQP_ERR_CUDA; }
        c.has_norm = tab->has_norm;
        c.lb = c.ub = nullptr;
        // the parameter rows: one shared row (stride 0), a host array copied with an even pitch, or a device array in place
        if (np > 0 && (!tab->per_problem || host)) {
            double* dp = reinterpret_cast<double*>(take(szP));
            const long long rows = tab->per_problem ? batch : 1;
            if (ppitch == np) BCU(cudaMemcpyAsync(dp, tab->params, (size_t)rows * np * 8, cudaMemcpyHostToDevice, stream));
            else BCU(cudaMemcpy2DAsync(dp, (size_t)ppitch * 8, tab->params, (size_t)np * 8, (size_t)np * 8, (size_t)rows,
                                       cudaMemcpyHostToDevice, stream));
            c.params = dp;
            c.param_stride = tab->per_problem ? ppitch : 0;
        } else {
            c.params = np > 0 ? tab->params : nullptr;
            c.param_stride = np;
        }
    }
    c.n_uniforms = (solver == CCQP_SOLVER_SPG) ? n_uniforms : 0;
    c.out = dout; c.counter = counter;
    c.batch = (int)batch; c.n = (int)n;
    c.tma_ok = ((n * 8) % 16 == 0 && (reinterpret_cast<uintptr_t>(c.A) & 15) == 0) ? 1 : 0;
    c.vec_ok = (n % 4 == 0 && (reinterpret_cast<uintptr_t>(c.A) & 31) == 0) ? 1 : 0;
    c.pf_ok = ((n * n * 8) % 16 == 0 && (reinterpret_cast<uintptr_t>(c.A) & 15) == 0) ? 1 : 0;
    c.vtma_ok = (n % 2 == 0 && ((reinterpret_cast<uintptr_t>(c.b) | reinterpret_cast<uintptr_t>(c.lb) | reinterpret_cast<uintptr_t>(c.ub)) & 15) == 0) ? 1 : 0;
    if (tab) {        // a parameter row is staged with b when every row is 16-byte aligned and fits vstage[1..2] (2 N doubles)
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
    cudaError_t le;
    const bool wreg = prm.m == kBWinReg;
    const bool use_sym = sym && !tab && batched_sym_supported(solver, n);
    if (use_sym) le = launch_batched_sym(c, solver, wreg, sm_count, stream);
    else if (tab) switch (solver) {
        case CCQP_SOLVER_PGD: le = launch_batched<CCQP_SOLVER_PGD, true, true>(c, sm_count, stream); break;
        case CCQP_SOLVER_APGD: le = launch_batched<CCQP_SOLVER_APGD, true, true>(c, sm_count, stream); break;
        case CCQP_SOLVER_APGD_AR: le = launch_batched<CCQP_SOLVER_APGD_AR, true, true>(c, sm_count, stream); break;
        case CCQP_SOLVER_BBPGD: le = launch_batched<CCQP_SOLVER_BBPGD, true, true>(c, sm_count, stream); break;
        case CCQP_SOLVER_BBPGDF: le = launch_batched<CCQP_SOLVER_BBPGDF, true, true>(c, sm_count, stream); break;
        case CCQP_SOLVER_SPG:
            le = wreg ? launch_batched<CCQP_SOLVER_SPG, true, true>(c, sm_count, stream)
                      : launch_batched<CCQP_SOLVER_SPG, false, true>(c, sm_count, stream);
            break;
        default: return CCQP_ERR_INVALID_ARG;
    }
    else switch (solver) {
        case CCQP_SOLVER_PGD: le = launch_batched<CCQP_SOLVER_PGD, true>(c, sm_count, stream); break;
        case CCQP_SOLVER_APGD: le = launch_batched<CCQP_SOLVER_APGD, true>(c, sm_count, stream); break;
        case CCQP_SOLVER_APGD_AR: le = launch_batched<CCQP_SOLVER_APGD_AR, true>(c, sm_count, stream); break;
        case CCQP_SOLVER_BBPGD: le = launch_batched<CCQP_SOLVER_BBPGD, true>(c, sm_count, stream); break;
        case CCQP_SOLVER_BBPGDF: le = launch_batched<CCQP_SOLVER_BBPGDF, true>(c, sm_count, stream); break;
        case CCQP_SOLVER_MPRGP: le = launch_batched<CCQP_SOLVER_MPRGP, true>(c, sm_count, stream); break;
        case CCQP_SOLVER_SPG:
            le = wreg ? launch_batched<CCQP_SOLVER_SPG, true>(c, sm_count, stream)
                      : launch_batched<CCQP_SOLVER_SPG, false>(c, sm_count, stream);
            break;
        default: return CCQP_ERR_INVALID_ARG;
    }
    BCU(le);
    *launches = 1;
    BCU(cudaEventRecord(ev1, stream));
    if (host) BCU(cudaMemcpyAsync(x_out, c.x_out, szV, cudaMemcpyDeviceToHost, stream));
    std::vector<BatchedOut> hout((size_t)batch);
    BCU(cudaMemcpyAsync(hout.data(), dout, szO, cudaMemcpyDeviceToHost, stream));
    BCU(cudaStreamSynchronize(stream));
    float ms = 0.f;
    BCU(cudaEventElapsedTime(&ms, ev0, ev1));
    long long tot_mv = 0, tot_gemv = 0, tot_it = 0, tot_dr = 0, nconv = 0;
    int first_status = 0;
    double hbmA = 8.0 * n * n;                  // bytes of A[i] the kernel reads
    if (use_sym) { hbmA = 0; for (long long i = 0; i < n; ++i) hbmA += 8.0 * (double)(n - 8 * (i / 8)); }
    if (tab && tab->per_problem) hbmA += 8.0 * (double)np;     // the problem's parameter row
    for (long long i = 0; i < batch; ++i) {
        const BatchedOut& o = hout[(size_t)i];
        if (results) {
            ccqp_result& r = results[i];
            std::memset(&r, 0, sizeof(r));
            r.residual = o.residual; r.mv_count = o.mv; r.gemv_count = o.gemv; r.iterations = o.iters;
            r.uniforms_used = o.draws; r.converged = o.converged; r.status = o.status;
            r.hbm_bytes = hbmA + 8.0 * n * (x0 ? 5 : 4);
        }
        tot_mv += o.mv; tot_gemv += o.gemv; tot_it += o.iters; tot_dr += o.draws; nconv += o.converged;
        if (o.status && !first_status) first_status = o.status;
    }
    if (summary) {
        std::memset(summary, 0, sizeof(*summary));
        summary->gpu_seconds = ms * 1e-3;
        summary->mv_count = tot_mv; summary->gemv_count = tot_gemv; summary->iterations = tot_it;
        summary->uniforms_used = tot_dr; summary->converged = (nconv == batch) ? 1 : 0;
        summary->status = first_status;
        summary->hbm_bytes = (double)batch * (hbmA + 8.0 * n * (x0 ? 5 : 4)) + 8.0 * (double)tot_dr;
        summary->kernel_launches = 1;
        summary->residual = NAN;
    }
    return CCQP_OK;
#undef BCU
}
#endif  // CCQP_BATCHED_DEVICE_ONLY

}  // namespace ccqp
