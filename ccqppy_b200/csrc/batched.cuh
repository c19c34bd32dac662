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
//     15 + 15), then the warps swap through shared memory (one barrier).  A variant that ran the 32-lane sums on the FP64
//     tensor path measured equal and was removed (DESIGN.md 2.2).
//   * stopping tests compare the SQUARED residual with a host-computed threshold that is exactly equivalent to the
//     reference's sqrt(.) < tol (sqrt is monotone), so no sqrt is on the per-iteration critical path; the reported
//     residual is computed once at the end.
//   * everything else (projection, axpy, step lengths) is per-thread register arithmetic, with the reference's rounding
//     (compiled with -fmad=false; explicit fma() only in the sums).
//   Problems are handed out through an atomic counter (iteration counts differ per problem); results do not depend on the
//   schedule.
//
// fp32 Hessians (the _f32 entry points): the same kernels with A's element type TA = float.  Only the staging changes -- a
// float tile, 4 bytes per entry on the mbarrier, and a register fill that widens every entry exactly (cvt.f64.f32) -- so the
// registers hold what the fp64 kernel holds for the widened matrix and solve_one, which never sees TA, returns the same bits.
//
// Bounds: HBM bytes/problem = 8 n^2 + 32 n (fp32 A: 4 n^2 + 32 n) (+8 n for x0, + uniforms read by SPG);
//         fp64 flops/problem = 2 n^2 * (mat-vecs executed).
#pragma once
#include <cmath>

#include "proj.cuh"
#include "../../include/ccqp_b200.h"

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
    static constexpr int PITCH_F32 = N + 4;            // ... (floats, rows 16-byte aligned): NT = 64 conflict-free (4 wavefronts per
                                                       // LDS.128); NT = 256 2 per quarter warp, 8 per LDS.128 at any pitch (the
                                                       // lane pairs that share a row sit 32 bytes apart), the fp64 fill's total
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
    const void* A;          // [batch][n][n] of the kernel's element type (double, or float for the _f32 entry points)
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
    int tma_ok;             // rows of A can be moved with 16-byte bulk copies (n * sizeof(entry) % 16 == 0, 16-byte aligned base)
    int vec_ok;             // rows of A can be read with 256-bit loads (fp64 A, n % 4 == 0, 32-byte aligned base)
    int pf_ok;              // whole problems can be bulk-prefetched into L2 (n^2 * sizeof(entry) % 16 == 0, 16-byte aligned base)
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

template <bool GEN, int NT, class TA>
struct BatchedSmem {
    static constexpr int PITCH = sizeof(TA) == 8 ? BL<NT>::PITCH : BL<NT>::PITCH_F32;
    TA tile[BL<NT>::N * PITCH];               // the NEXT problem's A, landed by TMA while the current one iterates
    double vstage[3][BL<NT>::N];              // ... and its b / lower / upper bounds (general table: b / parameter row
                                              // of up to 2 N entries in vstage[1..2]) on the same mbarrier
    double xs[2][BL<NT>::XS];                 // mat-vec input, double buffered
    double red[2][BL<NT>::WARPS][4];          // [parity][warp][slot]
    double pj[GEN ? 2 : 1][GEN ? BL<NT>::N : 2];   // general table: the vector being projected, for the members of norm blocks
    uint64_t mbar;
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
// four floats of an fp32 tile, widened exactly: d[0..3] <- (double)tile[addr .. addr + 15]
__device__ __forceinline__ void lds_f32x4_widen(uint32_t addr, double* d) {
    float f0, f1, f2, f3;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(f0), "=f"(f1), "=f"(f2), "=f"(f3) : "r"(addr) : "memory");
    d[0] = (double)f0; d[1] = (double)f1; d[2] = (double)f2; d[3] = (double)f3;
}

__device__ __forceinline__ double shfl_xor_f64(double v, int mask) { return __shfl_xor_sync(0xffffffffu, v, mask); }

// Sum K (<= 4) values over the 64 threads; result in every thread; ONE __syncthreads.
// Exchange butterfly: after the first stages each lane carries ONE of the K sums, so the tree
// costs max(K,2)+3 shuffles and adds instead of 5K.  Fixed order => deterministic.

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

constexpr int kBatchedCtas = 6;         // resident CTAs per SM the register budget is cut for (6 -> 168 registers)
constexpr int batched_min_ctas(int solver) {
    return (solver == CCQP_SOLVER_PGD || solver == CCQP_SOLVER_BBPGD || solver == CCQP_SOLVER_SPG) ? kBatchedCtas : 5;
}

extern __shared__ __align__(16) unsigned char batched_dyn_smem[];       // NT = 256: the 141 KB of BatchedSmem are dynamic

// TA: the element type of A in memory (double / float); the registers and everything after the fill are fp64 either way
template <int SOLVER, bool WREG, bool GEN, int NT, class TA>
__global__ void __launch_bounds__(NT, NT == 64 ? (GEN ? 5 : batched_min_ctas(SOLVER)) : 1) batched_kernel(const BatchedCtx c) {
    using L = BL<NT>;
    using Smem = BatchedSmem<GEN, NT, TA>;
    constexpr uint32_t ESZ = sizeof(TA);
    Smem* smp;
    if constexpr (NT == 64) { __shared__ __align__(16) Smem sm_static; smp = &sm_static; }
    else smp = reinterpret_cast<Smem*>(batched_dyn_smem);
    Smem& sm = *smp;
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
    // (c.A is cast to const TA* where it is used: a typed copy taken here moves the load of c.A, and with it the schedule
    // ptxas picks for the fp64 instantiations)

    auto prefetch_l2 = [&](int prob) {      // the whole next problem, one instruction (TMA engine)
        if (c.pf_ok && t == 0)
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;"
                         ::"l"(static_cast<const TA*>(c.A) + (size_t)prob * prob_elems), "r"((unsigned)(prob_elems * ESZ)) : "memory");
    };
    const bool staged = c.tma_ok != 0;
    const bool vstaged = staged && c.vtma_ok != 0;
    unsigned phase = 0;
    if (t == 0) { mbar_init(&sm.mbar, 1); mbar_fence_init(); }
    auto issue_load = [&](int prob) {       // one n * ESZ-byte bulk copy per row into the padded tile (+ 3 for the vectors), one mbarrier
        if constexpr (GEN) {
            // b into vstage[0], the problem's parameter row into vstage[1..2].  bb / pb are the one definition of what is
            // copied: thread 0 announces exactly bb + pb bytes besides A, and a copy is issued iff its size is non-zero
            // (announced bytes that never arrive would leave mbar_wait spinning forever).
            const uint32_t bb = vstaged ? (uint32_t)(n * 8) : 0u, pb = vstaged ? (uint32_t)c.prow_bytes : 0u;
            if (t == 0) mbar_expect_tx(&sm.mbar, (uint32_t)(prob_elems * ESZ) + bb + pb);
            if (t < n)
                bulk_g2s(sm.tile + t * Smem::PITCH, static_cast<const TA*>(c.A) + (size_t)prob * prob_elems + (size_t)t * n,
                         (uint32_t)n * ESZ, &sm.mbar);
            if (bb != 0u && t == NT - 1) bulk_g2s(sm.vstage[0], c.b + (size_t)prob * n, bb, &sm.mbar);
            if (pb != 0u && t == NT - 2) bulk_g2s(sm.vstage[1], c.params + (size_t)prob * c.param_stride, pb, &sm.mbar);
        } else {
            if (t == 0) mbar_expect_tx(&sm.mbar, (uint32_t)(prob_elems * ESZ) + (vstaged ? 3u * (uint32_t)(n * 8) : 0u));
            if (t < n)
                bulk_g2s(sm.tile + t * Smem::PITCH, static_cast<const TA*>(c.A) + (size_t)prob * prob_elems + (size_t)t * n,
                         (uint32_t)n * ESZ, &sm.mbar);
            if (vstaged && t >= NT - 3) {   // three otherwise idle-ish threads (the mbarrier's expect_tx is program-ordered only in thread 0,
                const int w = t - (NT - 3); // but a complete_tx that arrives first just drives the pending count negative: legal)
                const double* src = w == 0 ? c.b + (size_t)prob * n : (w == 1 ? c.lb : c.ub) + (size_t)prob * c.bound_stride;
                bulk_g2s(sm.vstage[w], src, (uint32_t)(n * 8), &sm.mbar);
            }
        }
    };
    // Work queue, two problems deep: `cur` is being solved, `nxt` is known (its A is in flight), and the index after that is
    // fetched by thread 0 at the start of a solve and published at its end -- the atomic's round trip hides behind the solve.
    if (t == 0) { sm.first = (int)atomicAdd(c.counter, 1u); sm.next = (int)atomicAdd(c.counter, 1u); }
    __syncthreads();
    int cur = sm.first;
    if (staged && cur < c.batch) { fence_proxy_async(); issue_load(cur); }
    while (cur < c.batch) {
        // ---- register fill: this thread's sub-block; register row r <- row row0 + (r ^ key) (see matvec)
        double a[kBRows][kBCols];
        const TA* Ap = static_cast<const TA*>(c.A) + (size_t)cur * prob_elems;
        BState s;
        s.u = u;
        s.act = u < n;
        s.own = s.act && primary;
        const size_t vo = (size_t)cur * n + u;
        const size_t bo = (size_t)cur * c.bound_stride + u;
        if (staged) {
            mbar_wait(&sm.mbar, phase);
            phase ^= 1u;
            const uint32_t tb = smem_u32(sm.tile);
#pragma unroll
            for (int r = 0; r < kBRows; ++r) {
                const int row = row0 + (r ^ key);
                if constexpr (ESZ == 8) {
#pragma unroll
                    for (int j = 0; j < kBCols; j += 2) {
                        if (row < n && col0 + j < n) lds_f64x2(tb + (uint32_t)(row * L::PITCH + col0 + j) * 8u, a[r][j], a[r][j + 1]);
                        else { a[r][j] = 0.0; a[r][j + 1] = 0.0; }
                    }
                } else {            // staged implies n % 4 == 0: a 4-float group is inside the row or wholly past its end
#pragma unroll
                    for (int j = 0; j < kBCols; j += 4) {
                        if (row < n && col0 + j < n) lds_f32x4_widen(tb + (uint32_t)(row * Smem::PITCH + col0 + j) * 4u, &a[r][j]);
                        else { a[r][j] = 0.0; a[r][j + 1] = 0.0; a[r][j + 2] = 0.0; a[r][j + 3] = 0.0; }
                    }
                }
            }
            if (vstaged) {
                s.b = s.act ? sm.vstage[0][u] : 0.0;
                if constexpr (!GEN) {
                    s.lo = s.act ? sm.vstage[1][u] : 0.0;
                    s.hi = s.act ? sm.vstage[2][u] : 0.0;
                }
            }
        } else if (ESZ == 8 && c.vec_ok) {       // fp64 only (the host never sets vec_ok for an fp32 A)
            if constexpr (ESZ == 8) {
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
            }
        } else {
#pragma unroll
            for (int r = 0; r < kBRows; ++r)
#pragma unroll
                for (int j = 0; j < kBCols; ++j)
                    a[r][j] = (row0 + (r ^ key) < n && col0 + j < n) ? (double)ldg_stream(Ap + (size_t)(row0 + (r ^ key)) * n + col0 + j) : 0.0;
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
                if (vstaged) return lds_f64(smem_u32(&sm.vstage[1][0]) + (uint32_t)k * 8u);   // the row runs on into vstage[2]
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
            if (staged) { fence_proxy_async(); issue_load(nxt); }
            else prefetch_l2(nxt);
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

// batched.cu: launches a persistent batched kernel (batched_kernel / batched_sym_kernel, `threads` per CTA, `dyn` bytes of
// dynamic shared memory) with as many CTAs as fit on the device, at most one per problem
cudaError_t launch_persistent(const void* kern, int threads, size_t dyn, const BatchedCtx& c, int sm_count, cudaStream_t stream);

// n <= 64: 64 threads per problem, A in 128 registers per thread, up to 6 problems per SM; 64 < n <= 128: 256 threads, one per SM
template <int SOLVER, bool WREG, bool GEN, class TA>
cudaError_t launch_nt(const BatchedCtx& c, int sm_count, cudaStream_t stream) {
    if (c.n <= kBN) return launch_persistent((const void*)batched_kernel<SOLVER, WREG, GEN, 64, TA>, 64, 0, c, sm_count, stream);
    return launch_persistent((const void*)batched_kernel<SOLVER, WREG, GEN, 256, TA>, 256, sizeof(BatchedSmem<GEN, 256, TA>), c,
                             sm_count, stream);
}

// GEN: the general table instead of a Box per problem; TA: A's element type.  Unknown solvers, and MPRGP with a table, are
// rejected before.  The fp64 kernels are instantiated in batched.cu, the fp32 ones in batched_f32.cu.
template <bool GEN, class TA>
cudaError_t launch_batched(const BatchedCtx& c, int solver, bool wreg, int sm_count, cudaStream_t stream) {
    switch (solver) {
        case CCQP_SOLVER_PGD: return launch_nt<CCQP_SOLVER_PGD, true, GEN, TA>(c, sm_count, stream);
        case CCQP_SOLVER_APGD: return launch_nt<CCQP_SOLVER_APGD, true, GEN, TA>(c, sm_count, stream);
        case CCQP_SOLVER_APGD_AR: return launch_nt<CCQP_SOLVER_APGD_AR, true, GEN, TA>(c, sm_count, stream);
        case CCQP_SOLVER_BBPGD: return launch_nt<CCQP_SOLVER_BBPGD, true, GEN, TA>(c, sm_count, stream);
        case CCQP_SOLVER_BBPGDF: return launch_nt<CCQP_SOLVER_BBPGDF, true, GEN, TA>(c, sm_count, stream);
        case CCQP_SOLVER_SPG:
            return wreg ? launch_nt<CCQP_SOLVER_SPG, true, GEN, TA>(c, sm_count, stream)
                        : launch_nt<CCQP_SOLVER_SPG, false, GEN, TA>(c, sm_count, stream);
        case CCQP_SOLVER_MPRGP:
            if constexpr (!GEN) return launch_nt<CCQP_SOLVER_MPRGP, true, false, TA>(c, sm_count, stream);
            else return cudaErrorInvalidValue;
        default: return cudaErrorInvalidValue;
    }
}
extern template cudaError_t launch_batched<false, float>(const BatchedCtx&, int, bool, int, cudaStream_t);
extern template cudaError_t launch_batched<true, float>(const BatchedCtx&, int, bool, int, cudaStream_t);

// batched_sym.cu: the one-warp-per-problem kernels for symmetric Hessians (n <= 64; PGD / BBPGD / BBPGDf / SPG, Box per
// problem), TA = double / float
bool batched_sym_supported(int solver, long long n);
template <class TA>
cudaError_t launch_batched_sym(const BatchedCtx& c, int solver, bool wreg, int sm_count, cudaStream_t stream);

}  // namespace ccqp
