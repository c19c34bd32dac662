// Batched mode for SYMMETRIC Hessians, n <= 64: one WARP per problem, eight problems in flight per SM.
//
// Problem i is  CCQPSolverX(tol,max_mv).solve(A[i], b[i], x0[i], BoxProjOp(n, lb[i], ub[i]))  (solvers.py:94/583/719/878 with
// solution_spaces.py:280-366), as in batched.cuh, for a caller that declares every A[i] symmetric (ccqp_solve_batched_sym; the
// objective 0.5 x'Ax + b'x of the reference only has the gradient Ax + b it iterates with when A is).  Only the upper
// block triangle of A[i] is ever read -- entries A[r][c] with c >= 8 * (r / 8), the dsymv('U') contract at 8 x 8 granularity.
//
// Why a second kernel: batched.cuh keeps the full 64 x 64 Hessian in the registers of 64 threads (32 KB of the 256 KB register
// file per problem), so six problems share an SM, and it is bound by the latency of ONE problem's dependent chain times the
// problems in flight (DESIGN.md 2.2: 1 -> 6 resident problems scale 13.8 -> 61.2 M QP/s almost linearly).  Half of a symmetric
// matrix is enough:
//   * the 8 x 8 grid of 8 x 8 blocks has 28 blocks above the diagonal: lane l < 28 keeps block (r, c), r < c, in 128 registers
//     and uses it TWICE per mat-vec -- s1 = B x_c is a partial sum of y_r, s2 = B' x_r one of y_c (the same 4096 DFMAs per
//     mat-vec as the full layout, from half the registers);
//   * the 8 diagonal blocks are spread over all lanes by rows: lane l keeps rows 2l, 2l+1 of diagonal block l / 4 (16 doubles)
//     -- exactly the two unknowns it owns, so that part needs no exchange;
//   * the 2 x 8 partial sums a lane produces go through 5 KB of shared memory (slot s of y_k holds the contribution of block
//     (k, s+1) for s >= k and of block (s, k) for s < k: seven slots per unknown, each written exactly once), a lane then adds
//     the seven slots of its two unknowns in a fixed order.  One warp = one problem: the two __syncwarp() of the mat-vec are
//     the only synchronisation, the dot products are pure shuffle butterflies (no shared-memory exchange, no CTA barrier).
//   * 20 KB (the upper block triangle, compact) of the NEXT problem's A and its b / lb / ub rows land in shared memory by TMA row
//     copies on one mbarrier while the current problem iterates; HBM traffic per problem drops from 32 KB to 18 KB.
// Launch shape: 32 threads per CTA, 8 CTAs per SM (<= 255 registers, 28 KB of shared memory each; b / lb / ub of the current
// problem live in shared memory: with them in registers ptxas split the row sums into two-chain groups).
//
// Measured (65 536 problems of n = 64, tol 1e-8, profiles/README.md): SPG 13.8 M QP/s against 12.9 M for batched.cuh (+7 %),
// BBPGD 51.8 M against 61.0 M (-15 %).  Eight problems are in flight instead of six, but one problem's iteration is a longer
// chain here: the mat-vec of a lone warp takes 930 cycles (x slices + diagonal rows 124, s1 308, s2 304, slots read + added
// 196; CCQP_BSYM_TIMING build, tools/bsym_timing.py) against ~480 for the two warps of batched.cuh, because 144 DFMAs per lane
// issue from ONE warp (2.9 cycles each out of a 64-entry register block: ccqp_microbench) where the full layout spreads 128
// over two sub-partitions.  The DFMA count per problem is the same in both layouts, so is their operand traffic; what the
// symmetric layout buys is register space (and half of the HBM reads), what it costs is the exchange through shared memory.
// Hence: an opt-in for callers whose solver is SPG (or whose batch is HBM- or capacity-bound), not the default.
//
// fp32 Hessians (ccqp_solve_batched_sym_f32): the same kernel with TA = float -- a compact float tile (rows padded by 4 floats,
// 16-byte aligned), row pieces of (n - c0) * 4 bytes, and a fill that widens every entry exactly; registers and solver loop
// are those of the fp64 kernel on the widened matrix, so the results are the same bits.
#include "batched.cuh"

namespace ccqp {
namespace bsym {

constexpr int kN = 64;                  // padded problem size
constexpr int kSlice = 10;              // pitch of an 8-entry slice of a vector in shared memory (conflict-free LDS.128, see batched.cuh)
constexpr int kXS = 8 * kSlice;
constexpr int kSlots = 7;
constexpr int kCtPitch = 82;            // doubles per slot: 41 16-byte chunks = 1 (mod 8), so that a lane's slot and its row block both move
                                        // its 16-byte chunk inside the 128-byte bank window (6 wavefronts per store instead of 9 at 90)
constexpr int kRowPad = 2;
constexpr int kRowPadF32 = 4;           // floats: rows start 16-byte aligned; register fill 174 wavefronts (fp64 tile: 516)
template <class TA> constexpr int kRowPadOf = sizeof(TA) == 8 ? kRowPad : kRowPadF32;
constexpr int kCtas = 8;                // resident CTAs (= problems) per SM

// offset (entries) of row i inside the compact tile: row block rb = i / 8 stores columns 8 rb .. 63 (+ pad)
__host__ __device__ constexpr int tile_row_off(int i, int pad = kRowPad) {
    const int rb = i >> 3;
    return 8 * rb * (kN + pad) - 32 * rb * (rb - 1) + (i & 7) * (kN - 8 * rb + pad);
}
constexpr int kTile = tile_row_off(kN);
static_assert(kTile == 2432, "compact tile");
static_assert(tile_row_off(kN, kRowPadF32) % 4 == 0, "fp32 tile: the vectors behind it stay 16-byte aligned");

template <class TA>
struct Smem {
    TA tile[tile_row_off(kN, kRowPadOf<TA>)];   // the NEXT problem: upper block triangle, row by row
    double vstage[3][kN];           // ... its b / lb / ub
    double vcur[3][kN];             // b / lb / ub of the problem being solved (12 registers per lane that the mat-vec needs more)
    double xs[kXS];                 // mat-vec input
    double ct[kSlots * kCtPitch];   // partial sums of the mat-vec
    uint64_t mbar;
    int next, first;
};

struct V2 { double a, b; };
__device__ __forceinline__ V2 operator+(V2 x, V2 y) { return {x.a + y.a, x.b + y.b}; }
__device__ __forceinline__ V2 operator-(V2 x, V2 y) { return {x.a - y.a, x.b - y.b}; }
__device__ __forceinline__ V2 operator*(V2 x, V2 y) { return {x.a * y.a, x.b * y.b}; }
__device__ __forceinline__ V2 operator*(double s, V2 y) { return {s * y.a, s * y.b}; }
__device__ __forceinline__ double hs(V2 x) { return x.a + x.b; }
__device__ __forceinline__ V2 clamp2(V2 t, V2 lo, V2 hi) { return {clampd(t.a, lo.a, hi.a), clampd(t.b, lo.b, hi.b)}; }

__device__ __forceinline__ void sts_f64x2(uint32_t addr, double x, double y) {
    asm volatile("st.shared.v2.f64 [%0], {%1,%2};" ::"r"(addr), "d"(x), "d"(y) : "memory");
}

// two neighbouring 16-byte stores as ONE statement: all four values are due at the same point, which keeps the compiler from
// sinking the row sums into two groups of two dependent chains (it did: 4.2 instead of 2.2 cycles per DFMA)
__device__ __forceinline__ void sts_f64x4(uint32_t addr, double x, double y, double z, double w) {
    asm volatile("st.shared.v2.f64 [%0], {%1,%2};\n\tst.shared.v2.f64 [%0+16], {%3,%4};" ::"r"(addr), "d"(x), "d"(y), "d"(z), "d"(w) : "memory");
}

// Sum K (<= 4) values over the warp; the result in every lane.  The exchange butterfly of batched.cuh's bsum (after two stages a
// lane carries ONE of the K sums), closed by K broadcasts instead of a shared-memory exchange.  Fixed order => deterministic.
template <int K>
__device__ __forceinline__ void wsum(double (&a)[K]) {
    static_assert(K >= 1 && K <= 4, "K");
    const int lane = threadIdx.x & 31;
    if constexpr (K == 1) {
        a[0] = warp_sum(a[0]);
    } else if constexpr (K == 2) {
        const bool odd = lane & 1;
        const double keep = odd ? a[1] : a[0], send = odd ? a[0] : a[1];
        double v = keep + shfl_xor_f64(send, 1);
        v += shfl_xor_f64(v, 2);
        v += shfl_xor_f64(v, 4);
        v += shfl_xor_f64(v, 8);
        v += shfl_xor_f64(v, 16);
        a[0] = __shfl_sync(0xffffffffu, v, 0);
        a[1] = __shfl_sync(0xffffffffu, v, 1);
    } else {
        const bool odd = lane & 1;
        const double a3 = (K == 4) ? a[K - 1] : 0.0;
        double k0 = odd ? a[2] : a[0], k1 = odd ? a3 : a[1];
        const double s0 = odd ? a[0] : a[2], s1 = odd ? a[1] : a3;
        k0 += shfl_xor_f64(s0, 1);
        k1 += shfl_xor_f64(s1, 1);
        const bool up = lane & 2;
        const double keep = up ? k1 : k0, send = up ? k0 : k1;
        double v = keep + shfl_xor_f64(send, 2);       // lane carries sum 2 * (lane & 1) + ((lane >> 1) & 1)
        v += shfl_xor_f64(v, 4);
        v += shfl_xor_f64(v, 8);
        v += shfl_xor_f64(v, 16);
        a[0] = __shfl_sync(0xffffffffu, v, 0);
        a[1] = __shfl_sync(0xffffffffu, v, 2);
        a[2] = __shfl_sync(0xffffffffu, v, 1);
        if constexpr (K == 4) a[3] = __shfl_sync(0xffffffffu, v, 3);
    }
}

struct Lane {                   // shared-window addresses of this lane, fixed for the whole kernel
    uint32_t xs_wr;             // its two unknowns in xs
    uint32_t xs_c, xs_r, xs_d;  // slices of the column block, the row block and the diagonal block it multiplies with
    uint32_t ct_w1, ct_w2;      // where s1 (-> y of row block r) and s2 (-> y of row block c) go
    uint32_t ct_rd;             // slot 0 of its two unknowns
    bool has_blk;               // lanes 28..31 hold no off-diagonal block
    bool act0, act1;            // its unknowns exist (index < n)
};

// y = A v for the two unknowns of the lane.  a: the off-diagonal block (r, c); dg: rows 2l, 2l+1 of the diagonal block.
#ifdef CCQP_BSYM_TIMING
struct MvT { long long t[6]; };
__device__ MvT g_mvt_dummy;
#define MVT_AT(k) if (mt) mt->t[k] += clock64() - t_in
#else
#define MVT_AT(k)
#endif
__device__ __forceinline__ V2 matvec(const double (&a)[8][8], const double (&dg)[2][8], const Lane& L, V2 v
#ifdef CCQP_BSYM_TIMING
                                     , MvT* mt = nullptr
#endif
) {
#ifdef CCQP_BSYM_TIMING
    const long long t_in = clock64();
#endif
    // padding (index >= n) is published as an exact zero whatever v is (batched.cuh matvec)
    sts_f64x2(L.xs_wr, L.act0 ? v.a : 0.0, L.act1 ? v.b : 0.0);
    __syncwarp();
    double xc[8], xr[8], xd[8];
#pragma unroll
    for (int j = 0; j < 8; j += 2) lds_f64x2(L.xs_c + j * 8, xc[j], xc[j + 1]);
#pragma unroll
    for (int j = 0; j < 8; j += 2) lds_f64x2(L.xs_d + j * 8, xd[j], xd[j + 1]);
    // the diagonal block's rows of the two owned unknowns: four chains of four
    double d00 = dg[0][0] * xd[0], d01 = dg[0][4] * xd[4], d10 = dg[1][0] * xd[0], d11 = dg[1][4] * xd[4];
#pragma unroll
    for (int j = 1; j < 4; ++j) {
        d00 = fma(dg[0][j], xd[j], d00); d01 = fma(dg[0][j + 4], xd[j + 4], d01);
        d10 = fma(dg[1][j], xd[j], d10); d11 = fma(dg[1][j + 4], xd[j + 4], d11);
    }
    d00 += d01; d10 += d11;
    MVT_AT(0);
    // s1[i] = sum_j a[i][j] x_c[j], four rows (= four independent chains: DFMA latency 8 cycles, issue 2) at a time
#pragma unroll
    for (int h = 0; h < 8; h += 4) {
        double s[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) s[i] = a[h + i][0] * xc[0];
#pragma unroll
        for (int j = 1; j < 8; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) s[i] = fma(a[h + i][j], xc[j], s[i]);
        if (L.has_blk) sts_f64x4(L.ct_w1 + h * 8, s[0], s[1], s[2], s[3]);
        if (h == 0) {
#pragma unroll
            for (int j = 0; j < 8; j += 2) lds_f64x2(L.xs_r + j * 8, xr[j], xr[j + 1]);
        }
    }
    MVT_AT(1);
    // s2[j] = sum_i a[i][j] x_r[i], four columns at a time
#pragma unroll
    for (int h = 0; h < 8; h += 4) {
        double s[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) s[j] = a[0][h + j] * xr[0];
#pragma unroll
        for (int i = 1; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) s[j] = fma(a[i][h + j], xr[i], s[j]);
        if (L.has_blk) sts_f64x4(L.ct_w2 + h * 8, s[0], s[1], s[2], s[3]);
    }
    MVT_AT(2);
    __syncwarp();
    double p[kSlots], q[kSlots];
#pragma unroll
    for (int k = 0; k < kSlots; ++k) lds_f64x2(L.ct_rd + (uint32_t)k * (kCtPitch * 8u), p[k], q[k]);
    V2 y;
    y.a = ((p[0] + p[1]) + (p[2] + p[3])) + ((p[4] + p[5]) + (p[6] + d00));
    y.b = ((q[0] + q[1]) + (q[2] + q[3])) + ((q[4] + q[5]) + (q[6] + d10));
    MVT_AT(3);
    return y;
}

struct State {
    V2 x0;
    double cs;
    uint32_t vcur;              // this lane's pair in Smem::vcur[0]
    __device__ __forceinline__ V2 ld(uint32_t off) const { V2 r; lds_f64x2(vcur + off, r.a, r.b); return r; }
    __device__ __forceinline__ V2 b() const { return ld(0); }
    __device__ __forceinline__ V2 lo() const { return ld(kN * 8); }
    __device__ __forceinline__ V2 hi() const { return ld(2 * kN * 8); }
};

#ifdef CCQP_BSYM_TIMING     // debug build: cycles of the pieces of a BBPGD iteration, returned in the result record
#define BSYM_T(var) const long long var = clock64()
#else
#define BSYM_T(var)
#endif
template <int SOLVER, bool WREG>
__device__ __forceinline__ void solve_one(const BatchedCtx& c, const double (&a)[8][8], const double (&dg)[2][8], const Lane& L,
                                          const State& s, const double* uni, V2& xsol, BatchedOut& o) {
    int mv = 0, gemv = 0, iters = 0, draws = 0, status = 0;
#ifdef CCQP_BSYM_TIMING
    long long tc_mv = 0, tc_sum = 0, tc_div = 0, tc_all = 0;
    MvT mvt = {{0, 0, 0, 0, 0, 0}};
    const long long tc_begin = clock64();
#endif
    double res = NAN;
    const int maxmv = c.max_mv_i;
    auto P = [&](V2 t) { return clamp2(t, s.lo(), s.hi()); };
    auto MV = [&](V2 v) { gemv++; return matvec(a, dg, L, v); };
    auto resid2 = [&](V2 x, V2 g) { const V2 d = s.cs * (x - P(x - kGd * g)); return hs(d * d); };

    if constexpr (SOLVER == CCQP_SOLVER_PGD || SOLVER == CCQP_SOLVER_BBPGD || SOLVER == CCQP_SOLVER_BBPGDF) {
        // solvers.py:114-170, 606-669, 741-819 (batched.cuh solve_one, two unknowns per lane)
        V2 x = s.x0, xm = s.x0, g, gm, xmin = s.x0, gmin = s.x0;
        double resmin = INFINITY;
        gm = MV(xm) + s.b(); mv = 1;
        double r1[1] = {resid2(xm, gm)};
        wsum<1>(r1);
        double res2 = r1[0];
        if (!(res2 < c.thr_lt)) {
            double step = c.step;
            if (SOLVER != CCQP_SOLVER_PGD) {
                const V2 ag = MV(gm);                                  // not counted (:635)
                double q[2] = {hs(gm * gm), hs(gm * ag)};
                wsum<2>(q);
                step = q[0] / q[1];
            }
            for (;;) {
                BSYM_T(t0);
                x = P(xm - step * gm);
                BSYM_T(t1);
#ifdef CCQP_BSYM_TIMING
                gemv++; g = matvec(a, dg, L, x, &mvt) + s.b(); mv++;
#else
                g = MV(x) + s.b(); mv++;
#endif
                BSYM_T(t2);
                if (mv >= maxmv) break;
                const V2 sx = x - xm, sy = g - gm;
                double q[3] = {resid2(x, g), hs(sx * sx), hs(sx * sy)};
                BSYM_T(t3);
                if (SOLVER == CCQP_SOLVER_PGD) { double q1[1] = {q[0]}; wsum<1>(q1); q[0] = q1[0]; }
                else wsum<3>(q);
                BSYM_T(t4);
#ifdef CCQP_BSYM_TIMING
                tc_mv += t2 - t1; tc_sum += t4 - t3; tc_div += (t1 - t0) ; tc_all += t3 - t2;
#endif
                res2 = q[0];
                iters++;
                if (res2 < c.thr_lt) break;
                if (SOLVER == CCQP_SOLVER_BBPGDF) {                   // :793-800
                    res = sqrt(res2);
                    if (res < resmin) { resmin = res; xmin = x; gmin = g; }
                    if (step < 10 * kEps) {
                        x = P(xmin - kGd * gmin);
                        const V2 sx2 = x - xm;
                        double q2[2] = {hs(sx2 * sx2), hs(sx2 * sy)};
                        wsum<2>(q2);
                        q[1] = q2[0]; q[2] = q2[1];
                    }
                }
                if (SOLVER != CCQP_SOLVER_PGD) step = q[1] / (q[2] + 10 * kEps);
                xm = x; gm = g;
            }
        }
        res = sqrt(res2);
        xsol = x;
    } else {
        static_assert(SOLVER == CCQP_SOLVER_SPG, "solver");
        // solvers.py:906-975
        V2 x = s.x0;
        V2 g = MV(x) + s.b();
        const V2 ag = MV(g);
        double q0[3] = {hs(g * x), hs(g * g), hs(g * ag)};
        wsum<3>(q0);
        double f = q0[0];
        double alpha = q0[1] / q0[2];
        mv = 2;
        SpgWindow<WREG> win;
        win.init(f);
        double dd_rep = NAN;
        double u_next = (c.n_uniforms > 0) ? __ldg(uni) : 0.0;           // the sample of iteration k+1 travels during iteration k
        for (;;) {
            const V2 d = P(x - alpha * g) - x;
            const V2 ad = MV(d); mv++;
            if (mv >= maxmv) break;
            double q[3] = {hs(d * d), hs(d * ad), hs(d * g)};
            wsum<3>(q);
            const double dd = q[0], dAd = q[1], dgs = q[2];
            dd_rep = dd;
            if (dd <= c.thr_le) break;                                // sqrt(dd) <= tol (:949)
            const double fmax = win.max();
            double xi, beta, alpha_next;                              // (fmax - f)/dAd, -dg/dAd, dd/dAd (:954,:955,:966)
            div3_same_divisor(fmax - f, -dgs, dd, dAd, xi, beta, alpha_next);
            const double bhat = c.tau * beta + sqrt((c.tau * c.tau) * (beta * beta) + 2 * xi);
            const double hi = (c.sig2 < bhat) ? c.sig2 : bhat;        // Python min(bhat, sig2)
            if (hi != hi) { status = CCQP_ERR_RANGE; break; }
            if (draws >= c.n_uniforms) { status = CCQP_ERR_UNIFORMS_EXHAUSTED; break; }
            const double bk = c.sig1 + (hi - c.sig1) * u_next;
            draws++;
            u_next = (draws < c.n_uniforms) ? __ldg(uni + draws) : 0.0;
            x = x + bk * d;
            g = g + bk * ad;
            f += bk * bk * dgs + 0.5 * (bk * bk) * dAd;               // :963 as written
            win.push(f, c.m);
            alpha = alpha_next;
            iters++;
        }
        res = sqrt(dd_rep);
        xsol = x;
    }
    o.residual = res;
    o.mv = mv; o.gemv = gemv; o.iters = iters; o.draws = draws;
    o.converged = (mv < maxmv && status == 0) ? 1 : 0;
    o.status = status;
#ifdef CCQP_BSYM_TIMING
    {   // residual <- cycles of the whole solve; gemv <- per-iteration mat-vec; iters <- reduction; draws <- products; (projection in mv)
        const int it = iters > 0 ? iters : 1;
        o.residual = (double)(clock64() - tc_begin);
        if (SOLVER == CCQP_SOLVER_BBPGD) {      // cumulative cycles inside the mat-vec, packed: after diag | after s1 | after s2 | end (12 bits each, /4)
            long long pk = 0;
            for (int k = 0; k < 4; ++k) pk |= ((mvt.t[k] / it / 4) & 0xfff) << (12 * k);
            o.residual = (double)pk;
        }
        o.gemv = (int)(tc_mv / it); o.iters = (int)(tc_sum / it); o.draws = (int)(tc_all / it); o.mv = (int)(tc_div / it) + 1000000 * iters;
    }
#endif
}

template <int SOLVER, bool WREG, class TA>
__global__ void __launch_bounds__(32, kCtas) batched_sym_kernel(const BatchedCtx c) {
    __shared__ __align__(16) Smem<TA> sm;
    constexpr int PAD = kRowPadOf<TA>;
    constexpr uint32_t ESZ = sizeof(TA);
    const int lane = threadIdx.x, n = c.n;
    // lane -> block (r, cc), r < cc, row-major over the 28 blocks above the diagonal
    int r = 0, cc = 1;
    {
        int l = lane;
        while (r < 7 && l >= 7 - r) { l -= 7 - r; r++; }
        cc = r + 1 + l;
    }
    Lane L;
    L.has_blk = lane < 28;
    if (!L.has_blk) { r = 0; cc = 1; }
    const int k = lane >> 2;                // diagonal block of the two unknowns u0 = 2 lane, u0 + 1
    const int u0 = 2 * lane;
    L.act0 = u0 < n; L.act1 = u0 + 1 < n;
    const uint32_t xs0 = smem_u32(sm.xs), ct0 = smem_u32(sm.ct);
    L.xs_wr = xs0 + (uint32_t)(u0 + 2 * k) * 8u;
    L.xs_c = xs0 + (uint32_t)(kSlice * cc) * 8u;
    L.xs_r = xs0 + (uint32_t)(kSlice * r) * 8u;
    L.xs_d = xs0 + (uint32_t)(kSlice * k) * 8u;
    L.ct_w1 = ct0 + (uint32_t)((cc - 1) * kCtPitch + kSlice * r) * 8u;
    L.ct_w2 = ct0 + (uint32_t)(r * kCtPitch + kSlice * cc) * 8u;
    L.ct_rd = ct0 + (uint32_t)(u0 + 2 * k) * 8u;
    const size_t prob_elems = (size_t)n * n;

    const bool staged = c.tma_ok != 0;                  // n * ESZ % 16 == 0, 16-byte aligned A: every row piece is a legal bulk copy
    const bool vstaged = staged && c.vtma_ok != 0;
    uint32_t tx_bytes = vstaged ? 3u * (uint32_t)(n * 8) : 0u;
    for (int i = 0; i < n; ++i) tx_bytes += (uint32_t)(n - 8 * (i >> 3)) * ESZ;
    unsigned phase = 0;
    if (lane == 0) { mbar_init(&sm.mbar, 1); mbar_fence_init(); }
    __syncwarp();
    auto issue_load = [&](int prob) {       // one bulk copy per row: columns 8 * (i / 8) .. n-1 (+ 3 for the vectors), one mbarrier
        const TA* Ap = static_cast<const TA*>(c.A) + (size_t)prob * prob_elems;
        if (lane == 0) mbar_expect_tx(&sm.mbar, tx_bytes);
        __syncwarp();
        for (int i = lane; i < n; i += 32) {
            const int c0 = 8 * (i >> 3);
            bulk_g2s(sm.tile + tile_row_off(i, PAD), Ap + (size_t)i * n + c0, (uint32_t)(n - c0) * ESZ, &sm.mbar);
        }
        if (vstaged && lane >= 29) {
            const int w = lane - 29;
            const double* src = w == 0 ? c.b + (size_t)prob * n : (w == 1 ? c.lb : c.ub) + (size_t)prob * c.bound_stride;
            bulk_g2s(sm.vstage[w], src, (uint32_t)(n * 8), &sm.mbar);
        }
    };
    if (lane == 0) { sm.first = (int)atomicAdd(c.counter, 1u); sm.next = (int)atomicAdd(c.counter, 1u); }
    __syncwarp();
    int cur = sm.first;
    if (staged && cur < c.batch) { fence_proxy_async(); issue_load(cur); }
    while (cur < c.batch) {
        double a[8][8], dg[2][8];
        const TA* Ap = static_cast<const TA*>(c.A) + (size_t)cur * prob_elems;
        State s;
        const size_t vo = (size_t)cur * n + u0;
        const size_t bo = (size_t)cur * c.bound_stride + u0;
        if (staged) {
            mbar_wait(&sm.mbar, phase);
            phase ^= 1u;
            const uint32_t tb = smem_u32(sm.tile);
            // fp64: two doubles per LDS.128; fp32 (staged implies n % 4 == 0): four floats, widened -- a group of
            // 16 / ESZ entries lies inside the row or wholly past its end
            constexpr int V = 16 / ESZ;
            auto ld = [&](uint32_t addr, double* d) {
                if constexpr (ESZ == 8) lds_f64x2(addr, d[0], d[1]);
                else lds_f32x4_widen(addr, d);
            };
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const uint32_t ro = tb + (uint32_t)(tile_row_off(8 * r, PAD) + i * (kN - 8 * r + PAD) + 8 * (cc - r)) * ESZ;
#pragma unroll
                for (int j = 0; j < 8; j += V) {
                    if (L.has_blk && 8 * r + i < n && 8 * cc + j < n) ld(ro + j * ESZ, &a[i][j]);
                    else {
#pragma unroll
                        for (int q = 0; q < V; ++q) a[i][j + q] = 0.0;
                    }
                }
            }
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                const uint32_t ro = tb + (uint32_t)tile_row_off(u0 + t, PAD) * ESZ;
#pragma unroll
                for (int j = 0; j < 8; j += V) {
                    if (u0 + t < n && 8 * k + j < n) ld(ro + j * ESZ, &dg[t][j]);
                    else {
#pragma unroll
                        for (int q = 0; q < V; ++q) dg[t][j + q] = 0.0;
                    }
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    a[i][j] = (L.has_blk && 8 * r + i < n && 8 * cc + j < n) ? (double)ldg_stream(Ap + (size_t)(8 * r + i) * n + 8 * cc + j) : 0.0;
#pragma unroll
            for (int t = 0; t < 2; ++t)
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    dg[t][j] = (u0 + t < n && 8 * k + j < n) ? (double)ldg_stream(Ap + (size_t)(u0 + t) * n + 8 * k + j) : 0.0;
        }
        {
            V2 vb, vl, vh;
            if (vstaged) {
                vb = {sm.vstage[0][u0], sm.vstage[0][u0 + 1]}; vl = {sm.vstage[1][u0], sm.vstage[1][u0 + 1]};
                vh = {sm.vstage[2][u0], sm.vstage[2][u0 + 1]};
            } else {
                vb = {L.act0 ? c.b[vo] : 0.0, L.act1 ? c.b[vo + 1] : 0.0};
                vl = {L.act0 ? c.lb[bo] : 0.0, L.act1 ? c.lb[bo + 1] : 0.0};
                vh = {L.act0 ? c.ub[bo] : 0.0, L.act1 ? c.ub[bo + 1] : 0.0};
            }
            s.vcur = smem_u32(&sm.vcur[0][u0]);     // read back by this lane only: no synchronisation needed
            sts_f64x2(s.vcur, L.act0 ? vb.a : 0.0, L.act1 ? vb.b : 0.0);
            sts_f64x2(s.vcur + kN * 8, L.act0 ? vl.a : 0.0, L.act1 ? vl.b : 0.0);
            sts_f64x2(s.vcur + 2 * kN * 8, L.act0 ? vh.a : 0.0, L.act1 ? vh.b : 0.0);
        }
        s.x0 = {(L.act0 && c.x0) ? c.x0[vo] : 0.0, (L.act1 && c.x0) ? c.x0[vo + 1] : 0.0};
        s.cs = 1.0 / (3 * (double)n * kGd);
        __syncwarp();                          // every lane has read its part of the tile / the staged vectors; sm.next is visible
        const int nxt = sm.next;
        unsigned after = 0;
        if (nxt < c.batch) {                   // the next problem travels while this one iterates
            if (staged) { fence_proxy_async(); issue_load(nxt); }
            else if (c.pf_ok && lane == 0)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(static_cast<const TA*>(c.A) + (size_t)nxt * prob_elems),
                             "r"((unsigned)(prob_elems * ESZ)) : "memory");
            if (c.x0 && L.act0) asm volatile("prefetch.global.L2 [%0];" ::"l"(c.x0 + (size_t)nxt * n + u0));
            if (lane == 0) after = atomicAdd(c.counter, 1u);     // consumed at the end of the solve
        } else if (lane == 0) after = (unsigned)c.batch;

        V2 xsol = {0.0, 0.0};
        BatchedOut o;
        solve_one<SOLVER, WREG>(c, a, dg, L, s, c.uniforms ? c.uniforms + (size_t)cur * c.n_uniforms : nullptr, xsol, o);
        if (L.act0) c.x_out[vo] = xsol.a;
        if (L.act1) c.x_out[vo + 1] = xsol.b;
        if (lane == 0) { c.out[cur] = o; sm.next = (int)after; }
        cur = nxt;
    }
}

}  // namespace bsym

bool batched_sym_supported(int solver, long long n) {
    return n <= bsym::kN && (solver == CCQP_SOLVER_PGD || solver == CCQP_SOLVER_BBPGD || solver == CCQP_SOLVER_BBPGDF ||
                             solver == CCQP_SOLVER_SPG);
}

template <class TA>
cudaError_t launch_batched_sym(const BatchedCtx& c, int solver, bool wreg, int sm_count, cudaStream_t stream) {
    const void* kern;
    switch (solver) {
        case CCQP_SOLVER_PGD: kern = (const void*)bsym::batched_sym_kernel<CCQP_SOLVER_PGD, true, TA>; break;
        case CCQP_SOLVER_BBPGD: kern = (const void*)bsym::batched_sym_kernel<CCQP_SOLVER_BBPGD, true, TA>; break;
        case CCQP_SOLVER_BBPGDF: kern = (const void*)bsym::batched_sym_kernel<CCQP_SOLVER_BBPGDF, true, TA>; break;
        case CCQP_SOLVER_SPG:
            kern = wreg ? (const void*)bsym::batched_sym_kernel<CCQP_SOLVER_SPG, true, TA>
                        : (const void*)bsym::batched_sym_kernel<CCQP_SOLVER_SPG, false, TA>;
            break;
        default: return cudaErrorInvalidValue;
    }
    return launch_persistent(kern, 32, 0, c, sm_count, stream);
}
template cudaError_t launch_batched_sym<double>(const BatchedCtx&, int, bool, int, cudaStream_t);
template cudaError_t launch_batched_sym<float>(const BatchedCtx&, int, bool, int, cudaStream_t);

}  // namespace ccqp
