"""Solver trajectories step by step against a high-precision oracle, on every kernel path.

The parity tests compare converged answers: a solver with a slightly wrong step, momentum coefficient, SPG window or
line-search bound still converges to the same minimiser, and the exits on the mat-vec limit (where the reference has
deliberate quirks: APGD returns the old iterate after its buffer swap, the PGD family the residual of the previous
iterate, MPRGP has four exits and reads a stale gradient in its proportioning branch, ccqp_oracle.py) are hardly
reached.  Here every solver of every path runs with max_mv = k for every k = 1..K, and each stop is compared with the
oracle stopped at the same k:

  * mv, the converged flag and (SPG) the uniforms consumed are equal;
  * the residual is NaN exactly when the oracle's is (SURVEY Q16), otherwise it agrees to RES_GATE relative;
  * |x_gpu - x_hp| <= X_GATE |x_hp|.

The oracle runs unchanged on a matrix whose products are summed in np.longdouble and rounded once, so it is the
trajectory of exact mat-vecs to within one rounding.  A point (case, k) where the oracle on plain NumPy products
disagrees with it is order-unstable (a branch flipped on rounding): it is skipped and counted, and the count is capped.
So are the stops from a tie of the tolerance test on: GPU and oracle residuals that agree to the residual gate but lie
on opposite sides of tol (the residual c |x - P(x - gd g)| cancels, so its last digits follow the rounding of x).

The file also mirrors the mat-vec tiling of the dense kernels (`choose_tiling`, csrc/capi.cu) and forces every branch of
it through CCQP_CW / CCQP_SW."""
import ctypes
import inspect
import sys

import numpy as np
import pytest

import problems as pr
from ccqppy_b200 import _capi
from emulated import EmulatedBox
from helpers import make_solver, op_from_table
from oracle import ccqp_oracle as orc

TOL = 1e-8
X_GATE = 1e-11           # |x_gpu - x_hp| / |x_hp|
RES_GATE = 1e-9          # |res_gpu - res_hp| / res_hp, above the floor below
RES_FLOOR = 64.0         # in units of c eps |x|: the rounding of x - P(x - gd g) scaled by c = 1 / (3 n gd)
STABLE = 1e-13           # the two oracle runs agree to this (relative, on x) at a stable point
GUARD_CAP = 0.05         # at most this fraction of the points of a test may be order-unstable
EPS = np.finfo(np.float64).eps


# ---- the high-precision oracle ------------------------------------------------------------------------------------
class LongDoubleMatrix:
    """A.dot(v) accumulated in np.longdouble and rounded once to float64, for a dense array or a scipy sparse matrix.
    A large dense A is widened in row blocks, never whole at 16 bytes per entry."""
    BLOCK_BYTES = 64 << 20

    def __init__(self, A):
        assert np.finfo(np.longdouble).nmant >= 63, "np.longdouble has no 64-bit mantissa on this host"
        self.shape = A.shape
        self.sparse = hasattr(A, "tocsr")
        if self.sparse:
            self.A = A.tocsr().astype(np.longdouble)
        else:
            A = np.asarray(A)
            n = A.shape[1]
            self.rows = max(1, self.BLOCK_BYTES // (16 * n))
            self.A = A.astype(np.longdouble) if self.rows >= A.shape[0] else A

    def dot(self, v):
        v = np.asarray(v, dtype=np.longdouble)
        if self.sparse or self.A.dtype == np.longdouble:
            return np.asarray(self.A.dot(v), dtype=np.float64)
        out = np.empty(self.shape[0])
        for r0 in range(0, self.shape[0], self.rows):
            out[r0:r0 + self.rows] = self.A[r0:r0 + self.rows].astype(np.longdouble) @ v
        return out


class LowRankMatrix:
    """A = diag(d) + u u^T + z z^T with u, z multiples of 1/16 and d of 1/256: every entry is exact in float64, so the
    product can be formed from the factors -- in np.longdouble (rounded once) or in float64 (a different rounding).
    The wide tiling cases generate such matrices on the device and never copy them to the host."""

    def __init__(self, d, u, z, longdouble):
        self.shape = (d.size, d.size)
        t = np.longdouble if longdouble else np.float64
        self.d, self.u, self.z = (np.asarray(a, dtype=t) for a in (d, u, z))
        self.t = t

    def dot(self, v):
        v = np.asarray(v, dtype=self.t)
        return np.asarray(self.d * v + self.u * self.u.dot(v) + self.z * self.z.dot(v), dtype=np.float64)


# ---- which exits of the oracle a sweep took --------------------------------------------------------------------
FAMILY = {pr.PGD: orc._pgd_family, pr.BBPGD: orc._pgd_family, pr.BBPGDF: orc._pgd_family, pr.APGD: orc._apgd_family,
          pr.APGD_AR: orc._apgd_family, pr.SPG: orc._spg, pr.MPRGP: orc._mprgp}


def _lines_after(func, text):
    """Line numbers of the statements that follow each line of `func` reading `text`."""
    src, first = inspect.getsourcelines(func)
    return {first + i + 1 for i, line in enumerate(src) if line.strip().startswith(text)}


# the `break` of every `if mv >= max_mv:`; for MPRGP also the first statement of the CG and expansion steps.
# MPRGP's proportioning step and its exit are not required: isclose(x, P(x)) holds for every feasible x (SURVEY Q8), so
# its chopped gradient is zero on the iterates, and the step runs only when the gradient is exactly zero (|g|^2 == 0 <
# |chopped g|^2 fails only then; SURVEY appendix B: proportioning is never taken).
EXIT_BREAKS = {f: _lines_after(f, "if mv >= max_mv:") for f in set(FAMILY.values())}
MPRGP_PROPORTIONING_EXIT = max(EXIT_BREAKS[orc._mprgp])
MPRGP_BRANCHES = {line - 1 for text in ("xn = np.copy(y)", "xh = xk - af * p") for line in _lines_after(orc._mprgp, text)}
assert all(len(v) >= 1 for v in EXIT_BREAKS.values()) and len(EXIT_BREAKS[orc._mprgp]) == 4 and len(MPRGP_BRANCHES) == 2
assert MPRGP_PROPORTIONING_EXIT - 2 in _lines_after(orc._mprgp, "gk = pb.mul(xk) + pb.b")


def required_lines(solver):
    f = FAMILY[solver]
    if solver == pr.MPRGP:
        return (EXIT_BREAKS[f] - {MPRGP_PROPORTIONING_EXIT}) | MPRGP_BRANCHES
    return EXIT_BREAKS[f]


class ExitTrace:
    """sys.settrace limited to the oracle's solver functions: records (solver, line) for the watched lines."""

    def __init__(self):
        self.hit = set()
        self.solver = None
        self.watch = {f.__code__: required_lines(s) for s, f in FAMILY.items() if s in (pr.PGD, pr.APGD, pr.SPG, pr.MPRGP)}

    def _local(self, frame, event, arg):
        if event == "line" and frame.f_lineno in self.watch[frame.f_code]:
            self.hit.add((self.solver, frame.f_lineno))
        return self._local

    def _global(self, frame, event, arg):
        return self._local if frame.f_code in self.watch else None

    def run(self, solver, fn):
        self.solver = solver
        prev = sys.gettrace()
        sys.settrace(self._global)
        try:
            return fn()
        finally:
            sys.settrace(prev)

    def missing(self, solvers):
        return {pr.SOLVER_NAMES[s]: sorted(required_lines(s) - {l for t, l in self.hit if t == s}) for s in solvers
                if required_lines(s) - {l for t, l in self.hit if t == s}}


# ---- the comparison ---------------------------------------------------------------------------------------------
def _xnorm(x):
    return float(np.linalg.norm(np.asarray(x, dtype=np.float64)))


def stable_point(o, p):
    """The oracle on long-double and on plain products took the same path to this stop."""
    if o["mv"] != p["mv"] or o["converged"] != p["converged"] or o["draws"] != p["draws"]:
        return False
    if np.isnan(o["residual"]) != np.isnan(p["residual"]):
        return False
    return _xnorm(o["solution"] - p["solution"]) <= STABLE * _xnorm(o["solution"])


def _res_gate(ro, sx, n):
    """How far the GPU's residual may be from the oracle's ro (|x_hp| = sx)."""
    return RES_GATE * abs(ro) + RES_FLOOR * max(1.0, 1.0 / (3 * n * orc.GD)) * EPS * sx


def convergence_tie(g, o, n):
    """The GPU and the oracle stopped on opposite sides of the tolerance test with residuals that agree to the gate: a
    rounding-level tie of that test, whose outcome no summation order decides."""
    rg, ro = float(g["residual"]), o["residual"]
    return (bool(g["converged"]) != o["converged"] and np.isfinite(rg) and np.isfinite(ro) and min(rg, ro) <= TOL <= max(rg, ro)
            and abs(rg - ro) <= _res_gate(ro, _xnorm(o["solution"]), n))


def compare(g, o, n, solver):
    """Failures of a GPU stop `g` against the oracle stop `o`, the relative deviation of x, and the deviation of the
    residual as a fraction of its gate."""
    errs = []
    if int(g["mv"]) != o["mv"]:
        errs.append("mv %d, oracle %d" % (g["mv"], o["mv"]))
    if bool(g["converged"]) != o["converged"]:
        errs.append("converged %s, oracle %s" % (bool(g["converged"]), o["converged"]))
    if solver == pr.SPG and int(g["draws"]) != o["draws"]:
        errs.append("uniforms used %d, oracle %d" % (g["draws"], o["draws"]))
    sx = _xnorm(o["solution"])
    dx = _xnorm(np.asarray(g["solution"], dtype=np.float64) - o["solution"])
    rx = dx / sx if sx > 0 else (0.0 if dx == 0 else np.inf)
    if not dx <= X_GATE * sx:
        errs.append("|dx|/|x| = %.3g" % rx)
    rg, ro = float(g["residual"]), o["residual"]
    rr = 0.0
    if np.isnan(rg) != np.isnan(ro):
        errs.append("residual %r, oracle %r" % (rg, ro))
    elif not np.isnan(ro):
        dr = abs(rg - ro)
        rr = dr / _res_gate(ro, sx, n) if dr else 0.0
        if not rr <= 1.0:
            errs.append("residual %.17g, oracle %.17g (%.3g x the gate)" % (rg, ro, rr))
    return errs, rx, rr


class Sweep:
    """Runs the k sweeps of one test, collects deviations, skips and failures, and reports them at the end."""

    def __init__(self, path):
        self.path = path
        self.trace = ExitTrace()
        self.rows = {}           # case -> [points, skipped, max x dev, max res dev]
        self.failures = []
        self.solvers = set()

    def run(self, case, solver, K, gpu_at, problems, step=0.01):
        """gpu_at(solver, k) -> list of GPU stops, one per problem; problems: list of dicts with the oracle's inputs
        (A_hp, A_plain, b, blocks, params, x0, uniforms)."""
        row = self.rows.setdefault(case, [0, 0, 0.0, 0.0])
        self.solvers.add(solver)
        tied = set()             # problems whose trajectory went past a tie of the tolerance test: the rest differs
        for k in range(1, K + 1):
            gs = gpu_at(solver, k)
            assert len(gs) == len(problems)
            for i, (g, q) in enumerate(zip(gs, problems)):
                kw = dict(x0=q.get("x0"), blocks=q["blocks"], params=q["params"], tol=TOL, max_mv=k, step_size=step,
                          uniforms=q.get("uniforms"))
                o = self.trace.run(solver, lambda: orc.solve(solver, q["A_hp"], q["b"], **kw))
                p = orc.solve(solver, q["A_plain"], q["b"], **kw)
                row[0] += 1
                if i in tied or not stable_point(o, p):
                    row[1] += 1
                    continue
                errs, rx, rr = compare(g, o, q["b"].shape[0], solver)
                if errs and convergence_tie(g, o, q["b"].shape[0]):
                    tied.add(i)
                    row[1] += 1
                    continue
                row[2], row[3] = max(row[2], rx), max(row[3], rr)
                if errs:
                    self.failures.append("%s %s k=%d problem %d: %s" % (case, pr.SOLVER_NAMES[solver], k, i, "; ".join(errs)))

    def finish(self):
        for case, (pts, skipped, mx, mr) in self.rows.items():
            print("[trajectories] %s %s: %d points, %d order-unstable skipped, max |dx|/|x| %.3g, max residual dev / gate %.3g"
                  % (self.path, case, pts, skipped, mx, mr))
        assert not self.failures, "%d stops differ from the oracle:\n%s" % (len(self.failures), "\n".join(self.failures[:40]))
        pts = sum(r[0] for r in self.rows.values())
        skipped = sum(r[1] for r in self.rows.values())
        assert skipped <= GUARD_CAP * pts, (skipped, pts)
        missing = self.trace.missing(self.solvers)
        assert not missing, "oracle exit sites / MPRGP branches never reached: %s" % missing


# ---- the mat-vec tiling of the dense kernels: a mirror of choose_tiling (csrc/capi.cu) ---------------------------
SMEM_TARGET, SMEM_LIMIT = 200 * 1024, 220 * 1024


def dense_smem_bytes(CW, rows_max, nseg):                           # csrc/dense.cuh
    return 2 * CW * 8 + rows_max * nseg * 8 + 8 * 32 * 8 + 32 * 8 + 8 * 8 + 128


def mirror_tiling(n, sm_count, nrows=None, world=1, cw=None, sw=None, csr_nnz=None, doubling="divisor"):
    """The tiling choose_tiling picks for n columns, this rank's nrows rows and `world` ranks; cw / sw: CCQP_CW /
    CCQP_SW.  doubling="divisor" is the rule of the code (double SW only while 2 SW divides CW), "any" the rule before
    it (double while SW < CW).  CSR: only the grid."""
    nrows = n if nrows is None else nrows
    rows_ref = max(1, n // world) if world > 1 else nrows
    if csr_nnz is not None:
        work = rows_ref if world > 1 else csr_nnz // 16384
    else:
        work = rows_ref * n // 8192
    t = dict(grid=max(1, min(sm_count, rows_ref, max(1, work))), accum=0)
    if csr_nnz is not None:
        return t
    t["rows_max"] = -(-nrows // t["grid"]) + 1
    cw_cap = -(-n // 128) * 128
    ok = lambda v: v is not None and 128 <= v <= 16384 and v % 128 == 0
    CW = min(cw if ok(cw) else min(8192, cw_cap), cw_cap)
    SW = min(sw if ok(sw) else min(2048, CW), CW)
    if CW % SW:
        SW = CW
    sw0 = SW

    def layout(SW, accum):
        npan = -(-n // CW)
        spp_full = CW // SW
        last = n - (npan - 1) * CW
        nseg = spp_full if accum else (npan - 1) * spp_full + -(-last // SW)
        t.update(CW=CW, SW=SW, np=npan, nseg=nseg, accum=accum, smem=dense_smem_bytes(CW, t["rows_max"], nseg))

    while True:
        layout(SW, 0)
        if t["smem"] <= SMEM_TARGET or (CW % (2 * SW) if doubling == "divisor" else SW >= CW):
            break
        SW *= 2
    if t["smem"] > SMEM_TARGET:
        layout(sw0, 1)
    return t


def psum_slots_ok(t, n):
    """Every (panel, segment) task of gemv_phase (csrc/dense.cuh) writes its own partial-sum slot below nseg, and every
    slot the row sum reads is written: one slot per segment of the whole row, or (accum) per segment of a panel, whose
    first panel writes them all."""
    CW, SW, nseg = t["CW"], t["SW"], t["nseg"]
    if not (SW <= CW and CW % SW == 0):
        return False
    seen = []
    for p in range(t["np"]):
        spp = -(-min(CW, n - p * CW) // SW)
        slots = [s if t["accum"] else p * (CW // SW) + s for s in range(spp)]
        if t["accum"] and (len(set(slots)) != len(slots) or (p == 0 and sorted(slots) != list(range(nseg)))):
            return False
        seen += slots
    if t["accum"]:
        return max(seen) < nseg
    return sorted(seen) == list(range(nseg))


def test_tiling_mirror_invariants():
    """CPU only: the partial-sum layout holds for every tiling the code can launch, over a grid of (n, CW, SW, SMs);
    the rule before the fix breaks it (CW 384 / 640, SW 128, n = 24000); the default tilings did not change."""
    for n in (1, 100, 127, 128, 129, 1000, 2049, 8191, 8193, 20000, 24000, 53000, 60000, 105000, 140000):
        for sms in (1, 2, 16, 132, 148, 160):
            for cw in (None, 128, 256, 384, 640, 1024, 2048, 3072, 6144, 8192, 16384):
                for sw in (None, 128, 256, 384, 512, 2048, 4096):
                    t = mirror_tiling(n, sms, cw=cw, sw=sw)
                    if t["smem"] <= SMEM_LIMIT:
                        assert psum_slots_ok(t, n), (n, sms, cw, sw, t)
    for cw in (384, 640):
        old = mirror_tiling(24000, 148, cw=cw, sw=128, doubling="any")
        assert old["smem"] <= SMEM_LIMIT and not psum_slots_ok(old, 24000), old
        new = mirror_tiling(24000, 148, cw=cw, sw=128)
        assert new["accum"] == 1 and new["SW"] == 128 and psum_slots_ok(new, 24000), new
    changed = [n for n in range(1, 140001) if mirror_tiling(n, 148) != mirror_tiling(n, 148, doubling="any")]
    assert not changed, changed[:10]
    # at 148 SMs the default tiling doubles SW from n = 51201 (4096) and 72965 (8192); from n = 101085 it adds panels up
    assert [(mirror_tiling(n, 148)["SW"], mirror_tiling(n, 148)["accum"]) for n in (51200, 51201, 72965, 101084, 101085)] == \
        [(2048, 0), (4096, 0), (8192, 0), (8192, 0), (2048, 1)]


def _assert_tiling(h, n, **kw):
    info = h.info()
    t = mirror_tiling(n, info["sm_count"], **kw)
    assert info["dense_grid"] == t["grid"], (info, t)
    if "smem" in t:
        assert info["dense_smem_bytes"] == t["smem"], (info, t)
    return t


# ---- GPU runners: each returns gpu_at(solver, k) -> [stop, ...] -------------------------------------------------
def _ptr(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


class DenseRun:
    """One handle whose matrix is set by `set_matrix(h)` (it returns what must stay alive) and a table; runs ccqp_solve
    with host vectors."""

    def __init__(self, set_matrix, tab, n, b, x0=None, step=0.01, uniforms=None):
        self.h = _capi.Handle()
        self.keep = set_matrix(self.h)
        self.blocks = _capi.make_blocks(tab.blocks)
        self.par = np.ascontiguousarray(tab.params if tab.params.size else np.zeros(1))
        _capi.check(self.h.h, self.h.lib.ccqp_set_projection(self.h.h, self.blocks.ptr, len(self.blocks), _ptr(self.par),
                                                             tab.params.size))
        self.n, self.b, self.x0, self.step, self.uni = n, np.ascontiguousarray(b, dtype=np.float64), x0, step, uniforms

    def __call__(self, solver, k):
        prm = make_solver(solver, TOL, k, self.step)._params()
        res = _capi.Result()
        x = np.empty(self.n)
        uni = self.uni if solver == pr.SPG else None
        _capi.check(self.h.h, self.h.lib.ccqp_solve(self.h.h, solver, ctypes.byref(prm), _ptr(self.b), _ptr(self.x0), _ptr(uni),
                                                    0 if uni is None else uni.size, _ptr(x), _capi.MEM_HOST, ctypes.byref(res)))
        return [dict(solution=x, residual=res.residual, converged=res.converged, mv=res.mv_count, draws=res.uniforms_used)]

    def close(self):
        self.h.close()


def _set_dense_host(A):
    A = np.ascontiguousarray(A, dtype=np.float64)
    n = A.shape[0]
    return lambda h: (_capi.check(h.h, h.lib.ccqp_set_matrix(h.h, _ptr(A), n, n, 0, n, _capi.MEM_HOST)), A)


def _set_dense_device(t, n, lda):
    return lambda h: (_capi.check(h.h, h.lib.ccqp_set_matrix(h.h, ctypes.c_void_p(t.data_ptr()), n, lda, 0, n, _capi.MEM_DEVICE)), t)


def _problem(A, b, tab, x0=None, uniforms=None, A_hp=None):
    return dict(A_hp=A_hp if A_hp is not None else LongDoubleMatrix(A), A_plain=A, b=np.asarray(b, dtype=np.float64),
                blocks=tab.blocks, params=tab.params, x0=x0, uniforms=uniforms)


def _step(A):
    A = np.asarray(A, dtype=np.float64) if not hasattr(A, "tocsr") else A
    return 1.0 / float(abs(A).sum(axis=1).max())


def _suite3():
    """The five 3x3 problems of the suite (problem_suite.py; integer A as in the reference)."""
    A = np.array([[2, -1, 0], [-1, 2, -1], [0, -1, 2]])
    out = []
    for name, tab, xs in (("unconstrained", pr.identity_table(3), (1, 0, 1)),
                          ("unconstrained_split", pr.Table().add(pr.IDENTITY, 1).add(pr.IDENTITY, 1).add(pr.IDENTITY, 1), (1, 0, 1)),
                          ("box", pr.box_table(3, 0.0, 2.0), (1, 0, 1)),
                          ("thin_box", pr.Table().add(pr.BOX, 3, [-10, -0.1, 0.9], [10, 0.1, 1.1]), (1, 0, 1)),
                          ("active_box", pr.box_table(3, 9.0, 10.0), (1, 1, 1))):
        out.append((name, A, -A.dot(np.array(xs)), tab))
    return out


def _box_problem(n, seed, lo=-1.0, hi=1.0):
    """shift_problem's minimiser lies in [-3, 1]^n: about half of the box constraints are active at the solution."""
    A, b = pr.shift_problem(n, seed)
    return A, b, pr.box_table(n, lo, hi)


ALL = list(range(7))


def _dense_sweep(sw, case, A, b, tab, set_matrix, K, x0=None, step=None, solvers=ALL, tiling=None):
    n = b.shape[0]
    step = _step(A) if step is None else step
    uni = pr.spg_uniforms(7, K + 8)
    run = DenseRun(set_matrix, tab, n, b, x0=x0, step=step, uniforms=uni)
    if tiling is not None:
        _assert_tiling(run.h, n, **tiling)
    prob = [_problem(A, b, tab, x0=x0, uniforms=uni)]
    for solver in solvers:
        sw.run(case, solver, K, run, prob, step=step)
    run.close()


@pytest.mark.gpu
def test_dense_fp64_trajectories():
    """One-CTA runs (the suite's 3x3 problems, n = 64 with x0), a multi-CTA run, and the scalar mat-vec loop (a CUDA
    tensor of odd n, and a window of a CUDA buffer with lda > n)."""
    import torch
    sw = Sweep("dense fp64")
    # K = 38: on the unconstrained 3x3 problems APGD-AR converges at mv = 39 after a Lipschitz test (l1 + l2 <= r1 + .. + r4)
    # whose two sides agree to rounding: the GPU's own dot products may reject it and spend one more product.  That tie
    # lies in the vector reductions, which the guard (a second oracle run on other mat-vec roundings) does not vary.
    for name, A, b, tab in _suite3():
        _dense_sweep(sw, "3x3 " + name, A, b, tab, _set_dense_host(A), K=38, step=0.1, tiling={})
    A, b, tab = _box_problem(64, 1)
    x0 = 0.5 * np.random.default_rng(2).standard_normal(64)
    _dense_sweep(sw, "n64 x0", A, b, tab, _set_dense_host(A), K=40, x0=x0, tiling={})
    A, b, tab = _box_problem(1100, 3)
    _dense_sweep(sw, "n1100 multi-CTA", A, b, tab, _set_dense_host(A), K=24, tiling={})
    A, b, tab = _box_problem(129, 4)
    _dense_sweep(sw, "n129 cuda odd n", A, b, tab, _set_dense_device(torch.from_numpy(A).cuda(), 129, 129), K=30, tiling={})
    A, b, tab = _box_problem(256, 5)
    buf = torch.zeros((256, 259), dtype=torch.float64, device="cuda")
    buf[:, :256] = torch.from_numpy(A)
    buf[:, 256:] = float("nan")                          # never read
    _dense_sweep(sw, "n256 window lda 259", A, b, tab, _set_dense_device(buf, 256, 259), K=30, tiling={})
    sw.finish()


@pytest.mark.gpu
def test_dense_fp32_trajectories():
    """ccqp_set_matrix_f32 against the oracle on the widened matrix (one CTA and multi-CTA, Box and a mixed table)."""
    sw = Sweep("dense fp32")
    for case, n, tab_of in (("n96 wide box", 96, lambda n: pr.box_table(n, -4.0, 2.0)), ("n700 mixed", 700, pr.mixed_table)):
        A, b = pr.shift_problem(n, 6)
        A32 = A.astype(np.float32)
        tab = tab_of(n)
        def set32(h, A32=A32, n=n):
            h.set_matrix_f32(A32, n)
            return A32
        _dense_sweep(sw, case, A32.astype(np.float64), b, tab, set32, K=30, tiling={})
    sw.finish()


def csr_problem(n, seed):
    """An SPD scipy CSR Hessian with empty rows (their unknowns are linear terms, held by the box) and one row and
    column with n - 1 entries (longer than a 4096-entry tile of the CSR stream)."""
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    D = sp.random(n, n, density=4.0 / n, random_state=np.random.RandomState(seed), format="csr",
                  data_rvs=lambda k: rng.standard_normal(k))
    A = (D.T @ D + sp.identity(n)).tolil()
    w = 0.01 * rng.standard_normal(n)
    A[1, :] = w
    A[:, 1] = w[:, None]
    A[1, 1] = 2.0 + np.abs(w).sum()
    empty = rng.choice(np.arange(2, n), size=max(1, n // 50), replace=False)
    A = A.tocsr()
    keep = np.ones(n)
    keep[empty] = 0
    K = sp.diags(keep)
    A = (K @ A @ K).tocsr()
    A.eliminate_zeros()
    A.sort_indices()
    assert A.indptr[2] - A.indptr[1] > 4096 and (np.diff(A.indptr) == 0).sum() == empty.size
    b = -(A @ (1 - 4 * rng.random(n))) + rng.standard_normal(n) * (keep == 0)
    return A, b


@pytest.mark.gpu
def test_csr_trajectories():
    from ccqppy_b200.solvers import _set_sparse_matrix
    sw = Sweep("csr")
    n = 5000
    A, b = csr_problem(n, 8)
    for case, tab in (("box", pr.box_table(n)), ("wide box", pr.box_table(n, -4.0, 2.0))):
        _dense_sweep(sw, "n5000 empty rows, row of 4999, " + case, A, b, tab, lambda h: _set_sparse_matrix(h, A, n), K=30,
                     tiling=dict(csr_nnz=A.nnz))
    sw.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_emulated_ranks_trajectories(world):
    """Row-sharded solves, ranks emulated on one GPU: every rank returns the same stop, and it is the oracle's."""
    sw = Sweep("emulated world %d" % world)
    for case, (A, b), tab in (("dense n300", pr.shift_problem(300, 9), pr.box_table(300)),
                              ("csr n5000 wide box", csr_problem(5000, 10), pr.box_table(5000, -4.0, 2.0))):
        n = b.shape[0]
        step = _step(A)
        uni = pr.spg_uniforms(11, 40)
        box = EmulatedBox(A, op_from_table(tab), world)
        for r, h in enumerate(box.handles):
            r0, r1 = box.ranges[r]
            _assert_tiling(h, n, nrows=r1 - r0, world=world, csr_nnz=A.nnz if hasattr(A, "nnz") else None)

        def at(solver, k):
            rs = box.solve(make_solver(solver, TOL, k, step), b, uniforms=uni if solver == pr.SPG else None)
            for r in rs[1:]:
                assert np.array_equal(r["solution"].view(np.int64), rs[0]["solution"].view(np.int64)), (case, solver, k)
                assert (r["mv"], r["converged"], r["draws"]) == (rs[0]["mv"], rs[0]["converged"], rs[0]["draws"])
                assert np.array_equal(np.float64(r["residual"]).view(np.int64), np.float64(rs[0]["residual"]).view(np.int64))
            return rs[:1]
        prob = [_problem(A, b, tab, uniforms=uni)]
        for solver in ALL:
            sw.run(case, solver, 28, at, prob, step=step)
        box.close()
    sw.finish()


# ---- batched solves: each k is ONE call for the whole batch ------------------------------------------------------
BATCH = 4
BSTEP = 0.1


def _batch(n, seed0, batch=BATCH, symmetric=False, wide=False):
    A = np.empty((batch, n, n))
    b = np.empty((batch, n))
    for i in range(batch):
        A[i], b[i] = pr.shift_problem(n, seed0 + i)
    if symmetric:
        A = 0.5 * (A + A.transpose(0, 2, 1))
    rng = np.random.default_rng(seed0)
    lb = -1.0 - 0.2 * rng.random((batch, n)) - 3.0 * wide
    ub = 1.0 + 0.2 * rng.random((batch, n)) + wide
    return A, b, lb, ub


def _batched_at(A, b, K, **kw):
    """gpu_at for solve_batched; SPG takes the explicit streams pr.spg_uniforms(i, K + 4)."""
    uni = np.stack([pr.spg_uniforms(i, K + 4) for i in range(b.shape[0])])

    def at(solver, k):
        s = make_solver(solver, TOL, k, BSTEP)
        s.solve_batched(A, b, uniforms=uni, **kw)
        x = s.solution.cpu().numpy() if hasattr(s.solution, "cpu") else np.asarray(s.solution)
        return [dict(solution=x[i], residual=s.solution_residual[i], converged=s.solution_converged[i],
                     mv=s.solution_num_matrix_vector_multiplications[i], draws=s._uniforms_used[i]) for i in range(b.shape[0])]
    return at, uni


def _box_problems(A, b, lb, ub, uni):
    out = []
    for i in range(b.shape[0]):
        tab = pr.Table().add(pr.BOX, b.shape[1], lb[i], ub[i])
        out.append(_problem(np.asarray(A[i], dtype=np.float64), b[i], tab, uniforms=uni[i]))
    return out


@pytest.mark.gpu
def test_batched_general_trajectories():
    """The general batched kernel with a Box per problem, all seven solvers: NT = 64 for n <= 64, NT = 256 above."""
    sw = Sweep("batched general")
    K = 30
    for n in (1, 2, 3, 7, 8, 9, 31, 63, 64, 65, 127, 128):
        A, b, lb, ub = _batch(n, 100 * n)
        at, uni = _batched_at(A, b, K, lower_bound=lb, upper_bound=ub)
        probs = _box_problems(A, b, lb, ub, uni)
        for solver in ALL:
            sw.run("n%d" % n, solver, K, at, probs, step=BSTEP)
    sw.finish()


@pytest.mark.gpu
def test_batched_symmetric_trajectories():
    """The one-warp-per-problem kernels for symmetric A: odd n loads directly, even n stages the tile by TMA."""
    sw = Sweep("batched symmetric")
    K = 30
    for n in (5, 8, 17, 63, 64):
        A, b, lb, ub = _batch(n, 100 * n + 1, symmetric=True)
        at, uni = _batched_at(A, b, K, lower_bound=lb, upper_bound=ub, symmetric=True)
        probs = _box_problems(A, b, lb, ub, uni)
        for solver in (pr.PGD, pr.BBPGD, pr.BBPGDF, pr.SPG):
            sw.run("n%d" % n, solver, K, at, probs, step=BSTEP)
    sw.finish()


def _small_mixed(n, rng):
    """Box, Lower, Upper, Sphere(3) blocks and an Identity tail on n >= 24 unknowns."""
    nb, nl, nu = n // 4, n // 8, n // 8
    t = pr.Table()
    lo = -1.0 - 0.5 * rng.random(nb)
    t.add(pr.BOX, nb, lo, lo + 1.5 + rng.random(nb))
    t.add(pr.LOWER, nl, -0.5 - rng.random(nl))
    t.add(pr.UPPER, nu, 0.5 + rng.random(nu))
    while t.n + 3 <= n - 2:
        t.add(pr.SPHERE, 3, 0.3 + rng.random())
    t.add(pr.IDENTITY, n - t.n)
    return t


TABLES = {"sphere3": (63, lambda n, rng: pr.sphere3_table(n, 0.3 + 0.4 * rng.random())),
          "mixed": (47, _small_mixed),
          "soc3": (30, lambda n, rng: pr.soc3_table(n, 0.3 + 0.5 * rng.random()))}
TABLE_SOLVERS = (pr.PGD, pr.APGD, pr.APGD_AR, pr.BBPGD, pr.BBPGDF, pr.SPG)


def _table_sweep(sw, name, form, K, f32=False):
    n, make = TABLES[name]
    A, b, _, _ = _batch(n, 7 * n + (form == "tables"))
    rng = np.random.default_rng(n)
    tabs = [make(n, rng) for _ in range(b.shape[0])] if form == "tables" else [make(n, rng)] * b.shape[0]
    ops = [op_from_table(t) for t in tabs]
    for t, op in zip(tabs, ops):
        assert np.array_equal(op.descriptor()[1], t.params)
    Ain = A.astype(np.float32) if f32 else A
    Aw = Ain.astype(np.float64)
    if form == "tables":
        P = np.stack([t.params for t in tabs])
        at, uni = _batched_at(Ain, b, K, convex_proj_op=ops[0], op_params=P)
    else:
        at, uni = _batched_at(Ain, b, K, convex_proj_op=ops[0])
    probs = [_problem(Aw[i], b[i], tabs[i], uniforms=uni[i]) for i in range(b.shape[0])]
    for solver in TABLE_SOLVERS:
        sw.run("%s %s" % (form, name), solver, K, at, probs, step=BSTEP)


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["table", "tables"])
def test_batched_table_trajectories(form):
    """One block table shared by the batch (`table`), and one block structure with parameters per problem (`tables`,
    op_params): Sphere(3) discs, a mixed table and SOC(3) cones, six solvers."""
    sw = Sweep("batched " + form)
    for name in TABLES:
        _table_sweep(sw, name, form, K=30)
    sw.finish()


@pytest.mark.gpu
def test_batched_f32_trajectories():
    """One representative per form for the float32 twins of the batched entry points."""
    sw = Sweep("batched fp32")
    K = 24
    for case, n, wide, kw, solvers in (("box n64", 64, False, {}, ALL), ("wide box n128", 128, True, {}, ALL),
                                       ("sym n63", 63, False, dict(symmetric=True), (pr.PGD, pr.BBPGD, pr.BBPGDF, pr.SPG))):
        A, b, lb, ub = _batch(n, 5 * n, symmetric="symmetric" in kw, wide=wide)
        A32 = A.astype(np.float32)
        at, uni = _batched_at(A32, b, K, lower_bound=lb, upper_bound=ub, **kw)
        probs = _box_problems(A32, b, lb, ub, uni)
        for solver in solvers:
            sw.run(case, solver, K, at, probs, step=BSTEP)
    _table_sweep(sw, "sphere3", "table", K, f32=True)
    _table_sweep(sw, "mixed", "tables", K, f32=True)
    sw.finish()


# ---- the gate rejects a perturbed trajectory -----------------------------------------------------------------------
@pytest.mark.gpu
def test_gate_rejects_perturbed_oracle():
    """The comparison rejects an oracle run whose PGD step, SPG sigma1 or x0 is off by 1e-6 relative."""
    n = 64
    A, b, tab = _box_problem(n, 12)
    step = _step(A)
    uni = pr.spg_uniforms(3, 40)
    x0 = 0.5 * np.random.default_rng(4).standard_normal(n)
    run = DenseRun(_set_dense_host(A), tab, n, b, x0=x0, step=step, uniforms=uni)
    hp = LongDoubleMatrix(A)
    base = dict(x0=x0, step_size=step, sigma1=0.01)
    for solver, change, first in ((pr.PGD, dict(step_size=step * (1 + 1e-6)), 1), (pr.SPG, dict(sigma1=0.01 * (1 + 1e-6)), 4),
                                  (pr.BBPGD, dict(x0=x0 * (1 + 1e-6)), 1)):
        for k in range(1, 9):                            # before the solves converge (which damps a change of x0)
            g = run(solver, k)[0]
            exact = orc.solve(solver, hp, b, blocks=tab.blocks, params=tab.params, tol=TOL, max_mv=k, uniforms=uni, **base)
            assert not compare(g, exact, n, solver)[0], (pr.SOLVER_NAMES[solver], k)
            bad = orc.solve(solver, hp, b, blocks=tab.blocks, params=tab.params, tol=TOL, max_mv=k, uniforms=uni,
                            **dict(base, **change))
            if k >= first:
                assert compare(g, bad, n, solver)[0], (pr.SOLVER_NAMES[solver], k)
    run.close()


# ---- forced tilings of the dense mat-vec -----------------------------------------------------------------------------
TILINGS = [("multi_panel", 20000, 2048, 512), ("doubling_to_divisor", 20000, 2048, 128), ("cw384_sw128", 24000, 384, 128),
           ("cw640_sw128", 24000, 640, 128), ("accum", 24000, 128, 128), ("default_doubling", 60000, None, None)]


def _expected_branch(name, t):
    if name == "multi_panel":
        return t["np"] > 1 and t["SW"] == 512 and not t["accum"]
    if name == "doubling_to_divisor":
        return t["SW"] > 128 and not t["accum"]
    if name in ("cw384_sw128", "cw640_sw128"):       # no width that divides CW fits: one slot per segment of a panel
        return t["SW"] == 128 and t["accum"] == 1
    if name == "accum":
        return t["accum"] == 1
    return t["SW"] > 2048 and not t["accum"]          # the default tiling doubles SW for n of ~53k to ~105k


@pytest.mark.gpu
@pytest.mark.parametrize("name, n, cw, sw", TILINGS, ids=[t[0] for t in TILINGS])
def test_forced_tilings(name, n, cw, sw, monkeypatch):
    """Every branch of choose_tiling, forced through CCQP_CW / CCQP_SW: the mirror proves which branch runs and must
    give the grid and shared-memory bytes of Handle.info().  A = diag(d) + u u^T + z z^T is generated on the device;
    its product is checked against the factors with the |A||v| bound, and a short SPG trajectory against the oracle."""
    import torch
    for var, val in (("CCQP_CW", cw), ("CCQP_SW", sw)):
        if val is None:
            monkeypatch.delenv(var, raising=False)
        else:
            monkeypatch.setenv(var, str(val))
    rng = np.random.default_rng(n + (cw or 0))
    u = rng.integers(-16, 17, n) / 16.0
    z = rng.integers(-16, 17, n) / 16.0
    d = 1.0 + rng.integers(0, 257, n) / 256.0
    dev = torch.device("cuda")
    ud, zd = torch.from_numpy(u).to(dev), torch.from_numpy(z).to(dev)
    A = torch.outer(ud, ud)
    A.addr_(zd, zd)
    A.diagonal().add_(torch.from_numpy(d).to(dev))
    torch.cuda.synchronize()
    h = _capi.Handle()
    _capi.check(h.h, h.lib.ccqp_set_matrix(h.h, ctypes.c_void_p(A.data_ptr()), n, n, 0, n, _capi.MEM_DEVICE))
    v = np.random.default_rng(1).standard_normal(n)
    y = np.empty(n)
    _capi.check(h.h, h.lib.ccqp_gemv(h.h, _ptr(v), _ptr(y), _capi.MEM_HOST))
    ref = LowRankMatrix(d, u, z, True).dot(v)
    scale = np.abs(d) * np.abs(v) + np.abs(u) * np.abs(u).dot(np.abs(v)) + np.abs(z) * np.abs(z).dot(np.abs(v))
    err = np.max(np.abs(y - ref) / scale)
    print("[trajectories] tiling %s: max |y - Av| / |A||v| = %.3g" % (name, err))
    assert err < 1e-14, err
    t = _assert_tiling(h, n, cw=cw, sw=sw)
    print("[trajectories] tiling %s: %s" % (name, t))
    assert _expected_branch(name, t), t
    h.close()
    # a short SPG trajectory on the same matrix
    xs = 1.0 - 4.0 * rng.random(n)
    b = -LowRankMatrix(d, u, z, True).dot(xs)
    tab = pr.box_table(n)
    uni = pr.spg_uniforms(5, 16)
    run = DenseRun(lambda hh: (_capi.check(hh.h, hh.lib.ccqp_set_matrix(hh.h, ctypes.c_void_p(A.data_ptr()), n, n, 0, n,
                                                                        _capi.MEM_DEVICE)), A), tab, n, b, uniforms=uni)
    _assert_tiling(run.h, n, cw=cw, sw=sw)
    sw_ = Sweep("tiling " + name)
    prob = [dict(A_hp=LowRankMatrix(d, u, z, True), A_plain=LowRankMatrix(d, u, z, False), b=b, blocks=tab.blocks,
                 params=tab.params, uniforms=uni)]
    sw_.run(name, pr.SPG, 6, run, prob)
    run.close()
    sw_.finish()
    del A
    torch.cuda.empty_cache()
