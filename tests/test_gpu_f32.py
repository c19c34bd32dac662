"""Dense Hessians stored as float32 (ccqp_set_matrix_f32, csrc/dense_f32.cu).

The reference's only use of A is A.dot(v) (solvers.py:133); NumPy widens a float32 A exactly and runs the product in
float64.  The fp32 kernels stream A at 4 bytes per entry, widen every entry in a register and keep the fp64 loop's
summation order, so everything here is checked BIT FOR BIT against the same call on A.astype(np.float64): the mat-vec
hook on both loops, every tiling branch and both memtypes, whole solves of all seven solvers, host / pinned / device
inputs, the pipelined stream and the emulated ranks of a sharded solve."""
import ctypes

import numpy as np
import pytest

import problems as pr
from ccqppy_b200 import _capi
from emulated import EmulatedBox
from helpers import make_solver, op_from_table
from oracle import ccqp_oracle as orc

pytestmark = pytest.mark.gpu

GEMV_N = [1, 3, 5, 127, 128, 129, 1000, 2047, 2048, 2049, 8191, 8192, 8193, 20000]


def _bits_equal(x, y):
    x, y = (np.ascontiguousarray(v.cpu().numpy() if hasattr(v, "cpu") else v, dtype=np.float64) for v in (x, y))
    return x.shape == y.shape and np.array_equal(x.view(np.int64), y.view(np.int64))


def _same_scalar(a, b):
    return a == b or (np.isnan(a) and np.isnan(b))


def _gemv(h, set_matrix, v, memtype):
    """y = A v through the C ABI after `set_matrix(h)`; v / y NumPy (host) or torch (device)."""
    set_matrix(h)
    if memtype == 0:
        y = np.empty(v.shape[0])
        _capi.check(h.h, h.lib.ccqp_gemv(h.h, ctypes.c_void_p(v.ctypes.data), ctypes.c_void_p(y.ctypes.data), 0))
        return y
    import torch
    y = torch.empty_like(v)
    _capi.check(h.h, h.lib.ccqp_gemv(h.h, ctypes.c_void_p(v.data_ptr()), ctypes.c_void_p(y.data_ptr()), 1))
    torch.cuda.synchronize()
    return y.cpu().numpy()


def _set64(ptr, n, lda, mem):
    return lambda h: _capi.check(h.h, h.lib.ccqp_set_matrix(h.h, ctypes.c_void_p(ptr), n, lda, 0, n, mem))


def _set32(ptr, n, lda, mem):
    return lambda h: _capi.check(h.h, h.lib.ccqp_set_matrix_f32(h.h, ctypes.c_void_p(ptr), n, lda, 0, n, mem))


@pytest.mark.parametrize("n", GEMV_N)
def test_gemv_f32_equals_widened_gemv(n):
    """Host and device memtype; device: the vector loop (rows 16 / 32-byte aligned, n % 4 == 0) and the scalar loop
    (odd n, and an fp32 view at a 4-byte offset against an fp64 view at an 8-byte offset)."""
    import torch
    rng = np.random.default_rng(n)
    A32 = rng.standard_normal((n, n)).astype(np.float32)
    A64 = A32.astype(np.float64)
    v = rng.standard_normal(n)
    h = _capi.Handle()
    y32 = _gemv(h, _set32(A32.ctypes.data, n, n, 0), v, 0)
    assert h.upload_info() == (4 * n * n, False)
    y64 = _gemv(h, _set64(A64.ctypes.data, n, n, 0), v, 0)
    assert _bits_equal(y32, y64), n
    ref = A32.dot(v)                                     # NumPy: the same widened products, its own summation order
    scale = np.abs(A64) @ np.abs(v)
    assert np.max(np.abs(y32 - ref) / scale) < 4e-16 * max(4, np.log2(n + 1))
    vd = torch.from_numpy(v).cuda()
    d32, d64 = torch.from_numpy(A32).cuda(), torch.from_numpy(A64).cuda()
    y32 = _gemv(h, _set32(d32.data_ptr(), n, n, 1), vd, 1)
    assert h.upload_info() == (0, False)
    y64 = _gemv(h, _set64(d64.data_ptr(), n, n, 1), vd, 1)
    assert _bits_equal(y32, y64), n
    if n % 4 == 0:
        assert _bits_equal(y32, _gemv(h, _set32(A32.ctypes.data, n, n, 0), v, 0))     # padded host upload: same loop
    o32 = torch.empty(n * n + 1, dtype=torch.float32, device="cuda")
    o64 = torch.empty(n * n + 1, dtype=torch.float64, device="cuda")
    o32[1:] = d32.reshape(-1)
    o64[1:] = d64.reshape(-1)
    y32 = _gemv(h, _set32(o32.data_ptr() + 4, n, n, 1), vd, 1)
    y64 = _gemv(h, _set64(o64.data_ptr() + 8, n, n, 1), vd, 1)
    assert _bits_equal(y32, y64), n
    assert np.max(np.abs(y32 - ref) / scale) < 4e-16 * max(4, np.log2(n + 1))
    h.close()


@pytest.mark.parametrize("n, cw, sw, accum", [(20000, 2048, 512, False), (20000, 1024, 1024, False), (8193, 8192, 128, False),
                                              (24000, 128, 128, True)])
def test_gemv_f32_tilings(n, cw, sw, accum, monkeypatch):
    """Multi-panel tilings and the branch that adds the panels' partial sums up in panel order (very wide rows)."""
    import torch
    monkeypatch.setenv("CCQP_CW", str(cw))
    monkeypatch.setenv("CCQP_SW", str(sw))
    g = torch.Generator(device="cuda").manual_seed(n)
    d32 = torch.randn((n, n), generator=g, device="cuda", dtype=torch.float32)
    d64 = d32.double()
    vd = torch.randn(n, generator=g, device="cuda", dtype=torch.float64)
    h = _capi.Handle()
    y32 = _gemv(h, _set32(d32.data_ptr(), n, n, 1), vd, 1)
    smem32 = h.info()["dense_smem_bytes"]
    y64 = _gemv(h, _set64(d64.data_ptr(), n, n, 1), vd, 1)
    assert smem32 == h.info()["dense_smem_bytes"]            # the same tiling
    if accum:                                                 # one partial-sum slot per (row, segment of a panel)
        assert smem32 < 16 * 1024, smem32
    assert _bits_equal(y32, y64)
    ref = (d64 @ vd).cpu().numpy()
    scale = (d64.abs() @ vd.abs()).cpu().numpy()
    assert np.max(np.abs(y32 - ref) / scale) < 1e-14
    h.close()


def test_set_matrix_f32_rejects_bad_arguments():
    h = _capi.Handle()
    A = np.ones((4, 4), dtype=np.float32)
    p = ctypes.c_void_p(A.ctypes.data)
    assert h.lib.ccqp_set_matrix_f32(h.h, None, 4, 4, 0, 4, 0) == 1           # CCQP_ERR_INVALID_ARG
    assert h.lib.ccqp_set_matrix_f32(h.h, p, 4, 3, 0, 4, 0) == 1              # lda < n
    assert h.lib.ccqp_set_matrix_f32(h.h, p, 4, 4, 2, 3, 0) == 1              # rows beyond n
    assert h.lib.ccqp_set_matrix_f32(h.h, p, 4, 4, 0, 4, 0) == 0
    h.close()


# ---- whole solves -------------------------------------------------------------------------------------------------
def _solve(solver, A, b, op, x0=None, tol=1e-6, max_mv=2000, step=0.01, **kw):
    s = make_solver(solver, tol, max_mv, step)
    uni = pr.spg_uniforms(3, int(max_mv)) if solver == pr.SPG else None
    s.solve(A, b, x0=x0, convex_proj_op=op, uniforms=uni, **kw)
    return s


def _assert_same_solve(s1, s2, what):
    assert _bits_equal(s1.solution, s2.solution), what
    assert _same_scalar(s1.solution_residual, s2.solution_residual), what
    assert s1.solution_num_matrix_vector_multiplications == s2.solution_num_matrix_vector_multiplications, what
    assert s1.solution_converged == s2.solution_converged, what
    assert s1.solution_gemv_count == s2.solution_gemv_count, what


def test_problem_suite_with_float32_A():
    from ccqppy_b200 import problem_suite
    for cls in ("UnconstrainedSPD1", "UnconstrainedSPD2", "BoxConstrainedSPD", "ThinBoxConstrainedSPD", "ActiveBoxConstrainedSPD"):
        p = getattr(problem_suite, cls)()
        A32 = np.asarray(p.A, dtype=np.float32)
        for solver in range(7):
            s32 = _solve(solver, A32, p.b, p.convex_proj_op, tol=1e-8, max_mv=10000, step=0.1)
            s64 = _solve(solver, A32.astype(np.float64), p.b, p.convex_proj_op, tol=1e-8, max_mv=10000, step=0.1)
            _assert_same_solve(s32, s64, (cls, solver))
            assert s32.solution_converged and np.linalg.norm(s32.solution - p.exact_solution) < 1e-5


SOLVE_CASES = [("shift_box_4096", pr.shift_problem, pr.box_table, 4096, False, np.inf),
               ("shift_mixed_1023_x0", pr.shift_problem, pr.mixed_table, 1023, True, np.inf),
               ("wishart_sphere3_2050", pr.wishart_problem, pr.sphere3_table, 2050, False, np.inf),
               ("shift_box_3001_maxmv", pr.shift_problem, pr.box_table, 3001, True, 9)]


@pytest.mark.parametrize("case", SOLVE_CASES, ids=[c[0] for c in SOLVE_CASES])
def test_solves_equal_widened_solves(case):
    name, gen, table, n, with_x0, max_mv = case
    A, b = gen(n, 11)
    A32 = A.astype(np.float32)
    A64 = A32.astype(np.float64)
    op = op_from_table(table(n))
    x0 = 0.5 * np.random.default_rng(4).standard_normal(n) if with_x0 else None
    step = 1.0 / np.abs(A64).sum(axis=1).max()
    limit = 3000 if np.isinf(max_mv) else max_mv
    stopped = 0
    for solver in range(7):
        s32 = _solve(solver, A32, b, op, x0=x0, tol=1e-6, max_mv=limit, step=step)
        s64 = _solve(solver, A64, b, op, x0=x0, tol=1e-6, max_mv=limit, step=step)
        _assert_same_solve(s32, s64, (name, solver))
        stopped += not s32.solution_converged
    assert stopped > 0 or np.isinf(max_mv)                   # the max_mv-limited case does stop solves


def test_solves_match_oracle_on_the_float32_matrix():
    n = 1023
    A, b = pr.shift_problem(n, 12)
    A32 = A.astype(np.float32)
    tab = pr.mixed_table(n)
    op = op_from_table(tab)
    step = 1.0 / np.abs(A32.astype(np.float64)).sum(axis=1).max()
    for solver in range(7):
        s = _solve(solver, A32, b, op, tol=1e-6, max_mv=1500, step=step)
        o = orc.solve(solver, A32, b, blocks=tab.blocks, params=tab.params, tol=1e-6, max_mv=1500, step_size=step,
                      uniforms=pr.spg_uniforms(3, 1500) if solver == pr.SPG else None)
        assert o["mv"] == s.solution_num_matrix_vector_multiplications and o["converged"] == s.solution_converged, solver
        assert np.linalg.norm(s.solution - o["solution"]) <= 1e-9 * np.linalg.norm(o["solution"]), solver


def test_cuda_float32_matrix_is_used_in_place():
    import torch
    n = 16384
    g = torch.Generator(device="cuda").manual_seed(3)
    G = torch.randn((n, n), generator=g, device="cuda", dtype=torch.float32)
    A = (G @ G.T) / n
    A.diagonal().add_(1.0)
    del G
    b = torch.randn(n, generator=g, device="cuda", dtype=torch.float64)
    op = op_from_table(pr.box_table(n))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    s32 = _solve(pr.BBPGD, A, b, op, tol=1e-6, max_mv=300)
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    assert extra < 0.01 * 4 * n * n, extra
    assert _capi.default_handle(A.device.index).upload_info() == (0, False)
    assert s32.solution_hbm_bytes == s32.solution_gemv_count * (4.0 * n * n + 16.0 * n)
    s64 = _solve(pr.BBPGD, A.double(), b, op, tol=1e-6, max_mv=300)
    _assert_same_solve(s32, s64, "in place")


def test_host_float32_inputs():
    """NumPy, pageable and pinned torch float32: 4 n^2 bytes cross PCIe, results equal the widened solve."""
    import torch
    n = 2048
    A, b = pr.shift_problem(n, 13)
    A32 = A.astype(np.float32)
    op = op_from_table(pr.mixed_table(n))
    for solver in (pr.SPG, pr.MPRGP):
        s64 = _solve(solver, A32.astype(np.float64), b, op)
        for A_in in (A32, torch.from_numpy(A32), torch.from_numpy(A32).pin_memory()):
            s32 = _solve(solver, A_in, b, op)
            assert _capi.default_handle(-1).upload_info() == (4 * n * n, False)
            _assert_same_solve(s32, s64, (solver, type(A_in)))
            assert s32.solution_hbm_bytes == s32.solution_gemv_count * (4.0 * n * n + 16.0 * n)


def test_pipeline_of_pinned_float32_problems():
    import torch
    from ccqppy_b200.pipeline import SolvePipeline
    n = 2048
    op = op_from_table(pr.box_table(n))
    problems = []
    for k in range(4):
        A, b = pr.shift_problem(n, 20 + k)
        problems.append((torch.from_numpy(A.astype(np.float32)).pin_memory(), b))
    uni = pr.spg_uniforms(5, 2000)
    pipe = SolvePipeline(make_solver(pr.SPG, 1e-7, 2000), depth=2)
    for A, b in problems:
        pipe.submit(A, b, convex_proj_op=op, uniforms=uni)
    out = pipe.results()
    pipe.close()
    for (A, b), r in zip(problems, out):
        s = make_solver(pr.SPG, 1e-7, 2000)
        s.solve(A, b, convex_proj_op=op, uniforms=uni)
        assert r.solution_hbm_bytes == r.solution_gemv_count * (4.0 * n * n + 16.0 * n)
        _assert_same_solve(r, s, "pipeline")


class _F32Box(EmulatedBox):
    """EmulatedBox whose ranks hold float32 row shards (ccqp_set_matrix_f32) instead of the widened ones."""

    def __init__(self, A32, op, world):
        super().__init__(A32, op, world)
        for r, h in enumerate(self.handles):
            r0, r1 = self.ranges[r]
            shard = np.ascontiguousarray(A32[r0:r1])
            self.keep.append(shard)
            h.set_matrix_f32(shard, self.n, r0, r1 - r0)


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("n, table", [(3050, pr.box_table), (1200, pr.mixed_table)], ids=["box_uneven", "mixed"])
def test_emulated_ranks_with_float32_shards(n, table, world):
    A, b = pr.shift_problem(n, 5)
    A32 = A.astype(np.float32)
    op = op_from_table(table(n))
    step = 1.0 / np.abs(A32.astype(np.float64)).sum(axis=1).max()
    box32, box64 = _F32Box(A32, op, world), EmulatedBox(A32.astype(np.float64), op, world)
    for solver in range(7):
        uni = pr.spg_uniforms(2, 1500)
        r32 = box32.solve(make_solver(solver, 1e-6, 1500, step), b, uniforms=uni)
        r64 = box64.solve(make_solver(solver, 1e-6, 1500, step), b, uniforms=uni)
        for r in range(world):
            assert _bits_equal(r32[r]["solution"], r32[0]["solution"]), (solver, r)
            assert _bits_equal(r32[r]["solution"], r64[r]["solution"]), (solver, r)
            assert r32[r]["mv"] == r64[r]["mv"] and r32[r]["converged"] == r64[r]["converged"], (solver, r)
            assert _same_scalar(r32[r]["residual"], r64[r]["residual"]), (solver, r)
    box32.close()
    box64.close()


def test_routes_that_still_widen():
    """symmetric=True, solve_batched and scipy.sparse take a float32 A through today's float64 path: same results."""
    import scipy.sparse as sp
    n = 2304
    A, b = pr.shift_problem(n, 14)
    A = 0.5 * (A + A.T)
    A32 = A.astype(np.float32)
    op = op_from_table(pr.box_table(n))
    _assert_same_solve(_solve(pr.BBPGD, A32, b, op, symmetric=True),
                       _solve(pr.BBPGD, A32.astype(np.float64), b, op, symmetric=True), "symmetric")
    batch, nb = 16, 48
    Ab = np.empty((batch, nb, nb), dtype=np.float32)
    bb = np.empty((batch, nb))
    for i in range(batch):
        Ai, bb[i] = pr.shift_problem(nb, i)
        Ab[i] = Ai
    lb, ub = -np.ones((batch, nb)), np.ones((batch, nb))
    s32 = make_solver(pr.SPG, 1e-8, 3000).solve_batched(Ab, bb, lb, ub)
    s64 = make_solver(pr.SPG, 1e-8, 3000).solve_batched(Ab.astype(np.float64), bb, lb, ub)
    assert _bits_equal(s32.solution, s64.solution)
    assert np.array_equal(s32.solution_num_matrix_vector_multiplications, s64.solution_num_matrix_vector_multiplications)
    S, bs = pr.sparse_problem(400, 3)
    S32 = S.astype(np.float32)
    opS = op_from_table(pr.box_table(400))
    _assert_same_solve(_solve(pr.MPRGP, S32, bs, opS), _solve(pr.MPRGP, S32.astype(np.float64), bs, opS), "sparse")


def test_sharded_solver_with_host_float32_A():
    """ShardedSolver (one rank) from a NumPy float32 A and a CPU float32 tensor, and set_matrix with a NumPy float32
    shard: float32 shards on the device, the bits of the solve of the widened matrix."""
    import torch
    from ccqppy_b200.dist import ShardedSolver
    n = 1500
    A, b = pr.shift_problem(n, 9)
    A32 = A.astype(np.float32)
    op = op_from_table(pr.mixed_table(n))
    uni = pr.spg_uniforms(6, 1500)
    out = {}
    for label, A_in in (("fp64", A32.astype(np.float64)), ("numpy_f32", A32), ("torch_cpu_f32", torch.from_numpy(A32))):
        runner = ShardedSolver(make_solver(pr.SPG, 1e-7, 1500), A_in, op, rank=0, world=1)
        assert runner.shard.is_cuda and runner.shard.dtype == (torch.float64 if label == "fp64" else torch.float32)
        out[label] = runner.solve(b, uniforms=uni)
        if label == "numpy_f32":
            runner.set_matrix(A32)
            out["set_matrix_f32"] = runner.solve(b, uniforms=uni)
        runner.close()
    for label, r in out.items():
        _assert_same_solve(r, out["fp64"], label)
