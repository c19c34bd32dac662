"""Batched solves on float32 Hessians (the `_f32` entry points) on the GPU: every solver, launch shape, load path and
feasible-set form returns the bits of the same call on the widened batch; the oracle agrees; the C twins report the fp64
functions' status codes."""
import ctypes

import numpy as np
import pytest

import problems as pr
from helpers import make_solver, op_from_table
from oracle import ccqp_oracle as orc
from ccqppy_b200 import _capi

pytestmark = pytest.mark.gpu

ALL = [pr.PGD, pr.APGD, pr.APGD_AR, pr.BBPGD, pr.BBPGDF, pr.SPG, pr.MPRGP]
TABLE_SOLVERS = [pr.PGD, pr.APGD, pr.APGD_AR, pr.BBPGD, pr.BBPGDF, pr.SPG]
K = 512


def batch32(batch, n, seed0=0, mu=1.0, symmetric=False):
    """float32 Hessians (rounded from the shift problems), fp64 b and boxes."""
    A = np.empty((batch, n, n), dtype=np.float32)
    b = np.empty((batch, n))
    for i in range(batch):
        Ai, b[i] = pr.shift_problem(n, seed0 + i, mu)
        A[i] = Ai
    if symmetric:
        A = (0.5 * (A + A.transpose(0, 2, 1))).astype(np.float32)
    rng = np.random.default_rng(1234 + seed0)
    lb = -1.0 - 0.2 * rng.random((batch, n))
    ub = 1.0 + 0.2 * rng.random((batch, n))
    return A, b, lb, ub


def run(solver, A, *args, tol=1e-8, max_mv=5000, **kw):
    s = make_solver(solver, tol, max_mv, 0.1)
    if solver == pr.SPG:
        kw.setdefault("seeds", np.arange(A.shape[0]))
        kw.setdefault("n_uniforms", K)
    return s.solve_batched(A, *args, **kw)


def host(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def assert_same(s32, s64):
    assert np.array_equal(host(s32.solution), host(s64.solution))
    assert np.array_equal(s32.solution_residual, s64.solution_residual, equal_nan=True)
    assert np.array_equal(s32.solution_num_matrix_vector_multiplications, s64.solution_num_matrix_vector_multiplications)
    assert np.array_equal(s32.solution_converged, s64.solution_converged)
    assert np.array_equal(s32.solution_status, s64.solution_status)
    r32, r64 = s32._batched_records, s64._batched_records
    for f in ("gemv", "it", "draws"):
        assert np.array_equal(r32[f], r64[f]), f


@pytest.mark.parametrize("solver", ALL)
@pytest.mark.parametrize("n", [64, 63, 62, 36, 17, 5, 128, 126, 65])
def test_box_bits_equal_the_widened_call(solver, n):
    """n = 64, 36: TMA-staged float tile; 62: staged in fp64, not in fp32 (4 n % 16 != 0); odd n: global loads; n > 64:
    the 256-thread shape."""
    batch = 40 if solver != pr.MPRGP else 24
    tol = 1e-6 if solver in (pr.APGD, pr.APGD_AR) else 1e-8
    A, b, lb, ub = batch32(batch, n, seed0=10 * n)
    s32 = run(solver, A, b, lb, ub, tol=tol)
    s64 = run(solver, A.astype(np.float64), b, lb, ub, tol=tol)
    assert_same(s32, s64)
    if solver != pr.MPRGP:          # (MPRGP at tol 1e-8 runs into max_mv on these problems, fp64 and fp32 alike)
        assert s32.solution_converged.mean() >= 0.9
    assert s64.solution_hbm_bytes - s32.solution_hbm_bytes == 4.0 * n * n * batch


@pytest.mark.parametrize("solver", [pr.PGD, pr.BBPGD, pr.BBPGDF, pr.SPG])
@pytest.mark.parametrize("n", [64, 62, 17])
def test_symmetric_bits_equal_the_widened_call(solver, n):
    """The one-warp-per-problem kernels read only the upper block triangle: poisoned with NaN below it, the float32 batch
    still gives the bits of the widened clean batch."""
    batch = 64
    A, b, lb, ub = batch32(batch, n, seed0=500 + n, symmetric=True)
    poisoned = A.copy()
    rr, cc = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    poisoned[:, cc < 8 * (rr // 8)] = np.nan
    s32 = run(solver, poisoned, b, lb, ub, symmetric=True)
    s64 = run(solver, A.astype(np.float64), b, lb, ub, symmetric=True)
    assert_same(s32, s64)
    assert s32.solution_converged.all()
    tri = sum(n - 8 * (i // 8) for i in range(n))
    assert s64.solution_hbm_bytes - s32.solution_hbm_bytes == 4.0 * tri * batch


def table_batch(struct, n, batch, seed):
    from test_gpu_batched_tables import tables
    tabs = tables(struct, n, batch, seed)
    A, b, _, _ = batch32(batch, n, seed0=seed)
    P = np.stack([t.params for t in tabs])
    return A, b, tabs, P


@pytest.mark.parametrize("solver", TABLE_SOLVERS)
@pytest.mark.parametrize("struct", ["sphere3", "mixed", "soc3"])
@pytest.mark.parametrize("n", [63, 126])
def test_tables_bits_equal_the_widened_call(solver, struct, n):
    batch = 24
    A, b, tabs, P = table_batch(struct, n, batch, seed=7 * n)
    op = op_from_table(tabs[0])
    tol = 1e-6 if solver in (pr.APGD, pr.APGD_AR) else 1e-8
    # one operator shared by the batch
    assert_same(run(solver, A, b, convex_proj_op=op, tol=tol), run(solver, A.astype(np.float64), b, convex_proj_op=op, tol=tol))
    # one block structure, per-problem parameters
    assert_same(run(solver, A, b, convex_proj_op=op, op_params=P, tol=tol),
                run(solver, A.astype(np.float64), b, convex_proj_op=op, op_params=P, tol=tol))


def test_x0_and_mv_limit():
    batch, n = 48, 64
    A, b, lb, ub = batch32(batch, n, seed0=900, mu=0.01)
    x0 = 0.5 * np.random.default_rng(3).standard_normal((batch, n))
    for solver in ALL:
        assert_same(run(solver, A, b, lb, ub, x0=x0), run(solver, A.astype(np.float64), b, lb, ub, x0=x0))
        s32 = run(solver, A, b, lb, ub, tol=1e-14, max_mv=9)
        assert_same(s32, run(solver, A.astype(np.float64), b, lb, ub, tol=1e-14, max_mv=9))
        assert not s32.solution_converged.any()


@pytest.mark.parametrize("n", [64, 36, 63])
def test_every_load_path_returns_the_same_bits(n):
    """Host NumPy, pinned host, a 16-byte aligned CUDA tensor, one 4 bytes past a 16-byte boundary (element-wise loads) and
    a non-contiguous CUDA tensor (one contiguous copy)."""
    import torch
    batch = 96
    A, b, lb, ub = batch32(batch, n, seed0=77)
    ref = run(pr.BBPGD, A, b, lb, ub)
    pinned = torch.from_numpy(A).pin_memory()
    bufs = [torch.empty(A.size + 8, dtype=torch.float32, device="cuda") for _ in range(2)]
    base = [(16 - buf.data_ptr() % 16) % 16 // 4 for buf in bufs]
    aligned = bufs[0][base[0]:base[0] + A.size].view(A.shape)
    shifted = bufs[1][base[1] + 1:base[1] + 1 + A.size].view(A.shape)
    assert aligned.data_ptr() % 16 == 0 and shifted.data_ptr() % 16 == 4
    aligned.copy_(torch.from_numpy(A))
    shifted.copy_(torch.from_numpy(A))
    strided = torch.from_numpy(A.transpose(0, 2, 1).copy()).cuda().transpose(1, 2)
    assert not strided.is_contiguous()
    dev = [torch.from_numpy(v).cuda() for v in (b, lb, ub)]
    assert_same(run(pr.BBPGD, pinned, b, lb, ub), ref)
    for a in (aligned, shifted, strided):
        assert_same(run(pr.BBPGD, a, *dev), ref)
    # a contiguous CUDA tensor is read in place, whatever its alignment: no float32 or float64 copy of it is made (the
    # peak grows by the solution array only)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    run(pr.BBPGD, shifted, *dev)
    assert torch.cuda.max_memory_allocated() - before <= batch * n * 8 + 4096


def test_oracle_parity_on_float32_hessians():
    """The reference's A.dot(v) with a float32 A widens to float64: the oracle given the float32 A agrees, with the
    acceptance of test_gpu_batched.test_batched_matches_oracle."""
    batch, n = 24, 36
    A, b, lb, ub = batch32(batch, n, seed0=4242)
    for solver in (pr.PGD, pr.BBPGD, pr.SPG, pr.MPRGP):
        s = run(solver, A, b, lb, ub)
        same = 0
        m = 12 if solver == pr.MPRGP else batch       # the oracle's MPRGP is slow (per-element Python loops)
        for i in range(m):
            tab = pr.Table().add(pr.BOX, n, lb[i], ub[i])
            o = orc.solve(solver, A[i], b[i], blocks=tab.blocks, params=tab.params, tol=1e-8, max_mv=5000, step_size=0.1,
                          uniforms=pr.spg_uniforms(i, K))
            assert bool(s.solution_converged[i]) == o["converged"]
            mv = int(s.solution_num_matrix_vector_multiplications[i])
            scale = max(np.linalg.norm(o["solution"]), 1e-300)
            if mv == o["mv"]:
                same += 1
                assert np.linalg.norm(s.solution[i] - o["solution"]) <= 1e-9 * scale
            else:
                assert abs(mv - o["mv"]) <= max(2, round(0.1 * o["mv"])), (i, mv, o["mv"])
                assert np.linalg.norm(s.solution[i] - o["solution"]) <= 1e-5 * scale
        assert same >= 0.9 * m, (solver, same)


def test_scale_65536_problems_from_a_device_float32_tensor():
    import torch
    batch, n = 65536, 64
    g = torch.Generator(device="cuda").manual_seed(0)
    G = torch.randn((batch, n, n), generator=g, device="cuda", dtype=torch.float32)
    A = G @ G.transpose(1, 2) / n + torch.eye(n, device="cuda", dtype=torch.float32)
    del G
    xs = 1 - 4 * torch.rand((batch, n), generator=g, device="cuda", dtype=torch.float64)
    b = -(A.double() @ xs.unsqueeze(-1)).squeeze(-1)
    lb, ub = -torch.ones_like(b), torch.ones_like(b)
    s32 = run(pr.BBPGD, A, b, lb, ub)
    s64 = run(pr.BBPGD, A.double(), b, lb, ub)
    assert_same(s32, s64)
    assert s32.solution_converged.mean() > 0.99
    assert s64.solution_hbm_bytes - s32.solution_hbm_bytes == 4.0 * n * n * batch


def _status(name, A, n, solver, table=None, batch=4):
    """Status of one call of a batched C entry point on device arrays."""
    import torch
    h = _capi.default_handle(0)
    lib = h.lib
    d = lambda *shape: torch.zeros(shape, dtype=torch.float64, device="cuda")     # noqa: E731
    b, x, lo, hi = d(batch, n), d(batch, n), d(batch, n) - 1, d(batch, n) + 1
    prm = make_solver(solver, 1e-8, 100)._params()
    p = lambda t: ctypes.c_void_p(t.data_ptr())       # noqa: E731
    res = (_capi.Result * batch)()
    summ = _capi.Result()
    uni = d(batch, 8)
    if "table" in name:
        blocks = table
        P = d(batch, 2 * n)
        return getattr(lib, name)(h.h, solver, ctypes.byref(prm), batch, n, p(A), p(b), None, blocks.ptr, len(blocks), p(P),
                                  2 * n, p(uni), 8, p(x), _capi.MEM_DEVICE, res, ctypes.byref(summ))
    return getattr(lib, name)(h.h, solver, ctypes.byref(prm), batch, n, p(A), p(b), None, p(lo), p(hi), p(uni), 8, p(x),
                              _capi.MEM_DEVICE, res, ctypes.byref(summ))


def test_c_twins_return_the_fp64_status_codes():
    import torch
    for n in (16, 130):
        A64 = torch.eye(n, dtype=torch.float64, device="cuda").repeat(4, 1, 1).contiguous()
        A32 = A64.float()
        good = _capi.make_blocks([(_capi.BOX, 0, n, 0)])
        short = _capi.make_blocks([(_capi.BOX, 0, n - 1, 0)])          # does not cover [0, n)
        cases = [("ccqp_solve_batched", pr.BBPGD, None), ("ccqp_solve_batched_sym", pr.SPG, None),
                 ("ccqp_solve_batched_table", pr.MPRGP, good), ("ccqp_solve_batched_tables", pr.MPRGP, good),
                 ("ccqp_solve_batched_table", pr.BBPGD, short), ("ccqp_solve_batched_tables", pr.BBPGD, short)]
        for name, solver, tab in cases:
            st64 = _status(name, A64, n, solver, tab)
            st32 = _status(name + "_f32", A32, n, solver, tab)
            assert st64 == st32, (name, n, solver, st64, st32)
            # n > 128 and MPRGP with a table: CCQP_ERR_UNSUPPORTED; a table that does not cover [0, n): CCQP_ERR_INVALID_ARG
            assert st64 == (4 if n > 128 or solver == pr.MPRGP else 1 if tab is short else 0), (name, n, solver, st64)
        torch.cuda.synchronize()
