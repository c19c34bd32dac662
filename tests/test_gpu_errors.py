"""Error behaviour of the boundary on a real device: status codes instead of exceptions across the ABI,
the two exceptions the reference itself can raise, and the edge cases of SURVEY.md section 9."""
import ctypes

import numpy as np
import pytest

import problems as pr
from helpers import op_from_table, make_solver
from ccqppy_b200 import _capi, solvers, solution_spaces as ss

pytestmark = pytest.mark.gpu
P = lambda a: ctypes.c_void_p(a.ctypes.data)


def test_status_codes_of_the_c_abi():
    h = _capi.Handle()
    lib = h.lib
    n = 8
    A, b = pr.shift_problem(n, 0)
    x = np.empty(n)
    prm, res = make_solver(pr.BBPGD, 1e-6, 100)._params(), _capi.Result()
    solve = lambda: lib.ccqp_solve(h.h, _capi.BBPGD, ctypes.byref(prm), P(b), None, None, 0, P(x), _capi.MEM_HOST, ctypes.byref(res))
    assert solve() == 5                                                   # CCQP_ERR_NOT_READY: no matrix, no projection
    assert lib.ccqp_set_matrix(h.h, P(A), n, n - 1, 0, n, _capi.MEM_HOST) == 1          # lda < n
    assert lib.ccqp_set_matrix(h.h, P(A), n, n, 4, n, _capi.MEM_HOST) == 1              # rows outside the matrix
    assert lib.ccqp_set_matrix(h.h, None, n, n, 0, n, _capi.MEM_HOST) == 1
    assert lib.ccqp_set_matrix(h.h, P(A), n, n, 0, n, _capi.MEM_HOST) == 0
    assert solve() == 5                                                   # still no projection
    blocks = _capi.make_blocks([(_capi.BOX, 0, n - 1, 0)])
    par = np.concatenate([-np.ones(n), np.ones(n)])
    assert lib.ccqp_set_projection(h.h, blocks.ptr, 1, P(par), par.size) == 0
    assert solve() == 1                                                   # table covers n-1 unknowns, matrix has n
    gap = _capi.make_blocks([(_capi.BOX, 0, 4, 0), (_capi.BOX, 5, 3, 8)])
    assert lib.ccqp_set_projection(h.h, gap.ptr, 2, P(par), par.size) == 1              # blocks must tile [0, n)
    short = _capi.make_blocks([(_capi.BOX, 0, n, 4)])
    assert lib.ccqp_set_projection(h.h, short.ptr, 1, P(par), par.size) == 1            # parameters run past the array
    unknown = _capi.make_blocks([(9, 0, n, 0)])
    assert lib.ccqp_set_projection(h.h, unknown.ptr, 1, P(par), par.size) == 1
    good = _capi.make_blocks([(_capi.BOX, 0, n, 0)])
    assert lib.ccqp_set_projection(h.h, good.ptr, 1, P(par), par.size) == 0
    assert solve() == 0 and res.converged == 1
    assert lib.ccqp_solve(h.h, 7, ctypes.byref(prm), P(b), None, None, 0, P(x), _capi.MEM_HOST, ctypes.byref(res)) == 1   # unknown solver
    assert lib.ccqp_solve_wait(h.h, ctypes.byref(res)) == 5              # nothing in flight
    A_shard = np.ascontiguousarray(A[:4])
    assert lib.ccqp_set_matrix(h.h, P(A_shard), n, n, 0, 4, _capi.MEM_HOST) == 0
    assert solve() == 4                                                   # CCQP_ERR_UNSUPPORTED: a row shard needs ccqp_comm_attach
    assert lib.ccqp_status_string(4) == b"unsupported request" and lib.ccqp_status_string(99) == b"unknown status"
    big = np.zeros((3, 129, 129))
    v = np.zeros((3, 129))
    assert lib.ccqp_solve_batched(h.h, _capi.BBPGD, ctypes.byref(prm), 3, 129, P(big), P(v), None, P(v), P(v), None, 0, P(v),
                                  _capi.MEM_HOST, None, None) == 4        # n > 128
    assert lib.ccqp_solve_batched(h.h, 7, ctypes.byref(prm), 3, 8, P(big), P(v), None, P(v), P(v), None, 0, P(v),
                                  _capi.MEM_HOST, None, None) == 1        # unknown solver
    h.close()


def test_spg_uniform_stream_and_range_errors():
    n = 40
    A, b = pr.shift_problem(n, 1)
    op = ss.BoxProjOp(n)
    s = solvers.CCQPSolverSPG(1e-12, 5000)
    s.quiet = True
    with pytest.raises(_capi.CCQPError) as e:                             # the stream runs dry: a status, not a hang
        s.solve(A, b, convex_proj_op=op, uniforms=np.random.RandomState(0).random_sample(3))
    assert e.value.status == _capi.ERR_UNIFORMS_EXHAUSTED
    # np.random.uniform(lo, nan) raises OverflowError in the reference (solvers.py:959): a NaN problem does the same here
    bn = b.copy()
    bn[0] = np.nan
    with pytest.raises(OverflowError):
        s.solve(A, bn, convex_proj_op=op)


def test_mv_limit_edge_cases_do_not_raise():
    """SURVEY Q16: where the reference would die with NameError (limit hit before the first residual exists) the
    result is residual = NaN, converged = False.  test_gpu_trajectories.py compares every such stop with the oracle."""
    n = 30
    A, b = pr.shift_problem(n, 2)
    tab = pr.box_table(n)
    for solver, limit in ((pr.APGD, 2), (pr.SPG, 3), (pr.APGD_AR, 2)):
        s = make_solver(solver, 1e-9, limit)
        s.solve(A, b, convex_proj_op=op_from_table(tab), uniforms=pr.spg_uniforms(0, 10))
        assert not s.solution_converged and np.isnan(s.solution_residual)
        assert np.all(np.isfinite(np.asarray(s.solution)))
    for solver in (pr.PGD, pr.BBPGD, pr.MPRGP):
        s = make_solver(solver, 1e-9, 1)                                   # the limit is reached by the very first product
        s.solve(A, b, convex_proj_op=op_from_table(tab))
        assert not s.solution_converged


def test_infinite_bounds_mean_no_bound():
    """SURVEY Q10: the reference's mask-multiply projections turn infinite bounds into NaN; here they are 'no bound'."""
    n = 50
    A, b = pr.shift_problem(n, 3)
    lo, hi = np.full(n, -np.inf), np.full(n, np.inf)
    hi[:10] = 0.25
    op = ss.BoxProjOp(n, lo, hi)
    s = make_solver(pr.BBPGD, 1e-8, 500)
    s.solve(A, b, convex_proj_op=op)
    ref = make_solver(pr.BBPGD, 1e-8, 500)
    ref.solve(A, b, convex_proj_op=ss.DisjointProjOp(ss.UpperBoundProjOp(10, hi[:10]), ss.IdentityProjOp(n - 10)))
    assert s.solution_converged and np.array_equal(np.asarray(s.solution), np.asarray(ref.solution))


def test_batched_problem_that_runs_out_of_uniforms_is_reported_not_converged():
    """ADVICE r1: a batched SPG problem that used up its uniform stream must not come back as converged."""
    batch, n = 6, 32
    A = np.empty((batch, n, n)); b = np.empty((batch, n))
    for i in range(batch):
        A[i], b[i] = pr.shift_problem(n, 40 + i, 0.05)
    lb, ub = -np.ones((batch, n)), np.ones((batch, n))
    s = make_solver(pr.SPG, 1e-12, 5000)
    with pytest.raises(_capi.CCQPError) as e:
        s.solve_batched(A, b, lb, ub, seeds=np.arange(batch), n_uniforms=3)
    assert e.value.status == _capi.ERR_UNIFORMS_EXHAUSTED
    st = s.solution_status
    assert np.any(st == _capi.ERR_UNIFORMS_EXHAUSTED)
    assert not np.any(np.asarray(s.solution_converged)[st != 0])          # status != 0  =>  not converged
    # the default stream length (max_mv samples) cannot run out
    s2 = make_solver(pr.SPG, 1e-8, 400)
    s2.solve_batched(A, b, lb, ub, seeds=np.arange(batch))
    assert np.all(s2.solution_status == 0)
    bn = b.copy()
    bn[2, 0] = np.nan
    with pytest.raises(OverflowError):                                    # np.random.uniform(lo, nan), solvers.py:959
        make_solver(pr.SPG, 1e-8, 400).solve_batched(A, bn, lb, ub, seeds=np.arange(batch))


def test_sharded_solve_without_prepare_is_refused():
    """ADVICE r1: the C-ABI refuses a sharded solve whose exchange buffer was not cleared by ccqp_comm_prepare()."""
    h = _capi.Handle()
    lib = h.lib
    n = 64
    A, b = pr.shift_problem(n, 0)
    desc = (ctypes.c_ubyte * 128)()
    assert lib.ccqp_comm_export(h.h, 0, 2, n, desc) == 0
    assert lib.ccqp_comm_prepare(h.h) == 5                                # not attached yet
    h.close()


def test_two_devices_from_one_process():
    """VERDICT r1: kernel attributes are per device.  One process solves n = 4096 (> 48 KB of dynamic shared
    memory) on device 0, then on device 1, then through a SolvePipeline bound to device 1."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    from ccqppy_b200.pipeline import SolvePipeline
    n = 4096
    A, b = pr.shift_problem(n, 3)
    op = ss.BoxProjOp(n)
    sols = []
    for dev in (0, 1):
        s = make_solver(pr.BBPGD, 1e-7, 500)
        s.solve(A, b, convex_proj_op=op, device=dev)
        assert s.solution_converged
        sols.append(np.asarray(s.solution).copy())
        Ad = torch.from_numpy(A).to("cuda:%d" % dev)
        s.solve(Ad, torch.from_numpy(b).to(Ad.device), convex_proj_op=op)
        assert np.array_equal(s.solution.cpu().numpy(), sols[-1])
    assert np.array_equal(sols[0], sols[1])
    pipe = SolvePipeline(make_solver(pr.BBPGD, 1e-7, 500), depth=2, device=1)
    for _ in range(3):
        pipe.submit(torch.from_numpy(A).pin_memory(), torch.from_numpy(b).pin_memory(), convex_proj_op=op)
    res = pipe.results()
    pipe.close()
    assert len(res) == 3 and all(np.array_equal(np.asarray(r.solution), sols[0]) for r in res)
