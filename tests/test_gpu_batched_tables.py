"""Batched solves with one block structure and per-problem operator parameters (`ccqp_solve_batched_tables`,
`solve_batched(convex_proj_op=op, op_params=P)` or a sequence of operators) on the GPU: problem by problem against the
oracle, bit for bit against the shared-table and Box-per-problem kernels, and at scale."""
import ctypes

import numpy as np
import pytest

import problems as pr
from helpers import make_solver, op_from_table
from oracle import ccqp_oracle as orc
from ccqppy_b200 import _capi, solution_spaces as ss

pytestmark = pytest.mark.gpu

SOLVERS = [pr.PGD, pr.APGD, pr.APGD_AR, pr.BBPGD, pr.BBPGDF, pr.SPG]


def tables(struct, n, batch, seed=0):
    """`batch` tables of one block structure, each with its own randomly drawn parameters."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(batch):
        t = pr.Table()
        if struct == "sphere3":                         # friction discs, radii in [0.1, 1]
            for _ in range(n // 3):
                t.add(pr.SPHERE, 3, 0.1 + 0.9 * rng.random())
        elif struct == "soc3":                          # friction cones, per-problem mu
            for _ in range(n // 3):
                t.add(pr.SOC, 3, 0.2 + 1.3 * rng.random())
        elif struct == "cone":                          # the reference's Cone, per-problem aspect ratio
            for _ in range(n // 3):
                t.add(pr.CONE_REF, 3, 0.3 + rng.random())
        elif struct == "mixed":                         # the structure of test_gpu_batched.small_mixed_table
            nb, nl, nu = n // 4, n // 8, n // 8
            lo = -1.0 - 0.5 * rng.random(nb)
            t.add(pr.BOX, nb, lo, lo + 1.5 + rng.random(nb))
            t.add(pr.LOWER, nl, -0.5 - rng.random(nl))
            t.add(pr.UPPER, nu, 0.5 + rng.random(nu))
            while t.n + 3 <= n - 3:
                t.add(pr.SPHERE, 3, 0.3 + rng.random())
            t.add(pr.SPHERE, 2, 0.4 + rng.random())
        elif struct == "box":
            lo = -1.0 - 0.5 * rng.random(n)
            t.add(pr.BOX, n, lo, lo + 1.2 + rng.random(n))
        if t.n < n:
            t.add(pr.IDENTITY, n - t.n)
        out.append(t)
    for t in out[1:]:
        assert np.array_equal(t.blocks, out[0].blocks)
    return out


def problems(batch, n, seed0):
    A = np.empty((batch, n, n))
    b = np.empty((batch, n))
    for i in range(batch):
        A[i], b[i] = pr.shift_problem(n, seed0 + i, 1.0)
    return A, b


def stacked(tabs):
    return op_from_table(tabs[0]), np.stack([t.params for t in tabs])


def same_bits(s1, s2):
    x1, x2 = (np.asarray(s.solution.cpu() if hasattr(s.solution, "cpu") else s.solution) for s in (s1, s2))
    assert np.array_equal(x1, x2)
    assert np.array_equal(s1.solution_num_matrix_vector_multiplications, s2.solution_num_matrix_vector_multiplications)
    assert np.array_equal(s1.solution_residual, s2.solution_residual, equal_nan=True)
    assert np.array_equal(s1.solution_status, s2.solution_status)
    assert np.array_equal(s1.solution_converged, s2.solution_converged)


# ---- 1. oracle parity, problem by problem ----------------------------------------------------------------------------
CASES = {"sphere3_63": ("sphere3", 63, 5000), "sphere3_47x0": ("sphere3", 47, 5000), "mixed_47": ("mixed", 47, 5000),
         "soc3_63": ("soc3", 63, 5000), "cone_36": ("cone", 36, 40), "sphere3_126": ("sphere3", 126, 5000),
         "mixed_126": ("mixed", 126, 5000)}


@pytest.mark.parametrize("solver", SOLVERS)
@pytest.mark.parametrize("case", list(CASES))
def test_per_problem_tables_match_oracle(solver, case):
    """Problem i equals solve(A[i], b[i], x0[i], op_i) with op_i's own parameters.  The reference's Cone never converges
    (its map is not a projection), so that case runs a fixed budget of 40 mat-vecs."""
    struct, n, max_mv = CASES[case]
    batch = 24 if n <= 64 else 12
    step, K = 0.1, 512
    tol = 1e-6 if solver in (pr.APGD, pr.APGD_AR) else 1e-8
    tabs = tables(struct, n, batch, seed=list(CASES).index(case))
    A, b = problems(batch, n, 1000)
    x0 = 0.3 * np.random.default_rng(12).standard_normal((batch, n)) if case == "sphere3_47x0" else None
    op, P = stacked(tabs)
    s = make_solver(solver, tol, max_mv, step)
    s.solve_batched(A, b, x0=x0, seeds=np.arange(batch), n_uniforms=K, convex_proj_op=op, op_params=P)
    same = 0
    for i in range(batch):
        o = orc.solve(solver, A[i], b[i], x0=None if x0 is None else x0[i], blocks=tabs[i].blocks, params=tabs[i].params,
                      tol=tol, max_mv=max_mv, step_size=step, uniforms=pr.spg_uniforms(i, K))
        assert bool(s.solution_converged[i]) == o["converged"]
        mv = int(s.solution_num_matrix_vector_multiplications[i])
        scale = max(np.linalg.norm(o["solution"]), 1e-300)
        if mv == o["mv"]:
            same += 1
            assert np.linalg.norm(s.solution[i] - o["solution"]) <= 1e-9 * scale, i
        else:
            assert abs(mv - o["mv"]) <= max(2, round(0.1 * o["mv"])), (i, mv, o["mv"])
            assert np.linalg.norm(s.solution[i] - o["solution"]) <= 1e-5 * scale
    assert same >= 0.9 * batch, (same, batch)


# ---- 2. bit identities -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("solver", SOLVERS)
@pytest.mark.parametrize("struct,n", [("sphere3", 63), ("mixed", 64), ("sphere3", 126)])
def test_rows_equal_to_shared_params_give_shared_bits(solver, struct, n):
    """Every row of P equal to the shared operator's parameters: the same bits, counts and statuses as the shared table
    (n = 63: unstaged rows; 64 and 126: rows staged next to b)."""
    batch = 40
    tab = tables(struct, n, 1, seed=3)[0]
    op = op_from_table(tab)
    A, b = problems(batch, n, 2000)
    P = np.tile(op.descriptor()[1], (batch, 1))
    tol = 1e-6 if solver in (pr.APGD, pr.APGD_AR) else 1e-8
    shared = make_solver(solver, tol, 3000, 0.1).solve_batched(A, b, seeds=np.arange(batch), n_uniforms=400, convex_proj_op=op)
    per = make_solver(solver, tol, 3000, 0.1).solve_batched(A, b, seeds=np.arange(batch), n_uniforms=400, convex_proj_op=op,
                                                            op_params=P)
    same_bits(shared, per)
    assert shared.solution_converged.any()


@pytest.mark.parametrize("solver", [pr.PGD, pr.APGD, pr.BBPGD, pr.SPG])
@pytest.mark.parametrize("n", [64, 47, 126])
def test_box_only_table_equals_box_per_problem(solver, n):
    """A Box-only table with per-problem bounds clamps with the same compare/select as the Box-per-problem kernels."""
    batch = 40
    tabs = tables("box", n, batch, seed=n)
    op, P = stacked(tabs)
    lb, ub = P[:, :n].copy(), P[:, n:].copy()
    A, b = problems(batch, n, 3000)
    tol = 1e-6 if solver == pr.APGD else 1e-8
    box = make_solver(solver, tol, 3000, 0.1).solve_batched(A, b, lb, ub, seeds=np.arange(batch), n_uniforms=400)
    tab = make_solver(solver, tol, 3000, 0.1).solve_batched(A, b, seeds=np.arange(batch), n_uniforms=400, convex_proj_op=op,
                                                            op_params=P)
    same_bits(box, tab)


@pytest.mark.parametrize("solver", [pr.BBPGD, pr.SPG])
def test_permuted_batch_gives_permuted_bits(solver):
    batch, n = 64, 63
    tabs = tables("mixed", n, batch, seed=9)
    op, P = stacked(tabs)
    A, b = problems(batch, n, 4000)
    uni = np.random.default_rng(5).random((batch, 400))
    perm = np.random.default_rng(6).permutation(batch)
    s1 = make_solver(solver, 1e-8, 3000).solve_batched(A, b, uniforms=uni, convex_proj_op=op, op_params=P)
    s2 = make_solver(solver, 1e-8, 3000).solve_batched(A[perm], b[perm], uniforms=uni[perm], convex_proj_op=op,
                                                       op_params=P[perm])
    assert np.array_equal(s1.solution[perm], s2.solution)
    assert np.array_equal(s1.solution_num_matrix_vector_multiplications[perm], s2.solution_num_matrix_vector_multiplications)


@pytest.mark.parametrize("struct", ["sphere3", "mixed"])
@pytest.mark.parametrize("n", [64, 126])
def test_staged_unstaged_host_device_and_sequence_agree(struct, n):
    """One batch through every way its parameter rows can travel: a host array (copied with an even pitch, rows staged
    next to b), a CUDA tensor used in place (staged when n_params is even, read from global memory when it is odd), the
    same tensor at an 8-byte offset (never staged), and the sequence of operators.  All give the same bits."""
    import torch
    batch = 48
    tabs = tables(struct, n, batch, seed=n + len(struct))
    op, P = stacked(tabs)
    A, b = problems(batch, n, 5000)
    np_ = P.shape[1]
    for solver in (pr.BBPGD, pr.SPG, pr.APGD):
        tol = 1e-6 if solver == pr.APGD else 1e-8
        run = lambda *a, **k: make_solver(solver, tol, 3000).solve_batched(*a, seeds=np.arange(batch), n_uniforms=400, **k)
        host = run(A, b, convex_proj_op=op, op_params=P)
        assert host.solution_converged.mean() > 0.9
        Ad, bd = torch.from_numpy(A).cuda(), torch.from_numpy(b).cuda()
        Pd = torch.from_numpy(P).cuda()
        dev = run(Ad, bd, convex_proj_op=op, op_params=Pd)
        assert dev.solution.is_cuda
        same_bits(host, dev)
        buf = torch.empty(batch * np_ + 1, dtype=torch.float64, device="cuda")
        Poff = buf[1:].view(batch, np_)
        Poff.copy_(Pd)
        assert Poff.data_ptr() % 16 == 8
        off = run(Ad, bd, convex_proj_op=op, op_params=Poff)
        same_bits(host, off)
        seq = run(A, b, convex_proj_op=[op_from_table(t) for t in tabs])
        same_bits(host, seq)
        # CPU tensors take the host path
        cpu = run(torch.from_numpy(A), torch.from_numpy(b), convex_proj_op=op, op_params=torch.from_numpy(P))
        same_bits(host, cpu)


def test_device_params_with_host_problem_and_odd_n():
    """n odd: b is not staged, so neither is the parameter row; a CUDA P with a host A is brought to the host."""
    import torch
    batch, n = 32, 47
    tabs = tables("mixed", n, batch, seed=21)
    op, P = stacked(tabs)
    A, b = problems(batch, n, 6000)
    h = make_solver(pr.BBPGD, 1e-8, 3000).solve_batched(A, b, convex_proj_op=op, op_params=P)
    d = make_solver(pr.BBPGD, 1e-8, 3000).solve_batched(A, b, convex_proj_op=op, op_params=torch.from_numpy(P).cuda())
    same_bits(h, d)
    assert h.solution_converged.all()


# ---- 3. constraint property at scale ---------------------------------------------------------------------------------
def test_per_problem_discs_at_scale():
    """65 536 contact-style problems of n = 63 (21 friction discs each, radius mu * f_n drawn on the device): every problem
    converges and every disc holds its own radius."""
    import torch
    batch, n, k = 65536, 63, 21
    g = torch.Generator(device="cuda").manual_seed(0)
    G = torch.randn((batch, n, n), generator=g, device="cuda", dtype=torch.float64)
    A = G @ G.transpose(1, 2) / n + torch.eye(n, device="cuda", dtype=torch.float64)
    del G
    xs = 1 - 4 * torch.rand((batch, n), generator=g, device="cuda", dtype=torch.float64)
    b = -(A @ xs.unsqueeze(-1)).squeeze(-1)
    mu = 0.2 + 0.6 * torch.rand((batch, 1), generator=g, device="cuda", dtype=torch.float64)
    fn = 0.5 + torch.rand((batch, k), generator=g, device="cuda", dtype=torch.float64)
    radii = (mu * fn).contiguous()
    op = ss.DisjointProjOp(*[ss.SphereProjOp(3, 1.0) for _ in range(k)])
    assert op.descriptor()[1].size == k
    uni = torch.rand((batch, 1000), generator=g, device="cuda", dtype=torch.float64)
    for solver in (pr.BBPGD, pr.SPG):
        s = make_solver(solver, 1e-8, 5000).solve_batched(A, b, uniforms=uni, convex_proj_op=op, op_params=radii)
        assert s.solution_converged.all(), int((~s.solution_converged).sum())
        norms = s.solution.view(batch, k, 3).norm(dim=2)
        assert bool((norms <= radii * (1 + 1e-12)).all())
        assert bool((norms >= radii * (1 - 1e-9)).any())        # the constraints are active somewhere
        assert s.solution_hbm_bytes > batch * 8.0 * (n * n + 4 * n + k) * 0.999


# ---- 4. C ABI errors -------------------------------------------------------------------------------------------------
def test_capi_errors():
    h = _capi.Handle()
    lib = h.lib
    P = lambda a: ctypes.c_void_p(a.ctypes.data)
    prm = make_solver(pr.BBPGD, 1e-8, 100)._params()
    batch, n = 4, 9
    A, b = problems(batch, n, 7000)
    x = np.zeros((batch, n))
    par = np.full((batch, 3), 0.5)
    res = (_capi.Result * batch)()
    summ = _capi.Result()

    def call(blocks, params, n_params, solver=_capi.BBPGD, nn=n, AA=A, bb=b, xx=x, entry=lib.ccqp_solve_batched_tables):
        return entry(h.h, solver, ctypes.byref(prm), batch, nn, P(AA), P(bb), None, blocks.ptr, len(blocks), params, n_params,
                     None, 0, P(xx), _capi.MEM_HOST, res, ctypes.byref(summ))
    S, I31, I64 = _capi.SPHERE, 2**31 - 1, 2**63 - 1
    good = _capi.make_blocks([(S, 0, 3, 0), (S, 3, 3, 1), (S, 6, 3, 2)])
    assert call(good, P(par), 3) == 0 and summ.converged == 1
    assert call(good, None, 3) == 1                                                        # null block_params
    assert call(_capi.make_blocks([(S, 0, 3, 0), (S, 3, 3, 1)]), P(par), 3) == 1          # [0, 6) only
    # a table malformed by itself: the same code from the projection of a handle and from both batched table entries
    malformed = {"a block overruns n_params": ([(S, 0, 3, 0), (S, 3, 3, 1), (S, 6, 3, 2)], 2),
                 "a gap at 3": ([(S, 0, 3, 0), (S, 4, 3, 1), (S, 7, 2, 2)], 3),
                 "unknown kind": ([(S, 0, 3, 0), (S, 3, 3, 1), (99, 6, 3, 2)], 3),
                 "zero dim": ([(S, 0, 3, 0), (S, 3, 0, 1), (S, 3, 6, 2)], 3),
                 "negative param_off": ([(S, 0, 3, 0), (S, 3, 3, -1), (S, 6, 3, 2)], 3),
                 # 64-bit wrap-around: the dims sum to 9 modulo 2^64, a parameter range ends past INT64_MAX
                 "n wraps around": ([(_capi.LOWER, 0, I31, 0), (_capi.IDENTITY, I31, I64 - I31, 0), (_capi.IDENTITY, I64, 1, 0),
                                     (_capi.IDENTITY, -I64 - 1, I64, 0), (_capi.IDENTITY, -1, 10, 0)], I31 + 1),
                 "param_off + need wraps around": ([(S, 0, 3, 0), (S, 3, 3, 1), (S, 6, 3, I64)], 3)}
    for what, (rows, n_params) in malformed.items():
        bad = _capi.make_blocks(rows)
        codes = (lib.ccqp_set_projection(h.h, bad.ptr, len(bad), P(par), n_params),
                 call(bad, P(par), n_params, entry=lib.ccqp_solve_batched_table), call(bad, P(par), n_params))
        assert codes == (1, 1, 1), (what, codes)
        for entry in (lib.ccqp_solve_batched_table, lib.ccqp_solve_batched_tables):      # malformed wins over MPRGP
            assert call(bad, P(par), n_params, solver=_capi.MPRGP, entry=entry) == 1, what
    assert call(good, P(par), 3, solver=_capi.MPRGP) == 4                                  # MPRGP: unsupported
    big, vb = np.zeros((batch, 129, 129)), np.zeros((batch, 129))
    wide = _capi.make_blocks([(S, 0, 129, 0)])
    assert call(wide, P(par), 3, nn=129, AA=big, bb=vb, xx=vb) == 4                       # n > 128
    assert call(wide, P(par), 3, solver=99, nn=129, AA=big, bb=vb, xx=vb) == 4            # ... wins over an unknown solver
    assert lib.ccqp_solve_batched(h.h, 99, ctypes.byref(prm), batch, 129, P(big), P(vb), None, P(vb), P(vb), None, 0,
                                  P(vb), _capi.MEM_HOST, res, ctypes.byref(summ)) == 4    # the same for a Box per problem
    assert call(good, P(par), 3, solver=99) == 1                                           # unknown solver
    h.close()
