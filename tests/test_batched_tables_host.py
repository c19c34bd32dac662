"""Batched solves with per-problem operator parameters (`solve_batched(convex_proj_op=op, op_params=P)` or a sequence of
operators): the argument checks that run before anything reaches the device, and the stacking of a sequence of
operators into the parameter array.  No GPU needed."""
import numpy as np
import pytest

from ccqppy_b200 import _capi, solution_spaces as ss, solvers


@pytest.fixture
def no_device(monkeypatch):
    """Every check below must fire before a handle (and so a device context) is created."""
    def fail(*a, **k):
        raise AssertionError("a handle was created before the arguments were checked")
    monkeypatch.setattr(_capi, "default_handle", fail)


def discs(radii):
    return ss.DisjointProjOp(*[ss.SphereProjOp(3, r) for r in radii])


def mixed(rng):
    lo = -1.0 - rng.random(4)
    return ss.DisjointProjOp(ss.BoxProjOp(4, lo, lo + 2.0), ss.LowerBoundProjOp(2, -rng.random(2)),
                             ss.UpperBoundProjOp(2, rng.random(2)), ss.SphereProjOp(3, 0.5 + rng.random()),
                             ss.SOCProjOp(3, rng.random()), ss.ConeProjOp(2, 1.0), ss.IdentityProjOp(2))


def problem(batch, n):
    A = np.broadcast_to(np.eye(n), (batch, n, n)).copy()
    return A, np.ones((batch, n))


def solver():
    s = solvers.CCQPSolverBBPGD(1e-8, 100)
    s.quiet = True
    return s


def test_op_params_shape(no_device):
    batch, n = 5, 12
    A, b = problem(batch, n)
    op = discs([0.5] * 4)
    for shape in [(batch, 5), (batch - 1, 4), (batch,), (batch, 4, 1), (4, batch)]:
        with pytest.raises(ValueError, match="op_params has shape"):
            solver().solve_batched(A, b, convex_proj_op=op, op_params=np.ones(shape))


def test_op_params_needs_the_structure_and_no_bounds(no_device):
    batch, n = 3, 6
    A, b = problem(batch, n)
    P = np.ones((batch, 2))
    with pytest.raises(ValueError, match="needs convex_proj_op"):
        solver().solve_batched(A, b, op_params=P)
    with pytest.raises(ValueError, match="needs convex_proj_op"):
        solver().solve_batched(A, b, -np.ones((batch, n)), np.ones((batch, n)), op_params=P)
    with pytest.raises(ValueError, match="either lower_bound"):
        solver().solve_batched(A, b, -np.ones((batch, n)), np.ones((batch, n)), convex_proj_op=discs([1, 1]), op_params=P)
    with pytest.raises(ValueError, match="either lower_bound"):
        solver().solve_batched(A, b, upper_bound=np.ones((batch, n)), convex_proj_op=discs([1, 1]), op_params=P)


def test_operator_dimension(no_device):
    batch, n = 3, 9
    A, b = problem(batch, n)
    with pytest.raises(ValueError, match="dimension 6, the problems 9"):
        solver().solve_batched(A, b, convex_proj_op=discs([1, 1]), op_params=np.ones((batch, 2)))
    ops = [discs([1, 1, 1]), discs([1, 1, 1]), discs([1, 1])]
    with pytest.raises(ValueError, match=r"convex_proj_op\[2\] has dimension 6"):
        solver().solve_batched(A, b, convex_proj_op=ops)


def test_sequence_length_and_structure(no_device):
    batch, n = 4, 9
    A, b = problem(batch, n)
    with pytest.raises(ValueError, match="3 operators for 4 problems"):
        solver().solve_batched(A, b, convex_proj_op=[discs([1, 2, 3])] * 3)
    with pytest.raises(ValueError, match="0 operators for 4 problems"):
        solver().solve_batched(A, b, convex_proj_op=[])
    # same dimension, different kinds / dims / parameter layout: the first index that differs is named
    other = [ss.DisjointProjOp(ss.SOCProjOp(3, 1.0), ss.SphereProjOp(3, 1.0), ss.SphereProjOp(3, 1.0)),
             ss.DisjointProjOp(ss.SphereProjOp(6, 1.0), ss.SphereProjOp(3, 1.0)),
             ss.DisjointProjOp(ss.BoxProjOp(3), ss.SphereProjOp(3, 1.0), ss.SphereProjOp(3, 1.0))]
    for bad in other:
        ops = [discs([1, 2, 3]), discs([2, 3, 4]), bad, ss.IdentityProjOp(9)]
        with pytest.raises(ValueError, match="operator 2 has a different block structure"):
            solver().solve_batched(A, b, convex_proj_op=ops)
    # a repeated member object shares its parameters in descriptor(): another layout than distinct members
    s = ss.SphereProjOp(3, 1.0)
    ops = [discs([1, 2, 3]), ss.DisjointProjOp(s, s, s), discs([1, 2, 3]), discs([1, 2, 3])]
    with pytest.raises(ValueError, match="operator 1 has a different block structure"):
        solver().solve_batched(A, b, convex_proj_op=ops)
    with pytest.raises(ValueError, match="ONE operator"):
        solver().solve_batched(A, b, convex_proj_op=[discs([1, 2, 3])] * batch, op_params=np.ones((batch, 3)))


def test_sequence_stacks_descriptor_rows():
    rng = np.random.default_rng(0)
    ops = [mixed(rng) for _ in range(6)]
    blocks, P = ss.stacked_descriptor(ops)
    b0, p0, rows0 = ops[0].descriptor()
    assert P.shape == (6, p0.size) and P.dtype == np.float64
    for i, op in enumerate(ops):
        _, p, rows = op.descriptor()
        assert rows == rows0
        assert np.array_equal(P[i], p)
    assert np.array_equal(blocks.arr, b0.arr)
    assert not np.array_equal(P[0], P[1])          # the parameters really are per problem
    with pytest.raises(ValueError):
        ss.stacked_descriptor([])
