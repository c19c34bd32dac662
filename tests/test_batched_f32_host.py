"""Batched solves on float32 Hessians, the host side (no GPU needed): which C entry point `solve_batched` calls for which
A, which buffer it passes, the errors for malformed A, and the argument checks of the four `_f32` C entry points."""
import ctypes

import numpy as np
import pytest

from ccqppy_b200 import _capi, solution_spaces as ss, solvers

ENTRIES = ("ccqp_solve_batched", "ccqp_solve_batched_sym", "ccqp_solve_batched_table", "ccqp_solve_batched_tables")


class _RecordingLib:
    """Stands in for the library: every batched entry point records (name, A pointer, memtype) and returns ok."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        if name not in ENTRIES and name[:-4] not in ENTRIES:
            raise AttributeError(name)

        def entry(h, solver, prm, batch, n, pa, *rest):
            mem = rest[-3]
            self.calls.append((name, pa.value, mem))
            return _capi.OK
        return entry


class _FakeHandle:
    def __init__(self):
        self.lib = _RecordingLib()
        self.h = ctypes.c_void_p(1)


@pytest.fixture
def fake(monkeypatch):
    h = _FakeHandle()
    monkeypatch.setattr(_capi, "default_handle", lambda device=-1: h)
    return h.lib


def solver():
    s = solvers.CCQPSolverBBPGD(1e-8, 100)
    s.quiet = True
    return s


def box(A, **kw):
    batch, n = A.shape[0], A.shape[1]
    return solver().solve_batched(A, np.ones((batch, n)), -np.ones((batch, n)), np.ones((batch, n)), **kw)


def discs(k):
    return ss.DisjointProjOp(*[ss.SphereProjOp(3, 0.5 + i) for i in range(k)])


def test_float32_numpy_goes_to_the_f32_twin_in_place(fake):
    A = np.ones((4, 6, 6), dtype=np.float32)
    box(A)
    assert fake.calls == [("ccqp_solve_batched_f32", A.ctypes.data, _capi.MEM_HOST)]


@pytest.mark.parametrize("dtype", [np.float64, np.float16, np.int64])
def test_other_dtypes_widen_to_float64_as_before(fake, dtype):
    box(np.ones((3, 5, 5), dtype=dtype))
    assert [c[0] for c in fake.calls] == ["ccqp_solve_batched"]


def test_every_feasible_set_form_routes_to_its_twin(fake):
    batch, n = 3, 6
    A = np.ones((batch, n, n), dtype=np.float32)
    b = np.ones((batch, n))
    box(A, symmetric=True)
    solver().solve_batched(A, b, convex_proj_op=discs(2))
    solver().solve_batched(A, b, convex_proj_op=discs(2), op_params=np.ones((batch, 2)))
    solver().solve_batched(A, b, convex_proj_op=[discs(2)] * batch)
    assert [c[0] for c in fake.calls] == ["ccqp_solve_batched_sym_f32", "ccqp_solve_batched_table_f32",
                                          "ccqp_solve_batched_tables_f32", "ccqp_solve_batched_tables_f32"]
    assert all(c[1] == A.ctypes.data for c in fake.calls)


def test_non_contiguous_float32_gets_one_float32_copy(fake):
    big = np.arange(4 * 6 * 12, dtype=np.float32).reshape(4, 6, 12)
    A = big[:, :, ::2]
    box(A)
    (name, ptr, mem), = fake.calls
    assert name == "ccqp_solve_batched_f32" and mem == _capi.MEM_HOST
    assert ptr not in (A.ctypes.data, big.ctypes.data)


def test_torch_host_float32(fake):
    torch = pytest.importorskip("torch")
    A = torch.ones((4, 6, 6), dtype=torch.float32)
    box(A)
    assert fake.calls[-1] == ("ccqp_solve_batched_f32", A.data_ptr(), _capi.MEM_HOST)
    At = A.transpose(1, 2)                       # strided, not contiguous: one contiguous float32 copy
    box(At)
    name, ptr, _ = fake.calls[-1]
    assert name == "ccqp_solve_batched_f32" and ptr != A.data_ptr()
    box(torch.ones((4, 6, 6), dtype=torch.float64))
    assert fake.calls[-1][0] == "ccqp_solve_batched"


@pytest.mark.parametrize("shape", [(4, 6, 5), (6, 6), (2, 3, 6, 6)])
def test_malformed_float32_shape_raises_value_error(fake, shape):
    with pytest.raises(ValueError, match=r"\[batch, n, n\]"):
        solver().solve_batched(np.ones(shape, dtype=np.float32), np.ones((shape[0], 6)), -np.ones((shape[0], 6)),
                               np.ones((shape[0], 6)))
    assert fake.calls == []


def test_sparse_float32_tensor_raises_type_error(fake):
    torch = pytest.importorskip("torch")
    A = torch.eye(6, dtype=torch.float32).repeat(2, 1, 1).to_sparse()
    with pytest.raises(TypeError, match="dense A"):
        box(A)
    assert fake.calls == []


def _call(name, A, h=None, n=4, batch=2, table=None):
    """One call of a batched entry point with valid vectors; A is a pointer (or None)."""
    lib = _capi.load()
    b = np.ones((batch, n))
    x = np.empty((batch, n))
    prm = _capi.Params(tol=1e-8, max_mv=100.0, step_size=0.01, tau=0.5, sigma1=0.01, sigma2=0.5, m=5)
    vp = lambda a: ctypes.c_void_p(a.ctypes.data)      # noqa: E731
    if "table" in name:
        blocks = table if table is not None else _capi.make_blocks([(_capi.BOX, 0, n, 0)])
        P = np.tile(np.r_[-np.ones(n), np.ones(n)], (batch, 1))
        return getattr(lib, name)(h, _capi.BBPGD, ctypes.byref(prm), batch, n, A, vp(b), None, blocks.ptr, len(blocks),
                                  vp(P), P.shape[1], None, 0, vp(x), _capi.MEM_HOST, None, None)
    lo, hi = -np.ones((batch, n)), np.ones((batch, n))
    return getattr(lib, name)(h, _capi.BBPGD, ctypes.byref(prm), batch, n, A, vp(b), None, vp(lo), vp(hi), None, 0, vp(x),
                              _capi.MEM_HOST, None, None)


@pytest.mark.parametrize("name", ENTRIES)
def test_c_twins_check_arguments_like_their_fp64_functions(name):
    """Without a device there is no handle: the checks that run first (null handle, null A) agree between the twins."""
    A64, A32 = np.eye(4).repeat(2, 0), np.eye(4, dtype=np.float32).repeat(2, 0)
    for A in (None, ctypes.c_void_p(A64.ctypes.data)):
        st64 = _call(name, A)
        st32 = _call(name + "_f32", None if A is None else ctypes.c_void_p(A32.ctypes.data))
        assert st64 == st32 == 1                      # CCQP_ERR_INVALID_ARG


def test_f32_twins_take_the_fp64_argument_types_except_a():
    lib = _capi.load()
    for name in ENTRIES:
        assert getattr(lib, name + "_f32").argtypes == getattr(lib, name).argtypes
        assert name + "_f32" in _capi.EXPORTS
