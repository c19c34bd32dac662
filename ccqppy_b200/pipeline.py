"""A stream of independent dense solves whose inputs live in host memory (extension; the reference has
no counterpart -- its `solve()` is one synchronous NumPy loop).

`solve()` from host arrays is PCIe-bound for large problems: at n = 32768 the 8.59 GB Hessian takes
~156 ms to reach the GPU and the solve itself ~70 ms.  With several solves to do, the upload of the
next Hessian can run on the copy engine while the current solve occupies the SMs.  `SolvePipeline`
keeps `depth` handles (each with its own CUDA stream, device copy of A and work buffers) and hands
the solves to them round-robin through `ccqp_solve_async` / `ccqp_solve_wait`:

    pipe = SolvePipeline(solvers.CCQPSolverSPG(1e-5, 2000), depth=2)
    for A, b in problems:                       # pinned host tensors / arrays
        pipe.submit(A, b, convex_proj_op=op, uniforms=u)
    for r in pipe.results():                    # in submission order
        r.solution, r.solution_converged, r.solution_num_matrix_vector_multiplications, ...

Every solve is the same computation as `solver.solve(...)` (same kernel, same arguments); only the
scheduling differs.  Host buffers must stay alive until their result has been collected; pinned
memory (`torch.Tensor.pin_memory()`) is what makes the copies asynchronous.  A float32 A is uploaded as float32
straight from the caller's buffer (`ccqp_set_matrix_f32`: half the PCIe bytes, the same result bits as its widening).
"""
import ctypes

import numpy as np

from . import _capi
from . import solution_spaces as ss
from .solvers import _as_f32_matrix, _as_f64, _is_torch


class SolveResult:
    """Result fields of one pipelined solve: the names of the solver properties (solvers.py:172-194)."""
    solution = None
    solution_converged = None
    solution_residual = None
    solution_num_matrix_vector_multiplications = None
    solution_gpu_time = None
    solution_hbm_bytes = None
    solution_gemv_count = None
    solution_kernel_launches = None


class _Slot:
    def __init__(self, device):
        self.handle = _capi.Handle(device)
        self.keep = None          # host objects of the solve in flight
        self.xout = None
        self.ticket = None


class SolvePipeline:
    def __init__(self, solver, depth=2, device=-1):
        if depth < 1:
            raise ValueError("depth must be at least 1")
        self.solver = solver
        self.slots = [_Slot(device) for _ in range(depth)]
        self._next = 0
        self._done = {}
        self._collected = 0

    def _pinned(self, n):
        try:
            import torch
            return torch.empty(n, dtype=torch.float64, pin_memory=True)
        except Exception:
            return np.empty(n, dtype=np.float64)

    def _collect(self, slot):
        res = _capi.Result()
        st = slot.handle.lib.ccqp_solve_wait(slot.handle.h, ctypes.byref(res))
        if st == _capi.ERR_NORMAL_NOT_IMPLEMENTED:
            raise NotImplementedError("Cone normal not implemented, yet.")
        if st == _capi.ERR_RANGE:
            raise OverflowError("Range exceeds valid bounds")
        _capi.check(slot.handle.h, st)
        r = SolveResult()
        r.solution = slot.xout
        r.solution_converged = bool(res.converged)
        r.solution_residual = float(res.residual)
        r.solution_num_matrix_vector_multiplications = int(res.mv_count)
        r.solution_gpu_time = float(res.gpu_seconds)
        r.solution_hbm_bytes = float(res.hbm_bytes)
        r.solution_gemv_count = int(res.gemv_count)
        r.solution_kernel_launches = int(res.kernel_launches)
        self._done[slot.ticket] = r
        slot.keep = slot.xout = slot.ticket = None

    def submit(self, A, b, x0=None, convex_proj_op=None, uniforms=None, symmetric=False):
        """Enqueue one solve; returns its ticket (0, 1, 2, ...).  Blocks if the slot it lands on still has a solve in
        flight (that one is collected first) and for the host-side symmetry test of a large A (`solve()`'s docstring);
        `symmetric=True` declares the symmetry and skips the test."""
        s = self.solver
        n = int(b.shape[0])
        if convex_proj_op is None:
            convex_proj_op = ss.IdentityProjOp(n)
        if s._solver_id == _capi.SPG and uniforms is None:
            raise ValueError("pipelined SPG solves need an explicit `uniforms` stream (the global NumPy RNG cannot be "
                             "left where the reference would leave it before the solve has finished)")
        slot = self.slots[self._next % len(self.slots)]
        if slot.ticket is not None:
            self._collect(slot)
        h, lib = slot.handle, slot.handle.lib
        A32 = None if symmetric else _as_f32_matrix(A)
        Ah = A32 if A32 is not None else _as_f64(A)
        b64 = _as_f64(b)
        x064 = None if x0 is None else _as_f64(x0)
        uni = None if uniforms is None else _as_f64(uniforms)
        if any(_is_torch(v) and v.is_cuda for v in (Ah, b64, x064, uni) if v is not None):
            raise TypeError("SolvePipeline is for host-resident inputs; device tensors go through solve()")
        blocks, params, _rows = convex_proj_op.descriptor()
        par = params if params.size else np.zeros(1)
        # the (small) projection table first: ccqp_set_projection synchronises the handle's stream, which is idle here
        _capi.check(h.h, lib.ccqp_set_projection(h.h, blocks.ptr, len(blocks), ctypes.c_void_p(par.ctypes.data), params.size))
        if A32 is not None:
            h.set_matrix_f32(A32, n)                                                  # asynchronous from pinned memory too
        else:
            pa, mem, _ = _capi.f64_ptr(Ah)
            lda = Ah.stride(0) if _is_torch(Ah) else n
            if symmetric:
                _capi.check(h.h, lib.ccqp_set_matrix_symmetric(h.h, pa, n, lda, mem))
            else:
                _capi.check(h.h, lib.ccqp_set_matrix(h.h, pa, n, lda, 0, n, mem))  # the copies are asynchronous from pinned memory
        xout = self._pinned(n)
        ptr = lambda v: None if v is None else _capi.f64_ptr(v)[0]
        prm = s._params()
        _capi.check(h.h, lib.ccqp_solve_async(h.h, s._solver_id, ctypes.byref(prm), ptr(b64), ptr(x064), ptr(uni),
                                              0 if uni is None else int(uni.shape[0]), ptr(xout), _capi.MEM_HOST))
        slot.keep = (Ah, b64, x064, uni, blocks, par, prm)
        slot.xout = xout
        slot.ticket = self._next
        self._next += 1
        return slot.ticket

    def results(self):
        """Collect everything in flight; returns the results not yet handed out, in submission order."""
        for slot in self.slots:
            if slot.ticket is not None:
                self._collect(slot)
        out = [self._done.pop(t) for t in sorted(self._done)]
        self._collected += len(out)
        return out

    def close(self):
        self.results()
        for slot in self.slots:
            slot.handle.close()
