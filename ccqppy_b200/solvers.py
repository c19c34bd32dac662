"""Solvers: host-side mirror of the reference's `ccqppy.solvers`
(/root/reference/src/ccqppy/solvers.py) in front of the B200 solver kernels.

Same class names, constructor signatures, `solve(A, b, x0=None, convex_proj_op=None)` (returns
the solver object), result properties and `name` strings as the reference (SURVEY.md section 8b).
Under the surface ONE C-ABI call (`ccqp_solve`) runs the whole solve in a persistent CUDA kernel:
the per-iteration fp64 mat-vec, the projection, the step-length dot products and the residual
reductions never leave the device and there is no per-iteration host round trip.

There is no CPU path.  Inputs the device path cannot take (an `A` that only offers `.dot`, a
projection that is an arbitrary Python callable) raise TypeError instead of silently running on
the host.

Extensions beyond the reference API (all optional):
  * `solve(..., uniforms=...)`      explicit U[0,1) stream for SPG instead of the global NumPy RNG
  * `solve_batched(A, b, lb, ub)`   many small QPs in one persistent kernel (n <= 128; per-problem boxes, one shared table,
                                    or one block structure with per-problem parameters: `convex_proj_op=op, op_params=P`
                                    or a sequence of operators)
  * `solution_gpu_time`, `solution_hbm_bytes`, `solution_gemv_count` after a solve
  * A / b / x0 may be torch tensors; a CUDA tensor A is used in place (no copy) when it is float64, or float32,
    contiguous and 16-byte aligned
  * a float32 dense A stays float32 (`ccqp_set_matrix_f32`): the kernels stream it at 4 bytes per entry and widen every
    entry exactly in a register, which is what NumPy does for the reference's `A.dot(v)` with a float32 A -- the result
    has the same bits as the solve of `A.astype(np.float64)`, for half the HBM and PCIe bytes and half the device memory.
    `symmetric=True` and sparse A widen a float32 A to float64 as before.
  * `solve_batched` keeps a float32 dense A [batch, n, n] float32 as well, for every feasible-set form (the `_f32` batched
    entry points): the kernels widen each entry exactly in a register when they load the problem, so the results are the
    bits of the widened call, for half the bytes of A moved over PCIe and HBM and no float64 copy on the device.
"""
import ctypes
import time
from abc import ABC, abstractmethod

import numpy as np

from . import _capi
from . import solution_spaces as ss

__all__ = ["CCQPSolverBase", "CCQPSolverPGD", "CCQPSolverAPGD", "CCQPSolverAPGDAntiRelaxation",
           "CCQPSolverBBPGD", "CCQPSolverBBPGDf", "CCQPSolverSPG", "CCQPSolverMPRGP", "CCQPSolverMPRGPBB"]

_MAX_DRAWS_UNBOUNDED = 1 << 20


def _is_torch(a):
    return a is not None and not isinstance(a, np.ndarray) and hasattr(a, "data_ptr")


def _is_sparse(a):
    """scipy.sparse matrix / array, or a torch sparse-CSR tensor: the operator-form Hessians the reference can take
    through `A.dot` (solvers.py:133)."""
    if _is_torch(a) or hasattr(a, "layout"):
        return str(getattr(a, "layout", "")) == "torch.sparse_csr"
    return hasattr(a, "tocsr") and hasattr(a, "nnz")


def _set_sparse_matrix(h, A, n):
    """CSR arrays of A -> ccqp_set_matrix_csr.  Returns objects that must stay alive during the solve."""
    lib = h.lib
    if hasattr(A, "layout"):                                  # torch.sparse_csr
        import torch
        ptr = A.crow_indices().to(torch.int64).contiguous()
        idx = A.col_indices().to(torch.int32).contiguous()
        val = A.values().to(torch.float64).contiguous()
        mem = _capi.MEM_DEVICE if val.is_cuda else _capi.MEM_HOST
        keep = (ptr, idx, val)
        args = (ptr.data_ptr(), idx.data_ptr(), val.data_ptr(), int(val.numel()))
    else:
        csr = A.tocsr()
        csr.sum_duplicates()
        ptr = np.ascontiguousarray(csr.indptr, dtype=np.int64)
        idx = np.ascontiguousarray(csr.indices, dtype=np.int32)
        val = np.ascontiguousarray(csr.data, dtype=np.float64)
        mem = _capi.MEM_HOST
        keep = (ptr, idx, val)
        args = (ptr.ctypes.data, idx.ctypes.data, val.ctypes.data, int(val.size))
    _capi.check(h.h, lib.ccqp_set_matrix_csr(h.h, ctypes.c_void_p(args[0]), ctypes.c_void_p(args[1]), ctypes.c_void_p(args[2]),
                                              n, args[3], 0, n, mem))
    return keep


def _as_f64(a, like_device=None):
    """float64, C-contiguous view/copy of a NumPy array or torch tensor (README passes int64)."""
    if _is_torch(a):
        import torch
        t = a.to(dtype=torch.float64).contiguous()
        if like_device is not None and t.device != like_device:
            t = t.to(like_device)
        return t
    if hasattr(a, "dot") and not hasattr(a, "__array__"):
        raise TypeError("A must be a dense array / tensor or a sparse (CSR-convertible) matrix: arbitrary objects that "
                        "only offer .dot cannot run inside the CUDA solver and there is no CPU fallback")
    arr = np.ascontiguousarray(a, dtype=np.float64)
    if like_device is not None:
        import torch
        return torch.from_numpy(arr).to(like_device)
    return arr


def _as_f32_matrix(a, aligned=True):
    """A float32 dense NumPy array / torch tensor as the C-contiguous float32 array / tensor ccqp_set_matrix_f32 takes
    (no widening); None for any other input.  A CUDA tensor is used as it is when it is contiguous and 16-byte aligned;
    otherwise ONE contiguous copy is made, so its rows take the same mat-vec loop as a widened copy of `a` would.
    aligned=False (batched solves, whose load path never changes the values): a contiguous CUDA tensor is used as it is
    at any alignment."""
    if isinstance(a, np.ndarray):
        return np.ascontiguousarray(a) if a.dtype == np.float32 else None
    if not _is_torch(a) or str(a.dtype) != "torch.float32" or str(a.layout) != "torch.strided":
        return None
    if a.is_contiguous() and (not a.is_cuda or not aligned or a.data_ptr() % 16 == 0):
        return a
    import torch
    return a.clone(memory_format=torch.contiguous_format)


class CCQPSolverBase(ABC):
    """solvers.py:11-68.  Concrete classes set `_solver_id`, `_label` and `_name`."""

    _solver_id = None
    _label = None     # what the reference prints: "solving <label>"
    _name = None
    quiet = False     # set True to suppress the reference's print (Q12)

    @abstractmethod
    def __init__(self, desired_residual_tol, max_matrix_vector_multiplications=np.inf):
        pass

    def _init_common(self, tol, max_mv):
        self.desired_residual_tol = tol
        self.max_matrix_vector_multiplications = max_mv
        self._solution = None
        self._solution_residual = None
        self._solution_converged = None
        self._solution_time = None
        self._solution_num_matrix_vector_mults = None
        self._gpu_time = None
        self._hbm_bytes = None
        self._gemv_count = None
        self._launches = None

    def _params(self):
        p = _capi.Params()
        p.tol = float(self.desired_residual_tol)
        p.max_mv = float(self.max_matrix_vector_multiplications)
        p.step_size = float(getattr(self, "step_size", 0.01))
        p.tau = float(getattr(self, "t", 0.5))
        p.sigma1 = float(getattr(self, "sigma1", 0.01))
        p.sigma2 = float(getattr(self, "sigma2", 0.5))
        p.m = int(getattr(self, "m", 5))
        return p

    def _checkSolveInput(self, A, b, x0):   # solvers.py:42 (a no-op there too)
        pass

    # -- SPG's random stream (Q5): draw from the GLOBAL NumPy RNG, then leave the global state
    #    exactly where the reference would have left it (one sample per completed iteration) --
    def _draw_uniforms(self):
        mx = self.max_matrix_vector_multiplications
        count = int(mx) if np.isfinite(mx) else _MAX_DRAWS_UNBOUNDED
        count = max(count, 1)
        state = np.random.get_state()
        return state, np.random.random_sample(count)

    @staticmethod
    def _restore_rng(state, used):
        np.random.set_state(state)
        if used:
            np.random.random_sample(int(used))

    def solve(self, A, b, x0=None, convex_proj_op=None, *, uniforms=None, device=-1, symmetric=False):
        """min 1/2 x^T A x + b^T x  s.t. x in Omega   (the gradient is A x + b, solvers.py:133).

        A : (n, n) dense array / tensor; b : (n,); x0 : (n,) or None (zeros);
        convex_proj_op : an operator of `ccqppy_b200.solution_spaces` (default Identity).
        Returns self; results are the `solution*` properties, as in the reference.

        A host-resident dense A that is symmetric crosses PCIe as its upper block triangle only (found out by a host-side
        test that runs while the copy engine works; the device copy is bit-identical to a full upload, and any other A is
        uploaded whole -- `ccqp_set_matrix`).  `symmetric=True` (extension) declares the symmetry instead: no test, the
        blocks below the block diagonal of A are never read (`ccqp_set_matrix_symmetric`).

        A float32 dense A (NumPy array, host or CUDA tensor; `symmetric=False`) is neither widened nor copied on the device
        (`ccqp_set_matrix_f32`): the solution, residual and counts are bit-identical to those of `A.astype(np.float64)`."""
        num_unknowns = b.shape[0]
        if convex_proj_op is None:
            convex_proj_op = ss.IdentityProjOp(num_unknowns)
        if not isinstance(convex_proj_op, ss.ProjOpBase):
            raise TypeError("convex_proj_op must be an operator from ccqppy_b200.solution_spaces; arbitrary "
                            "callables cannot run inside the CUDA solver and there is no CPU fallback")
        time_start = time.time()
        self._checkSolveInput(A, b, x0)
        if not self.quiet:
            print("solving " + self._label)

        sparse = _is_sparse(A)
        on_device = (_is_torch(A) or hasattr(A, "layout")) and A.is_cuda
        dev = A.device if on_device else None
        if on_device:
            device = A.device.index if A.device.index is not None else -1
        A32 = None if (sparse or symmetric) else _as_f32_matrix(A)
        A64 = None if (sparse or A32 is not None) else _as_f64(A)
        Ad = A32 if A32 is not None else A64
        # the vectors live where A lives (or where b lives, if only b is a CUDA tensor)
        vec_dev = dev if on_device else (b.device if (_is_torch(b) and b.is_cuda) else None)
        b64 = _as_f64(b, vec_dev)
        x064 = None if x0 is None else _as_f64(x0, vec_dev)
        if tuple(A.shape if sparse else Ad.shape) != (num_unknowns, num_unknowns):
            raise ValueError("A must be (n, n) with n = b.shape[0]")

        h = _capi.default_handle(device)
        lib = h.lib
        if on_device or vec_dev is not None:
            import torch
            with torch.cuda.device(dev if on_device else vec_dev):
                _capi.check(h.h, lib.ccqp_set_stream(h.h, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        if sparse:
            _ka = _set_sparse_matrix(h, A, num_unknowns)
        elif A32 is not None:
            h.set_matrix_f32(A32, num_unknowns)      # a host A is copied on the handle's stream before the solve's own copies
        else:
            pa, mem_a, _ka = _capi.f64_ptr(A64)
            lda = A64.stride(0) if _is_torch(A64) else num_unknowns
            if symmetric:
                _capi.check(h.h, lib.ccqp_set_matrix_symmetric(h.h, pa, num_unknowns, lda, mem_a))
            else:
                _capi.check(h.h, lib.ccqp_set_matrix(h.h, pa, num_unknowns, lda, 0, num_unknowns, mem_a))
        blocks, params, _rows = convex_proj_op.descriptor()
        pp, _, _kp = _capi.f64_ptr(params if params.size else np.zeros(1))
        _capi.check(h.h, lib.ccqp_set_projection(h.h, blocks.ptr, len(blocks), pp, params.size))

        rng_state = None
        uni = None
        if self._solver_id == _capi.SPG:
            if uniforms is None:
                rng_state, uni = self._draw_uniforms()
            else:
                uni = uniforms
            uni = _as_f64(uni, vec_dev)
        if vec_dev is not None:
            import torch
            xout = torch.empty(num_unknowns, dtype=torch.float64, device=vec_dev)
        else:
            xout = np.empty(num_unknowns, dtype=np.float64)
        pb, mem_v, _kb = _capi.f64_ptr(b64)
        px0, _, _kx = _capi.f64_ptr(x064)
        pu, _, _ku = _capi.f64_ptr(uni)
        pxo, _, _ko = _capi.f64_ptr(xout)
        prm = self._params()
        res = _capi.Result()
        st = lib.ccqp_solve(h.h, self._solver_id, ctypes.byref(prm), pb, px0, pu,
                            0 if uni is None else int(uni.shape[0]), pxo, mem_v, ctypes.byref(res))
        if rng_state is not None:
            self._restore_rng(rng_state, res.uniforms_used if st in (_capi.OK, _capi.ERR_RANGE) else 0)
        if st == _capi.ERR_NORMAL_NOT_IMPLEMENTED:
            raise NotImplementedError("Cone normal not implemented, yet.")      # solution_spaces.py:465
        if st == _capi.ERR_RANGE:
            raise OverflowError("Range exceeds valid bounds")                   # np.random.uniform(lo, nan)
        _capi.check(h.h, st)

        self._solution = xout
        self._solution_converged = bool(res.converged)
        self._solution_residual = float(res.residual)
        self._solution_num_matrix_vector_mults = int(res.mv_count)
        self._gpu_time = float(res.gpu_seconds)
        self._hbm_bytes = float(res.hbm_bytes)
        self._gemv_count = int(res.gemv_count)
        self._launches = int(res.kernel_launches)
        self._uniforms_used = int(res.uniforms_used)
        self._solution_time = time.time() - time_start
        return self

    def _batched_draws(self, batch):
        """Length of the per-problem U[0,1) stream for batched SPG when the caller gives none: one sample per
        iteration is consumed, iterations <= max_mv, so max_mv samples can never run out; capped so the
        host-drawn streams of the whole batch stay below 1 GiB (a problem that does run out is reported,
        never returned as converged)."""
        mx = self.max_matrix_vector_multiplications
        cap = max(256, (1 << 30) // (8 * max(int(batch), 1)))
        return max(1, int(min(mx, cap))) if np.isfinite(mx) else min(cap, 4096)

    def solve_batched(self, A, b, lower_bound=None, upper_bound=None, x0=None, seeds=None, uniforms=None, n_uniforms=None,
                      device=-1, convex_proj_op=None, symmetric=False, op_params=None):
        """Extension: solve `batch` independent constrained QPs in one persistent kernel.

        The feasible set is one of
          * per-problem boxes (`lower_bound` / `upper_bound` [batch, n]);
          * ONE operator of `ccqppy_b200.solution_spaces` shared by all problems (`convex_proj_op=op`, any block kinds:
            the contact-style case where every problem has the same friction-disc structure);
          * one block structure with per-problem parameters: `convex_proj_op=op, op_params=P`, P [batch, n_params]
            (NumPy or torch, host or device; a CUDA tensor is used in place when A is on the device), row i laid out as
            `op.descriptor()[1]` -- problem i is solved with op's blocks and the bounds / radii / aspect ratios of P[i],
            e.g. friction discs of radius mu * f_n computed on the GPU;
          * a sequence of `batch` operators `[op_0, ..., op_{batch-1}]` with identical `descriptor()` rows (kind, offset,
            dim, param_off): problem i is `solve(A[i], b[i], x0[i], op_i)`.  Their parameters are stacked into P.
        Tables run every solver except MPRGP (CCQPError).  A P of the wrong shape, a sequence of the wrong length or
        structure, `op_params` without `convex_proj_op` or together with bounds, and an operator of the wrong dimension
        raise ValueError before anything reaches the device.

        A [batch, n, n], b / lower_bound / upper_bound / x0 [batch, n] (NumPy or torch, host or
        device).  Problem i equals `type(self)(tol, max_mv).solve(A[i], b[i], x0[i],
        BoxProjOp(n, lb[i], ub[i]))` of the reference run after `np.random.seed(seeds[i])`.
        For SPG pass either `seeds` (the streams are drawn on the host with RandomState(seed))
        or `uniforms` [batch, K].  Results are per-problem arrays on the `solution*` properties;
        `solution_status` holds the per-problem ccqp_status raised inside the kernel.  A problem whose
        SPG step bound is NaN raises OverflowError (np.random.uniform does, solvers.py:959); a problem
        that used up its uniform stream raises CCQPError naming the problems (pass more samples).

        `symmetric=True` declares every A[i] symmetric (what the reference's objective assumes): with per-problem
        boxes, n <= 64 and PGD / BBPGD / BBPGDf / SPG the one-warp-per-problem kernels then read only the upper block
        triangle of A[i] (entries [r][c] with c >= 8 * (r // 8); `ccqp_solve_batched_sym`); every other case runs the
        general kernels.  The caller vouches for the symmetry: it is not checked.

        A float32 A (NumPy array, or a strided torch tensor on the host or on CUDA) is not widened: it goes to the `_f32`
        twin of the entry point (a contiguous CUDA tensor is read in place at any alignment, anything non-contiguous gets
        one contiguous float32 copy) and the results equal bit for bit those of `A.astype(np.float64)`.  Any other dtype
        is widened to float64.  An A that is not [batch, n, n] raises ValueError, a sparse torch tensor TypeError."""
        time_start = time.time()
        if not self.quiet:
            print("solving " + self._label)
        on_device = _is_torch(A) and A.is_cuda
        dev = A.device if on_device else None
        if on_device:
            device = A.device.index if A.device.index is not None else -1
        if _is_torch(A) and str(A.layout) != "torch.strided":
            raise TypeError("solve_batched takes a dense A [batch, n, n], got a %s tensor" % A.layout)
        A32 = _as_f32_matrix(A, aligned=False)      # a float32 batch stays float32 (the _f32 entry points)
        Ad = A32 if A32 is not None else _as_f64(A, dev)
        if Ad.ndim != 3 or Ad.shape[1] != Ad.shape[2]:
            raise ValueError("A must be [batch, n, n], got shape %s" % (tuple(Ad.shape),))
        batch, n = int(Ad.shape[0]), int(Ad.shape[1])
        b64 = _as_f64(b, dev)
        P64 = None          # per-problem parameter rows [batch, n_params], where A lives
        if op_params is not None and convex_proj_op is None:
            raise ValueError("op_params needs convex_proj_op: the operator that supplies the block structure")
        if convex_proj_op is not None:
            if lower_bound is not None or upper_bound is not None:
                raise ValueError("give either lower_bound / upper_bound or convex_proj_op")
            seq = isinstance(convex_proj_op, (list, tuple))     # one operator per problem
            ops = list(convex_proj_op) if seq else [convex_proj_op]
            if seq and op_params is not None:
                raise ValueError("give op_params with ONE operator (the structure), not with a sequence of operators")
            if seq and len(ops) != batch:
                raise ValueError("convex_proj_op has %d operators for %d problems" % (len(ops), batch))
            for i, op in enumerate(ops):
                if not isinstance(op, ss.ProjOpBase):
                    raise TypeError("convex_proj_op must be an operator from ccqppy_b200.solution_spaces (or a sequence of them)")
                if op.embedded_dimension != n:
                    raise ValueError("convex_proj_op%s has dimension %d, the problems %d" % (
                        "[%d]" % i if seq else "", op.embedded_dimension, n))
            if seq:
                blocks, op_params = ss.stacked_descriptor(ops)
                n_params = op_params.shape[1]
            else:
                blocks, params, _rows = convex_proj_op.descriptor()
                n_params = params.size
            if op_params is not None:
                shape = tuple(op_params.shape) if hasattr(op_params, "shape") else np.shape(op_params)
                if tuple(shape) != (batch, n_params):
                    raise ValueError("op_params has shape %s, expected (batch, n_params) = (%d, %d) (rows laid out as "
                                     "convex_proj_op.descriptor()[1])" % (tuple(shape), batch, n_params))
                P64 = _as_f64(op_params, dev)
                if dev is None and _is_torch(P64) and P64.is_cuda:
                    P64 = P64.cpu()                     # the rows live where A lives
            lb64 = ub64 = None
        else:
            if lower_bound is None or upper_bound is None:
                raise ValueError("lower_bound and upper_bound (or convex_proj_op) are required")
            lb64 = _as_f64(np.broadcast_to(lower_bound, (batch, n)) if isinstance(lower_bound, np.ndarray) else lower_bound, dev)
            ub64 = _as_f64(np.broadcast_to(upper_bound, (batch, n)) if isinstance(upper_bound, np.ndarray) else upper_bound, dev)
        x064 = None if x0 is None else _as_f64(x0, dev)
        uni = None
        K = 0
        if self._solver_id == _capi.SPG:
            if uniforms is None:
                if seeds is None:
                    seeds = np.arange(batch)
                if n_uniforms is None:
                    n_uniforms = self._batched_draws(batch)
                uniforms = np.empty((batch, n_uniforms))
                for i, s in enumerate(seeds):
                    uniforms[i] = np.random.RandomState(int(s)).random_sample(n_uniforms)
            uni = _as_f64(uniforms, dev)
            K = int(uni.shape[1])
        h = _capi.default_handle(device)
        lib = h.lib
        if on_device:
            import torch
            with torch.cuda.device(dev):
                _capi.check(h.h, lib.ccqp_set_stream(h.h, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
            xout = torch.empty((batch, n), dtype=torch.float64, device=dev)
        else:
            xout = np.empty((batch, n), dtype=np.float64)
        ptrs = [_capi.f64_ptr(Ad, "float64" if A32 is None else "float32")]
        ptrs += [_capi.f64_ptr(v) for v in (b64, x064, lb64, ub64, uni, xout)]
        f32 = "" if A32 is None else "_f32"            # the twin of each entry point that takes a float32 A
        mem = ptrs[0][1]
        results = (_capi.Result * batch)()
        summary = _capi.Result()
        prm = self._params()
        if P64 is not None:
            pp, _, _kp = _capi.f64_ptr(P64)
            entry = getattr(lib, "ccqp_solve_batched_tables" + f32)
            st = entry(h.h, self._solver_id, ctypes.byref(prm), batch, n, ptrs[0][0], ptrs[1][0], ptrs[2][0], blocks.ptr,
                       len(blocks), pp, int(P64.shape[1]), ptrs[5][0], K, ptrs[6][0], mem, results, ctypes.byref(summary))
        elif convex_proj_op is not None:
            pp, _, _kp = _capi.f64_ptr(params if params.size else np.zeros(1))
            entry = getattr(lib, "ccqp_solve_batched_table" + f32)
            st = entry(h.h, self._solver_id, ctypes.byref(prm), batch, n, ptrs[0][0], ptrs[1][0], ptrs[2][0], blocks.ptr,
                       len(blocks), pp, params.size, ptrs[5][0], K, ptrs[6][0], mem, results, ctypes.byref(summary))
        else:
            entry = getattr(lib, ("ccqp_solve_batched_sym" if symmetric else "ccqp_solve_batched") + f32)
            st = entry(h.h, self._solver_id, ctypes.byref(prm), batch, n, ptrs[0][0], ptrs[1][0],
                       ptrs[2][0], ptrs[3][0], ptrs[4][0], ptrs[5][0], K, ptrs[6][0], mem, results,
                       ctypes.byref(summary))
        _capi.check(h.h, st)
        rec = np.frombuffer(results, dtype=np.dtype([("residual", "f8"), ("gpu_seconds", "f8"), ("hbm_bytes", "f8"),
                                                     ("mv", "i8"), ("gemv", "i8"), ("it", "i8"), ("draws", "i8"),
                                                     ("conv", "i4"), ("status", "i4"), ("launches", "i8")]))
        self._solution = xout
        self._solution_residual = rec["residual"].copy()
        self._solution_converged = rec["conv"].astype(bool)
        self._solution_num_matrix_vector_mults = rec["mv"].copy()
        self._batched_status = rec["status"].copy()
        self._batched_records = rec.copy()          # every field of the per-problem ccqp_result (tools/)
        self._gpu_time = float(summary.gpu_seconds)
        self._hbm_bytes = float(summary.hbm_bytes)
        self._gemv_count = int(summary.gemv_count)
        self._launches = int(summary.kernel_launches)
        self._uniforms_used = rec["draws"].copy()
        self._solution_time = time.time() - time_start
        bad = np.flatnonzero(self._batched_status != _capi.OK)
        if bad.size:
            first = int(self._batched_status[bad[0]])
            which = ", ".join(str(int(i)) for i in bad[:8]) + (" ..." if bad.size > 8 else "")
            if first == _capi.ERR_RANGE:
                raise OverflowError("Range exceeds valid bounds (problems %s)" % which)     # np.random.uniform(lo, nan)
            raise _capi.CCQPError(first, "%s in %d of %d problems (%s); their results are marked not converged%s" % (
                _capi.load().ccqp_status_string(first).decode(), bad.size, batch, which,
                "; pass a longer `uniforms` stream / larger n_uniforms (used K = %d)" % K if first == _capi.ERR_UNIFORMS_EXHAUSTED else ""))
        return self

    # -- result properties, solvers.py:172-194 ---------------------------------------------------
    @property
    def name(self):
        return self._name

    @property
    def solution(self):
        return self._solution

    @property
    def solution_residual(self):
        return self._solution_residual

    @property
    def solution_converged(self):
        return self._solution_converged

    @property
    def solution_time(self):
        return self._solution_time

    @property
    def solution_num_matrix_vector_multiplications(self):
        return self._solution_num_matrix_vector_mults

    # -- accounting for the roofline (extension) -------------------------------------------------
    @property
    def solution_gpu_time(self):
        """Device seconds of the solver kernel (CUDA events)."""
        return self._gpu_time

    @property
    def solution_hbm_bytes(self):
        """Algorithmic bytes streamed: executed mat-vecs x (8 n^2 + 16 n)."""
        return self._hbm_bytes

    @property
    def solution_gemv_count(self):
        """Mat-vec products actually executed (the reported count skips some, SURVEY Q4)."""
        return self._gemv_count

    @property
    def solution_kernel_launches(self):
        return self._launches

    @property
    def solution_status(self):
        """Batched solves: per-problem ccqp_status raised inside the kernel (0 = none)."""
        return getattr(self, "_batched_status", None)


class CCQPSolverPGD(CCQPSolverBase):
    """solvers.py:71-194: fixed-step projected gradient."""
    _solver_id, _label, _name = _capi.PGD, "PGD", "PGD"

    def __init__(self, desired_residual_tol, max_matrix_vector_multiplications=np.inf, step_size=0.01):
        self._init_common(desired_residual_tol, max_matrix_vector_multiplications)
        self.step_size = step_size


class CCQPSolverAPGD(CCQPSolverBase):
    """solvers.py:197-367: accelerated projected gradient with Lipschitz backtracking."""
    _solver_id, _label, _name = _capi.APGD, "APGD", "APGD"

    def __init__(self, desired_residual_tol, max_matrix_vector_multiplications=np.inf):
        self._init_common(desired_residual_tol, max_matrix_vector_multiplications)


class CCQPSolverAPGDAntiRelaxation(CCQPSolverBase):
    """solvers.py:370-557: APGD with best-iterate tracking and adaptive restart."""
    _solver_id, _label, _name = _capi.APGD_AR, "APGD", "Anti-relaxation APGD"

    def __init__(self, desired_residual_tol, max_matrix_vector_multiplications=np.inf):
        self._init_common(desired_residual_tol, max_matrix_vector_multiplications)


class CCQPSolverBBPGD(CCQPSolverBase):
    """solvers.py:560-693: Barzilai-Borwein projected gradient.  (Name and print strings carry
    the reference's typos on purpose, Q11.)"""
    _solver_id, _label, _name = _capi.BBPGD, "BBPGDf", "BBGPD"

    def __init__(self, desired_residual_tol, max_matrix_vector_multiplications=np.inf):
        self._init_common(desired_residual_tol, max_matrix_vector_multiplications)


class CCQPSolverBBPGDf(CCQPSolverBase):
    """solvers.py:696-843: BBPGD with fallback to the best iterate on stagnation."""
    _solver_id, _label, _name = _capi.BBPGDF, "BBPGDf", "BBPDGf"

    def __init__(self, desired_residual_tol, max_matrix_vector_multiplications=np.inf):
        self._init_common(desired_residual_tol, max_matrix_vector_multiplications)


class CCQPSolverSPG(CCQPSolverBase):
    """solvers.py:846-999: spectral projected gradient with a non-monotone window and a random
    step drawn from the global NumPy RNG."""
    _solver_id, _label, _name = _capi.SPG, "SPG", "SPG-QP"

    def __init__(self, desired_residual_tol, max_matrix_vector_multiplications=np.inf,
                 m=5, tau=0.5, sigma1=0.01, sigma2=0.5):
        self._init_common(desired_residual_tol, max_matrix_vector_multiplications)
        self.m = m
        self.t = tau
        self.sigma1 = sigma1
        self.sigma2 = sigma2


class CCQPSolverMPRGP(CCQPSolverBase):
    """solvers.py:1002-1224: MPRGP with BB / expansion steps."""
    _solver_id, _label, _name = _capi.MPRGP, "MPRGP", "MPRGP"

    def __init__(self, desired_residual_tol, max_matrix_vector_multiplications=np.inf):
        self._init_common(desired_residual_tol, max_matrix_vector_multiplications)


# The README and north_star call it MPRGP-BB; the live reference class is CCQPSolverMPRGP (which
# already uses BB steps).  The old name only survives in stale docs (SURVEY.md section 0.1).
CCQPSolverMPRGPBB = CCQPSolverMPRGP
