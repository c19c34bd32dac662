"""Feasible sets: host-side mirror of the reference's `ccqppy.solution_spaces`
(/root/reference/src/ccqppy/solution_spaces.py) in front of the CUDA projection kernels.

Same class names, constructor arguments, public attributes and `name` strings as the reference
(SURVEY.md section 8b), so `ss.BoxProjOp(3, lb, ub)` etc. are drop-ins.  What differs is where the
arithmetic happens: `op(x)` and `op.normal_vector(x)` run on the GPU through the C-ABI
(`ccqp_project` / `ccqp_normal`); inside a solve the operator is never called from Python at all,
it is handed to the solver kernel as a flat block table (`descriptor()`).

`projected_gradient(x, g)` (SURVEY.md section 8 row f-4; no live solver of the reference calls it) is
mirrored too, behaviour for behaviour: Lower / Upper / Box / Disjoint run on the GPU
(`ccqp_projected_gradient`), Identity returns None, Sphere raises NotImplementedError, Cone has no such
method (only `proximal_gradient`, which raises), a Disjoint with an Identity member raises TypeError.
Out of scope, as in SURVEY.md section 2: `plot` (presentation code).
"""
from abc import ABC, abstractmethod

import numpy as np

from . import _capi

__all__ = ["ProjOpBase", "IdentityProjOp", "LowerBoundProjOp", "UpperBoundProjOp", "BoxProjOp",
           "SphereProjOp", "ConeProjOp", "SOCProjOp", "DisjointProjOp"]

_proj_handle = None


def _handle():
    global _proj_handle
    if _proj_handle is None:
        _proj_handle = _capi.Handle()
    return _proj_handle


class _ParamBuf:
    """Growing parameter array of a block table (chunks are concatenated once at the end)."""

    def __init__(self):
        self.chunks, self.size = [], 0

    def __len__(self):
        return self.size

    def extend(self, arr):
        arr = np.asarray(arr, dtype=np.float64).ravel()
        self.chunks.append(arr)
        self.size += arr.size

    def append(self, value):
        self.extend([float(value)])

    def array(self):
        return np.concatenate(self.chunks) if self.chunks else np.zeros(0)


def _per_element(value, dim, default):
    if value is None:
        return np.full(dim, float(default))
    return np.ascontiguousarray(np.broadcast_to(np.asarray(value, dtype=np.float64), (dim,)))


class ProjOpBase(ABC):
    """solution_spaces.py:9-74.  Subclasses provide `_blocks(offset, params)`."""

    def __init__(self, embedded_dimension):
        self.dim = embedded_dimension

    @property
    @abstractmethod
    def name(self):
        """Name of the projection operator."""

    @property
    def embedded_dimension(self):
        return self.dim

    @abstractmethod
    def _blocks(self, offset, params):
        """Append this operator's parameters to `params` (a _ParamBuf) and return its block rows
        [(kind, offset, dim, param_off), ...]."""

    def descriptor(self):
        """Flat block table for the C-ABI: (ctypes ccqp_block array, float64 params array)."""
        params = _ParamBuf()
        rows = self._blocks(0, params)
        return _capi.make_blocks(rows), params.array(), rows

    # -- GPU evaluation through the unit-test hooks of the ABI --------------------------------
    def _run(self, fn_name, x):
        is_torch = not isinstance(x, np.ndarray) and hasattr(x, "data_ptr")
        if is_torch:
            xin = x.to(dtype=__import__("torch").float64).contiguous()
            out = xin.new_empty(xin.shape)
        else:
            xin = np.ascontiguousarray(x, dtype=np.float64)
            out = np.empty_like(xin)
        if xin.shape[0] != self.dim:
            raise ValueError("expected a vector of length %d" % self.dim)
        h = _handle()
        blocks, params, _ = self.descriptor()
        pp, _, _k1 = _capi.f64_ptr(params if params.size else np.zeros(1))
        _capi.check(h.h, h.lib.ccqp_set_projection(h.h, blocks.ptr, len(blocks), pp, params.size))
        px, mem, _k2 = _capi.f64_ptr(xin)
        po, _, _k3 = _capi.f64_ptr(out)
        st = getattr(h.lib, fn_name)(h.h, px, po, mem)
        if st == _capi.ERR_NORMAL_NOT_IMPLEMENTED:
            raise NotImplementedError("Cone normal not implemented, yet.")   # solution_spaces.py:465
        _capi.check(h.h, st)
        return out

    def __call__(self, x):
        """P(x), evaluated by the CUDA projection kernel."""
        return self._run("ccqp_project", x)

    def normal_vector(self, x):
        """Outward unit normal at x (zero inside / when x is infeasible), on the GPU."""
        return self._run("ccqp_normal", x)

    def _projected_gradient_gpu(self, x, g):
        """(free gradient, chopped gradient) through ccqp_projected_gradient; NumPy in, NumPy out."""
        xin = np.ascontiguousarray(x, dtype=np.float64)
        gin = np.ascontiguousarray(g, dtype=np.float64)
        if xin.shape[0] != self.dim or gin.shape[0] != self.dim:
            raise ValueError("expected vectors of length %d" % self.dim)
        free, chopped = np.empty_like(xin), np.empty_like(xin)
        h = _handle()
        blocks, params, _ = self.descriptor()
        pp, _, _k1 = _capi.f64_ptr(params if params.size else np.zeros(1))
        _capi.check(h.h, h.lib.ccqp_set_projection(h.h, blocks.ptr, len(blocks), pp, params.size))
        P = lambda a: _capi.f64_ptr(a)[0]
        _capi.check(h.h, h.lib.ccqp_projected_gradient(h.h, P(xin), P(gin), P(free), P(chopped), _capi.MEM_HOST))
        return free, chopped

    def plot(self, *args, **kwargs):
        raise NotImplementedError("plot() is presentation code of the reference and out of scope here")


class IdentityProjOp(ProjOpBase):
    """solution_spaces.py:77-125"""

    @property
    def name(self):
        return "Identity"

    def _blocks(self, offset, params):
        return [(_capi.IDENTITY, offset, self.dim, len(params))]

    def __call__(self, x):
        return x            # the reference returns its argument (alias), :125

    def projected_gradient(self, x, g):
        """solution_spaces.py:100-109: the reference's method has a docstring and no body, so it returns None."""
        return None


class LowerBoundProjOp(ProjOpBase):
    """solution_spaces.py:128-201; default bound -1."""

    def __init__(self, embedded_dimension, lower_bound=None):
        self.dim = embedded_dimension
        self.lower_bound = lower_bound if lower_bound is not None else -np.ones(embedded_dimension)

    @property
    def name(self):
        return "Lower Bound"

    def _blocks(self, offset, params):
        poff = len(params)
        params.extend(_per_element(self.lower_bound, self.dim, -1.0))
        return [(_capi.LOWER, offset, self.dim, poff)]

    def projected_gradient(self, x, g):
        """(free gradient, chopped gradient) at x, solution_spaces.py:162-184, on the GPU."""
        return self._projected_gradient_gpu(x, g)


class UpperBoundProjOp(ProjOpBase):
    """solution_spaces.py:204-277; default bound +1."""

    def __init__(self, embedded_dimension, upper_bound=None):
        self.dim = embedded_dimension
        self.upper_bound = upper_bound if upper_bound is not None else np.ones(embedded_dimension)

    @property
    def name(self):
        return "Upper Bound"

    def _blocks(self, offset, params):
        poff = len(params)
        params.extend(_per_element(self.upper_bound, self.dim, 1.0))
        return [(_capi.UPPER, offset, self.dim, poff)]

    def projected_gradient(self, x, g):
        """(free gradient, chopped gradient) at x, solution_spaces.py:238-260, on the GPU."""
        return self._projected_gradient_gpu(x, g)


class BoxProjOp(ProjOpBase):
    """solution_spaces.py:280-366; defaults [-1, 1].  Like the reference, ub > lb is not enforced."""

    def __init__(self, embedded_dimension, lower_bound=None, upper_bound=None):
        self.dim = embedded_dimension
        self.lower_bound = lower_bound if lower_bound is not None else -np.ones(embedded_dimension)
        self.upper_bound = upper_bound if upper_bound is not None else np.ones(embedded_dimension)

    @property
    def name(self):
        return "Box"

    def _blocks(self, offset, params):
        poff = len(params)
        params.extend(_per_element(self.lower_bound, self.dim, -1.0))
        params.extend(_per_element(self.upper_bound, self.dim, 1.0))
        return [(_capi.BOX, offset, self.dim, poff)]

    def projected_gradient(self, x, g):
        """(free gradient, chopped gradient) at x, solution_spaces.py:324-347 (the activity test of :339-340 as written), on the GPU."""
        return self._projected_gradient_gpu(x, g)


class SphereProjOp(ProjOpBase):
    """solution_spaces.py:369-435; default radius 1."""

    def __init__(self, embedded_dimension, radius=None):
        self.dim = embedded_dimension
        self.radius = radius if radius is not None else 1

    @property
    def name(self):
        return "Sphere"

    def _blocks(self, offset, params):
        poff = len(params)
        params.append(float(self.radius))
        return [(_capi.SPHERE, offset, self.dim, poff)]

    def projected_gradient(self, x, g):
        raise NotImplementedError("Cone proximal gradient not implemented, yet.")     # solution_spaces.py:415, as written


class ConeProjOp(ProjOpBase):
    """solution_spaces.py:438-492.  Bug-compatible with the reference, whose own source says
    "This projection op is bugged" (:439): the norm runs over the whole vector and the result is
    not a projection.  `normal_vector` raises NotImplementedError like the reference (:465), so
    MPRGP cannot be used with it.  Use `SOCProjOp` for a correct second-order cone."""

    def __init__(self, embedded_dimension, aspect_ratio=None):
        self.dim = embedded_dimension
        self.aspect_ratio = aspect_ratio if aspect_ratio is not None else 1

    @property
    def name(self):
        return "Cone"

    def _blocks(self, offset, params):
        poff = len(params)
        params.append(float(self.aspect_ratio))
        return [(_capi.CONE_REF, offset, self.dim, poff)]

    def proximal_gradient(self, x, g):
        raise NotImplementedError("Cone proximal gradient not implemented, yet.")     # solution_spaces.py:467-468


class SOCProjOp(ProjOpBase):
    """Extension (not in the reference; parity unpinned): Euclidean projection onto the
    second-order cone {(u, z) : |u| <= mu z}, the friction cone of contact problems."""

    def __init__(self, embedded_dimension, aspect_ratio=None):
        self.dim = embedded_dimension
        self.aspect_ratio = aspect_ratio if aspect_ratio is not None else 1

    @property
    def name(self):
        return "SOC"

    def _blocks(self, offset, params):
        poff = len(params)
        params.append(float(self.aspect_ratio))
        return [(_capi.SOC, offset, self.dim, poff)]


def stacked_descriptor(ops):
    """Extension (not star-exported).  Block table shared by a sequence of operators and their parameter arrays stacked
    row by row: (ctypes ccqp_block array, float64 [len(ops), n_params]).  Row i is exactly `ops[i].descriptor()[1]`.  The operators must have the same
    block structure -- identical `descriptor()` rows (kind, offset, dim, param_off) -- or ValueError names the first one
    that differs.  This is the input of a batched solve with per-problem parameters (`solve_batched`)."""
    ops = list(ops)
    if not ops:
        raise ValueError("stacked_descriptor needs at least one operator")
    blocks, first, rows = ops[0].descriptor()
    ref = np.asarray(rows, dtype=np.int64).reshape(-1, 4)
    P = np.empty((len(ops), first.size))
    P[0] = first
    for i, op in enumerate(ops[1:], 1):
        _, par, r = op.descriptor()
        r = np.asarray(r, dtype=np.int64).reshape(-1, 4)
        if r.shape != ref.shape or not np.array_equal(r, ref) or par.size != first.size:
            raise ValueError("operator %d has a different block structure (kind, offset, dim, param_off) than operator 0" % i)
        P[i] = par
    return blocks, P


class DisjointProjOp(ProjOpBase):
    """solution_spaces.py:495-560: concatenation of operators acting on consecutive slices."""

    def __init__(self, *convex_proj_ops):
        self.proj_ops = convex_proj_ops
        self.dim = 0
        for op in self.proj_ops:
            self.dim += op.embedded_dimension
        self._desc = None

    def descriptor(self):
        # flattening ~1e4 Python operator objects costs tens of ms; the tuple of operators is fixed
        # at construction, so the table is built once (call invalidate() after mutating a member)
        if self._desc is None:
            self._desc = super().descriptor()
        return self._desc

    def invalidate(self):
        self._desc = None

    @property
    def name(self):
        return "DisjointUnion"

    def projected_gradient(self, x, g):
        """solution_spaces.py:527-538: every member's projected_gradient on its slice.  Like the reference: a member
        without the method (Cone) raises AttributeError, Sphere raises NotImplementedError, and an Identity member --
        whose method returns None -- makes the tuple unpacking raise TypeError.  Otherwise one GPU pass."""
        def check(members):
            for op in members:
                if isinstance(op, DisjointProjOp):
                    check(op.proj_ops)
                elif not hasattr(op, "projected_gradient"):
                    raise AttributeError("'%s' object has no attribute 'projected_gradient'" % type(op).__name__)
                elif isinstance(op, SphereProjOp):
                    raise NotImplementedError("Cone proximal gradient not implemented, yet.")
                elif isinstance(op, IdentityProjOp):
                    raise TypeError("cannot unpack non-iterable NoneType object")
        check(self.proj_ops)
        return self._projected_gradient_gpu(x, g)

    def _blocks(self, offset, params):
        rows = []
        cache = {}
        for op in self.proj_ops:
            # benchmarks build [Op(3)] * (n // 3): share the parameters of repeated objects
            key = id(op)
            if key in cache and not isinstance(op, DisjointProjOp):
                kind, dim, poff = cache[key]
                rows.append((kind, offset, dim, poff))
            else:
                sub = op._blocks(offset, params)
                if len(sub) == 1:
                    cache[key] = (sub[0][0], sub[0][2], sub[0][3])
                rows.extend(sub)
            offset += op.embedded_dimension
        return rows
