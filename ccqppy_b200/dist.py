"""Row-sharded dense solves on several B200s of one box (one process per GPU, e.g. torchrun).

Nothing in the reference corresponds to this module (it is single-process NumPy); it is the
"scale n" mechanism of SURVEY.md section 8(e).  The Hessian is split by rows; every rank runs the
SAME persistent solver kernel on its rows and, inside the kernel, writes its slice of each mat-vec
input vector and its scalar partial sums directly into the peers' buffers over NVLink.
torch.distributed is only plumbing here: it carries the 128-byte CUDA-IPC descriptors at setup and
provides the host barrier in front of each launch.

    runner = ShardedSolver(solvers.CCQPSolverSPG(1e-5, 2000), A_rows_or_full, op)
    r = runner.solve(b)            # every rank gets the full solution and identical fields
"""
import ctypes

import numpy as np

from . import _capi
from . import solution_spaces as ss
from .solvers import _as_f32_matrix

NORM_KINDS = (_capi.SPHERE, _capi.CONE_REF, _capi.SOC)


def shard_rows(rows, n, world):
    """Row ranges [(r0, r1)] * world, as even as possible, with every boundary on a projection
    block boundary (a norm-type block must live on one rank; elementwise blocks can be cut
    anywhere).  rows: [(kind, offset, dim, param_off)]."""
    if world < 1 or world > n:
        raise ValueError("cannot split %d rows over %d ranks" % (n, world))
    spans = [(int(off), int(off) + int(dim)) for kind, off, dim, _ in rows if int(kind) in NORM_KINDS and int(dim) > 1]
    starts = np.array([a for a, _ in spans], dtype=np.int64)
    ends = np.array([b for _, b in spans], dtype=np.int64)
    bounds = [0]
    for r in range(1, world):
        cut = (r * n + world // 2) // world
        if len(starts):
            k = int(np.searchsorted(starts, cut, side="right")) - 1
            if k >= 0 and starts[k] < cut < ends[k]:          # inside a norm block: move to its nearer end
                lo, hi = int(starts[k]), int(ends[k])
                cut = lo if (cut - lo) <= (hi - cut) else hi
        bounds.append(int(cut))
    bounds.append(n)
    if any(b1 <= b0 for b0, b1 in zip(bounds[:-1], bounds[1:])):
        raise ValueError("projection blocks are too coarse to give each of %d ranks some rows" % world)
    return [(bounds[i], bounds[i + 1]) for i in range(world)]


def exchange_descriptors(desc, group=None):
    """All-gather the opaque per-rank descriptors (bytes).  Works on any backend."""
    import torch.distributed as dist
    out = [None] * dist.get_world_size(group)
    dist.all_gather_object(out, bytes(desc), group=group)
    return b"".join(out)


def batch_range(batch, rank, world):
    """Contiguous share [i0, i1) of `batch` independent problems for `rank` (sizes differ by at most 1)."""
    base, extra = divmod(int(batch), int(world))
    i0 = rank * base + min(rank, extra)
    return i0, i0 + base + (1 if rank < extra else 0)


def solve_batched_sharded(solver, A, b, lower_bound, upper_bound, x0=None, seeds=None, uniforms=None, n_uniforms=None,
                          gather=True, group=None):
    """Batched mode on several GPUs: the problems are independent, so every rank solves its contiguous
    share on its own GPU and there is NO communication on the data path (SURVEY.md section 8e).
    The arguments are the FULL batch (NumPy / torch; each rank only touches its share).  With
    `gather` the per-problem results are all-gathered afterwards so that every rank returns the whole
    batch; otherwise each rank keeps its share.  Returns (solution, residual, converged, mv, (i0, i1))."""
    import torch
    import torch.distributed as dist
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    batch = int(A.shape[0])
    i0, i1 = batch_range(batch, rank, world)
    cut = lambda v: None if v is None else v[i0:i1]
    if seeds is None and uniforms is None:
        seeds = np.arange(batch)
    solver.solve_batched(cut(A), cut(b), cut(lower_bound), cut(upper_bound), x0=cut(x0), seeds=cut(seeds),
                         uniforms=cut(uniforms), n_uniforms=n_uniforms)
    dev = torch.device("cuda", torch.cuda.current_device())
    x = solver.solution if hasattr(solver.solution, "is_cuda") else torch.from_numpy(np.ascontiguousarray(solver.solution))
    x = x.to(dev)
    res = torch.from_numpy(np.ascontiguousarray(solver.solution_residual)).to(dev)
    conv = torch.from_numpy(solver.solution_converged.astype(np.int64)).to(dev)
    mv = torch.from_numpy(np.ascontiguousarray(solver.solution_num_matrix_vector_multiplications, dtype=np.int64)).to(dev)
    if not gather or world == 1:
        return x, res, conv.bool(), mv, (i0, i1)
    n = int(x.shape[1])
    cap = (batch + world - 1) // world                      # all_gather wants equal shapes: pad the short shares
    pack = torch.zeros((cap, n + 3), dtype=torch.float64, device=dev)
    pack[:i1 - i0, :n] = x
    pack[:i1 - i0, n] = res
    pack[:i1 - i0, n + 1] = conv.double()
    pack[:i1 - i0, n + 2] = mv.double()
    parts = [torch.empty_like(pack) for _ in range(world)]
    dist.all_gather(parts, pack, group=group)
    full = torch.cat([parts[r][:batch_range(batch, r, world)[1] - batch_range(batch, r, world)[0]] for r in range(world)])
    return full[:, :n].contiguous(), full[:, n].contiguous(), full[:, n + 1] > 0.5, full[:, n + 2].long(), (i0, i1)


class ShardedResult:
    """Result fields of one sharded solve (same names as the solver properties)."""


class ShardedSolver:
    """Binds a solver object (its tolerance / limits / hyper-parameters), one row shard of A and the
    full projection table to this rank's GPU.  `A` is either this rank's rows (`row_range` given)
    or the full matrix (the shard is sliced out; nothing is copied for a CUDA tensor).  A float32 A keeps float32
    shards (`ccqp_set_matrix_f32`), with the bits of the widened matrix's solve."""

    def __init__(self, solver, A, convex_proj_op=None, rank=None, world=None, device=None, row_range=None, group=None):
        import torch
        import torch.distributed as dist
        self.solver = solver
        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world = dist.get_world_size(group) if world is None else world
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        n = int(A.shape[1])
        self.n = n
        self.op = convex_proj_op if convex_proj_op is not None else ss.IdentityProjOp(n)
        blocks, params, rows = self.op.descriptor()
        self.ranges = shard_rows(rows, n, self.world)
        r0, r1 = self.ranges[self.rank]
        self.h = _capi.Handle(self.device.index)
        lib = self.h.lib
        stream = torch.cuda.current_stream(self.device).cuda_stream
        _capi.check(self.h.h, lib.ccqp_set_stream(self.h.h, ctypes.c_void_p(stream)))
        if hasattr(A, "tocsr"):
            # operator-form Hessian (scipy.sparse): this rank keeps rows [r0, r1) of the CSR arrays
            if row_range is not None:
                raise ValueError("a sparse A is given in full; the shard is sliced here")
            csr = A.tocsr()[r0:r1]
            csr.sum_duplicates()
            self.shard = (torch.from_numpy(np.ascontiguousarray(csr.indptr, dtype=np.int64)).to(self.device),
                          torch.from_numpy(np.ascontiguousarray(csr.indices, dtype=np.int32)).to(self.device),
                          torch.from_numpy(np.ascontiguousarray(csr.data, dtype=np.float64)).to(self.device))
            ptr, idx, val = self.shard
            _capi.check(self.h.h, lib.ccqp_set_matrix_csr(self.h.h, ctypes.c_void_p(ptr.data_ptr()), ctypes.c_void_p(idx.data_ptr()),
                                                          ctypes.c_void_p(val.data_ptr()), n, int(val.numel()), r0, r1 - r0,
                                                          _capi.MEM_DEVICE))
        else:
            if row_range is not None:
                if tuple(row_range) != (r0, r1):
                    raise ValueError("row_range %s does not match the block-aligned split %s" % (row_range, (r0, r1)))
                shard = A
            else:
                shard = A[r0:r1]
            A32 = _as_f32_matrix(shard)
            if A32 is not None:
                self.shard = A32 if (hasattr(A32, "is_cuda") and A32.is_cuda) else torch.as_tensor(A32).to(self.device)
                self.h.set_matrix_f32(self.shard, n, r0, r1 - r0)
            else:
                if not (hasattr(shard, "is_cuda") and shard.is_cuda):
                    shard = torch.as_tensor(np.ascontiguousarray(shard, dtype=np.float64)).to(self.device)
                self.shard = shard.to(dtype=torch.float64).contiguous()     # keeps the storage alive
                _capi.check(self.h.h, lib.ccqp_set_matrix(self.h.h, ctypes.c_void_p(self.shard.data_ptr()), n,
                                                          self.shard.stride(0), r0, r1 - r0, _capi.MEM_DEVICE))
        pp, _, _keep = _capi.f64_ptr(params if params.size else np.zeros(1))
        _capi.check(self.h.h, lib.ccqp_set_projection(self.h.h, blocks.ptr, len(blocks), pp, params.size))
        if self.world > 1:
            desc = (ctypes.c_ubyte * 128)()
            _capi.check(self.h.h, lib.ccqp_comm_export(self.h.h, self.rank, self.world, n, desc))
            alld = exchange_descriptors(bytes(desc), group)
            self._alld = ctypes.create_string_buffer(alld, len(alld))
            _capi.check(self.h.h, lib.ccqp_comm_attach(self.h.h, self._alld))

    def set_matrix(self, shard):
        """Replace this rank's rows of A.  `shard` is [r1 - r0, n]: a CUDA tensor (borrowed in place) or a
        host array / CPU tensor (copied to the device by the library; pinned memory makes the copy
        asynchronous); a float32 shard stays float32.  Every rank must call it before the next solve()."""
        import torch
        r0, r1 = self.ranges[self.rank]
        if tuple(shard.shape) != (r1 - r0, self.n):
            raise ValueError("shard must be %s" % ((r1 - r0, self.n),))
        lib = self.h.lib
        A32 = _as_f32_matrix(shard)
        if A32 is not None:
            self.shard = A32
            self.h.set_matrix_f32(A32, self.n, r0, r1 - r0)
            return
        if hasattr(shard, "is_cuda") and shard.is_cuda:
            self.shard = shard.to(dtype=torch.float64).contiguous()
            ptr, lda, mem = self.shard.data_ptr(), self.shard.stride(0), _capi.MEM_DEVICE
        else:
            if hasattr(shard, "numpy"):
                self.shard = shard.to(dtype=torch.float64).contiguous()
                ptr, lda = self.shard.data_ptr(), self.shard.stride(0)
            else:
                self.shard = np.ascontiguousarray(shard, dtype=np.float64)
                ptr, lda = self.shard.ctypes.data, self.n
            mem = _capi.MEM_HOST
        _capi.check(self.h.h, lib.ccqp_set_matrix(self.h.h, ctypes.c_void_p(ptr), self.n, lda, r0, r1 - r0, mem))

    def _to_dev(self, v):
        import torch
        if hasattr(v, "is_cuda"):
            return v.to(device=self.device, dtype=torch.float64).contiguous()
        return torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).to(self.device)

    def solve(self, b, x0=None, uniforms=None):
        import torch
        import torch.distributed as dist
        s, lib, h = self.solver, self.h.lib, self.h
        n, dev = self.n, self.device
        b64 = self._to_dev(b)
        x064 = None if x0 is None else self._to_dev(x0)
        uni, state = None, None
        if s._solver_id == _capi.SPG:
            if uniforms is None:
                # the reference draws from the global NumPy RNG: rank 0's stream is the one that counts
                state, u = s._draw_uniforms()
                uni = torch.from_numpy(u).to(dev)
                if self.world > 1:
                    dist.broadcast(uni, src=0, group=self.group)
            else:
                uni = self._to_dev(uniforms)
        xout = torch.empty(n, dtype=torch.float64, device=dev)
        if self.world > 1:
            _capi.check(h.h, lib.ccqp_comm_prepare(h.h))
            torch.cuda.synchronize(dev)
            dist.barrier(group=self.group)
        prm = s._params()
        res = _capi.Result()
        st = lib.ccqp_solve(h.h, s._solver_id, ctypes.byref(prm), ctypes.c_void_p(b64.data_ptr()),
                            None if x064 is None else ctypes.c_void_p(x064.data_ptr()),
                            None if uni is None else ctypes.c_void_p(uni.data_ptr()),
                            0 if uni is None else int(uni.shape[0]),
                            ctypes.c_void_p(xout.data_ptr()), _capi.MEM_DEVICE, ctypes.byref(res))
        if state is not None:
            s._restore_rng(state, res.uniforms_used)
        if st == _capi.ERR_NORMAL_NOT_IMPLEMENTED:
            raise NotImplementedError("Cone normal not implemented, yet.")
        if st == _capi.ERR_RANGE:
            raise OverflowError("Range exceeds valid bounds")
        _capi.check(h.h, st)
        r = ShardedResult()
        r.solution = xout
        r.solution_converged = bool(res.converged)
        r.solution_residual = float(res.residual)
        r.solution_num_matrix_vector_multiplications = int(res.mv_count)
        r.solution_gpu_time = float(res.gpu_seconds)
        r.solution_hbm_bytes = float(res.hbm_bytes)
        r.solution_gemv_count = int(res.gemv_count)
        r.solution_kernel_launches = int(res.kernel_launches)
        return r

    def close(self):
        self.h.close()
