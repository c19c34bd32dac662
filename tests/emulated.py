"""Driver of the C-ABI's emulated-ranks test vehicle (ccqp_debug_emulate_ranks / ccqp_debug_solve_emulated):
`world` handles on ONE GPU play the ranks of a row-sharded solve inside a single cooperative launch, so the
multi-GPU exchange protocol (fused all-gather into the peers' buffers, {data, epoch} packet all-reduce, cross-rank
barrier) is exercised on single-GPU test boxes.  Mirrors ccqppy_b200.dist.ShardedSolver."""
import ctypes

import numpy as np

from ccqppy_b200 import _capi
from ccqppy_b200.dist import shard_rows


class EmulatedBox:
    def __init__(self, A, op, world, device=-1):
        """A: dense (n, n) NumPy array or scipy.sparse matrix; op: a ccqppy_b200.solution_spaces operator."""
        self.world, self.op = world, op
        self.n = n = int(A.shape[0])
        blocks, params, rows = op.descriptor()
        self.ranges = shard_rows(rows, n, world)
        self.handles = [_capi.Handle(device) for _ in range(world)]
        self.lib = self.handles[0].lib
        self.harr = (ctypes.c_void_p * world)(*[h.h for h in self.handles])
        _capi.check(self.handles[0].h, self.lib.ccqp_debug_emulate_ranks(self.harr, world, n))
        self.keep = []
        par = np.ascontiguousarray(params if params.size else np.zeros(1))
        for r, h in enumerate(self.handles):
            r0, r1 = self.ranges[r]
            if hasattr(A, "tocsr"):
                csr = A.tocsr()[r0:r1]
                csr.sum_duplicates()
                ptr = np.ascontiguousarray(csr.indptr, dtype=np.int64)
                idx = np.ascontiguousarray(csr.indices, dtype=np.int32)
                val = np.ascontiguousarray(csr.data, dtype=np.float64)
                self.keep.append((ptr, idx, val))
                _capi.check(h.h, self.lib.ccqp_set_matrix_csr(h.h, ctypes.c_void_p(ptr.ctypes.data), ctypes.c_void_p(idx.ctypes.data),
                                                              ctypes.c_void_p(val.ctypes.data), n, int(val.size), r0, r1 - r0,
                                                              _capi.MEM_HOST))
            else:
                shard = np.ascontiguousarray(A[r0:r1], dtype=np.float64)
                self.keep.append(shard)
                _capi.check(h.h, self.lib.ccqp_set_matrix(h.h, ctypes.c_void_p(shard.ctypes.data), n, n, r0, r1 - r0, _capi.MEM_HOST))
            _capi.check(h.h, self.lib.ccqp_set_projection(h.h, blocks.ptr, len(blocks), ctypes.c_void_p(par.ctypes.data), params.size))
        self.keep.append((blocks, par))

    def solve(self, solver, b, x0=None, uniforms=None):
        """solver: a ccqppy_b200.solvers object (tolerance / limits / hyper-parameters).  Returns a list of
        per-rank dicts (solution, mv, gemv, converged, residual, status, draws = SPG uniforms consumed)."""
        n, world = self.n, self.world
        b64 = np.ascontiguousarray(b, dtype=np.float64)
        x064 = None if x0 is None else np.ascontiguousarray(x0, dtype=np.float64)
        uni = None if uniforms is None else np.ascontiguousarray(uniforms, dtype=np.float64)
        xout = np.empty((world, n))
        res = (_capi.Result * world)()
        prm = solver._params()
        P = lambda a: None if a is None else ctypes.c_void_p(a.ctypes.data)
        st = self.lib.ccqp_debug_solve_emulated(self.harr, world, solver._solver_id, ctypes.byref(prm), P(b64), P(x064), P(uni),
                                                0 if uni is None else int(uni.size), P(xout), _capi.MEM_HOST, res)
        if st == _capi.ERR_NORMAL_NOT_IMPLEMENTED:
            raise NotImplementedError("Cone normal not implemented, yet.")
        _capi.check(self.handles[0].h, st)
        return [dict(solution=xout[r].copy(), mv=int(res[r].mv_count), gemv=int(res[r].gemv_count), converged=bool(res[r].converged),
                     residual=float(res[r].residual), status=int(res[r].status), gpu_seconds=float(res[r].gpu_seconds),
                     draws=int(res[r].uniforms_used))
                for r in range(world)]

    def close(self):
        for h in self.handles:
            h.close()
