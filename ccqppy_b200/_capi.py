"""ctypes binding of the C-ABI in include/ccqp_b200.h (the only way the package computes).

There is deliberately no CPU fallback: if the shared library is missing, or there is no B200,
every compute entry point raises."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# CCQP_B200_LIB: tuning hook, points at a variant build of the same library (tools/sweep_*.py)
LIB_PATH = os.environ.get("CCQP_B200_LIB") or os.path.join(_HERE, "csrc", "libccqp_b200.so")

MEM_HOST, MEM_DEVICE = 0, 1
(IDENTITY, LOWER, UPPER, BOX, SPHERE, CONE_REF, SOC) = range(7)
(PGD, APGD, APGD_AR, BBPGD, BBPGDF, SPG, MPRGP) = range(7)

OK = 0
ERR_NORMAL_NOT_IMPLEMENTED = 6
ERR_UNIFORMS_EXHAUSTED = 7
ERR_RANGE = 8

EXPORTS = ["ccqp_abi_version", "ccqp_status_string", "ccqp_last_error", "ccqp_create", "ccqp_destroy",
           "ccqp_set_stream", "ccqp_get_info", "ccqp_set_matrix", "ccqp_set_matrix_csr", "ccqp_set_projection", "ccqp_solve", "ccqp_solve_async", "ccqp_solve_wait",
           "ccqp_solve_batched", "ccqp_gemv", "ccqp_gemv_timed", "ccqp_project", "ccqp_normal", "ccqp_comm_export",
           "ccqp_comm_attach", "ccqp_comm_prepare", "ccqp_comm_detach", "ccqp_debug_divide", "ccqp_fp64_peak",
           "ccqp_microbench", "ccqp_debug_emulate_ranks", "ccqp_debug_solve_emulated", "ccqp_projected_gradient", "ccqp_solve_batched_table", "ccqp_solve_batched_sym",
           "ccqp_get_upload_info", "ccqp_set_matrix_symmetric", "ccqp_host_matrix_is_block_symmetric", "ccqp_upload_block_rows",
           "ccqp_set_matrix_f32", "ccqp_solve_batched_tables", "ccqp_solve_batched_f32", "ccqp_solve_batched_sym_f32",
           "ccqp_solve_batched_table_f32", "ccqp_solve_batched_tables_f32"]


class Block(C.Structure):
    _fields_ = [("kind", C.c_int32), ("reserved", C.c_int32), ("offset", C.c_int64), ("dim", C.c_int64),
                ("param_off", C.c_int64)]


class Params(C.Structure):
    _fields_ = [("tol", C.c_double), ("max_mv", C.c_double), ("step_size", C.c_double), ("tau", C.c_double),
                ("sigma1", C.c_double), ("sigma2", C.c_double), ("m", C.c_int32), ("reserved", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("residual", C.c_double), ("gpu_seconds", C.c_double), ("hbm_bytes", C.c_double),
                ("mv_count", C.c_int64), ("gemv_count", C.c_int64), ("iterations", C.c_int64),
                ("uniforms_used", C.c_int64), ("converged", C.c_int32), ("status", C.c_int32),
                ("kernel_launches", C.c_int64)]


class CCQPError(RuntimeError):
    def __init__(self, status, text):
        super().__init__("ccqp_b200: %s (status %d)" % (text, status))
        self.status = status


_lib = None


def load():
    """Load the shared library (no GPU needed for that) and declare the signatures."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: run `python -m ccqppy_b200.build` (needs nvcc). "
                          "ccqppy_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, dp, i64, i32 = C.c_void_p, C.c_void_p, C.c_int64, C.c_int
    lib.ccqp_abi_version.restype = C.c_int
    lib.ccqp_status_string.restype = C.c_char_p
    lib.ccqp_status_string.argtypes = [C.c_int]
    lib.ccqp_last_error.restype = C.c_char_p
    lib.ccqp_last_error.argtypes = [vp]
    lib.ccqp_create.argtypes = [C.POINTER(vp), C.c_int]
    lib.ccqp_destroy.argtypes = [vp]
    lib.ccqp_set_stream.argtypes = [vp, vp]
    lib.ccqp_get_info.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                  C.POINTER(C.c_int64)]
    lib.ccqp_set_matrix.argtypes = [vp, dp, i64, i64, i64, i64, i32]
    lib.ccqp_set_matrix_csr.argtypes = [vp, dp, dp, dp, i64, i64, i64, i64, i32]
    lib.ccqp_set_projection.argtypes = [vp, C.POINTER(Block), i64, dp, i64]
    lib.ccqp_solve.argtypes = [vp, i32, C.POINTER(Params), dp, dp, dp, i64, dp, i32, C.POINTER(Result)]
    lib.ccqp_solve_async.argtypes = [vp, i32, C.POINTER(Params), dp, dp, dp, i64, dp, i32]
    lib.ccqp_solve_wait.argtypes = [vp, C.POINTER(Result)]
    lib.ccqp_solve_batched.argtypes = [vp, i32, C.POINTER(Params), i64, i64, dp, dp, dp, dp, dp, dp, i64, dp, i32,
                                       C.POINTER(Result), C.POINTER(Result)]
    lib.ccqp_solve_batched_sym.argtypes = lib.ccqp_solve_batched.argtypes
    lib.ccqp_solve_batched_table.argtypes = [vp, i32, C.POINTER(Params), i64, i64, dp, dp, dp, C.POINTER(Block), i64, dp, i64, dp, i64,
                                             dp, i32, C.POINTER(Result), C.POINTER(Result)]
    lib.ccqp_solve_batched_tables.argtypes = lib.ccqp_solve_batched_table.argtypes
    for name in ("ccqp_solve_batched", "ccqp_solve_batched_sym", "ccqp_solve_batched_table", "ccqp_solve_batched_tables"):
        getattr(lib, name + "_f32").argtypes = getattr(lib, name).argtypes      # the fp32 twins: A is a float pointer
    lib.ccqp_set_matrix_symmetric.argtypes = [vp, dp, i64, i64, i32]
    lib.ccqp_set_matrix_f32.argtypes = [vp, dp, i64, i64, i64, i64, i32]
    lib.ccqp_get_upload_info.argtypes = [vp, C.POINTER(i64), C.POINTER(i32)]
    lib.ccqp_host_matrix_is_block_symmetric.argtypes = [dp, i64, i64, i32]
    lib.ccqp_host_matrix_is_block_symmetric.restype = i32
    lib.ccqp_upload_block_rows.argtypes = []
    lib.ccqp_upload_block_rows.restype = i32
    lib.ccqp_gemv.argtypes = [vp, dp, dp, i32]
    lib.ccqp_gemv_timed.argtypes = [vp, dp, dp, i32, C.POINTER(C.c_double)]
    lib.ccqp_project.argtypes = [vp, dp, dp, i32]
    lib.ccqp_normal.argtypes = [vp, dp, dp, i32]
    lib.ccqp_projected_gradient.argtypes = [vp, dp, dp, dp, dp, i32]
    lib.ccqp_debug_divide.argtypes = [vp, dp, dp, dp, dp, dp, dp, dp, i64]
    lib.ccqp_fp64_peak.argtypes = [vp, i32, i32, C.POINTER(C.c_double)]
    lib.ccqp_microbench.argtypes = [vp, C.POINTER(C.c_double), C.c_int32]
    lib.ccqp_debug_emulate_ranks.argtypes = [C.POINTER(vp), i32, i64]
    lib.ccqp_debug_solve_emulated.argtypes = [C.POINTER(vp), i32, i32, C.POINTER(Params), dp, dp, dp, i64, dp, i32, C.POINTER(Result)]
    lib.ccqp_comm_export.argtypes = [vp, i32, i32, i64, vp]
    lib.ccqp_comm_attach.argtypes = [vp, vp]
    lib.ccqp_comm_prepare.argtypes = [vp]
    lib.ccqp_comm_detach.argtypes = [vp]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if fn.restype is C.c_int and name not in ("ccqp_abi_version",):
            fn.restype = C.c_int
    _lib = lib
    return lib


def check(handle, status):
    if status == OK:
        return
    lib = load()
    text = lib.ccqp_status_string(status).decode()
    if status in (3, 4, 5, 10) and handle:
        detail = lib.ccqp_last_error(handle).decode()
        if detail:
            text += ": " + detail
    if status == 9:
        text += " (the kernel trapped: this process's CUDA context is unusable from here on; restart the process)"
    raise CCQPError(status, text)


class Handle:
    """Owns one ccqp_handle (one device, one stream, its workspaces)."""

    def __init__(self, device=-1):
        self.lib = load()
        self.h = C.c_void_p()
        st = self.lib.ccqp_create(C.byref(self.h), int(device))
        if st != OK:
            self.h = C.c_void_p()
            check(None, st)

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.ccqp_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def fp64_peak(self, blocks_per_sm=8, threads_per_block=256):
        """Measured DFMA throughput of the device, TFLOP/s (ccqp_fp64_peak)."""
        out = C.c_double()
        check(self.h, self.lib.ccqp_fp64_peak(self.h, int(blocks_per_sm), int(threads_per_block), C.byref(out)))
        return out.value

    PROBES = ("dfma", "dadd", "dmul", "shfl64_dadd", "div_dadd", "sqrt_dadd", "lds128_bcast_dadd", "lds128_distinct_dadd",
              "sts_bar_lds_dadd_bar", "bar64", "dsetp_sel_dadd", "dmma884_dependent", "dmma884_x8_independent_plus_8_dadd",
              "warpsum_dmma_dadd_dmma", "warpsum_5_shfl64_dadd", "dmma_x8_with_dfma_x8",
              "dfma_independent_x8_one_fresh_operand", "dfma_independent_x8_two_fresh_operands", "dfma_matvec_8x8_register_block")

    def microbench(self):
        """SM cycles per dependent operation (ccqp_microbench), as a dict."""
        out = (C.c_double * len(self.PROBES))()
        check(self.h, self.lib.ccqp_microbench(self.h, out, len(self.PROBES)))
        return dict(zip(self.PROBES, [float(v) for v in out]))

    def upload_info(self):
        """(bytes, mirrored) of the last host -> device matrix copy (ccqp_get_upload_info)."""
        nbytes, mirrored = C.c_int64(), C.c_int32()
        check(self.h, self.lib.ccqp_get_upload_info(self.h, C.byref(nbytes), C.byref(mirrored)))
        return nbytes.value, bool(mirrored.value)

    def set_matrix_f32(self, a, n, row_begin=0, n_rows=None):
        """ccqp_set_matrix_f32 with rows [row_begin, row_begin + n_rows) of a float32 NumPy array or torch tensor of shape
        (n_rows, n) whose rows are contiguous (lda = its row stride; a CUDA tensor is borrowed, anything else is copied
        to the device)."""
        n_rows = n if n_rows is None else n_rows
        if isinstance(a, np.ndarray):
            if a.dtype != np.float32:
                raise TypeError("set_matrix_f32 takes float32, got %s" % a.dtype)
            strides = tuple(s // 4 for s in a.strides) if a.ndim == 2 and all(s % 4 == 0 for s in a.strides) else None
            ptr, mem = a.ctypes.data, MEM_HOST
        else:
            if str(a.dtype) != "torch.float32":
                raise TypeError("set_matrix_f32 takes float32, got %s" % a.dtype)
            strides = tuple(a.stride()) if a.dim() == 2 else None
            ptr, mem = a.data_ptr(), (MEM_DEVICE if a.is_cuda else MEM_HOST)
        if tuple(a.shape) != (n_rows, n) or strides is None or strides[1] != 1 or (n_rows > 1 and strides[0] < n):
            raise ValueError("set_matrix_f32 needs an (%d, %d) matrix with contiguous rows, got shape %s strides %s"
                             % (n_rows, n, tuple(a.shape), strides))
        lda = strides[0] if n_rows > 1 else n
        check(self.h, self.lib.ccqp_set_matrix_f32(self.h, C.c_void_p(ptr), int(n), int(lda), int(row_begin), int(n_rows), mem))

    def info(self):
        sm, grid, thr, smem = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
        check(self.h, self.lib.ccqp_get_info(self.h, C.byref(sm), C.byref(grid), C.byref(thr), C.byref(smem)))
        return dict(sm_count=sm.value, dense_grid=grid.value, dense_threads=thr.value, dense_smem_bytes=smem.value)


_default = {}


def default_handle(device=-1):
    key = int(device)
    if key not in _default:
        _default[key] = Handle(device)
    return _default[key]


BLOCK_DTYPE = np.dtype([("kind", "<i4"), ("reserved", "<i4"), ("offset", "<i8"), ("dim", "<i8"), ("param_off", "<i8")])


class BlockArray:
    """ccqp_block[] backed by a NumPy structured array (fast to build for ~1e4 blocks)."""

    def __init__(self, rows):
        rows = np.asarray(rows, dtype=np.int64).reshape(-1, 4)
        self.arr = np.zeros(rows.shape[0], dtype=BLOCK_DTYPE)
        self.arr["kind"], self.arr["offset"], self.arr["dim"], self.arr["param_off"] = rows.T
        self.ptr = self.arr.ctypes.data_as(C.POINTER(Block))

    def __len__(self):
        return self.arr.shape[0]

    def __getitem__(self, k):
        return self.ptr[k]


def make_blocks(rows):
    """rows: iterable of (kind, offset, dim, param_off) -> BlockArray (pass `.ptr` to the ABI)."""
    return BlockArray(rows)


def f64_ptr(a, dtype="float64"):
    """(pointer, memtype, keepalive) of a float64 (or `dtype`) C-contiguous NumPy array or torch tensor."""
    if a is None:
        return None, None, None
    if isinstance(a, np.ndarray):
        assert a.dtype == np.dtype(dtype) and a.flags["C_CONTIGUOUS"]
        return C.c_void_p(a.ctypes.data), MEM_HOST, a
    # torch tensor (duck-typed to avoid importing torch here)
    assert str(a.dtype) == "torch." + dtype and a.is_contiguous()
    return C.c_void_p(a.data_ptr()), (MEM_DEVICE if a.is_cuda else MEM_HOST), a
