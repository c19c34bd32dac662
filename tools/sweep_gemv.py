"""Tuning sweep of the dense mat-vec kernel (run under gpurun; build the variants here first).

    python tools/sweep_gemv.py --build         # cross-compile the (threads, unroll) variants, no GPU needed
    python tools/sweep_gemv.py --run           # on the B200: time every variant x tiling x shape

Shapes: the headline n=32768 (A = 8.6 GB), its 8-GPU row shard (4096 x 32768), and n=4096 (config 2).
Prints GB/s = (8*rows*n + 8*n + 8*rows) / mean kernel time (CUDA events, back-to-back launches;
inputs are far larger than L2 except n=4096, which is flagged)."""
import ctypes as C
import itertools
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "ccqppy_b200", "csrc")
VAR = os.path.join(CSRC, "variants")
VARIANTS = [(512, 8), (512, 4), (256, 8), (256, 16), (1024, 4), (1024, 2)]


def lib_path(t, u):
    return os.path.join(VAR, "libccqp_T%d_U%d.so" % (t, u))


def build():
    """Every unit of the library, with the tuning macros, and only the mat-vec hook instantiated (CCQP_SWEEP_BUILD)."""
    from concurrent.futures import ThreadPoolExecutor
    sys.path.insert(0, ROOT)
    from ccqppy_b200 import build as lib_build
    with ThreadPoolExecutor(len(VARIANTS)) as pool:
        list(pool.map(lambda tu: lib_build.build(lib=lib_path(*tu), defines=["CCQP_DENSE_THREADS=%d" % tu[0], "CCQP_UNROLL=%d" % tu[1],
                                                                            "CCQP_SWEEP_BUILD"]), VARIANTS))


def run():
    import torch
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int
    shapes = [("n32768", 32768, 32768), ("shard4096x32768", 4096, 32768), ("n4096(L2-resident)", 4096, 4096)]
    tilings = [(8192, 2048), (8192, 1024), (8192, 4096), (8192, 8192), (4096, 2048), (4096, 1024), (2048, 2048)]
    torch.manual_seed(0)
    Abig = torch.randn((32768, 32768), dtype=torch.float64, device="cuda")
    results = []
    for (t, u) in VARIANTS:
        lib = C.CDLL(lib_path(t, u))
        lib.ccqp_create.argtypes = [C.POINTER(vp), i32]
        lib.ccqp_set_matrix.argtypes = [vp, vp, i64, i64, i64, i64, i32]
        lib.ccqp_gemv_timed.argtypes = [vp, vp, vp, i32, C.POINTER(C.c_double)]
        for (cw, sw), ef in itertools.product(tilings, (1, 0)):
            os.environ["CCQP_CW"], os.environ["CCQP_SW"], os.environ["CCQP_EVICT_FIRST"] = str(cw), str(sw), str(ef)
            for name, rows, n in shapes:
                if ef == 0 and name != "n32768" and (cw, sw) != (8192, 2048):
                    continue
                h = vp()
                assert lib.ccqp_create(C.byref(h), -1) == 0
                A = Abig.view(-1)[: n * n].view(n, n) if rows == n else Abig[:rows]
                st = lib.ccqp_set_matrix(h, vp(A.data_ptr()), n, n, 0, rows, 1)
                assert st == 0, st
                v = torch.zeros(n + 64, dtype=torch.float64, device="cuda")
                v[:n] = torch.randn(n, dtype=torch.float64, device="cuda")
                y = torch.zeros(rows + 64, dtype=torch.float64, device="cuda")
                sec = C.c_double()
                reps = 20 if n > 4096 and rows > 4096 else 100
                st = lib.ccqp_gemv_timed(h, vp(v.data_ptr()), vp(y.data_ptr()), reps, C.byref(sec))
                if st != 0:
                    print("FAILED", t, u, cw, sw, name, st, flush=True)
                    continue
                ref = A[:rows] @ v[:n]
                err = float((y[:rows] - ref).abs().max() / ref.abs().max())
                gbs = (8.0 * rows * n + 8.0 * n + 8.0 * rows) / sec.value / 1e9
                results.append(dict(threads=t, unroll=u, CW=cw, SW=sw, evict_first=ef, shape=name, us=sec.value * 1e6,
                                    GBps=gbs, relerr=err))
                print("T%-4d U%-2d CW%-5d SW%-5d EF%d %-22s %9.1f us %8.1f GB/s err %.1e" %
                      (t, u, cw, sw, ef, name, sec.value * 1e6, gbs, err), flush=True)
                lib.ccqp_destroy(h)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(results, open(os.path.join(ROOT, "gpurun_out", "sweep_gemv.json"), "w"), indent=0)
    best = {}
    for r in results:
        if r["shape"] not in best or r["GBps"] > best[r["shape"]]["GBps"]:
            best[r["shape"]] = r
    for k, r in best.items():
        print("BEST", k, r)


if __name__ == "__main__":
    if "--build" in sys.argv:
        build()
    if "--run" in sys.argv:
        run()
