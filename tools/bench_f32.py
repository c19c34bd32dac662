"""fp32-stored dense Hessians against the fp64 path, in one GPU run (ccqp_set_matrix_f32, csrc/dense_f32.cu).

    python tools/bench_f32.py [--reps 5] [--stream-steps 4] [--big] [--out FILE]

* resident solves: the bench workload (n = 32768, A = G G^T / n + I symmetrised, seed 0) rounded to fp32; SPG and APGD,
  tol 1e-5, max 2000 mat-vecs.  Arm fp64 = the solve of the widened matrix, arm fp32 = the solve of the fp32 matrix; the
  arms alternate, every repeat is reported, and the two arms' outputs must be identical bit for bit.  Rates are device
  time (CUDA events around the solver kernel); bytes/s at 8 and at 4 bytes per entry of A.  Also the bare mat-vec
  (ccqp_gemv_timed) of both arms, to separate the stream from the solver's other phases.
* stream of host-resident problems: SolvePipeline (depth 2) from pinned memory -- fp32 A, the fp64 A of the bench (its
  automatic symmetric upload moves the upper block triangle) and the fp64 A uploaded whole (CCQP_SYM_UPLOAD=0, what a
  non-symmetric A costs).  Host wall clock around the stream, h2d bytes per step.
* --big: one SPG solve at n = 131072 (68.7 GB in fp32; its fp64 copy would need 137 GB more) from a CUDA fp32 tensor
  built on the device in blocks; it/s and the peak device memory.

Prints one JSON document (stdout, and --out) with the card's name and power limit."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from bench import MAX_MV, N_DENSE, TOL, make_dense_problem, spg_uniform_stream   # noqa: E402
from ccqppy_b200 import _capi, solution_spaces as ss, solvers                    # noqa: E402
from ccqppy_b200.pipeline import SolvePipeline                                   # noqa: E402


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return dict(name=torch.cuda.get_device_name(0), nvidia_smi=q)


def bits_equal(x, y):
    x, y = (np.ascontiguousarray(v.cpu().numpy() if hasattr(v, "cpu") else v) for v in (x, y))
    return bool(np.array_equal(x.view(np.int64), y.view(np.int64)))


def make_solver(name):
    s = solvers.CCQPSolverSPG(TOL, MAX_MV) if name == "SPG" else solvers.CCQPSolverAPGD(TOL, MAX_MV)
    s.quiet = True
    return s


def resident(A32, b, reps):
    n = A32.shape[0]
    A64w = A32.double()                   # what solve() made of an fp32 A before ccqp_set_matrix_f32
    torch.cuda.synchronize()
    op = ss.BoxProjOp(n)
    uni = torch.from_numpy(spg_uniform_stream(MAX_MV)).cuda()
    out = {}
    for name in ("SPG", "APGD"):
        arms = dict(fp64=A64w, fp32=A32)
        runs = {k: [] for k in arms}
        same = True
        first = {}
        for rep in range(reps + 1):                   # rep 0: warm-up of both arms
            for arm, A in arms.items():
                s = make_solver(name)
                s.solve(A, b, convex_proj_op=op, uniforms=uni)
                if arm not in first:
                    first[arm] = (s.solution.clone(), s.solution_num_matrix_vector_multiplications, s.solution_residual)
                else:
                    same &= bits_equal(s.solution, first[arm][0])
                if rep:
                    runs[arm].append(dict(gemv=s.solution_gemv_count, gpu_s=s.solution_gpu_time))
        same_arms = bits_equal(first["fp32"][0], first["fp64"][0]) and first["fp32"][1:] == first["fp64"][1:]
        rec = dict(mv=first["fp32"][1], identical_outputs=bool(same_arms), run_to_run_identical=bool(same))
        for arm, rs in runs.items():
            its = [r["gemv"] / r["gpu_s"] for r in rs]
            rec[arm] = dict(gemv_per_s=its, median=float(np.median(its)),
                            GBps_at_8B=[i * (8.0 * n * n + 16.0 * n) / 1e9 for i in its],
                            GBps_at_4B=[i * (4.0 * n * n + 16.0 * n) / 1e9 for i in its])
        rec["ratio_fp32_over_fp64"] = rec["fp32"]["median"] / rec["fp64"]["median"]
        out[name] = rec
        log("[bench_f32] %s n=%d: fp64 %.1f it/s, fp32 %.1f it/s, ratio %.3f, identical %s" %
            (name, n, rec["fp64"]["median"], rec["fp32"]["median"], rec["ratio_fp32_over_fp64"], same_arms))
    # the bare mat-vec of both arms (no solver phases around it)
    h = _capi.Handle(0)
    v = torch.zeros(n + 64, dtype=torch.float64, device="cuda")
    v[:n] = torch.rand(n, dtype=torch.float64, device="cuda")
    y = torch.empty(n, dtype=torch.float64, device="cuda")
    gemv = {}
    for rep in range(3):
        for arm, A in (("fp64", A64w), ("fp32", A32)):
            if arm == "fp32":
                h.set_matrix_f32(A, n)
            else:
                _capi.check(h.h, h.lib.ccqp_set_matrix(h.h, ctypes.c_void_p(A.data_ptr()), n, n, 0, n, _capi.MEM_DEVICE))
            sec = ctypes.c_double()
            _capi.check(h.h, h.lib.ccqp_gemv_timed(h.h, ctypes.c_void_p(v.data_ptr()), ctypes.c_void_p(y.data_ptr()), 20,
                                                   ctypes.byref(sec)))
            eb = 8.0 if arm == "fp64" else 4.0
            gemv.setdefault(arm, []).append(dict(us=sec.value * 1e6, GBps=(eb * n * n + 16.0 * n) / sec.value / 1e9))
    h.close()
    out["gemv_timed"] = gemv
    log("[bench_f32] mat-vec alone: %s" % json.dumps(gemv))
    del A64w
    torch.cuda.empty_cache()
    return out


def stream(A32h, b_h, steps):
    n = A32h.shape[0]
    A64h = A32h.double().pin_memory()          # exactly symmetric: the automatic symmetric upload applies
    op = ss.BoxProjOp(n)
    uni = torch.from_numpy(spg_uniform_stream(MAX_MV)).pin_memory()
    out = {}
    for label, A, env in (("fp32", A32h, None), ("fp64_auto_symmetric", A64h, None), ("fp64_whole", A64h, "0")):
        if env is None:
            os.environ.pop("CCQP_SYM_UPLOAD", None)
        else:
            os.environ["CCQP_SYM_UPLOAD"] = env
        pipe = SolvePipeline(make_solver("SPG"), depth=2)
        for _ in range(2):
            pipe.submit(A, b_h, convex_proj_op=op, uniforms=uni)
        pipe.results()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            pipe.submit(A, b_h, convex_proj_op=op, uniforms=uni)
        res = pipe.results()
        dt = time.perf_counter() - t0
        up = pipe.slots[0].handle.upload_info()
        pipe.close()
        mvs = sum(r.solution_gemv_count for r in res)
        out[label] = dict(gemv_per_s=mvs / dt, s_per_solve=dt / steps, steps=steps, h2d_matrix_bytes_per_step=up[0],
                          mirrored=up[1], h2d_bytes_per_step=up[0] + 8 * n + 8 * MAX_MV, solution=np.asarray(res[0].solution))
        log("[bench_f32] stream %s: %.1f it/s, %.3f s per solve, %.2f GB of A per step" % (label, mvs / dt, dt / steps, up[0] / 1e9))
    os.environ.pop("CCQP_SYM_UPLOAD", None)
    ref = out["fp64_auto_symmetric"]["solution"]
    for rec in out.values():
        rec["identical_to_fp64_auto_symmetric"] = bits_equal(rec.pop("solution"), ref)
    out["ratio_fp32_over_fp64_auto_symmetric"] = out["fp32"]["gemv_per_s"] / out["fp64_auto_symmetric"]["gemv_per_s"]
    out["ratio_fp32_over_fp64_whole"] = out["fp32"]["gemv_per_s"] / out["fp64_whole"]["gemv_per_s"]
    return out


def big(n=131072, blk=8192):
    """A = S / n + 2 I, S symmetric with U[0, 1) entries (Gershgorin: spectrum in [1, 3]), fp32, built block by block."""
    torch.cuda.reset_peak_memory_stats()
    A = torch.empty((n, n), dtype=torch.float32, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(1)
    for i in range(0, n, blk):
        for j in range(i, n, blk):
            B = torch.rand((blk, blk), generator=g, device="cuda", dtype=torch.float32).div_(n)
            A[i:i + blk, j:j + blk] = B
            if j != i:
                A[j:j + blk, i:i + blk] = B.t()
            else:
                A[i:i + blk, i:i + blk] = 0.5 * (B + B.t())
    A.diagonal().add_(2.0)
    b = torch.rand(n, generator=g, device="cuda", dtype=torch.float64).sub_(0.5)
    torch.cuda.synchronize()
    s = make_solver("SPG")
    s.solve(A, b, convex_proj_op=ss.BoxProjOp(n), uniforms=torch.from_numpy(spg_uniform_stream(MAX_MV)).cuda())
    torch.cuda.synchronize()
    free, total = torch.cuda.mem_get_info()
    rec = dict(n=n, A_bytes=4 * n * n, mv=s.solution_num_matrix_vector_multiplications, converged=s.solution_converged,
               gemv_per_s=s.solution_gemv_count / s.solution_gpu_time,
               GBps_at_4B=s.solution_hbm_bytes / s.solution_gpu_time / 1e9,
               torch_peak_allocated_bytes=torch.cuda.max_memory_allocated(), device_used_bytes_after=total - free,
               device_total_bytes=total)
    log("[bench_f32] big: %s" % json.dumps(rec))
    del A
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--stream-steps", type=int, default=4)
    ap.add_argument("--big", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_f32 needs a CUDA device")
    doc = dict(card=card(), n=N_DENSE, tol=TOL, max_mv=MAX_MV)
    A64, b = make_dense_problem(N_DENSE, "cuda:0")
    A32 = A64.float()                          # the bench workload rounded to fp32
    del A64
    doc["resident"] = resident(A32, b, args.reps)
    A32h, b_h = A32.cpu().pin_memory(), b.cpu().pin_memory()
    del A32, b
    torch.cuda.empty_cache()
    doc["stream"] = stream(A32h, b_h, args.stream_steps)
    del A32h, b_h
    if args.big:
        doc["big"] = big()
    doc["card_after"] = card()
    text = json.dumps(doc, indent=1, default=float)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
