"""Batched solves on float32 Hessians against the widened fp64 batch: kernel time, and the whole call from a float32 source.

The batches are A = G G^T / n + I generated in float32 on the device (seed 0), b = -A x* for x* uniform in [-3, 1], boxes
[-1, 1], tol 1e-8, SPG with 1000 device-drawn uniforms per problem.  Three measurements, each alternating its two arms over
`--rounds` rounds on the same batch (the spread between rounds is reported next to the difference between arms):
  1. kernel time (`summary.gpu_seconds`: CUDA events around the one solver kernel), device-resident inputs: the fp64 batch
     (`A.double()`) against the float32 batch, 65 536 x n = 64 and 16 384 x n = 128, BBPGD and SPG, plus symmetric=True at
     n = 64 (BBPGD); median of `--reps` calls per round;
  2. the whole call from a CUDA float32 tensor, wall clock ending in a device synchronise: `solve_batched(A32.double())`
     (what solve_batched did before it had an fp32 path: widen on the device, then the fp64 kernel) against
     `solve_batched(A32)`;
  3. the whole call from pinned host memory (solve_batched hands the pinned pointers to the C ABI: ccqp_solve_batched on a
     pinned widened copy made before the timed calls, against ccqp_solve_batched_f32 on the pinned float32 batch): bytes of
     A that cross PCIe, and wall clock.
Every call's solutions, mat-vec counts, residuals and converged flags are compared between the arms bit for bit.  The
card's name and power limit are read in the same run and written with the numbers.

Usage: python tools/bench_batched_f32.py [--rounds 5] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
K = 1000


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(name=torch.cuda.get_device_name(0),
                nvidia_smi=q.stdout.strip() if q.returncode == 0 else "unknown (nvidia-smi failed)")


def batch(b, n):
    import torch
    g = torch.Generator(device="cuda").manual_seed(0)
    G = torch.randn((b, n, n), generator=g, device="cuda", dtype=torch.float32)
    A = G @ G.transpose(1, 2) / n + torch.eye(n, device="cuda", dtype=torch.float32)
    del G
    A = 0.5 * (A + A.transpose(1, 2))           # exactly symmetric (the symmetric kernels read the upper block triangle)
    xs = 1 - 4 * torch.rand((b, n), generator=g, device="cuda", dtype=torch.float64)
    rhs = -(A.double() @ xs.unsqueeze(-1)).squeeze(-1)
    uni = torch.rand((b, K), generator=g, device="cuda", dtype=torch.float64)
    return A.contiguous(), rhs, -torch.ones_like(rhs), torch.ones_like(rhs), uni


def solver(name):
    from ccqppy_b200 import solvers
    s = {"BBPGD": lambda: solvers.CCQPSolverBBPGD(1e-8, 5000), "SPG": lambda: solvers.CCQPSolverSPG(1e-8, 5000)}[name]()
    s.quiet = True
    return s


def outputs(s):
    import torch
    x = s.solution
    x = x.cpu().numpy() if isinstance(x, torch.Tensor) else x
    return x, s.solution_num_matrix_vector_multiplications, s.solution_residual, s.solution_converged


def same(o1, o2):
    import numpy as np
    return all(np.array_equal(a, b, equal_nan=True) for a, b in zip(o1, o2))


def spread(v):
    med = statistics.median(v)
    return dict(median=med, min=min(v), max=max(v), rel_spread=(max(v) - min(v)) / med if med else None, rounds=v)


def kernel_times(args):
    import torch
    out = []
    for b, n, name, sym in [(65536, 64, "BBPGD", False), (65536, 64, "SPG", False), (16384, 128, "BBPGD", False),
                            (16384, 128, "SPG", False), (65536, 64, "BBPGD", True)]:
        A32, rhs, lb, ub, uni = batch(b, n)
        A64 = A32.double()
        kw = dict(symmetric=sym, uniforms=uni if name == "SPG" else None)
        arms = {"fp64": A64, "fp32": A32}
        t = {k: [] for k in arms}
        identical = True
        for r in range(args.rounds):
            outs = {}
            for arm in (("fp64", "fp32") if r % 2 == 0 else ("fp32", "fp64")):
                ts = []
                for rep in range(args.reps + 1):
                    s = solver(name).solve_batched(arms[arm], rhs, lb, ub, **kw)
                    if rep:                     # the first call of a round is a warm-up
                        ts.append(s.solution_gpu_time)
                outs[arm] = (outputs(s), s.solution_hbm_bytes)
                t[arm].append(statistics.median(ts))
            identical &= same(outs["fp64"][0], outs["fp32"][0])
        del A64
        torch.cuda.empty_cache()
        rec = dict(batch=b, n=n, solver=name, symmetric=sym, bit_identical=identical,
                   hbm_bytes=dict(fp64=outs["fp64"][1], fp32=outs["fp32"][1]),
                   kernel_seconds={k: spread(v) for k, v in t.items()},
                   fp32_over_fp64=statistics.median(t["fp32"]) / statistics.median(t["fp64"]))
        rec["qp_per_s"] = {k: b / rec["kernel_seconds"][k]["median"] for k in t}
        print(json.dumps(rec), flush=True)
        out.append(rec)
    return out


def whole_calls(args):
    import torch
    res = []
    b, n, name = 65536, 64, "BBPGD"
    A32, rhs, lb, ub, _ = batch(b, n)
    # 2. from a CUDA float32 tensor
    arms = {"widen_then_fp64": lambda: solver(name).solve_batched(A32.double(), rhs, lb, ub),
            "fp32": lambda: solver(name).solve_batched(A32, rhs, lb, ub)}
    res.append(alternate("cuda_float32_tensor", arms, args, dict(batch=b, n=n, solver=name)))
    # 3. from pinned host memory: the widened pinned copy is made before the timed calls
    hA32 = A32.cpu().pin_memory()
    hA64 = hA32.double().pin_memory()
    hv = [v.cpu().pin_memory() for v in (rhs, lb, ub)]
    arms = {"fp64_on_widened_pinned": lambda: solver(name).solve_batched(hA64, *hv),
            "fp32_pinned": lambda: solver(name).solve_batched(hA32, *hv)}
    rec = alternate("pinned_host_float32", arms, args, dict(batch=b, n=n, solver=name))
    rec["pcie_bytes_of_A"] = {"fp64_on_widened_pinned": b * n * n * 8, "fp32_pinned": b * n * n * 4}
    res.append(rec)
    return res


def alternate(label, arms, args, meta):
    import torch
    keys = list(arms)
    t = {k: [] for k in keys}
    identical = True
    for r in range(args.rounds):
        outs = {}
        for k in (keys if r % 2 == 0 else keys[::-1]):
            ts = []
            for rep in range(args.reps + 1):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                s = arms[k]()
                torch.cuda.synchronize()
                if rep:
                    ts.append(time.perf_counter() - t0)
            outs[k] = outputs(s)
            t[k].append(statistics.median(ts))
        identical &= same(outs[keys[0]], outs[keys[1]])
    rec = dict(meta, source=label, bit_identical=identical, wall_seconds={k: spread(v) for k, v in t.items()},
               speedup=statistics.median(t[keys[0]]) / statistics.median(t[keys[1]]))
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_batched_f32: needs a CUDA device")
    doc = dict(card=card(), rounds=args.rounds, reps=args.reps, kernel=kernel_times(args), whole_call=whole_calls(args))
    doc["all_bit_identical"] = all(r["bit_identical"] for r in doc["kernel"] + doc["whole_call"])
    text = json.dumps(doc, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
