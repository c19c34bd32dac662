"""Rate of batched solves with a projection table: one shared table against per-problem parameters.

The workload is a contact-style batch: 65 536 problems of n = 63, 21 Sphere(3) friction discs each, A = G G^T / n + I generated on the device, BBPGD and SPG (tol 1e-8, 1000 uniforms per
problem drawn on the device).  Arms:
  (a) shared table (`ccqp_solve_batched_table`) on a baseline library (`--baseline-lib`, e.g. the parent commit's build);
  (b) shared table on this tree's library;
  (c) per-problem radii mu * f_n (`ccqp_solve_batched_tables`, a device [batch, 21] array) on this tree's library;
  (c0) the per-problem entry point with every row equal to the shared row of (b): the same problems, the same bits as (b),
       so c0 / b is the cost of the per-problem path alone ((c) solves other problems: its mat-vec counts differ).
`--n 64` runs the same discs plus one free unknown and rows of 22 parameters (the last one unused): b and the parameter
rows then travel by TMA with A (n even, 16-byte aligned rows), while at n = 63 every thread reads them from global memory.
Every arm runs in a subprocess of its own (the C ABI is driven through ctypes, so a baseline library without the newer
entry point loads too); the arms alternate over `--rounds` rounds so that the spread between rounds is visible next to the
differences between arms.  The rate is problems / kernel time (CUDA events around the one solver kernel,
ccqp_result.gpu_seconds); the median over `--reps` calls per round is reported.  The solutions of (a) and (b) are compared
bit for bit (SHA-256 of x).  The card's name and power limit are read in the same run and written with the numbers.

Build a baseline library from another checkout with `python -m ccqppy_b200.build` there.
Usage: python tools/bench_batched_tables.py [--baseline-lib PATH] [--batch 65536] [--n 63] [--rounds 3] [--reps 5]
                                            [--out FILE]
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DISCS, K = 21, 1000
SOLVERS = {"BBPGD": 3, "SPG": 5}


def worker(lib_path, arm, batch, reps, N):
    import torch
    sys.path.insert(0, ROOT)
    from ccqppy_b200 import _capi
    lib = C.CDLL(lib_path)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int
    lib.ccqp_create.argtypes = [C.POINTER(vp), i32]
    lib.ccqp_set_stream.argtypes = [vp, vp]
    lib.ccqp_destroy.argtypes = [vp]
    entry = lib.ccqp_solve_batched_table if arm == "shared" else lib.ccqp_solve_batched_tables
    entry.argtypes = [vp, i32, C.POINTER(_capi.Params), i64, i64, vp, vp, vp, C.POINTER(_capi.Block), i64, vp, i64, vp, i64,
                      vp, i32, C.POINTER(_capi.Result), C.POINTER(_capi.Result)]
    h = vp()
    assert lib.ccqp_create(C.byref(h), 0) == 0
    assert lib.ccqp_set_stream(h, vp(torch.cuda.current_stream().cuda_stream)) == 0
    g = torch.Generator(device="cuda").manual_seed(0)
    G = torch.randn((batch, N, N), generator=g, device="cuda", dtype=torch.float64)
    A = G @ G.transpose(1, 2) / N + torch.eye(N, device="cuda", dtype=torch.float64)
    del G
    xs = 1 - 4 * torch.rand((batch, N), generator=g, device="cuda", dtype=torch.float64)
    b = -(A @ xs.unsqueeze(-1)).squeeze(-1)
    uni = torch.rand((batch, K), generator=g, device="cuda", dtype=torch.float64)
    mu = 0.2 + 0.6 * torch.rand((batch, 1), generator=g, device="cuda", dtype=torch.float64)
    n_params = DISCS + 1 if N % 2 == 0 else DISCS   # n = 64: even rows, so that device rows are 16-byte aligned
    radii = (mu * (0.5 + torch.rand((batch, n_params), generator=g, device="cuda", dtype=torch.float64))).contiguous()
    shared = radii[0].cpu().numpy().copy()          # the shared arm: problem 0's discs for every problem
    same = torch.from_numpy(shared).cuda().repeat(batch, 1).contiguous()
    rows = [(_capi.SPHERE, 3 * k, 3, k) for k in range(DISCS)]
    blocks = _capi.make_blocks(rows + ([(_capi.IDENTITY, 3 * DISCS, N - 3 * DISCS, DISCS)] if N > 3 * DISCS else []))
    x = torch.empty((batch, N), dtype=torch.float64, device="cuda")
    results = (_capi.Result * batch)()
    summary = _capi.Result()
    out = {}
    for name, sid in SOLVERS.items():
        prm = _capi.Params(tol=1e-8, max_mv=5000.0, step_size=0.01, tau=0.5, sigma1=0.01, sigma2=0.5, m=5)
        par = {"shared": shared.ctypes.data_as(vp), "per_problem": vp(radii.data_ptr()), "per_problem_same": vp(same.data_ptr())}[arm]

        def call():
            st = entry(h, sid, C.byref(prm), batch, N, vp(A.data_ptr()), vp(b.data_ptr()), None, blocks.ptr, len(blocks), par,
                       n_params, vp(uni.data_ptr()), K, vp(x.data_ptr()), _capi.MEM_DEVICE, results, C.byref(summary))
            assert st == 0 and summary.status == 0, (st, summary.status)
            return summary.gpu_seconds
        call()                                      # warm-up: module load, workspace
        t = [call() for _ in range(reps)]
        out[name] = dict(qps=[batch / s for s in t], converged=int(summary.converged), mv_total=int(summary.mv_count),
                         sha256=hashlib.sha256(x.cpu().numpy().tobytes()).hexdigest()[:16])
    lib.ccqp_destroy(h)
    print(json.dumps(out))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--baseline-lib", help="a second libccqp_b200.so for arm (a)")
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--n", type=int, default=63, choices=(63, 64))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", help="write the JSON report here too")
    ap.add_argument("--worker", nargs=2, metavar=("LIB", "ARM"), help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        return worker(a.worker[0], a.worker[1], a.batch, a.reps, a.n)
    sys.path.insert(0, ROOT)
    from ccqppy_b200 import build
    arms = [("b_shared", build.LIB, "shared"), ("c0_per_problem_same_rows", build.LIB, "per_problem_same"),
            ("c_per_problem", build.LIB, "per_problem")]
    if a.baseline_lib:
        arms.insert(0, ("a_shared_baseline", os.path.abspath(a.baseline_lib), "shared"))
    runs = {name: [] for name, _, _ in arms}
    for r in range(a.rounds):
        for name, lib, arm in arms:
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", lib, arm, "--batch", str(a.batch),
                                "--reps", str(a.reps), "--n", str(a.n)], capture_output=True, text=True)
            if p.returncode != 0:
                sys.exit("%s failed:\n%s" % (name, p.stderr[-3000:]))
            runs[name].append(json.loads(p.stdout.strip().splitlines()[-1]))
            print("round %d %s: %s" % (r, name, {s: round(statistics.median(v["qps"]) / 1e6, 3) for s, v in runs[name][-1].items()}),
                  file=sys.stderr)
    report = dict(card=card(), batch=a.batch, n=a.n, discs=DISCS, baseline_lib=a.baseline_lib, arms={})
    for name, rs in runs.items():
        report["arms"][name] = {}
        for s in SOLVERS:
            med = [statistics.median(r[s]["qps"]) for r in rs]
            report["arms"][name][s] = dict(qps_median_per_round=med, qps_median=statistics.median(med),
                                           spread=(max(med) - min(med)) / statistics.median(med),
                                           converged=all(r[s]["converged"] for r in rs), mv_total=rs[0][s]["mv_total"],
                                           sha256=sorted({r[s]["sha256"] for r in rs}))
    if a.baseline_lib:
        report["a_b_same_bits"] = {s: report["arms"]["a_shared_baseline"][s]["sha256"] == report["arms"]["b_shared"][s]["sha256"]
                                   for s in SOLVERS}
    report["b_c0_same_bits"] = {s: report["arms"]["b_shared"][s]["sha256"] == report["arms"]["c0_per_problem_same_rows"][s]["sha256"]
                                for s in SOLVERS}
    for s in SOLVERS:
        b_ = report["arms"]["b_shared"][s]["qps_median"]
        report.setdefault("c0_over_b", {})[s] = report["arms"]["c0_per_problem_same_rows"][s]["qps_median"] / b_
        report.setdefault("c_over_b", {})[s] = report["arms"]["c_per_problem"][s]["qps_median"] / b_
        if a.baseline_lib:
            report.setdefault("b_over_a", {})[s] = b_ / report["arms"]["a_shared_baseline"][s]["qps_median"]
    text = json.dumps(report, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
