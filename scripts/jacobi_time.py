"""Cost and effect of the Jacobi preconditioner of BlockPCG (b200_block_pcg_pc, pc = 1) on the GPU.

  1. CG-step time with and without Jacobi, alternating, n = m^3 (m = 200: 8 M rows), k = 40 columns, 30 steps per
     solve (rate = tol = 1e-30, so every step runs), on the P1 pencil (constant stencil) and on a lognormal-coefficient
     7-point lattice (variable coefficients).  CUDA events on the library stream around each solve.
  2. The diagonal kernel: its own device time (torch.profiler, CUDA activities), and the cost of forming D^-1 as a
     solve sees it (a solve with max_iter = 0 with Jacobi minus one without: kernel + the one read-back of its check).
  3. A whole GCG solve on the lognormal pencil with a random diagonal B at n = mg^3 (mg = 100: 1 M rows), with and
     without Jacobi: outer iterations, converged pairs and seconds.

Writes a log (default profiles/jacobi_time.log) that starts with the card's name and power limit.
    python scripts/jacobi_time.py [--m 200] [--k 40] [--reps 5] [--mg 100] [--nev 30] [--out FILE]"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import numpy as np                                  # noqa: E402

from gcge_b200 import api, problems as P           # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "not available"


def timed_solve(A, B, Bv, X, k, ws, precond, max_iter, shift=0.0):
    api.timer_start()
    api.block_pcg(A, Bv, X, (0, 0), (k, k), B=B, max_iter=max_iter, rate=1e-30, tol=1e-30, shift=shift, ws=ws,
                  precond=precond)
    return api.timer_stop()


def step_times(name, pen, k, reps, log):
    n = pen.A.ncols
    A = api.Mat(pen.A)
    Bv = api.MultiVec(n, k); X = api.MultiVec(n, k)
    api.libc_srand(1); Bv.set_random(0, k)
    ws = [api.MultiVec(n, k) for _ in range(3)]
    for pc in ("none", "jacobi"):                   # warm-up of both variants
        timed_solve(A, None, Bv, X, k, ws, pc, 30)
    ms = {"none": [], "jacobi": []}
    for _ in range(reps):
        for pc in ("none", "jacobi"):
            ms[pc].append(timed_solve(A, None, Bv, X, k, ws, pc, 30))
    zero = {"none": [], "jacobi": []}
    for _ in range(reps):
        for pc in ("none", "jacobi"):
            zero[pc].append(timed_solve(A, None, Bv, X, k, ws, pc, 0))
    st = A.storage()
    rec = {"what": "cg_step", "pencil": name, "n": n, "k": k, "storage": st, "steps_per_solve": 30,
           "per_step_ms": {pc: [round(v / 30, 4) for v in ms[pc]] for pc in ms},
           "median_per_step_ms": {pc: round(float(np.median(ms[pc])) / 30, 4) for pc in ms},
           "jacobi_over_none": round(float(np.median(ms["jacobi"]) / np.median(ms["none"])), 4),
           "spread_none": round(float((max(ms["none"]) - min(ms["none"])) / np.median(ms["none"])), 4),
           "max_iter0_solve_ms": {pc: [round(v, 4) for v in zero[pc]] for pc in zero},
           "forming_dinv_ms_median": round(float(np.median(zero["jacobi"]) - np.median(zero["none"])), 4)}
    log(rec)
    return A, Bv, X, ws


def diag_kernel_time(A, Bv, X, k, ws, log, name):
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                timed_solve(A, None, Bv, X, k, ws, "jacobi", 0)
            api.sync()
        ts = [e.device_time for e in prof.events() if "bpcg_jacobi_diag_kernel" in e.name]
        log({"what": "diag_kernel", "pencil": name, "source": "torch.profiler CUDA activities", "calls": len(ts),
             "us": [round(t, 2) for t in ts], "median_us": round(float(np.median(ts)), 2) if ts else "not measured"})
    except Exception as exc:                        # the timing above (max_iter = 0 difference) still stands
        log({"what": "diag_kernel", "pencil": name, "median_us": "not measured", "error": repr(exc)[:300]})


def gcg(mg, nev, log):
    pen = P.diffusion7_var(mg, "lognormal", mass=True)
    A, B = api.Mat(pen.A), api.Mat(pen.B)
    for pc in (0, 1):
        api.sync()
        t0 = time.perf_counter()
        o = api.gcg_solve(A, B, nev=nev, compW_cg_pc=pc)
        api.sync()
        secs = time.perf_counter() - t0
        log({"what": "gcg", "pencil": f"diffusion7_var({mg}, lognormal, mass=True)", "n": pen.A.ncols, "nev": nev,
             "compW_cg_pc": pc, "outer_iterations": o["num_iter"], "nev_conv": o["nev_conv"], "seconds": round(secs, 3),
             "linsol_s": round(o["stats"]["linsol"], 3), "eval_head": [float(v) for v in o["eval"][:3]]})
        api.gcg_free_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--m", type=int, default=200)
    ap.add_argument("--k", type=int, default=40)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--mg", type=int, default=100)
    ap.add_argument("--nev", type=int, default=30)
    ap.add_argument("--out", default=str(Path(__file__).resolve().parents[1] / "profiles" / "jacobi_time.log"))
    a = ap.parse_args()
    out = Path(a.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    f = out.open("w")

    def log(rec):
        line = rec if isinstance(rec, str) else json.dumps(rec)
        print(line, flush=True); f.write(line + "\n"); f.flush()

    api.init(0)
    log(f"# card (name, power limit, max SM clock): {card()}")
    log(f"# scripts/jacobi_time.py --m {a.m} --k {a.k} --reps {a.reps} --mg {a.mg} --nev {a.nev}")
    for name, pen in (("p1_fem_kuhn", lambda: P.p1_fem_kuhn(a.m)),
                      ("diffusion7_var lognormal", lambda: P.diffusion7_var(a.m, "lognormal"))):
        A, Bv, X, ws = step_times(name, pen(), a.k, a.reps, log)
        diag_kernel_time(A, Bv, X, a.k, ws, log, name)
        del A, Bv, X, ws
    gcg(a.mg, a.nev, log)
    f.close()


if __name__ == "__main__":
    main()
