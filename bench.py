#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on its own configuration.

metric   GCG solve seconds (lower is better): wall time of one whole block-GCG solve --
         ops->EigenSolver, i.e. InitializeX .. last Rayleigh-Ritz, matrix build/upload excluded
         (reference test/test_eig_sol_gcg.c:88-144 "Time is") -- of the P1-FEM stiffness/mass
         pencil A x = lambda B x on the Kuhn triangulation, n = m^3 (default m = 200, n = 8.0 M,
         ~15 nnz/row), nev = 200 (nevMax 400, block_size 40), reference default tolerances.
step     one whole solve of that pencil from srand(0).
value    seconds per solve, inputs (A, B) resident in HBM and the four GCG workspaces created
         beforehand (the reference's driver creates gcg_mv_ws[0..3] before its clock starts,
         test/test_eig_sol_gcg.c:57-68,88), CUDA events on the library stream.
e2e      the same solve through the C-ABI with HOST buffers: CCS arrays of A and B uploaded
         from page-locked host memory and turned into device matrices, workspaces allocated,
         solve, eigenvalues + the nev converged eigenvectors copied back to the host, workspaces
         freed -- all inside the timed region.
roofline the dominant kernel class of the timed region (device time from CUDA events around
         every launch of the class, algorithmic bytes/flops of SURVEY.md 8d / DESIGN.md).
cpu_baseline / --impl reference
         the UNMODIFIED reference (oracle/_ref: CCS + OpenMP GCG, OpenBLAS) on the box's host
         cores, on a bounded sample of the same workload (same pencil family, nev, block size
         and tolerances on a smaller lattice, solved to convergence), scaled linearly in n and
         in the outer-iteration count to the full workload -- see `sample` in the JSON line.

same_size  a MEASURED pair at one size both arms can run: the reference solves --same-m (default 40:
         n = 64 000, same nev / block size / tolerances) to convergence on the host cores, the device
         solver is timed on the same pencil in the same run -- beside the extrapolated full-size figure.
parity_vs_golden
         before the timed region EVERY rank solves two of the reference's recorded runs
         (tests/golden/gcg_reference.json: p1_fem_kuhn m = 12 nev = 10 and m = 24 nev = 200) and the line
         carries iteration counts, eigenvalue differences and whether all ranks hold identical bits.

--dump-outputs DIR
         after the timed steps, what the last timed solve handed its caller goes to DIR as .npy files (see
         dump_outputs); inputs are generated from fixed seeds, so two builds can be compared output for output.

Other workloads of BASELINE.json (same line format): --workload laplace7 --m 100 --nev 50 (config 2,
standard problem, analytic eigenvalues as the parity pin), --workload q1_27pt (config 4's operator), and
--kernel-sweep (config 5: per-kernel sweep at n = m^3, k = 16 ... 512, with the reference's slots timed on the host
cores at --sweep-cpu-m beside it; its own one-line format, `rows`).

Multi-GPU (torchrun, one rank per GPU): the SAME pencil is split into 1-D row blocks over the N
GPUs (strong scaling): SpMM halo rows travel by copy-engine peer-to-peer copies into IPC mailboxes
over NVLink (overlapped with the interior rows), the CG scalars are allreduced inside the streaming
kernels over NVLink, Gram blocks by ncclAllReduce, projected problem replicated.  value = seconds per
solve, max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# outer iterations the full workload needs (measured on B200 with this repo, kept in
# profiles/bench_iters.json; bench.py only reads it); the reference arm scales its bounded
# sample with it.  Iteration-count parity with the reference is a tested property (tests/).
ITERS_FILE = ROOT / "profiles" / "bench_iters.json"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index),
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except ValueError:
                continue
            for nm, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------- reference
def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def iters_full(m: int, nev: int, fallback: int) -> tuple[int, str]:
    try:
        d = json.loads(ITERS_FILE.read_text())
        return int(d[f"m{m}_nev{nev}"]["num_iter"]), f"{ITERS_FILE.name} (measured on B200 by this bench)"
    except Exception:
        return fallback, "fallback (no recorded B200 run for this size)"


WORKLOADS = {"p1_fem": "p1_fem_kuhn", "laplace7": "laplace3d_7pt", "q1_27pt": "q1_27pt", "cube4": "cube4_p1"}


def make_pencil(workload: str, m: int):
    from gcge_b200 import problems as P
    if workload == "cube4":                       # config 1: the reference's mesh, two refinements: 15^3 unknowns
        return P.cube4_p1(2)
    return getattr(P, WORKLOADS[workload])(m)


def reference_sample(workload: str, nev: int, m_ref: int, it_ref: int, threads: int) -> dict:
    """One bounded sample of the reference's own GCG (oracle/_ref, unmodified sources): the
    workload's pencil at m_ref^3, same nev / nevMax / block_size / tolerances, up to it_ref outer
    iterations from srand(0) (InitializeX included)."""
    from oracle import ref
    ref.set_threads(threads)
    pen = make_pencil(workload, m_ref)
    r = ref.gcg_solve(pen.A, pen.B, nev=nev, max_iter=it_ref, want_evec=False)
    return {"seconds": r["seconds"], "num_iter": r["num_iter"], "nev_conv": r["nev_conv"], "n": pen.A.ncols, "m": m_ref,
            "generator": WORKLOADS[workload], "eval": r["eval"]}


def scale_reference(sample: dict, m_full: int, nev: int) -> tuple[float, str]:
    n_full = m_full ** 3
    if sample["m"] == m_full:
        return sample["seconds"], (f"reference GCG (oracle/_ref, CCS+OpenMP, unmodified) solving {sample['generator']} "
                                   f"m={m_full} (n={n_full}), nev={nev}, AT FULL SIZE to convergence: {sample['num_iter']} outer "
                                   f"iterations, {sample['seconds']:.2f} s incl. InitializeX -- measured, not scaled")
    itf, src = iters_full(m_full, nev, fallback=100)
    per_row_iter = sample["seconds"] / sample["n"] / max(sample["num_iter"], 1)
    value = per_row_iter * n_full * itf
    desc = (f"reference GCG (oracle/_ref, CCS+OpenMP, unmodified) solving {sample['generator']} m={sample['m']} (n={sample['n']}), "
            f"nev={nev}, to convergence: {sample['num_iter']} outer iterations, {sample['seconds']:.2f} s incl. "
            f"InitializeX; scaled linearly x(n {n_full}/{sample['n']}) x(outer iterations {itf}/{sample['num_iter']}; "
            f"{itf} = full solve, {src}).  The sample fits the host caches, so this flatters the CPU.")
    return value, desc


def pick_reference_size(cal: dict, m_full: int, budget_s: float) -> int:
    """Largest lattice (multiple of 8) whose reference solve is expected to fit budget_s: seconds ~ rows x
    outer iterations; the calibration sample is cache-resident, so a factor 2 of margin."""
    per_row = cal["seconds"] / cal["n"]
    best = cal["m"]
    for m in range(cal["m"] + 8, m_full + 1, 8):
        if per_row * m ** 3 * 2.0 <= budget_s:
            best = m
    if m_full > best and per_row * m_full ** 3 * 2.0 <= budget_s:
        best = m_full
    return best


def reference_kernel_slices(gen: str, m: int, ks, budget_s: float, cores: int) -> dict:
    """BASELINE config 5 on the host cores (SURVEY 8d "per-kernel slices of config 5"): the reference's own slots --
    CCS MatDotMultiVec, MultiVecInnerProd, MultiVecLinearComb, MultiVecAxpby, MultiVecOrth -- on the same kind of pencil at
    a size the CPU finishes in seconds, same shapes as the GPU sweep (3k-wide left operand), OMP threads = cores."""
    from oracle import ref
    from gcge_b200 import problems as P
    ref.set_threads(cores)
    pen = getattr(P, gen)(m)
    n, nnz = pen.A.ncols, pen.A.nnz
    rows, t_begin = [], time.time()

    def best(fn, reps=3):
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
        return min(ts) * 1e3

    for k in ks:
        if time.time() - t_begin > budget_s:
            break
        p = 3 * k
        rng = np.random.default_rng(k)
        X = np.asfortranarray(rng.random((n, p))); Y = np.zeros((n, k), order="F")
        row = {"k": k, "p": p}
        ms = best(lambda: ref.mat_dot_multivec(pen.A, X, Y, (0, 0), (k, k)))
        row["spmm_ms"] = round(ms, 3); row["spmm_GBs"] = round((nnz * 12 + (n + 1) * 4 + 16 * n * k) / ms / 1e6, 2)
        ms = best(lambda: ref.multivec_axpby(0.5, X, 1.5, Y, (0, 0), (k, k)))
        row["axpby_ms"] = round(ms, 3); row["axpby_GBs"] = round(24 * n * k / ms / 1e6, 2)
        d = np.zeros(k)
        ms = best(lambda: ref.multivec_inner_prod("D", X, Y, (0, 0), (k, k), d, 1))
        row["dots_ms"] = round(ms, 3); row["dots_GBs"] = round(16 * n * k / ms / 1e6, 2)
        g = np.zeros((p, k), order="F")
        ms = best(lambda: ref.multivec_inner_prod("N", X, Y, (0, 0), (p, k), g, p))
        row["gram_ms"] = round(ms, 3); row["gram_TF"] = round(2.0 * n * p * k / ms / 1e9, 4)
        coef = np.asfortranarray(rng.random((p, k)))
        ms = best(lambda: ref.multivec_linear_comb(X, Y, (0, 0), (p, k), coef, p, None, 0))
        row["lincomb_ms"] = round(ms, 3); row["lincomb_TF"] = round(2.0 * n * p * k / ms / 1e9, 4)
        if time.time() - t_begin < budget_s:
            end0 = ref.multivec_orth(X, 0, 2 * k, B=pen.B, block_size=80)
            t0 = time.perf_counter(); end = ref.multivec_orth(X, 2 * k, 3 * k, B=pen.B, block_size=80)
            row["orth_ms"] = round((time.perf_counter() - t0) * 1e3, 3); row["orth_end"] = [int(end0), int(end)]
        rows.append(row)
    return {"kind": "reference", "cores": cores, "unit": "ms per call (see rows)", "value": rows[0]["spmm_ms"] if rows else None,
            "sample": f"the reference's slots on {gen} m={m} (n = {n}, nnz = {nnz}), k in {[r['k'] for r in rows]}, "
                      f"best of 3 calls each, {cores} OpenMP threads", "rows": rows}


def run_kernel_sweep(a) -> int:
    """BASELINE config 5 (`--kernel-sweep`): scripts/kernel_sweep.py's rows at n = m^3 and the reference's slots on
    the host cores at a reduced size, as ONE JSON line."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("kernel_sweep", str(ROOT / "scripts" / "kernel_sweep.py"))
    ks_mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(ks_mod)
    sa = ks_mod.arguments(["--m", str(a.m), "--ks", a.sweep_ks])
    sa.quiet = True
    head, rows = ks_mod.sweep(sa)
    line = {"metric": "kernel_sweep", "unit": "GB/s and TFLOP/s per kernel (rows)", "n_gpus": 1, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"BASELINE config 5: SpMM / axpby / dots / Gram (3k x k) / LinearComb (3k -> k) / B-orth of k "
                                   f"against 2k on the P1-FEM pencil, n = {head['n']}, k in {a.sweep_ks}", "m": a.m,
                       "l2": "L2 flushed between repetitions (b200_flush_l2)"},
            "peak_hbm_gbs": head["hbm_gbs"], "rows": rows}
    if not a.no_cpu:
        from oracle import ref
        if ref.available():
            cpu_ks = [int(v) for v in a.sweep_ks.split(",") if int(v) <= 128]
            line["cpu_baseline"] = reference_kernel_slices("p1_fem_kuhn", a.sweep_cpu_m, cpu_ks, a.ref_budget / 2, host_cores())
    print(json.dumps(line))
    return 0


def run_reference(a) -> int:
    """Reference arm: the UNMODIFIED reference on the host cores.  One calibration solve at --ref-m, then ONE
    real solve, to convergence, at the largest lattice expected to fit --ref-budget seconds (the whole arm
    must end within minutes, so the K timed steps of the launch are not K repetitions of it); `value` is
    that solve scaled to the full workload (rows x outer iterations), `measured` is the solve itself."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    from oracle import ref
    if not ref.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libgcge_ref.so was not built "
                          "(needs /root/reference at build time)"}))
        return 0
    cores = host_cores()
    cal = reference_sample(a.workload, a.nev, min(a.ref_m, a.m), a.ref_iters, cores)
    m_big = a.ref_big_m if a.ref_big_m > 0 else pick_reference_size(cal, a.m, a.ref_budget)
    big = cal if m_big == cal["m"] else reference_sample(a.workload, a.nev, m_big, a.ref_iters, cores)
    value, desc = scale_reference(big, a.m, a.nev)
    desc += (f"  [calibration: m={cal['m']} in {cal['seconds']:.2f} s; one solve measured, the --steps/--warmup of this "
             f"arm are not repetitions]")
    cfg = workload_config(a, 1)
    cfg["reference_ran"] = {"m": big["m"], "n": big["n"], "nev": a.nev, "scaled_to_m": a.m}
    line = {"impl": "reference", "metric": "gcg_solve_seconds", "value": value, "unit": "s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": value * 1e3, "higher_is_better": False,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "extrapolated": big["m"] != a.m,
            "measured": {"m": big["m"], "n": big["n"], "nev": a.nev, "seconds": big["seconds"],
                         "num_iter": big["num_iter"], "nev_conv": big["nev_conv"], "cores": cores},
            "cpu_baseline": {"value": value, "unit": "s", "cores": cores, "kind": "reference", "sample": desc},
            "e2e": {"value": value, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def workload_config(a, n_gpus: int) -> dict:
    nev, m = a.nev, a.m
    bs = nev // 5 if nev >= 30 else nev
    what = {"p1_fem": "3D P1-FEM stiffness/mass pencil A x = lambda B x (Kuhn triangulation)",
            "laplace7": "3D 7-point Laplacian, standard problem A x = lambda x (B = NULL)",
            "q1_27pt": "3D 27-point trilinear (Q1) stiffness/mass pencil A x = lambda B x",
            "cube4": "P1 stiffness/mass pencil on the reference's mesh data/cube4.dat after two regular refinements "
                     "(BASELINE config 1 restated)"}[a.workload]
    par = "single GPU" if n_gpus == 1 else (
        f"1-D row blocks over {n_gpus} GPUs (SpMM halos by copy-engine P2P mailboxes over NVLink, CG scalars "
        f"allreduced in-kernel over NVLink, Gram blocks by ncclAllReduce, replicated Rayleigh-Ritz)")
    mv_gb = 8.0 * m ** 3 * (2 * (2 * nev + 2 * bs) + 2 * nev + 3 * bs) / 1e9
    return {"workload": f"{what}, n = {m}^3 = {m ** 3}, nev = {nev} (nevMax {2 * nev}, block_size {bs}), "
                        f"{'B-orthogonal ' if a.workload != 'laplace7' else ''}GCG with BlockPCG, tol = (1e-1, 1e-8), srand(0)",
            "generator": f"gcge_b200.problems.{WORKLOADS[a.workload]}" + (" (pencil_rows: each rank its own planes)" if getattr(a, "local_gen", False) else ""),
            "m": m, "nev": nev,
            "parallelism": par,
            "l2": f"inputs >> L2 (multi-vectors {mv_gb:.1f} GB at m={m}); no flush needed" if mv_gb > 1.0 else
                  "L2 flushed between solves (b200_flush_l2)"}


def residual_check(api, A, B, evec, ev, npairs, prm, n, width=40) -> dict:
    """Residual norms of the first npairs returned eigenpairs, width columns at a time."""
    ta, tb = api.MultiVec(n, width), api.MultiVec(n, width)
    res = np.zeros(npairs)
    bnorm = np.zeros(npairs)
    one = np.array([1.0])
    try:
        for c0 in range(0, npairs, width):
            k = min(width, npairs - c0)
            api.mat_dot_multivec(A, evec, ta, (c0, 0), (c0 + k, k))
            api.mat_dot_multivec(B, evec, tb, (c0, 0), (c0 + k, k))
            d = np.zeros(k)
            api.multivec_inner_prod("D", evec, tb, (c0, 0), (c0 + k, k), d, 1)          # x^T B x
            bnorm[c0:c0 + k] = d
            coef = np.asfortranarray(np.diag(-np.asarray(ev[c0:c0 + k], dtype=np.float64)))
            api.multivec_linear_comb(tb, ta, (0, 0), (k, k), coef, k, one, 0)           # A x - lambda B x
            api.multivec_inner_prod("D", ta, ta, (0, 0), (k, k), d, 1)
            res[c0:c0 + k] = np.sqrt(d)
    finally:
        ta.close(); tb.close()
    lam = np.abs(np.asarray(ev[:npairs], dtype=np.float64))
    tol0, tol1 = float(prm.tol[0]), float(prm.tol[1])
    ok = (res <= 1.001 * tol0) & ((res <= 1.001 * lam * tol1) | (lam <= tol1))
    return {"pairs_checked": int(npairs), "pairs_meeting_reference_tolerance": int(ok.sum()),
            "max_residual": float(res.max()), "max_residual_over_lambda": float((res / np.maximum(lam, 1e-300)).max()),
            "max_abs_xBx_minus_1": float(np.abs(bnorm - 1.0).max()), "tol": [tol0, tol1]}


def golden_parity(api, dist, cases=(4, 9)) -> list:
    """Every rank solves recorded reference runs (tests/golden/gcg_reference.json, produced by the unmodified
    reference through tests/golden/make_golden.py) with the device solver -- row-partitioned over all ranks of
    the job -- and compares: outer iterations (contract: within 1), eigenvalues (1e-10 relative), converged
    count, and whether every rank ended with bit-identical eigenvalues."""
    import torch
    from gcge_b200 import problems as P
    gold = json.loads((ROOT / "tests" / "golden" / "gcg_reference.json").read_text())["cases"]
    out = []
    for idx in cases:
        c = gold[idx]
        pen = getattr(P, c["generator"])(**c["args"])
        A = api.Mat(pen.A); B = None if pen.B is None else api.Mat(pen.B)
        o = api.gcg_solve(A, B, nev=c["nev"])
        k = min(o["nev_conv"], c["nev_conv"])
        ref_ev = np.array(c["eval"][:k])
        err = float(np.max(np.abs(o["eval"][:k] - ref_ev) / np.abs(ref_ev))) if k else None
        same = True
        if dist is not None:
            ev = torch.from_numpy(o["eval"].copy()).cuda()
            ev0 = ev.clone()
            dist.broadcast(ev0, 0)
            flag = torch.tensor([1 if torch.equal(ev.view(torch.int64), ev0.view(torch.int64)) else 0], device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            same = bool(flag.item())
        out.append({"case": f"{c['generator']} {c['args']} nev={c['nev']}", "num_iter": int(o["num_iter"]),
                    "ref_num_iter": int(c["num_iter"]), "nev_conv": int(o["nev_conv"]), "ref_nev_conv": int(c["nev_conv"]),
                    "max_rel_eval": err, "bitwise_identical_across_ranks": same,
                    "ok": bool(abs(o["num_iter"] - c["num_iter"]) <= 1 and err is not None and err < 1e-10
                               and o["nev_conv"] >= c["nev"] and same)})
        o["evec_mv"].close(); A.close()
        if B is not None:
            B.close()
    return out


DUMP_EVEC_BYTES = 48 << 20          # eigenvector sample; with the eigenvalues the dump stays under 64 MB


def dump_outputs(out_dir: Path, out: dict, evec, nev: int) -> None:
    """--dump-outputs: the last timed solve's results as its caller receives them -- eigenvalues.npy (the nev
    wanted eigenvalues), eigenvectors_sample.npy (their eigenvectors on a fixed set of rows: every row when that fits
    DUMP_EVEC_BYTES, else rows drawn by numpy.random.default_rng(0) without replacement, ascending), num_iter.npy and
    nev_conv.npy (scalars); all float64."""
    n = evec.nrows
    if n * 8 * nev <= DUMP_EVEC_BYTES:
        rows = np.arange(n)
    else:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_EVEC_BYTES // (8 * nev), replace=False))
    sample = np.empty((rows.size, nev))
    chunk = max(1, (256 << 20) // (8 * n))             # columns per download: ~256 MB of host memory, one column if larger
    for c0 in range(0, nev, chunk):
        c1 = min(nev, c0 + chunk)
        sample[:, c0:c1] = evec.numpy(c0, c1)[rows]
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "eigenvalues.npy", np.asarray(out["eval"][:nev], dtype=np.float64))
    np.save(out_dir / "eigenvectors_sample.npy", sample)
    np.save(out_dir / "num_iter.npy", np.float64(out["num_iter"]))
    np.save(out_dir / "nev_conv.npy", np.float64(out["nev_conv"]))


# ------------------------------------------------------------------------------------- ours
def run_b200(a) -> int:
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if a.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes a single GPU's results: run bench.py as one process, without torchrun")
    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from gcge_b200 import api, problems as P
    api.init(local)
    if world > 1:
        api.comm_init_from_torch()

    # ---- parity against the reference's recorded runs, on all ranks, before anything is timed
    par_gold = None
    if not a.no_parity:
        try:
            par_gold = golden_parity(api, dist)
        except Exception as exc:
            par_gold = [{"error": str(exc)[:300], "ok": False}]

    t0 = time.time()
    n = a.m ** 3
    if a.local_gen:
        # every rank generates and uploads ONLY its own row block (whole lattice planes): what the reference's
        # distributed back ends do (app/app_phg.c:292-357); needed once the whole CCS no longer fits a host / a GPU
        if a.m % world:
            raise SystemExit(f"--local-gen needs the lattice size {a.m} to be a multiple of the rank count {world}")
        k0, k1 = (a.m // world) * rank, (a.m // world) * (rank + 1)
        rowsA, rowsB = P.pencil_rows(WORKLOADS[a.workload], a.m, k0, k1)
        pen = None
        host_arrays = list(rowsA) + ([] if rowsB is None else list(rowsB))
        nnz = int(rowsA[0][-1])

        def make_mats():
            Am = api.Mat.from_local_rows(n, k0 * a.m * a.m, *rowsA)
            return Am, (None if rowsB is None else api.Mat.from_local_rows(n, k0 * a.m * a.m, *rowsB))
    else:
        pen = make_pencil(a.workload, a.m)
        nnz = pen.A.nnz
        host_arrays = [pen.A.j_col, pen.A.i_row, pen.A.data] + ([] if pen.B is None else [pen.B.j_col, pen.B.i_row, pen.B.data])

        def make_mats():
            return api.Mat(pen.A), (None if pen.B is None else api.Mat(pen.B))
    for h in host_arrays:
        api.host_register(h)
    t_gen = time.time() - t0
    A, B = make_mats()
    prm = api.default_params(a.nev)
    evec = api.MultiVec(n, prm.nevMax)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        api.sync()

    def solve(Am, Bm, ws=None):
        return api.gcg_solve(Am, Bm, nev=a.nev, evec=evec, seed=0, ws=ws, numIterMax=a.max_iter if a.max_iter > 0 else 500)

    # the four GCG workspaces are created before the clock starts, as in the reference's driver
    # (test/test_eig_sol_gcg.c:57-68 allocates gcg_mv_ws[0..3] ahead of `time_start`, :88)
    ws = api.gcg_workspace(n, prm)
    for _ in range(a.warmup):
        out = solve(A, B, ws)
    # ---- timed region: K solves, matrices resident ---------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    api.prof_enable(True)
    l0 = api.kernel_launches()
    barrier()
    api.timer_start()
    w0 = time.time()
    step_wall = []
    for _ in range(a.steps):
        ws0 = time.time()
        out = solve(A, B, ws)
        step_wall.append({"wall_s": round(time.time() - ws0, 4), "solver_s": round(float(out["stats"]["time_total"]), 4)})
    ms = api.timer_stop()
    barrier()
    wall = time.time() - w0
    launches = api.kernel_launches() - l0
    prof = api.prof_report()
    api.prof_enable(False)
    clocks = sampler.stop() if rank == 0 else None
    sec = ms / 1e3 / a.steps
    if dist is not None:
        t = torch.tensor([sec], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t.item())
    stats = out["stats"]
    if a.dump_outputs:                                        # before the e2e solves below overwrite evec
        dump_outputs(Path(a.dump_outputs), out, evec, a.nev)

    # ---- parity at full size, outside the timed region: every returned pair against the reference's
    # own acceptance test (src/ops_eig_sol_gcg.c:229-252): ||A x - lambda B x||_2 <= tol[0] and
    # <= |lambda| tol[1], recomputed from scratch with the library's SpMM / LinearComb / dot kernels
    parity = None
    try:
        parity = residual_check(api, A, B, evec, out["eval"], min(a.nev, int(out["nev_conv"])), prm, n)
    except Exception as exc:                                  # never lose the bench line over the check
        parity = {"error": str(exc)[:200]}

    # ---- e2e: host CCS arrays -> upload -> workspaces -> solve -> eigenpairs back on the host
    A.close()
    if B is not None:
        B.close()
    for w in ws:
        w.close()
    nev_out = a.nev
    _, nloc = evec.local_range()
    host_vec = np.zeros((nloc, nev_out), order="F")          # this rank's rows of the eigenvectors
    api.host_register(host_vec)
    e2e_s = []
    for i in range(a.e2e_steps):
        barrier()
        w0 = time.time()
        A2, B2 = make_mats()
        o2 = solve(A2, B2)
        evec.numpy_local(0, nev_out, out=host_vec)
        ev_host = o2["eval"][:nev_out].copy()
        barrier()
        e2e_s.append(time.time() - w0)
        A2.close()
        if B2 is not None:
            B2.close()
    e2e = float(np.mean(e2e_s)) if e2e_s else None
    if dist is not None and e2e is not None:
        t = torch.tensor([e2e], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = float(t.item())
    # whole-CCS input: every rank receives the whole CCS and cuts out its slab on the device; --local-gen: its rows only
    h2d = sum(h.nbytes for h in host_arrays) * world
    d2h = 8 * n * nev_out + 8 * prm.nevMax            # all ranks together

    if rank != 0:
        api.comm_finalize()
        if dist is not None:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel class ---------------------------------------------
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "B200_PROFILING.md fallback"
    tot_ms = sum(v["ms"] for v in prof.values()) or 1.0
    classes = {k: {"ms": round(v["ms"] / a.steps, 3), "calls": v["calls"] // a.steps,
                   "share": round(v["ms"] / tot_ms, 4),
                   "GBs": round(v["bytes"] / v["ms"] / 1e6, 1) if v["ms"] > 0 else None,
                   "TFs": round(v["flops"] / v["ms"] / 1e9, 2) if v["ms"] > 0 else None,
                   "gap_before_ms": round(v.get("gap_before_ms", 0.0) / a.steps, 3)}
               for k, v in prof.items()}
    top = max(prof, key=lambda k: prof[k]["ms"])
    tv = prof[top]
    if top in ("gram", "lincomb"):
        dmma_peak = api.measure_dmma_peak()
        roof = {"kernel": top, "bound": "tensor", "achieved": tv["flops"] / tv["ms"] / 1e9, "peak": dmma_peak,
                "unit": "TFLOP/s", "peak_source": "b200_measure_dmma_peak (FP64 DMMA m8n8k4 issue ceiling, measured in this run)"}
    else:
        roof = {"kernel": top, "bound": "hbm", "achieved": tv["bytes"] / tv["ms"] / 1e6, "peak": hbm_peak, "unit": "GB/s",
                "peak_source": hbm_src}
    roof["frac"] = roof["achieved"] / roof["peak"]
    # DRAM traffic per launch of the class's main kernel from the committed ncu --set full capture
    # (profiles/ncu_traffic.json), only when this run is the workload the capture was taken on
    roof["traffic"] = None
    try:
        tr = json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text())
        if tr.get("workload", {}).get("m") == a.m and world == 1 and top in tr:
            roof["traffic"] = tr[top]["traffic_bytes_per_launch"]
            roof["traffic_algorithmic_at_capture"] = tr[top].get("algorithmic_bytes_per_launch")
            roof["traffic_source"] = f'{tr[top]["kernel"]}: {tr[top]["source"]}'
    except Exception:
        pass
    roof["launches"] = tv["calls"] // a.steps
    roof["avg_launch_ms"] = tv["ms"] / max(tv["calls"], 1)
    roof["algorithmic_per_launch"] = (tv["flops"] if roof["bound"] == "tensor" else tv["bytes"]) / max(tv["calls"], 1)
    # secondary rooflines: always report SpMM (HBM) and the DMMA contractions
    spmm = prof.get("spmm")
    extra = {}
    if spmm and spmm["ms"] > 0:
        extra["spmm_GBs"] = round(spmm["bytes"] / spmm["ms"] / 1e6, 1)
        extra["spmm_frac_hbm"] = round(spmm["bytes"] / spmm["ms"] / 1e6 / hbm_peak, 4)

    # ---- CPU baseline: the reference itself on the host cores, bounded sample, and the same-size pair -----
    # the full-size device buffers go first (cudaFree of tens of GB takes seconds and must not land inside the small
    # timed solves below: the solver's cached [X P W] buffer, the eigenvector block, whatever Python still holds)
    import gc
    try:
        api.host_unregister(host_vec)
    except Exception:
        pass
    evec.close()
    api.gcg_free_cache()
    gc.collect()
    api.sync()
    cpu, same = None, None
    if world == 1 and not a.no_cpu and pen is not None:
        try:
            from oracle import ref
            if ref.available():
                cores = host_cores()
                m_s = min(a.same_m, a.m)
                s = reference_sample(a.workload, a.nev, m_s, a.ref_iters, cores)
                v, desc = scale_reference(s, a.m, a.nev)
                cpu = {"value": v, "unit": "s", "cores": cores, "kind": "reference", "sample": desc}
                # the device solver on the very same pencil, in the same run: a measured pair
                pen_s = pen if m_s == a.m else make_pencil(a.workload, m_s)
                w0 = time.time()
                As, Bs = api.Mat(pen_s.A), (None if pen_s.B is None else api.Mat(pen_s.B))
                ev_s = api.MultiVec(pen_s.A.ncols, prm.nevMax)
                o_w = api.gcg_solve(As, Bs, nev=a.nev, evec=ev_s, seed=0)           # warm-up (and the e2e-style wall time)
                host_s = ev_s.numpy(0, a.nev)
                api.sync()
                e2e_same = time.time() - w0
                dev_all = []
                for _ in range(2):                                                    # two timed solves, the faster one counts
                    api.timer_start()
                    o_s = api.gcg_solve(As, Bs, nev=a.nev, evec=ev_s, seed=0)
                    dev_all.append(api.timer_stop() / 1e3)
                dev_s = min(dev_all)
                k = min(int(o_s["nev_conv"]), int(s["nev_conv"]))
                err = float(np.max(np.abs(o_s["eval"][:k] - s["eval"][:k]) / np.abs(s["eval"][:k]))) if k else None
                same = {"m": m_s, "n": pen_s.A.ncols, "nev": a.nev, "generator": WORKLOADS[a.workload],
                        "reference_s": s["seconds"], "reference_cores": cores, "reference_num_iter": s["num_iter"],
                        "reference_nev_conv": s["nev_conv"],
                        "b200_s": dev_s, "b200_s_all": dev_all, "b200_e2e_s": e2e_same, "b200_num_iter": int(o_s["num_iter"]),
                        "b200_phases_s": {k: round(float(v), 4) for k, v in o_s["stats"].items() if isinstance(v, float)},
                        "b200_nev_conv": int(o_s["nev_conv"]), "max_rel_eval_vs_reference": err,
                        "ratio_reference_over_b200": s["seconds"] / dev_s if dev_s > 0 else None,
                        "ratio_reference_over_b200_e2e": s["seconds"] / e2e_same if e2e_same > 0 else None,
                        "note": "both arms measured in this run on this box at the same size, both to convergence from srand(0); "
                                "b200_e2e_s = matrices from host CCS + workspaces + solve + eigenvectors back (first call: includes "
                                "one-time module loading for kernels of this width)"}
                del host_s
                ev_s.close(); As.close()
                if Bs is not None:
                    Bs.close()
            else:
                cpu = {"value": None, "unit": "s", "cores": 0, "kind": "reference",
                       "sample": "oracle/_ref not present on this box"}
        except Exception as e:  # the baseline must never take the GPU number down with it
            cpu = cpu or {"value": None, "unit": "s", "cores": 0, "kind": "reference", "sample": f"failed: {e}"}
            same = {"error": str(e)[:300]}

    line = {"metric": "gcg_solve_seconds", "value": sec, "unit": "s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": sec * 1e3, "higher_is_better": False,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(a, world),
            "parity_vs_golden": par_gold,
            "parity_at_full_size": parity,
            "same_size": same, "timed_steps": step_wall,
            "result": {"num_iter": int(out["num_iter"]), "nev_conv": int(out["nev_conv"]),
                       "eval_first": float(out["eval"][0]), "eval_nev": float(out["eval"][a.nev - 1]),
                       "wall_s_per_step": wall / a.steps},
            "phases_s": {k: round(stats[k], 3) for k in ("initX", "checkconv", "compP", "compRR", "rr_eig", "compRV",
                                                          "compW", "linsol", "compX")},
            "kernel_classes": classes,
            "roofline": roof, **extra,
            "cpu_baseline": cpu,
            "e2e": {"value": e2e, "unit": "s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "setup_s": {"generate_pencil": round(t_gen, 2)}}
    print(json.dumps(line))
    api.comm_finalize()
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="p1_fem", choices=sorted(WORKLOADS),
                    help="p1_fem: BASELINE config 3 (default); laplace7: config 2; q1_27pt: config 4's operator")
    ap.add_argument("--m", "--lattice", dest="m", type=int, default=200,
                    help="lattice size: n = m^3 unknowns (200 -> 8.0 M); under torchrun write --lattice (torchrun's own parser "
                         "takes --m for an abbreviation of its options)")
    ap.add_argument("--nev", type=int, default=200)
    ap.add_argument("--max-iter", type=int, default=0, help="cap on outer iterations (0 = reference default 500)")
    ap.add_argument("--e2e-steps", type=int, default=1)
    ap.add_argument("--ref-m", type=int, default=24, help="lattice size of the reference's bounded sample")
    ap.add_argument("--ref-iters", type=int, default=500, help="outer-iteration cap of the reference's bounded sample")
    ap.add_argument("--local-gen", action="store_true", help="every rank generates and uploads only its own row block "
                    "(b200_mat_create_from_local_rows); for sizes whose whole CCS does not fit (config 4: q1_27pt m=400)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / same_size leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the golden-vector parity solves before the timed region")
    ap.add_argument("--same-m", type=int, default=40, help="lattice size of the measured same-size pair (reference on the "
                    "host cores and device solver on the same pencil); also the sample the cpu_baseline is scaled from")
    ap.add_argument("--kernel-sweep", action="store_true", help="BASELINE config 5: per-kernel sweep at n = m^3 with the "
                    "reference's slots on the host cores beside it (one JSON line)")
    ap.add_argument("--sweep-ks", default="16,32,64,128,256,512")
    ap.add_argument("--sweep-cpu-m", type=int, default=64, help="lattice size of the CPU slices of --kernel-sweep")
    ap.add_argument("--ref-budget", type=float, default=240.0, help="--impl reference: seconds the one real solve may take")
    ap.add_argument("--ref-big-m", type=int, default=0, help="--impl reference: lattice size of the real solve (0: pick by budget)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed solve's eigenvalues, a "
                    "fixed row sample of its eigenvectors and its iteration counts to DIR as .npy (single GPU)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.kernel_sweep):
        ap.error("--dump-outputs applies to the timed device solve (--impl b200, no --kernel-sweep)")
    if a.workload == "cube4":
        a.m = 15
        a.same_m = 15
        a.ref_m = 15
    if a.impl == "reference":
        return run_reference(a)
    if a.kernel_sweep:
        return run_kernel_sweep(a)
    return run_b200(a)


if __name__ == "__main__":
    sys.exit(main())
