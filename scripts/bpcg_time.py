"""Times BlockPCG (30 iterations, k columns) on the P1-FEM pencil: per-class device time per iteration."""
import sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import numpy as np
from gcge_b200 import api, problems as P
api.init(0)
m = int(sys.argv[1]) if len(sys.argv) > 1 else 200
k = int(sys.argv[2]) if len(sys.argv) > 2 else 40
pen = P.p1_fem_kuhn(m)
A = api.Mat(pen.A)
n = pen.A.ncols
# 3rd argument "wide": x is a k-column block in the middle of a 480-column multi-vector, as in the eigensolver (x lives in
# [X P W]: k*8-byte row segments at a 3840-byte pitch), instead of a k-column multi-vector of its own
wide = len(sys.argv) > 3 and sys.argv[3] == "wide"
xo = 200 if wide else 0
Bv = api.MultiVec(n, k); X = api.MultiVec(n, 480 if wide else k)
api.libc_srand(1); Bv.set_random(0, k)
ws = [api.MultiVec(n, k) for _ in range(3)]
api.block_pcg(A, Bv, X, (0, xo), (k, xo + k), max_iter=30, rate=1e-30, tol=1e-30, ws=ws)
api.sync()
api.prof_enable(True)
api.block_pcg(A, Bv, X, (0, xo), (k, xo + k), max_iter=30, rate=1e-30, tol=1e-30, ws=ws)
api.sync()
pr = api.prof_report(); api.prof_enable(False)
tot = sum(v["ms"] for v in pr.values())
print({"x_layout": "block of 480 columns" if wide else "own multi-vector", "m": m, "k": k, "total_ms": round(tot, 2), "per_iter_ms": round(tot / 30, 4),
       "spmm_ms_per_call": round(pr["spmm"]["ms"] / max(pr["spmm"]["calls"], 1), 4), "spmm_GBs": round(pr["spmm"]["bytes"] / pr["spmm"]["ms"] / 1e6, 1),
       "bpcg_ms_per_iter": round(pr["bpcg_fused"]["ms"] / 30, 4), "bpcg_GBs": round(pr["bpcg_fused"]["bytes"] / pr["bpcg_fused"]["ms"] / 1e6, 1)}, flush=True)
