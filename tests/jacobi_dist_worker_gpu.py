"""Jacobi-preconditioned BlockPCG / GCG on several GPUs, one process per GPU, launched by torchrun from
tests/test_jacobi_dist_gpu.py (which passes the one-GPU results in the file named by JACOBI_ONE_GPU).  Every rank
builds the same global inputs; the library keeps its row block."""
import os
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
from gcge_b200 import api, problems as P                                     # noqa: E402
from test_jacobi_dist_gpu import BPCG_CASES, GCG_CASE, GCG_NEV, bpcg_inputs  # noqa: E402

local = int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
api.init(local)
rank, world = api.comm_init_from_torch()
L = api.lib()
one = np.load(os.environ["JACOBI_ONE_GPU"])


def check(cond, msg):
    if not cond:
        raise AssertionError(f"rank {rank}: {msg}")


def gather_rows(mv, k, n):
    full = np.zeros((n, k), order="F")
    api._chk(L.b200_mv_download(mv.h, 0, k, full.ctypes.data_as(api.c_dbl_p), n))     # own rows only
    t = torch.from_numpy(np.ascontiguousarray(full)).cuda()
    dist.all_reduce(t)
    return t.cpu().numpy()


def same_on_every_rank(a):
    t = torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.float64))).cuda()
    t0 = t.clone(); dist.broadcast(t0, 0)
    return bool(torch.equal(t, t0))


# ---- BlockPCG with pc = 1: the same bits on every rank, the one-GPU solve to 1e-10 ----------------------------------
for name, _, k, shift in BPCG_CASES:
    pen, b, x0 = bpcg_inputs(name)
    n = pen.A.ncols
    A = api.Mat(pen.A); B = None if pen.B is None else api.Mat(pen.B)
    X = api.MultiVec.from_numpy(x0)
    niter, res = api.block_pcg(A, api.MultiVec.from_numpy(b), X, (0, 0), (k, k), B=B, shift=shift, precond="jacobi")
    x = gather_rows(X, k, n)
    check(same_on_every_rank([niter, res]), f"{name}: iteration count / residual differ across ranks")
    check(niter == int(one[f"{name}_niter"][0]), f"{name}: {niter} iterations, one GPU {int(one[f'{name}_niter'][0])}")
    ref = one[f"{name}_x"]
    scale = np.abs(ref).max(axis=0)
    err = np.max(np.abs(x - ref).max(axis=0) / np.where(scale > 0, scale, 1.0))
    check(err < 1e-10, f"{name}: x differs from the one-GPU solve by {err:.2e}")
    check(abs(res - one[f"{name}_res"][0]) <= 1e-10 * one[f"{name}_res"][0], f"{name}: residual {res} vs {one[f'{name}_res'][0]}")
    if rank == 0:
        print(f"jacobi bpcg {name}: {niter} iterations, max rel dx vs one GPU {err:.1e}", flush=True)

# ---- a bad diagonal on the last rank's rows fails on every rank, with x untouched, and the library keeps working -----
pen, b, x0 = bpcg_inputs("k16")
n = pen.A.ncols
import scipy.sparse as sp                                                       # noqa: E402
S = pen.A.to_scipy().tolil(); S[n - 1, n - 1] = -1.0
S = sp.csc_matrix(S); S.sort_indices()
Abad = api.Mat(P.CCS(n, n, S.indptr.astype(np.int32), S.indices.astype(np.int32), S.data.astype(np.float64)))
X = api.MultiVec.from_numpy(x0)
failed = False
try:
    api.block_pcg(Abad, api.MultiVec.from_numpy(b), X, (0, 0), (16, 16), precond="jacobi")
except api.B200Error as exc:
    failed = True
    mine = rank == world - 1
    check(("first: row %d" % (n - 1) in str(exc)) == mine and ("another rank" in str(exc)) == (not mine), f"message: {exc}")
check(failed, "a negative diagonal on the last rank was accepted")
check(np.array_equal(gather_rows(X, 16, n), x0), "x moved in a failed call")
niter, _ = api.block_pcg(api.Mat(pen.A), api.MultiVec.from_numpy(b), X, (0, 0), (16, 16), precond="jacobi")
check(niter == int(one["k16_niter"][0]), "solve after a rejected one")

# ---- GCG with compW_cg_pc = 1 ------------------------------------------------------------------------------------
pen = P.diffusion7_var(**GCG_CASE)
o = api.gcg_solve(api.Mat(pen.A), api.Mat(pen.B), nev=GCG_NEV, compW_cg_pc=1)
check(same_on_every_rank(o["eval"]) and same_on_every_rank([o["num_iter"]]), "GCG results differ across ranks")
ev1 = one["gcg_eval"][:GCG_NEV]
err = np.max(np.abs(o["eval"][:GCG_NEV] - ev1) / np.abs(ev1))
check(o["nev_conv"] >= GCG_NEV and err < 1e-10, f"GCG eigenvalues differ from one GPU by {err:.2e}")
check(abs(o["num_iter"] - int(one["gcg_num_iter"][0])) <= 1, f"GCG {o['num_iter']} outer iterations, one GPU {int(one['gcg_num_iter'][0])}")

dist.barrier()
if rank == 0:
    print(f"jacobi dist ok: world={world} gcg outer {o['num_iter']} (one GPU {int(one['gcg_num_iter'][0])}), "
          f"max rel eigenvalue diff {err:.1e}")
api.comm_finalize()
dist.destroy_process_group()
