"""Jacobi-preconditioned BlockPCG and GCG on several GPUs (one process per GPU, NCCL): tests/jacobi_dist_worker_gpu.py
under torchrun at 2, 4 and 8 ranks.  This process solves the same problems on one GPU first and hands the results to
the workers, which check that every rank returns the same bits and that the row-partitioned solve agrees with the
one-GPU solve to 1e-10.  Skipped below the rank count."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
pytestmark = pytest.mark.gpu

# (name, pencil args of problems.diffusion7_var, k, shift): k = 16 keeps the reductions in the in-kernel allreduce
# (3k <= 256 values); k = 100 sends the initial 3k-value reduction through the NCCL path; k = 130 is split into chunks
BPCG_CASES = [
    ("k16", dict(m=16, coef="lognormal", seed=11), 16, 0.0),
    ("k100", dict(m=16, coef="jump", seed=12), 100, 0.0),
    ("k130", dict(m=16, coef="lognormal", seed=13), 130, 0.0),
    ("shift_B_k16", dict(m=16, coef="lognormal", seed=14, mass=True), 16, 2.0),
]
GCG_CASE = dict(m=16, coef="lognormal", seed=15, mass=True)
GCG_NEV = 10


def bpcg_inputs(name):
    """(pencil, b, x0) of a BlockPCG case: the same on every process"""
    from gcge_b200 import problems as P
    _, args, k, _ = next(c for c in BPCG_CASES if c[0] == name)
    pen = P.diffusion7_var(**args)
    n = pen.A.ncols
    rng = np.random.default_rng(len(name))
    b = np.asfortranarray(rng.standard_normal((n, k)) * 10.0 ** rng.uniform(-2, 2, k))
    x0 = np.zeros((n, k), order="F")
    x0[:, 1::4] = rng.standard_normal((n, len(range(1, k, 4))))
    return pen, b, x0


def one_gpu_results(api):
    """{key: array} of the one-GPU solves the workers compare with"""
    from gcge_b200 import problems as P
    out = {}
    for name, _, k, shift in BPCG_CASES:
        pen, b, x0 = bpcg_inputs(name)
        A = api.Mat(pen.A); B = None if pen.B is None else api.Mat(pen.B)
        X = api.MultiVec.from_numpy(x0)
        niter, res = api.block_pcg(A, api.MultiVec.from_numpy(b), X, (0, 0), (k, k), B=B, shift=shift, precond="jacobi")
        out[f"{name}_x"] = X.numpy(); out[f"{name}_niter"] = np.array([niter]); out[f"{name}_res"] = np.array([res])
    pen = P.diffusion7_var(**GCG_CASE)
    o = api.gcg_solve(api.Mat(pen.A), api.Mat(pen.B), nev=GCG_NEV, compW_cg_pc=1)
    out["gcg_eval"] = o["eval"]; out["gcg_num_iter"] = np.array([o["num_iter"]])
    return out


@pytest.mark.parametrize("nproc", [2, 4, 8])
def test_jacobi_row_partitioned(b200, nproc, tmp_path):
    if b200.device_count() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    ref = tmp_path / "one_gpu.npz"
    np.savez(ref, **one_gpu_results(b200))
    env = dict(os.environ, PYTHONPATH=str(ROOT), JACOBI_ONE_GPU=str(ref))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(29560 + nproc),
           str(ROOT / "tests" / "jacobi_dist_worker_gpu.py")]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "jacobi dist ok" in r.stdout
