"""The Jacobi-preconditioned BlockPCG and GCG in numpy: the reference side of the device's b200_block_pcg_pc (pc = 1)
and of the GCG's compW_cg_pc = 1.  Built on the numpy port of the reference (oracle/gcg_numpy.py), which stays the
reference's unpreconditioned algorithm.

Jacobi: z = D^-1 r with D = diag(A + shift B) (B None: diag(A) + shift), rho = r^T z drives alpha and beta,
p = z + beta p; the residual norms and the stop test stay on ||r||_2, so rate and tol mean what they mean without it.
The operations are those of the device, in its order (b200_bpcg.cu)."""
import contextlib

import numpy as np

from oracle import gcg_numpy as G


def jacobi_dinv(A, shift=0.0, B=None):
    """1 / diag(A + shift*B) (B None: diag(A) + shift) as a column, summed as bpcg_jacobi_diag_kernel does.  A and B
    only need .diagonal().  Raises when an entry is not > 0."""
    d = np.asarray(A.diagonal(), dtype=np.float64).copy()
    if shift != 0.0:
        d = d + shift * (np.ones_like(d) if B is None else np.asarray(B.diagonal(), dtype=np.float64))
    if not np.all(d > 0.0):
        raise ValueError(f"Jacobi: {int(np.sum(~(d > 0.0)))} diagonal entries of A + shift*B are not > 0")
    return (1.0 / d)[:, None]


def block_pcg(A, b, x, max_iter, rate, tol, tol_type="abs", shift=0.0, B=None, return_info=False, precond=None):
    """gcg_numpy.block_pcg (the reference's BlockPCG, src/ops_lin_sol.c:140-437) with a preconditioner: precond
    "jacobi" (D from jacobi_dinv), a dinv column, or None / "none" (then the same bits as gcg_numpy.block_pcg).
    x is updated in place; returns (niter, residual norms[, info]) like gcg_numpy.block_pcg."""
    k = b.shape[1]
    if precond is None or (isinstance(precond, str) and precond == "none"):
        dinv = None
    elif isinstance(precond, str) and precond == "jacobi":
        dinv = jacobi_dinv(A, shift, B)
    elif isinstance(precond, np.ndarray):
        dinv = precond.reshape(-1, 1)
    else:
        raise ValueError(f"block_pcg: precond {precond!r}")

    def op(v):
        y = G._matdot(A, v)
        if shift != 0.0:
            y += shift * (v if B is None else G._matdot(B, v))
        return y

    norm_b = np.sqrt(np.sum(b * b, axis=0)) if tol_type == "rel" else np.ones(k)
    r = b - op(x)
    rho2 = np.sum(r * r, axis=0)
    init_res = np.sqrt(rho2)
    if dinv is not None:
        rho2 = np.sum(r * (dinv * r), axis=0)
    last_res = init_res.copy()
    unconv = [i for i in range(k) if init_res[i] > tol * norm_b[i]]
    stop = np.zeros(k, dtype=int)
    ratios = [init_res[i] / (tol * norm_b[i]) for i in range(k) if tol * norm_b[i] > 0]
    p = np.zeros_like(r)
    rho1 = np.zeros(k)
    niter = 0
    while niter < max_iter and unconv:
        stop[unconv] += 1
        u = np.array(unconv)
        beta = np.zeros(len(u)) if niter == 0 else rho2[u] / rho1[u]
        p[:, u] = (r[:, u] if dinv is None else dinv * r[:, u]) + p[:, u] * beta
        w = op(p[:, u])
        ptw = np.sum(p[:, u] * w, axis=0)
        rho1[u] = rho2[u]
        alpha = rho2[u] / ptw
        x[:, u] += p[:, u] * alpha
        r[:, u] -= w * alpha
        rr = np.sum(r[:, u] * r[:, u], axis=0)
        last_res[u] = np.sqrt(rr)
        rho2[u] = rr if dinv is None else np.sum(r[:, u] * (dinv * r[:, u]), axis=0)
        if return_info:
            ratios += [last_res[i] / t for i in unconv for t in (rate * init_res[i], tol * norm_b[i]) if t > 0]
        unconv = [i for i in unconv if last_res[i] > rate * init_res[i] and last_res[i] > tol * norm_b[i]]
        niter += 1
    if return_info:
        return niter, last_res, {"stop": stop, "ratios": np.array(ratios)}
    return niter, last_res


@contextlib.contextmanager
def _inner_solve(precond):
    """gcg_numpy's ComputeW / ComputeW12 call the module's block_pcg: route those calls through this one"""
    orig = G.block_pcg
    G.block_pcg = lambda *a, **kw: block_pcg(*a, precond=precond, **kw)
    try:
        yield
    finally:
        G.block_pcg = orig


def gcg_solve(A, B=None, seed=0, cg_pc=0, **kw):
    """gcg_numpy.gcg_solve with the inner solve's preconditioner: cg_pc 0 none (the reference's), 1 Jacobi with the
    sigma of each ComputeW / ComputeW12 call -- the device's compW_cg_pc"""
    if cg_pc not in (0, 1):
        raise ValueError(f"cg_pc {cg_pc} (0 none, 1 Jacobi)")
    if cg_pc == 0:
        return G.gcg_solve(A, B, seed, **kw)
    with _inner_solve("jacobi"):
        return G.gcg_solve(A, B, seed, **kw)
