"""The Jacobi-preconditioned BlockPCG in numpy (tests/jacobi_numpy.block_pcg(precond="jacobi")), which the
device's b200_block_pcg_pc(pc = 1) is held to in tests/test_jacobi_pcg_gpu.py, and what it does for the GCG on
heterogeneous-coefficient pencils.  No GPU needed.

Jacobi here: z = D^-1 r with D = diag(A + shift B), rho = r^T z drives alpha and beta, p = z + beta p; the residual
norms and the stop test stay on ||r||_2, so rate and tol keep their meaning."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as sla

from gcge_b200 import problems as P
from oracle import gcg_numpy as G

import jacobi_numpy as J

SETTINGS = {            # (max_iter, rate, tol, tol_type), as tests/test_bpcg_gpu.py
    "gcg": (30, 1e-2, 1e-14, "abs"),
    "gcg_rel": (30, 1e-2, 1e-14, "rel"),
    "tight_abs": (300, 1e-30, 1e-7, "abs"),
}


def _block(n, k, seed):
    rng = np.random.default_rng(seed)
    b = np.asfortranarray(rng.standard_normal((n, k)) * 10.0 ** rng.uniform(-2, 2, k))
    x0 = np.zeros((n, k), order="F")
    x0[:, 1::3] = rng.standard_normal((n, len(range(1, k, 3))))          # warm starts
    return b, x0


def _run(A, b, x0, setting, precond=None, shift=0.0, B=None):
    max_iter, rate, tol, tol_type = SETTINGS[setting]
    x = x0.copy(order="F")
    niter, last, info = J.block_pcg(A, b.copy(order="F"), x, max_iter, rate, tol, tol_type, shift, B,
                                    return_info=True, precond=precond)
    return niter, last, info, x


def _rel_err(x, x_ref):
    scale = np.abs(x_ref).max(axis=0)
    return np.max(np.abs(x - x_ref).max(axis=0) / np.where(scale > 0, scale, 1.0))


@pytest.mark.parametrize("setting", ["gcg", "tight_abs"])
def test_jacobi_with_constant_diagonal_is_plain_cg(setting):
    """D = c I changes nothing but rounding: z = r / c, p and rho scale by 1/c, alpha by c, so x is the same.  With c a
    power of two every scaling is exact and the iterates are the same bits; with D = diag(7-point Laplacian) = 6 I they
    agree to rounding and every column stops at the same iteration."""
    A = P.laplace3d_7pt(12).A.to_scipy().tocsr()
    n = A.shape[0]
    b, x0 = _block(n, 12, 0)
    plain = _run(A, b, x0, setting)
    four = _run(A, b, x0, setting, precond=np.full(n, 0.25))
    assert four[0] == plain[0] and np.array_equal(four[2]["stop"], plain[2]["stop"])
    assert np.array_equal(four[3], plain[3]) and np.array_equal(four[1], plain[1])
    six = _run(A, b, x0, setting, precond="jacobi")
    assert np.allclose(J.jacobi_dinv(A), 1.0 / 6.0, rtol=0, atol=0)
    assert six[0] == plain[0] and np.array_equal(six[2]["stop"], plain[2]["stop"])
    assert _rel_err(six[3], plain[3]) < 1e-12
    assert np.max(np.abs(six[1] - plain[1]) / np.maximum(plain[1], 1e-300)) < 1e-10


def _textbook_pcg(op, b, x, dinv, max_iter, rate, tol, norm_b):
    """One column, the textbook preconditioned CG (Saad, Iterative Methods, Alg. 9.1) with the reference's stop test"""
    r = b - op(x)
    z = dinv * r
    rz = r @ z
    res0 = np.sqrt(r @ r)
    if not res0 > tol * norm_b:
        return 0, x
    p = z.copy()
    it = 0
    while it < max_iter:
        w = op(p)
        alpha = rz / (p @ w)
        x = x + alpha * p
        r = r - alpha * w
        it += 1
        res = np.sqrt(r @ r)
        if not (res > rate * res0 and res > tol * norm_b):
            break
        z = dinv * r
        rz_new = r @ z
        p = z + (rz_new / rz) * p
        rz = rz_new
    return it, x


@pytest.mark.parametrize("shift,with_B", [(0.0, False), (0.5, False), (2.0, True)])
def test_jacobi_block_pcg_is_textbook_pcg_per_column(shift, with_B):
    """Every column of the block solve is the single-column textbook PCG with M = D: same stop iteration, x to
    rounding.  On a heterogeneous-coefficient operator, plain, shifted by the identity, and shifted by a diagonal B."""
    pen = P.diffusion7_var(9, "lognormal", seed=3, mass=with_B)
    A = pen.A.to_scipy().tocsr()
    B = pen.B.to_scipy().tocsr() if with_B else None
    n = A.shape[0]
    S = A + shift * (B if with_B else sp.identity(n, format="csr")) if shift != 0.0 else A
    dinv = 1.0 / S.diagonal()
    b, x0 = _block(n, 9, 1)
    max_iter, rate, tol, tol_type = SETTINGS["gcg"]
    niter, _, info, x = _run(A, b, x0, "gcg", precond="jacobi", shift=shift, B=B)
    assert np.allclose(J.jacobi_dinv(A, shift, B)[:, 0], dinv, rtol=1e-15, atol=0)
    for c in range(b.shape[1]):
        it, xc = _textbook_pcg(lambda v: S @ v, b[:, c], x0[:, c].copy(), dinv, max_iter, rate, tol, 1.0)
        assert it == info["stop"][c], (c, it, info["stop"][c])
        scale = np.abs(xc).max()
        assert np.abs(x[:, c] - xc).max() <= 1e-11 * scale, (c, np.abs(x[:, c] - xc).max() / scale)
    assert niter == info["stop"].max()


def test_jacobi_oracle_rejects_a_bad_diagonal():
    A = P.diffusion7_var(5, "const").A.to_scipy().tolil()
    A[7, 7] = -1.0
    b, x0 = _block(A.shape[0], 2, 0)
    with pytest.raises(ValueError, match="not > 0"):
        _run(A.tocsr(), b, x0, "gcg", precond="jacobi")


def test_jacobi_numpy_without_preconditioner_is_the_reference_port():
    """precond None and "none" are gcg_numpy.block_pcg, the reference's iteration, bit for bit; so is the GCG with
    cg_pc = 0."""
    A = P.diffusion7_var(8, "jump", seed=2).A.to_scipy().tocsr()
    b, x0 = _block(A.shape[0], 6, 4)
    max_iter, rate, tol, tol_type = SETTINGS["gcg_rel"]
    x = x0.copy(order="F")
    niter, last, info = G.block_pcg(A, b.copy(order="F"), x, max_iter, rate, tol, tol_type, return_info=True)
    for pc in (None, "none"):
        other = _run(A, b, x0, "gcg_rel", precond=pc)
        assert other[0] == niter and np.array_equal(other[3], x) and np.array_equal(other[1], last)
        assert np.array_equal(other[2]["stop"], info["stop"]) and np.array_equal(other[2]["ratios"], info["ratios"])
    a = G.gcg_solve(A, None, nev=5)
    c = J.gcg_solve(A, None, nev=5, cg_pc=0)
    assert a["num_iter"] == c["num_iter"] and np.array_equal(a["eval"], c["eval"])
    assert G.block_pcg.__module__ == G.__name__                  # the Jacobi GCG restored the port's inner solve
    J.gcg_solve(A, None, nev=5, cg_pc=1)
    assert G.block_pcg.__module__ == G.__name__


def test_gcg_lognormal_jacobi_halves_the_outer_iterations():
    """The m = 12 lognormal-coefficient pencil with a random positive diagonal B: the GCG with the Jacobi inner solve
    needs at most half the outer iterations of the one without, and its eigenvalues agree with shift-invert Lanczos to
    1e-10."""
    nev = 10
    pen = P.diffusion7_var(12, "lognormal", mass=True)
    A = pen.A.to_scipy().tocsr(); B = pen.B.to_scipy().tocsr()
    ref = np.sort(sla.eigsh(pen.A.to_scipy().tocsc(), k=nev, M=pen.B.to_scipy().tocsc(), sigma=0.0, which="LM",
                            tol=0)[0])
    plain = J.gcg_solve(A, B, nev=nev)
    jac = J.gcg_solve(A, B, nev=nev, cg_pc=1)
    assert jac["nev_conv"] >= nev and plain["nev_conv"] >= nev
    assert 2 * jac["num_iter"] <= plain["num_iter"], (jac["num_iter"], plain["num_iter"])
    err = np.max(np.abs(np.sort(jac["eval"][:nev]) - ref) / np.abs(ref))
    assert err < 1e-10, err
    print(f"\nGCG lognormal m=12 nev=10: outer {plain['num_iter']} -> {jac['num_iter']} with Jacobi, "
          f"CG steps {sum(plain['cg_iters'])} -> {sum(jac['cg_iters'])}, max rel eigenvalue error {err:.1e}")
