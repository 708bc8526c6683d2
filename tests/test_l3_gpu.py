"""GPU parity of the fused L3 providers: orthogonalisation (reference test/test_orth.c:21-178
turned into assertions), BlockPCG (reference test/test_lin_sol.c:58-116) and the projected
eigen-solve that replaces dsyevx."""
import ctypes as C

import numpy as np
import pytest

from gcge_b200 import problems as P

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps


def gram_err(v, Bd, k):
    g = v[:, :k].T @ (Bd @ v[:, :k]) if Bd is not None else v[:, :k].T @ v[:, :k]
    return np.abs(g - np.eye(k)).max()


@pytest.mark.parametrize("with_B", [False, True])
def test_orth_rank_deficient_like_reference_TestOrth(b200, with_B):
    """reference test/test_orth.c:44-111: 10 vectors, columns 5-9 duplicated from 0-4;
    orthogonalise from 0 and from 2; X^T B X must be the identity on the surviving columns and
    the dependent ones must be dropped."""
    pen = P.p1_fem_kuhn(8)
    n = pen.A.ncols
    Bm = b200.Mat(pen.B) if with_B else None
    Bd = pen.B.to_scipy() if with_B else None
    rng = np.random.default_rng(4)
    x = np.asfortranarray(rng.random((n, 10)))
    x[:, 5:10] = x[:, 0:5]
    for start in (0, 2):
        X = b200.MultiVec.from_numpy(x)
        if start == 2:     # the first two must already be orthonormal
            e0 = b200.orth(X, 0, 2, B=Bm, block_size=8, max_reorth=5, orth_zero_tol=1e-8)
            assert e0 == 2
        end = b200.orth(X, start, 10, B=Bm, block_size=8, max_reorth=5, orth_zero_tol=1e-8)
        assert end == 5
        assert gram_err(X.numpy(), Bd, end) < 1e-12


@pytest.mark.parametrize("k,start", [(1, 0), (10, 0), (40, 60), (80, 100), (100, 20)])
def test_orth_against_previous_block(b200, k, start):
    pen = P.p1_fem_kuhn(10)
    n = pen.A.ncols
    Bm = b200.Mat(pen.B); Bd = pen.B.to_scipy()
    rng = np.random.default_rng(k + start)
    x = np.asfortranarray(rng.random((n, start + k)))
    X = b200.MultiVec.from_numpy(x)
    if start:
        assert b200.orth(X, 0, start, B=Bm, block_size=80) == start
    ws = b200.MultiVec(n, 80)
    end = b200.orth(X, start, start + k, B=Bm, ws=ws, block_size=80)
    assert end == start + k
    v = X.numpy()
    assert gram_err(v, Bd, end) < 1e-12
    # the span is preserved: the new columns reproduce the old ones
    old = x[:, start:start + k]
    coef = v.T @ (Bd @ old)
    assert np.abs(v @ coef - old).max() < 1e-10 * np.abs(old).max()


@pytest.mark.parametrize("with_B", [False, True])
def test_orth_bgs_rank_deficient_like_reference_TestOrth(b200, refmod, with_B):
    """BinaryGramSchmidt + OrthSelfEVP on the device (SURVEY 8f row 2; reference src/ops_orth.c:122-201,415-640):
    the TestOrth case with 20 columns of which 8 repeat earlier ones, and the same call to the live reference's
    BinaryGramSchmidt: same number of surviving columns, X^T B X = I, and the same span."""
    pen = P.p1_fem_kuhn(8)
    n = pen.A.ncols
    Bm = b200.Mat(pen.B) if with_B else None
    Bd = pen.B.to_scipy() if with_B else None
    rng = np.random.default_rng(4)
    x = np.asfortranarray(rng.random((n, 20)))
    x[:, 12:20] = x[:, 0:8]
    for start in (0, 3):
        X = b200.MultiVec.from_numpy(x)
        if start:
            assert b200.orth_bgs(X, 0, start, B=Bm, block_size=4, orth_zero_tol=1e-8) == start
        end = b200.orth_bgs(X, start, 20, B=Bm, block_size=4, max_reorth=3, orth_zero_tol=1e-8)
        assert end == 12
        v = X.numpy()
        assert gram_err(v, Bd, end) < 1e-12
        if refmod is not None:
            xr = x.copy(order="F")
            if start:
                assert refmod.multivec_orth(xr, 0, start, B=pen.B if with_B else None, method="bgs", block_size=4, orth_zero_tol=1e-8) == start
            er = refmod.multivec_orth(xr, start, 20, B=pen.B if with_B else None, method="bgs", block_size=4, max_reorth=3,
                                      orth_zero_tol=1e-8)
            assert er == end
            m = xr[:, :end].T @ ((Bd @ v[:, :end]) if Bd is not None else v[:, :end])
            assert np.linalg.svd(m, compute_uv=False).min() > 1 - 1e-10          # same span


@pytest.mark.parametrize("k,start,block", [(16, 0, -1), (40, 60, 8), (80, 100, 16), (100, 20, -1), (64, 0, 80)])
def test_orth_bgs_against_previous_block(b200, k, start, block):
    pen = P.p1_fem_kuhn(10)
    n = pen.A.ncols
    Bm = b200.Mat(pen.B); Bd = pen.B.to_scipy()
    rng = np.random.default_rng(k + start)
    x = np.asfortranarray(rng.random((n, start + k)))
    X = b200.MultiVec.from_numpy(x)
    if start:
        assert b200.orth_bgs(X, 0, start, B=Bm, block_size=16) == start
    end = b200.orth_bgs(X, start, start + k, B=Bm, block_size=block)
    assert end == start + k
    v = X.numpy()
    assert gram_err(v, Bd, end) < 1e-12
    old = x[:, start:start + k]
    coef = v.T @ (Bd @ old)
    assert np.abs(v @ coef - old).max() < 1e-10 * np.abs(old).max()


def test_orth_tiny_and_scaled_columns(b200):
    """Columns that are almost inside span(X0) (remainder 1e-12): the case the reference's
    absolute re-orthogonalisation test mishandles (tests/test_oracle.py)."""
    rng = np.random.default_rng(8)
    n = 4000
    q, _ = np.linalg.qr(rng.standard_normal((n, 30)))
    x = np.zeros((n, 30), order="F")
    x[:, :20] = q[:, :20]
    x[:, 20:] = q[:, :20] @ rng.standard_normal((20, 10)) + 1e-12 * q[:, 20:] * (10.0 ** rng.integers(-3, 3, 10))
    X = b200.MultiVec.from_numpy(x)
    end = b200.orth(X, 20, 30, block_size=80)
    assert end == 30
    assert gram_err(X.numpy(), None, 30) < 1e-10


def _geometric_hierarchy(m0=15, levels=3):
    """7-point Laplacian on m0^3 with trilinear interpolation to (m-1)/2 grids and Galerkin coarse operators"""
    import scipy.sparse as sp

    def p1d(mf):
        mc = (mf - 1) // 2
        Pm = sp.lil_matrix((mf, mc))
        for j in range(mc):
            f = 2 * j + 1
            Pm[f, j] = 1.0; Pm[f - 1, j] = 0.5; Pm[f + 1, j] = 0.5
        return Pm.tocsc()

    def ccs(M):
        M = M.tocsc(); M.sort_indices()
        return P.CCS(M.shape[0], M.shape[1], M.indptr.astype(np.int32), M.indices.astype(np.int32), M.data.astype(np.float64))

    A = [P.laplace3d_7pt(m0).A.to_scipy().tocsc()]
    Ps, m = [], m0
    for _ in range(levels - 1):
        p1 = p1d(m)
        Pm = sp.kron(p1, sp.kron(p1, p1)).tocsc()
        Ps.append(Pm); A.append((Pm.T @ A[-1] @ Pm).tocsc()); m = (m - 1) // 2
    return A, Ps, [ccs(a) for a in A], [ccs(p) for p in Ps]


def test_reference_block_amg_over_ops_b200(b200, refmod, drive_b200):
    """SURVEY 8f row 4: the reference's BlockAMG (src/ops_lin_sol.c:466-715; V-cycles with BlockPCG smoothing,
    MultiVecFromItoJ through the prolongation matrices, src/ops_multi_grid.c:69-117) runs UNCHANGED over
    OPS_B200_Set -- rectangular device matrices, true transposed multiply for the restriction -- and gives the same
    iterates as over the reference's own dense LAPACK back end on the same three-level hierarchy."""
    if drive_b200 is None:
        pytest.skip("oracle/_ref (reference + driver) not present on this box")
    A, Ps, Ac, Pc = _geometric_hierarchy()
    n = A[0].shape[0]
    rng = np.random.default_rng(11)
    sol = np.asfortranarray(rng.random((n, 6)))
    b = np.asfortranarray(A[0] @ sol)
    max_iter = [3, 4, 4, 4, 4, 60, 60]          # V-cycles; (pre, post) smoothing steps per level
    rate = [1e-36] * 3; tol = [1e-36] * 4
    x_ref = refmod.block_amg_dense([a.toarray() for a in A], [p.toarray() for p in Ps], b, np.zeros_like(b, order="F"),
                                   max_iter, rate, tol)
    x_dev = drive_b200.block_amg(Ac, Pc, b, np.zeros_like(b, order="F"), max_iter, rate, tol)
    res0 = np.linalg.norm(b)
    assert np.linalg.norm(A[0] @ x_ref - b) < 1e-3 * res0          # the V-cycles do converge
    assert np.abs(x_dev - x_ref).max() < 1e-9 * np.abs(x_ref).max()


def test_block_pcg_like_reference_TestMultiLinearSolver(b200, refmod):
    """reference test/test_lin_sol.c:58-116: manufactured right-hand side b = A x, 4 columns,
    "abs" 1e-8; and the GCG use: 30 iterations max, rate 1e-2 (per-column stop)."""
    from gcge_b200 import api
    pen = P.laplace3d_7pt(12)
    n = pen.A.ncols
    A = b200.Mat(pen.A); Ad = pen.A.to_scipy()
    rng = np.random.default_rng(6)
    xs = np.asfortranarray(rng.random((n, 4)))
    bh = np.asfortranarray(Ad @ xs)
    Bv = b200.MultiVec.from_numpy(np.hstack([np.zeros((n, 1)), bh]))
    X = b200.MultiVec(n, 6)
    niter, res = b200.block_pcg(A, Bv, X, (1, 2), (5, 6), max_iter=500, rate=1e-30, tol=1e-8)
    sol = X.numpy()[:, 2:6]
    assert np.abs(Ad @ sol - bh).max() < 1e-7
    assert niter < 200
    if refmod is not None:
        b2 = np.asfortranarray(np.hstack([np.zeros((n, 1)), bh])); x2 = np.zeros((n, 6), order="F")
        it_ref, _ = refmod.block_pcg(pen.A, b2, x2, (1, 2), (5, 6), max_iter=500, rate=1e-30, tol=1e-8)
        assert abs(niter - it_ref) <= 1
        assert np.abs(sol - x2[:, 2:6]).max() < 1e-6
        # the GCG setting: few iterations, rate stop, per-column masks -- same iterate
        for k in (1, 4):
            X = b200.MultiVec(n, 6); x3 = np.zeros((n, 6), order="F")
            it_dev, _ = b200.block_pcg(A, Bv, X, (1, 2), (1 + k, 2 + k), max_iter=30, rate=1e-2, tol=1e-14)
            it_ref, _ = refmod.block_pcg(pen.A, b2, x3, (1, 2), (1 + k, 2 + k), max_iter=30, rate=1e-2, tol=1e-14)
            assert it_dev == it_ref
            got = X.numpy()
            assert np.abs(got - x3).max() < 1e-11 * np.abs(x3).max()


@pytest.mark.parametrize("k", [10, 40])
def test_block_pcg_fused_dot_matches_streaming_dot(b200, k):
    """The SpMM with diag(p^T A p) in its epilogue (b200_spmm_lat.cu: spmm_lat_kernel<.., DOT>) against the SpMM +
    streaming dot kernel pair (option no_fused_dot): same iteration count, same iterate up to the rounding of the
    differently ordered dot products.  The profiler's call counts show that the two arms took different paths."""
    pen = P.p1_fem_kuhn(14)
    n = pen.A.ncols
    A = b200.Mat(pen.A)
    L = b200.lib()
    rng = np.random.default_rng(11)
    bh = np.asfortranarray(rng.random((n, k)))
    out = []
    for no_fused in (0, 1):
        old = C.c_int(0)
        assert L.b200_option_get(b"no_fused_dot", C.byref(old)) == 0
        assert L.b200_option_set(b"no_fused_dot", no_fused) == 0
        try:
            X = b200.MultiVec(n, k)
            b200.prof_enable(True)
            niter, res = b200.block_pcg(A, b200.MultiVec.from_numpy(bh), X, (0, 0), (k, k), max_iter=30, rate=1e-2,
                                        tol=1e-14)
            rep = b200.prof_report()
        finally:
            b200.prof_enable(False)
            L.b200_option_set(b"no_fused_dot", old.value)
        out.append((niter, X.numpy(), rep["small_dense"]["calls"], rep["bpcg_fused"]["calls"]))
    # fused: the one-CTA reduction of the SpMM's partial sums in each of the 30 launched steps; streaming: no such
    # reduction, one more streaming kernel (p^T w) per step instead
    assert out[0][2] == 30 and out[1][2] == 0, (out[0][2:], out[1][2:])
    assert out[1][3] == out[0][3] + 30, (out[0][2:], out[1][2:])
    assert out[0][0] == out[1][0]
    assert np.abs(out[0][1] - out[1][1]).max() < 1e-11 * np.abs(out[1][1]).max()
    # and it solves the system: 30 iterations at rate 1e-2 bring the residual down by > 10
    Ad = pen.A.to_scipy()
    assert np.linalg.norm(Ad @ out[0][1] - bh) < 0.1 * np.linalg.norm(bh)


def test_block_pcg_shifted_operator(b200):
    """(A + sigma B) x = b, the operator of reference src/ops_eig_sol_gcg.c:63-96."""
    pen = P.p1_fem_kuhn(8)
    n = pen.A.ncols
    A = b200.Mat(pen.A); B = b200.Mat(pen.B)
    Ad = pen.A.to_scipy(); Bd = pen.B.to_scipy()
    rng = np.random.default_rng(16)
    xs = rng.random((n, 3))
    for sigma, Bm, Bdd in ((2.5, B, Bd), (0.5, None, None)):
        op = Ad + sigma * (Bdd if Bdd is not None else 1.0 * np.eye(n))
        bh = np.asfortranarray(op @ xs)
        X = b200.MultiVec(n, 3)
        niter, res = b200.block_pcg(A, b200.MultiVec.from_numpy(bh), X, (0, 0), (3, 3), B=Bm, shift=sigma,
                                    max_iter=400, rate=1e-30, tol=1e-10)
        assert np.abs(op @ X.numpy() - bh).max() < 1e-8


@pytest.mark.parametrize("n", [1, 2, 3, 8, 33, 120, 241])
def test_dense_syev_vs_lapack(b200, n):
    """Replaces dsyevx (reference src/ops_eig_sol_gcg.c:1201): eigenvalues to 1e-13 of the
    spectral radius, eigenvectors orthonormal and A z = w z to the same level."""
    rng = np.random.default_rng(n)
    a = rng.standard_normal((n, n)); a = a + a.T
    if n > 8:       # a degenerate cluster and a near-diagonal block, as the projected matrix has
        a[:4, :4] = np.diag([1.0, 1.0, 1.0, 1.0]) * 3.0
        a[:4, 4:] *= 1e-9; a[4:, :4] *= 1e-9
    w, z, sweeps = b200.dense_syev(a)
    wl = np.linalg.eigvalsh(a)
    scale = max(np.abs(wl).max(), 1e-300)
    assert np.abs(w - wl).max() < 1e-13 * scale
    assert np.all(np.diff(w) >= 0)
    assert np.abs(z.T @ z - np.eye(n)).max() < 1e-12      # ~ n * eps * sweeps
    assert np.abs(a @ z - z * w).max() < 1e-12 * scale
    assert 1 <= sweeps <= 15


@pytest.mark.parametrize("n", [100, 280, 480])
def test_dense_syev_projected_matrix_shape(b200, n):
    """The matrix the solver actually sees (reference src/ops_eig_sol_gcg.c:1013-1033): a diagonal
    X block (the previous Ritz values, with clusters), a dense border and a dense P/W block; order
    up to nevMax + 2 block_size = 480 at the headline configuration."""
    rng = np.random.default_rng(n)
    nx = (n * 5) // 6
    a = np.zeros((n, n))
    lam = np.sort(rng.uniform(30, 650, nx)); lam[3:6] = lam[3]          # a triple eigenvalue
    a[np.arange(nx), np.arange(nx)] = lam
    bw = n - nx
    e = rng.standard_normal((nx, bw)) * 5
    c = rng.standard_normal((bw, bw)); c = c @ c.T * 50 + np.eye(bw) * 700
    a[:nx, nx:] = e; a[nx:, :nx] = e.T; a[nx:, nx:] = c
    w, z, sweeps = b200.dense_syev(a)
    wl = np.linalg.eigvalsh(a)
    scale = np.abs(wl).max()
    assert np.abs(w - wl).max() < 1e-12 * scale
    assert np.abs(z.T @ z - np.eye(n)).max() < 2e-12
    assert np.abs(a @ z - z * w).max() < 1e-12 * scale
    assert 1 <= sweeps <= 15


def test_dense_syev_uses_upper_triangle_like_dsyevx(b200):
    rng = np.random.default_rng(77)
    a = rng.standard_normal((20, 20)); s = np.triu(a) + np.triu(a, 1).T
    junk = np.triu(a) + np.tril(rng.standard_normal((20, 20)), -1)
    w, _, _ = b200.dense_syev(junk)
    assert np.abs(w - np.linalg.eigvalsh(s)).max() < 1e-13 * np.abs(s).max() * 20
