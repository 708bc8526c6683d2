"""CPU tests of the oracle itself (SURVEY.md §8c): the plain-C leaf restatement and the numpy
GCG port are pinned against the unmodified reference (oracle/_ref, when present) and against
the committed golden vectors the reference produced (tests/golden/gcg_reference.json), plus
the analytic spectra of the synthetic operators."""
import ctypes as C

import numpy as np
import pytest

from gcge_b200 import problems as P
from oracle import gcg_numpy as G

dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))


def rel(a, b):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


# ------------------------------------------------------------------ generators
def test_stencil_matches_kron_7pt():
    import scipy.sparse as sp
    m = 5
    T = sp.diags([-1.0, 2.0, -1.0], [-1, 0, 1], shape=(m, m)); I = sp.identity(m)
    K = sp.kron(sp.kron(I, I), T) + sp.kron(sp.kron(I, T), I) + sp.kron(sp.kron(T, I), I)
    A = P.laplace3d_7pt(m).A
    assert abs(A.to_scipy() - K).max() == 0.0
    assert A.nnz == 7 * m**3 - 6 * m**2


def test_p1_stencil_matches_element_assembly():
    A4, B4, _ = P.p1_kuhn_assemble(4)
    pen = P.p1_fem_kuhn(4)
    assert abs(pen.A.to_scipy() - A4).max() < 1e-14
    assert abs(pen.B.to_scipy() - B4).max() < 1e-18
    assert np.array_equal(pen.A.j_col, pen.B.j_col) and np.array_equal(pen.A.i_row, pen.B.i_row)
    for M in (pen.A, pen.B):     # rows ascending inside every column, as the CCS contract says
        for j in range(M.ncols):
            r = M.i_row[M.j_col[j]:M.j_col[j + 1]]
            assert np.all(np.diff(r) > 0)


def test_1d_pencil_is_the_reference_driver_matrix():
    pen = P.laplace1d_pencil(807)
    h = 1.0 / 808
    assert pen.A.nnz == 3 * 807 - 2 and pen.B.nnz == 807
    d = P.ccs_to_dense(pen.A)
    assert d[0, 0] == 2.0 / h and d[1, 0] == -1.0 / h and d[5, 6] == -1.0 / h
    assert np.all(pen.B.data == 1.0 * h)


# ------------------------------------------------------------------ plain-C leaves vs reference
@pytest.mark.parametrize("k", [1, 3, 10])
def test_c_oracle_spmm_bitexact_vs_reference(refmod, k):
    if refmod is None:
        pytest.skip("oracle/_ref not present")
    pen = P.p1_fem_kuhn(6)
    n = pen.A.ncols
    rng = np.random.default_rng(1)
    x = np.asfortranarray(rng.standard_normal((n, k)))
    y_ref = np.zeros((n, k), order="F")
    refmod.mat_dot_multivec(pen.A, x, y_ref, (0, 0), (k, k))
    y = np.zeros((n, k), order="F")
    G.clib().oracle_ccs_spmm(n, ip(pen.A.j_col), ip(pen.A.i_row), dp(pen.A.data), dp(x), dp(y), k)
    assert np.array_equal(y, y_ref)          # same loop order, no contraction: bit-exact


def test_c_oracle_dense_leaves_vs_reference(refmod):
    if refmod is None:
        pytest.skip("oracle/_ref not present")
    rng = np.random.default_rng(2)
    n, p, q = 300, 7, 5
    x = np.asfortranarray(rng.standard_normal((n, p))); y = np.asfortranarray(rng.standard_normal((n, q)))
    c_ref = np.zeros((p, q), order="F"); c = np.zeros((p, q), order="F")
    refmod.multivec_inner_prod("N", x, y, (0, 0), (p, q), c_ref, p)
    G.clib().oracle_gram(C.c_char(b"N"), n, p, q, dp(x), dp(y), dp(c), p)
    assert rel(c, c_ref) < 1e-12
    coef = np.asfortranarray(rng.standard_normal((p, q))); beta = rng.standard_normal(q)
    y1 = y.copy(order="F"); y2 = y.copy(order="F")
    refmod.multivec_linear_comb(x, y1, (0, 0), (p, q), coef, p, beta, 1)
    G.clib().oracle_linear_comb(n, p, q, dp(x), dp(coef), p, dp(beta), 1, dp(y2))
    assert rel(y2, y1) < 1e-12
    a1 = y.copy(order="F"); a2 = y.copy(order="F")
    refmod.multivec_axpby(0.7, np.asfortranarray(x[:, :q]), -1.3, a1, (0, 0), (q, q))
    xs = np.asfortranarray(x[:, :q])
    G.clib().oracle_axpby(C.c_size_t(n * q), C.c_double(0.7), dp(xs), C.c_double(-1.3), dp(a2))
    assert rel(a2, a1) < 1e-14


def test_c_oracle_rand_stream_is_the_references(refmod):
    if refmod is None:
        pytest.skip("oracle/_ref not present")
    a = np.zeros((50, 3), order="F"); b = np.zeros((50, 3), order="F")
    refmod.srand(0); refmod.multivec_set_random(a, 0, 3)
    G.srand(0); G.fill_random(b, 0, 3)
    assert np.array_equal(a, b)
    assert a[0, 0] == 1804289383 / 2147483648.0      # glibc rand() after srand(0)


# ------------------------------------------------------------------ numpy GCG port
def _gen(case):
    return getattr(P, case["generator"])(**case["args"])


@pytest.mark.parametrize("idx", [0, 2, 4])
def test_port_reference_algorithm_vs_golden(golden, idx):
    """The port run with the reference's own algorithm choices (column OrthSelf) reproduces
    the reference's iteration count and eigenvalues on its driver case and small lattices."""
    case = golden["cases"][idx]
    pen = _gen(case)
    o = G.gcg_solve(pen.A.to_scipy().tocsr(), None if pen.B is None else pen.B.to_scipy().tocsr(),
                    nev=case["nev"], orth_self="column")
    assert o["nev_conv"] >= case["nev"]
    assert abs(o["num_iter"] - case["num_iter"]) <= 1
    k = min(o["nev_conv"], case["nev_conv"])
    assert rel(o["eval"][:k], np.array(case["eval"][:k])) < 1e-10


@pytest.mark.parametrize("argv,kw", [(("-gcge_compW_cg_order", "2"), {"cg_order": 2}),
                                     (("-gcge_compW_cg_auto_shift", "1"), {"cg_auto_shift": 1}),
                                     (("-gcge_compW_cg_shift", "3.0"), {"cg_shift": 3.0})])
def test_port_options_vs_golden(golden, argv, kw):
    """SURVEY 8f options in the port (ComputeW12, automatic and fixed shift of the inner solve) against
    the reference's recorded runs with the same command-line options."""
    case = [c for c in golden["cases"] if c.get("argv") == list(argv)][0]
    pen = _gen(case)
    o = G.gcg_solve(pen.A.to_scipy().tocsr(), pen.B.to_scipy().tocsr(), nev=case["nev"], orth_self="column", **kw)
    assert o["nev_conv"] >= case["nev"]
    assert abs(o["num_iter"] - case["num_iter"]) <= 1, (o["num_iter"], case["num_iter"])
    k = min(o["nev_conv"], case["nev_conv"])
    assert rel(o["eval"][:k], np.array(case["eval"][:k])) < 1e-10


def test_port_device_variant_headline_block_structure(golden):
    """The device variant of the port at nev = 200 (nevMax 400, block_size 40, projected problems of order
    up to 480 -- the block structure of the headline benchmark) against the reference's recorded run."""
    case = [c for c in golden["cases"] if c["nev"] == 200][0]
    pen = _gen(case)
    o = G.gcg_solve(pen.A.to_scipy().tocsr(), pen.B.to_scipy().tocsr(), nev=200, orth_self="bcgs2")
    assert o["nev_conv"] >= 200
    assert abs(o["num_iter"] - case["num_iter"]) <= 1, (o["num_iter"], case["num_iter"])
    k = min(o["nev_conv"], case["nev_conv"])
    assert rel(o["eval"][:k], np.array(case["eval"][:k])) < 1e-10


@pytest.mark.parametrize("idx", [0, 1, 2, 3, 4, 5, 6, 7, 8])
def test_port_device_variant_vs_golden(golden, idx):
    """The variant the device code implements (BCGS2 + Gram/Cholesky panel) against the
    reference's recorded results, incl. the nev = 30 / 50 block structures (cases 1, 7, 8): eigenvalues
    1e-10, iteration count within 1 -- the north_star contract (BASELINE.md section 4)."""
    case = golden["cases"][idx]
    pen = _gen(case)
    o = G.gcg_solve(pen.A.to_scipy().tocsr(), None if pen.B is None else pen.B.to_scipy().tocsr(),
                    nev=case["nev"], orth_self="bcgs2")
    assert o["nev_conv"] >= case["nev"]
    assert abs(o["num_iter"] - case["num_iter"]) <= 1, (o["num_iter"], case["num_iter"])
    k = min(o["nev_conv"], case["nev_conv"])
    assert rel(o["eval"][:k], np.array(case["eval"][:k])) < 1e-10


def test_golden_matches_analytic_spectra(golden):
    for case in golden["cases"]:
        ev = np.array(case["eval"])
        if case["generator"] == "laplace1d_pencil":
            # the pencil is the FD matrix scaled: eigenvalues (2-2cos(k pi h))/h^2
            assert rel(ev, P.laplace1d_eigenvalues(case["args"]["n"], len(ev))) < 1e-9
        if case["generator"] == "laplace3d_7pt":
            assert rel(ev, P.laplace3d_7pt_eigenvalues(case["args"]["m"], len(ev))) < 1e-9


def test_port_against_live_reference(refmod):
    if refmod is None:
        pytest.skip("oracle/_ref not present")
    pen = P.p1_fem_kuhn(10)
    r = refmod.gcg_solve(pen.A, pen.B, nev=8, want_evec=False)
    o = G.gcg_solve(pen.A.to_scipy().tocsr(), pen.B.to_scipy().tocsr(), nev=8, orth_self="bcgs2")
    assert abs(o["num_iter"] - r["num_iter"]) <= 1
    k = min(o["nev_conv"], r["nev_conv"])
    assert rel(o["eval"][:k], r["eval"][:k]) < 1e-10


@pytest.mark.parametrize("nev_given,noise", [(10, 1e-3), (6, 1e-6)])
def test_port_warm_start_against_live_reference(refmod, golden, nev_given, noise):
    """Warm start (reference src/ops_eig_sol_gcg.c:107-109,140) in the port, pinned against the reference
    itself with the same given block in the first nevGiven columns of evec.  Without oracle/_ref: the warm start
    on the pencil of the reference's recorded cold solve (golden case 4, p1_fem_kuhn m = 12, nev = 10) gives
    that solve's eigenvalues in no more outer iterations (+1)."""
    import scipy.sparse.linalg as sla
    m, nev = (10, 8) if refmod is not None else (12, 10)
    pen = P.p1_fem_kuhn(m)
    A, B = pen.A.to_scipy().tocsc(), pen.B.to_scipy().tocsc()
    w, v = sla.eigsh(A, k=nev_given, M=B, sigma=0.0, which="LM")
    v = v[:, np.argsort(w)]
    given = np.asfortranarray(v + noise * np.abs(v).max() * np.random.default_rng(3).standard_normal(v.shape))
    o = G.gcg_solve(A.tocsr(), B.tocsr(), nev=nev, orth_self="bcgs2", evec_given=given)
    if refmod is not None:
        r = refmod.gcg_solve(pen.A, pen.B, nev=nev, want_evec=False, evec_given=given)
        assert abs(o["num_iter"] - r["num_iter"]) <= 1, (o["num_iter"], r["num_iter"])
    else:
        r = golden["cases"][4]
        assert (r["generator"], r["args"], r["nev"]) == ("p1_fem_kuhn", {"m": 12}, 10)
        assert o["num_iter"] <= r["num_iter"] + 1, (o["num_iter"], r["num_iter"])
    assert o["nev_conv"] >= nev and r["nev_conv"] >= nev
    k = min(o["nev_conv"], r["nev_conv"])
    assert rel(o["eval"][:k], np.asarray(r["eval"][:k])) < 1e-10


@pytest.mark.parametrize("nev,nev_max,nev_init", [(30, 48, 18)])
def test_port_moving_window_against_live_reference(refmod, nev, nev_max, nev_init):
    """nevInit < nevMax (reference src/ops_eig_sol_gcg.c:1281-1283,1400-1428) in the port against the reference
    with the same -nevMax / -nevInit.  Without oracle/_ref: the iteration count against the reference's recorded
    runs (tests/golden/reference_iteration_spread.json) and the eigenvalues against the pencil's own."""
    pen = P.p1_fem_kuhn(12)
    from conftest import pencil_eigenvalues, recorded_reference_runs, reference_runs_over_threads
    if refmod is not None:
        runs = reference_runs_over_threads(
            refmod, lambda: refmod.gcg_solve(pen.A, pen.B, nev=nev, nev_max=nev_max, nev_init=nev_init, want_evec=False))
    else:
        runs = recorded_reference_runs("p1_fem_kuhn", {"m": 12}, nev, nev_max, nev_init)
    its = [q["num_iter"] for q in runs]
    r = runs[0]
    o = G.gcg_solve(pen.A.to_scipy().tocsr(), pen.B.to_scipy().tocsr(), nev=nev, nev_max=nev_max, nev_init=nev_init,
                    block_size=nev // 5, orth_self="bcgs2")
    assert o["nev_conv"] >= nev and r["nev_conv"] >= nev
    # the reference's own count moves with its OpenMP thread count on this long run (69..72)
    assert min(its) - 1 <= o["num_iter"] <= max(its) + 1, (o["num_iter"], its)
    k = min(o["nev_conv"], r["nev_conv"])
    want = r["eval"][:k] if refmod is not None else pencil_eigenvalues(pen, k)
    assert rel(o["eval"][:k], want) < 1e-10


def test_reference_orth_loses_orthogonality_inside_gcg(refmod, monkeypatch):
    """Documents WHY the device orthogonalisation is BCGS2 + Gram/Cholesky panel instead of a
    transcription of ops_orth.c (DESIGN.md "Orthogonalisation").  The numpy port is run with the
    reference's algorithm on the 7-point 20^3 Laplacian; every coefficient block ComputeP is
    about to orthonormalise (reference src/ops_eig_sol_gcg.c:371-414) is ALSO handed, unchanged,
    to the reference's own ops_orth.c and to the device variant.  When the unconverged block is
    split inside a degenerate cluster the block mixes O(1) and O(1e-7) columns, and the
    reference's routine (column-wise OrthSelf without re-orthogonalisation, absolute
    re-projection test, reference src/ops_orth.c:93,262-267) returns a basis that is off
    orthonormal by ~1e-2 -- P then is not B-orthogonal to X and the Rayleigh-Ritz step, which
    assumes V^T B V = I, stalls.  The device variant stays at rounding level on the same input."""
    if refmod is None:
        pytest.skip("oracle/_ref not present")
    pen = P.laplace3d_7pt(20)
    A = pen.A.to_scipy().tocsr()
    n = A.shape[0]
    orig = G.mgs
    worst = {"ref": 0.0, "dev": 0.0, "x0": 0.0}
    gram_err = lambda y, e: np.abs(y[:, :e].T @ y[:, :e] - np.eye(e)).max()

    def spy(x, s, e, B, prm, orth_self="column"):
        if x.shape[0] != n:                       # coefficient-space call from compute_p
            xr = x.copy(order="F"); xd = x.copy(order="F")
            er = refmod.multivec_orth(xr, s, e, None, "mgs", prm.block_size, prm.max_reorth, prm.orth_zero_tol)
            ed = orig(xd, s, e, B, prm, "bcgs2")
            worst["x0"] = max(worst["x0"], gram_err(x, s))
            worst["ref"] = max(worst["ref"], gram_err(xr, er))
            worst["dev"] = max(worst["dev"], gram_err(xd, ed))
        return orig(x, s, e, B, prm, orth_self)

    monkeypatch.setattr(G, "mgs", spy)
    G.gcg_solve(A, None, nev=20, orth_self="column", num_iter_max=18)
    assert worst["x0"] < 1e-13, worst      # the columns it orthogonalises against ARE orthonormal
    assert worst["ref"] > 1e-6, worst      # the reference's weakness, reproduced with its own code
    assert worst["dev"] < 1e-12, worst
