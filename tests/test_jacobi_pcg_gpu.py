"""Jacobi-preconditioned BlockPCG on the device (b200_block_pcg_pc with pc = 1: gcge_b200/host/b200_bpcg.c,
gcge_b200/csrc/b200_bpcg.cu) against numpy (tests/jacobi_numpy.block_pcg(precond="jacobi")), and the device GCG
with compW_cg_pc = 1 on heterogeneous-coefficient pencils.

The comparison is the one of tests/test_bpcg_gpu.py, at its tolerances: the reference side multiplies through the
plain-C CCS scatter, whose bits every device SpMM kernel reproduces, and D^-1 = 1 / (a + shift b) is formed with a shift
that is a power of two, so the two runs differ only by the summation order of the dot products and FMA contraction.
Every case forces one SpMM path and asserts from the matrix storage and the profiler's call counts that it was taken."""
import ctypes as C
import functools

import numpy as np
import pytest
import scipy.sparse.linalg as sla

from gcge_b200 import problems as P
import jacobi_numpy as J

from test_bpcg_gpu import (Case, CcsOp, KINDS, MARGIN, RES_TOL, SETTINGS, SWEEP, X_TOL, _PerturbedOp, _worst_column_error,
                           _wide, matrices, options)
from test_gcg_gpu import residual_test


@functools.lru_cache(None)
def jmatrices(name):
    """(A, B) as problems.CCS: the matrices of tests/test_bpcg_gpu.py and two with lognormal coefficients"""
    if name == "dlog10":
        pen = P.diffusion7_var(10, "lognormal", seed=5)
        return pen.A, None
    if name == "dlog10B":
        pen = P.diffusion7_var(10, "lognormal", seed=6, mass=True)
        return pen.A, pen.B
    return matrices(name)


class DiagOp(CcsOp):
    """CcsOp with the diagonal the numpy port's Jacobi reads"""

    def diagonal(self):
        return self.M.to_scipy().diagonal()


JCASES = [
    # lattice SpMM, variable coefficients (the diagonal D varies), fused p^T w
    Case("jac_lat_var_7pt_k16", "var7", 16, "lat_var", True),
    Case("jac_lat_var_p1_k40", "varp1", 40, "lat_var", True, "tight_abs", b_off=2),
    Case("jac_lat_var_lognormal_k10", "dlog10", 10, "lat_var", True, "gcg_rel"),
    # lattice SpMM, constant stencil (D = c I)
    Case("jac_lat_const_p1_k16", "p1_12", 16, "lat_const", True, x_off=2),
    Case("jac_lat_const_7pt_k8_rel", "7pt14", 8, "lat_const", True, "tight_rel"),
    # 1-D diagonal kernel (no_lat), fused p^T w
    Case("jac_dia_var7_k16", "var7", 16, "dia", True, mat_opts=(("no_lat", 1),)),
    Case("jac_dia_banded_k10", "banded", 10, "dia", True, "gcg_rel"),
    # CSR kernels, streaming p^T w
    Case("jac_csr_var7_k16", "var7", 16, "csr", False, mat_opts=(("no_dia", 1),)),
    Case("jac_csr_irregular_k10", "irregular", 10, "csr", False, "tight_rel"),
    # SpMM then the streaming p^T w kernel
    Case("jac_stream_var7_k16", "var7", 16, "lat_var", False, call_opts=(("no_fused_dot", 1),)),
    Case("jac_stream_varp1_k3", "varp1", 3, "lat_var", False, "tight_rel"),
    Case("jac_stream_var7_k9_oddoff", "var7", 9, "lat_var", False, b_off=1, x_off=2, x_pad=1),
    # (A + shift B), D = diag(A) + shift diag(B), and (A + shift I)
    Case("jac_shift_B_lognormal_k16", "dlog10B", 16, "lat_var", False, shift=2.0, with_B=True),
    Case("jac_shift_B_p1_k16", "p1_12", 16, "lat_const", False, "gcg_rel", shift=0.25, with_B=True),
    Case("jac_shift_I_var7_k10", "var7", 10, "lat_var", False, "tight_rel", shift=0.5),
    # split into chunks: wider than 128, wider than the workspaces (one D^-1 for all of them)
    Case("jac_chunks_varp1_k130", "varp1", 130, "lat_var", False),
    Case("jac_chunks_var7_k200_ws40", "var7", 200, "lat_var", True, ws=40, seed=3),
]
JCASE_IDS = [c.id for c in JCASES]
JBY_ID = {c.id: c for c in JCASES}


def _ops(case):
    A, B = jmatrices(case.mat)
    Aop = DiagOp(A)
    Bop = DiagOp(B) if case.with_B else None

    def op(v):
        y = Aop @ v
        if case.shift != 0.0:
            y += case.shift * (v if Bop is None else Bop @ v)
        return y
    return Aop, Bop, op


@functools.lru_cache(None)
def jproblem(case_id):
    """(b, x0) of a case: the column kinds of tests/test_bpcg_gpu.py"""
    case = JBY_ID[case_id]
    A, B = jmatrices(case.mat)
    n, k = A.ncols, case.k
    _, _, op = _ops(case)
    rng = np.random.default_rng(100 + case.seed)
    S = A.to_scipy()
    if case.shift != 0.0:
        import scipy.sparse as sp
        S = S + case.shift * (B.to_scipy() if case.with_B else sp.identity(n))
    V = sla.eigsh(S.tocsc(), k=3, which="LA", tol=1e-12, v0=np.ones(n))[1]
    b = np.zeros((n, k), order="F"); x0 = np.zeros((n, k), order="F")
    for c in range(k):
        kind = KINDS[c % len(KINDS)]
        scale = 10.0 ** rng.uniform(-2, 2)
        if kind in ("random", "warm"):
            b[:, c] = scale * rng.standard_normal(n)
            if kind == "warm":
                x0[:, c] = scale * rng.standard_normal(n)
        elif kind == "eig":
            b[:, c] = op(V @ rng.standard_normal((3, 1)))[:, 0] * scale
        elif kind == "solved":
            x0[:, c] = scale * rng.standard_normal(n)
            b[:, c] = op(x0[:, c:c + 1])[:, 0]
        elif kind == "local":
            lo = int(rng.integers(0, n // 2))
            b[lo:lo + n // 5, c] = scale * rng.standard_normal(len(b[lo:lo + n // 5, c]))
        elif kind == "manufactured":
            b[:, c] = op(scale * rng.random((n, 1)))[:, 0]
    return b, x0


def jreference(case, max_iter, precond="jacobi"):
    """(niter, last_res, info, x) of the numpy port truncated at max_iter"""
    _, rate, tol, tol_type = SETTINGS[case.setting]
    Aop, Bop, _ = _ops(case)
    b, x0 = jproblem(case.id)
    x = x0.copy(order="F")
    niter, last, info = J.block_pcg(Aop, b.copy(order="F"), x, max_iter, rate, tol, tol_type, case.shift, Bop,
                                    return_info=True, precond=precond)
    return niter, last, info, x


@functools.lru_cache(None)
def jreference_full(case_id):
    case = JBY_ID[case_id]
    return jreference(case, SETTINGS[case.setting][0])


# ------------------------------------------------------------------------------------------------------ reference side
@pytest.mark.parametrize("case_id", JCASE_IDS)
def test_jacobi_reference_decisions_are_not_marginal(case_id):
    """Every stop decision of the numpy port's Jacobi run lies at least MARGIN away from its threshold, so the device's
    summation order cannot flip it; and the columns stop at several different iterations."""
    case = JBY_ID[case_id]
    niter, last, info, x = jreference_full(case_id)
    ratios = info["ratios"]
    assert np.all(np.isfinite(ratios)) and np.abs(ratios - 1.0).min() >= MARGIN, np.abs(ratios - 1.0).min()
    stop = info["stop"]
    assert niter == stop.max() and niter > 0
    if case.k >= 6:
        assert stop.min() == 0 and len(set(stop.tolist())) >= 3, stop


class _UlpOp(_PerturbedOp):
    """the CCS product moved by up to one ulp per entry after the initial residual, with the diagonal Jacobi reads"""

    def diagonal(self):
        return self.M.to_scipy().diagonal()


@pytest.mark.parametrize("case_id", JCASE_IDS)
def test_jacobi_reference_residual_is_determined(case_id):
    """The returned residual is compared at RES_TOL, so it must not be rounding: with every SpMM result moved by up to
    one ulp (more than the device's summation order brings) the port's largest final residual stays within RES_TOL / 4
    and the iteration count does not change.  A solve driven down to the attainable-accuracy floor fails here, on the
    CPU: there the residual is rounding and no tolerance of this size can tell a correct device run from a wrong one."""
    case = JBY_ID[case_id]
    max_iter, rate, tol, tol_type = SETTINGS[case.setting]
    niter, last, _, _ = jreference_full(case_id)
    A, B = jmatrices(case.mat)
    b, x0 = jproblem(case_id)
    worst = 0.0
    for seed in range(3):
        x = x0.copy(order="F")
        n2, last2 = J.block_pcg(_UlpOp(A, ulp_seed=seed), b.copy(order="F"), x, max_iter, rate, tol, tol_type, case.shift,
                                DiagOp(B) if case.with_B else None, precond="jacobi")
        assert n2 == niter, (seed, n2, niter)
        worst = max(worst, abs(last2.max() - last.max()) / last.max())
    assert worst <= RES_TOL / 4, worst


# --------------------------------------------------------------------------------------------------------- device side
class JDeviceCase:
    """The device matrices of a case, created under its creation-time options, and one solve at a time"""

    def __init__(self, b200, case):
        self.api, self.case = b200, case
        A, B = jmatrices(case.mat)
        with options(case.mat_opts):
            self.A = b200.Mat(A)
            self.B = b200.Mat(B) if case.with_B else None
        self.b, self.x0 = jproblem(case.id)
        self.b_in = _wide(self.b, case.b_off, case.b_pad, 1)
        self.x_in = _wide(self.x0, case.x_off, case.x_pad, 2)
        self.ws = [b200.MultiVec(A.ncols, case.ws) for _ in range(3)] if case.ws else None

    def solve(self, max_iter, precond="jacobi"):
        """(niter, residual, x block, b block, prof report)"""
        api, case = self.api, self.case
        _, rate, tol, tol_type = SETTINGS[case.setting]
        Bv = api.MultiVec.from_numpy(self.b_in); Xv = api.MultiVec.from_numpy(self.x_in)
        k = case.k
        with options(case.call_opts):
            api.prof_enable(True)
            try:
                niter, res = api.block_pcg(self.A, Bv, Xv, (case.b_off, case.x_off), (case.b_off + k, case.x_off + k),
                                           B=self.B, max_iter=max_iter, rate=rate, tol=tol, tol_type=tol_type,
                                           shift=case.shift, ws=self.ws, precond=precond)
                rep = api.prof_report()
            finally:
                api.prof_enable(False)
        return niter, res, Xv.numpy(), Bv.numpy(), rep


def _path_evidence(dev, case, rep, max_iter):
    """storage and per-class call counts: as tests/test_bpcg_gpu.py, plus the one diagonal kernel of the call"""
    st = dev.A.storage()
    if case.arm == "lat_const":
        assert st["lat_s1"] > 0 and st["lat_const"] == 1, st
    elif case.arm == "lat_var":
        assert st["lat_s1"] > 0 and st["lat_const"] == 0, st
    elif case.arm == "dia":
        assert st["dia_nd"] > 0 and st["lat_s1"] == 0, st
    else:
        assert st["dia_nd"] == 0, st
    steps = case.chunks * max_iter
    if case.fused:
        assert rep["small_dense"]["calls"] == steps, rep["small_dense"]
        assert rep["bpcg_fused"]["calls"] == 1 + 2 * case.chunks + 2 * steps, rep["bpcg_fused"]
    else:
        assert rep["small_dense"]["calls"] == 0, rep["small_dense"]
        assert rep["bpcg_fused"]["calls"] == 1 + 2 * case.chunks + 3 * steps, rep["bpcg_fused"]


def _compare(case, dev_out, ref, what):
    niter, res, x, _, _ = dev_out
    niter_r, last_r, _, x_r = ref
    xs = x[:, case.x_off:case.x_off + case.k]
    assert niter == niter_r, (what, niter, niter_r)
    err = np.abs(xs - x_r).max(axis=0)
    scale = np.abs(x_r).max(axis=0)
    bad = np.nonzero(err > X_TOL * scale)[0]
    assert bad.size == 0, (what, bad, err[bad], scale[bad])
    assert abs(res - last_r.max()) <= RES_TOL * last_r.max(), (what, res, last_r.max())
    return np.max(err / np.where(scale > 0, scale, 1.0))


@pytest.mark.gpu
@pytest.mark.parametrize("case_id", JCASE_IDS)
def test_jacobi_block_pcg_matches_reference(b200, case_id):
    """One forced path with pc = 1: the same iteration count as the numpy port, every column to X_TOL, the residual to
    RES_TOL; the same for max_iter = 0 ... 12 and on either side of every column's stop.  A stopped column never moves
    again, columns outside the range are untouched, a repeated call gives the same bits."""
    case = JBY_ID[case_id]
    max_iter = SETTINGS[case.setting][0]
    dev = JDeviceCase(b200, case)
    ref = jreference_full(case_id)
    stop = ref[2]["stop"]
    full = dev.solve(max_iter)
    _path_evidence(dev, case, full[4], max_iter)
    worst = _compare(case, full, ref, "full")
    again = dev.solve(max_iter)
    assert again[:2] == full[:2] and np.array_equal(again[2], full[2]) and np.array_equal(again[3], full[3])
    x_full = full[2]
    lo, hi = case.x_off, case.x_off + case.k
    assert np.array_equal(x_full[:, :lo], dev.x_in[:, :lo]) and np.array_equal(x_full[:, hi:], dev.x_in[:, hi:])
    if not (case.shift != 0.0 and case.with_B):
        assert np.array_equal(full[3], dev.b_in)
    ms = set(SWEEP) | {s + d for s in set(stop.tolist()) for d in (-1, 0)}
    for m in sorted(v for v in ms if 0 <= v <= max_iter):
        out = dev.solve(m)
        _path_evidence(dev, case, out[4], m)
        worst = max(worst, _compare(case, out, jreference(case, m), f"max_iter={m}"))
        xm = out[2][:, lo:hi]
        done = stop <= m
        assert np.array_equal(xm[:, done], x_full[:, lo:hi][:, done]), ("frozen column moved", m, np.nonzero(done)[0])
    print(f"\nJacobi BPCG {case_id}: niter {ref[0]} (unpreconditioned {jreference(case, max_iter, None)[0]}), "
          f"stops {sorted(set(stop.tolist()))}, worst max|dx|/max|x| {worst:.2e}")


def _column_pcg(op, b, x, dinv, max_iter, rate, tol, norm_b, rho_with_dinv=True):
    """One column of a Jacobi PCG; rho_with_dinv = False is the wrong variant rho = r^T r with p = D^-1 r + beta p"""
    r = b - op(x)
    z = dinv * r
    rho = (r @ z) if rho_with_dinv else (r @ r)
    res0 = np.sqrt(r @ r)
    if not res0 > tol * norm_b:
        return x
    p = z.copy()
    for _ in range(max_iter):
        w = op(p)
        alpha = rho / (p @ w)
        x = x + alpha * p
        r = r - alpha * w
        res = np.sqrt(r @ r)
        if not (res > rate * res0 and res > tol * norm_b):
            break
        z = dinv * r
        rho_new = (r @ z) if rho_with_dinv else (r @ r)
        p = z + (rho_new / rho) * p
        rho = rho_new
    return x


@pytest.mark.gpu
def test_jacobi_tolerance_is_sharp(b200):
    """The device result breaks X_TOL by far against the two nearest wrong preconditioners: D = diag(A) without the
    shift B term, and D^-1 left out of rho (rho = r^T r)."""
    case = JBY_ID["jac_shift_B_lognormal_k16"]
    max_iter, rate, tol, tol_type = SETTINGS[case.setting]
    dev = JDeviceCase(b200, case)
    x_dev = dev.solve(max_iter)[2][:, case.x_off:case.x_off + case.k]
    ref = jreference_full(case.id)[3]
    assert _worst_column_error(x_dev, ref) <= X_TOL
    Aop, Bop, op = _ops(case)
    b, x0 = jproblem(case.id)
    no_sigma = x0.copy(order="F")
    J.block_pcg(Aop, b.copy(order="F"), no_sigma, max_iter, rate, tol, tol_type, case.shift, Bop,
                precond=1.0 / Aop.diagonal())
    assert _worst_column_error(x_dev, no_sigma) > 100 * X_TOL
    dinv = J.jacobi_dinv(Aop, case.shift, Bop)[:, 0]
    opc = lambda v: op(v[:, None])[:, 0]
    rho_rr = np.column_stack([_column_pcg(opc, b[:, c], x0[:, c].copy(), dinv, max_iter, rate, tol, 1.0, False)
                              for c in range(case.k)])
    assert _worst_column_error(x_dev, rho_rr) > 100 * X_TOL
    print(f"\nsharpness: device vs port {_worst_column_error(x_dev, ref):.1e}, vs D = diag(A) "
          f"{_worst_column_error(x_dev, no_sigma):.1e}, vs rho = r^T r {_worst_column_error(x_dev, rho_rr):.1e}")


def _block_pcg_pc(api, A, B, b, x, start, end, prm, pc, ws):
    niter = C.c_int(0); res = C.c_double(0)
    s, e = api._se(start, end)
    api._chk(api.lib().b200_block_pcg_pc(A.h, None if B is None else B.h, b.h, x.h, s, e, C.byref(prm), pc,
                                         ws[0].h, ws[1].h, ws[2].h, C.byref(niter), C.byref(res)))
    return niter.value, res.value


def _block_pcg_plain(api, A, B, b, x, start, end, prm, ws):
    niter = C.c_int(0); res = C.c_double(0)
    s, e = api._se(start, end)
    api._chk(api.lib().b200_block_pcg(A.h, None if B is None else B.h, b.h, x.h, s, e, C.byref(prm),
                                      ws[0].h, ws[1].h, ws[2].h, C.byref(niter), C.byref(res)))
    return niter.value, res.value


@pytest.mark.gpu
@pytest.mark.parametrize("case_id", ["jac_lat_var_7pt_k16", "jac_shift_B_lognormal_k16", "jac_chunks_var7_k200_ws40"])
def test_pc0_is_block_pcg(b200, case_id):
    """b200_block_pcg_pc with pc = 0 is b200_block_pcg: the same bits in x, b and the residual, the same launches."""
    case = JBY_ID[case_id]
    max_iter, rate, tol, tol_type = SETTINGS[case.setting]
    dev = JDeviceCase(b200, case)
    prm = b200._BpcgParams(max_iter, rate, tol, 1 if tol_type == "rel" else 0, case.shift)
    k = case.k
    ws = dev.ws or [b200.MultiVec(dev.A.nrows, k) for _ in range(3)]
    se = ((case.b_off, case.x_off), (case.b_off + k, case.x_off + k))
    runs = []
    for fn in ("plain", "pc0", "plain"):
        Bv = b200.MultiVec.from_numpy(dev.b_in); Xv = b200.MultiVec.from_numpy(dev.x_in)
        b200.sync()
        l0 = b200.kernel_launches()
        if fn == "plain":
            out = _block_pcg_plain(b200, dev.A, dev.B, Bv, Xv, *se, prm, ws)
        else:
            out = _block_pcg_pc(b200, dev.A, dev.B, Bv, Xv, *se, prm, 0, ws)
        launches = b200.kernel_launches() - l0
        runs.append((out, launches, Xv.numpy(), Bv.numpy()))
    for r in runs[1:]:
        assert r[0] == runs[0][0] and r[1] == runs[0][1], (r[:2], runs[0][:2])
        assert np.array_equal(r[2], runs[0][2]) and np.array_equal(r[3], runs[0][3])


def _with_bad_diagonal(M, row, value):
    """M (problems.CCS) with entry (row, row) set to value, or removed when value is None"""
    import scipy.sparse as sp
    S = M.to_scipy().tolil()
    S[row, row] = 0.0 if value is None else value
    S = sp.csc_matrix(S)
    if value is None:
        S.eliminate_zeros()
    S.sort_indices()
    return P.CCS(S.shape[0], S.shape[1], S.indptr.astype(np.int32), S.indices.astype(np.int32), S.data.astype(np.float64))


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["negative", "zero_entry", "missing", "negative_shift", "B_missing"])
def test_jacobi_bad_diagonal_fails_and_leaves_x(b200, what):
    """A row whose diagonal of A + shift B is not > 0, or that stores no diagonal entry, fails the call with a message;
    x and b are untouched, and the next solve runs."""
    A, _ = jmatrices("var7")
    n = A.ncols
    B = None
    shift = 0.0
    if what == "negative":
        A = _with_bad_diagonal(A, 17, -1.0)
    elif what == "zero_entry":
        A = _with_bad_diagonal(A, n - 1, 0.0)
    elif what == "missing":
        A = _with_bad_diagonal(A, 3, None)
    elif what == "negative_shift":
        shift = -float(A.to_scipy().diagonal().min()) * 4.0
    else:
        import scipy.sparse as sp
        Bs = sp.identity(n, format="lil"); Bs[5, 5] = 0.0
        Bs = sp.csc_matrix(Bs); Bs.eliminate_zeros(); Bs.sort_indices()
        B = P.CCS(n, n, Bs.indptr.astype(np.int32), Bs.indices.astype(np.int32), Bs.data.astype(np.float64))
        shift = 2.0
    Am = b200.Mat(A); Bm = None if B is None else b200.Mat(B)
    rng = np.random.default_rng(0)
    b = np.asfortranarray(rng.standard_normal((n, 4))); x = np.asfortranarray(rng.standard_normal((n, 4)))
    Bv = b200.MultiVec.from_numpy(b); Xv = b200.MultiVec.from_numpy(x)
    with pytest.raises(b200.B200Error, match="no diagonal entry or one <= 0"):
        b200.block_pcg(Am, Bv, Xv, (0, 0), (4, 4), B=Bm, shift=shift, precond="jacobi")
    assert np.array_equal(Xv.numpy(), x) and np.array_equal(Bv.numpy(), b)
    good = b200.Mat(jmatrices("var7")[0])
    niter, res = b200.block_pcg(good, Bv, Xv, (0, 0), (4, 4), precond="jacobi")
    assert niter > 0 and np.isfinite(res)


# ------------------------------------------------------------------------------------------------------------- GCG
GCG_CASES = {           # id: (coef, mass, compW_cg_shift)
    "lognormal": ("lognormal", False, 0.0),
    "jump": ("jump", False, 0.0),
    "lognormal_B_shift": ("lognormal", True, 0.5),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case_id", list(GCG_CASES))
def test_device_gcg_with_jacobi(b200, case_id):
    """Device GCG with compW_cg_pc = 1 on m = 24 heterogeneous-coefficient pencils, nev = 30: outer iterations within 1
    of the numpy port with cg_pc = 1, eigenvalues within 1e-10 of shift-invert Lanczos, the reference's residual test on
    every pair, and fewer outer iterations than the same device solve without Jacobi."""
    coef, mass, shift = GCG_CASES[case_id]
    nev = 30
    pen = P.diffusion7_var(24, coef, mass=mass)
    A, B = b200.Mat(pen.A), (b200.Mat(pen.B) if pen.B is not None else None)
    plain = b200.gcg_solve(A, B, nev=nev, compW_cg_shift=shift)
    jac = b200.gcg_solve(A, B, nev=nev, compW_cg_shift=shift, compW_cg_pc=1)
    As = pen.A.to_scipy().tocsr(); Bs = None if pen.B is None else pen.B.to_scipy().tocsr()
    port = J.gcg_solve(As, Bs, nev=nev, cg_pc=1, cg_shift=shift)
    ref = np.sort(sla.eigsh(pen.A.to_scipy().tocsc(), k=nev, M=None if Bs is None else pen.B.to_scipy().tocsc(),
                            sigma=0.0, which="LM", tol=0)[0])
    assert jac["nev_conv"] >= nev
    assert abs(jac["num_iter"] - port["num_iter"]) <= 1, (jac["num_iter"], port["num_iter"])
    err = np.max(np.abs(jac["eval"][:nev] - ref) / np.abs(ref))
    assert err < 1e-10, err
    ok, r = residual_test(pen, jac["eval"][:nev], jac["evec_mv"].numpy(0, nev))
    assert ok, r
    assert jac["num_iter"] < plain["num_iter"], (jac["num_iter"], plain["num_iter"])
    print(f"\nGCG {case_id} m=24 nev=30: device outer {plain['num_iter']} -> {jac['num_iter']} with Jacobi "
          f"(numpy port {port['num_iter']}), max rel eigenvalue error {err:.1e}")


@pytest.mark.gpu
def test_device_gcg_jacobi_on_constant_stencil(b200):
    """On p1_fem_kuhn (constant diagonal of A + sigma B) Jacobi is a rescaling: outer iterations within 1 of the solve
    without it, and the same eigenvalues to 1e-10."""
    pen = P.p1_fem_kuhn(12)
    A, B = b200.Mat(pen.A), b200.Mat(pen.B)
    plain = b200.gcg_solve(A, B, nev=10)
    jac = b200.gcg_solve(A, B, nev=10, compW_cg_pc=1)
    assert jac["nev_conv"] >= 10
    assert abs(jac["num_iter"] - plain["num_iter"]) <= 1, (jac["num_iter"], plain["num_iter"])
    assert np.max(np.abs(jac["eval"][:10] - plain["eval"][:10]) / np.abs(plain["eval"][:10])) < 1e-10
