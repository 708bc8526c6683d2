"""BlockPCG on the device (b200_block_pcg: gcge_b200/host/b200_bpcg.c, gcge_b200/csrc/b200_bpcg.cu) against the
reference's BlockPCG restated in numpy (oracle/gcg_numpy.block_pcg, reference src/ops_lin_sol.c:140-437).

In the reference every column is an independent CG -- its own alpha, beta and stop test -- and only the SpMM is shared.
The reference here multiplies through the plain-C CCS scatter, which every device SpMM kernel reproduces bit for bit
(tests/test_slots_gpu.py), so the two runs differ only by the summation order of the dot products and FMA contraction.
That is what the tolerances below allow for, and all they allow for.

Every case forces one path through the solver -- lattice SpMM with constant or variable coefficients, the 1-D
diagonal kernel, CSR, each with diag(p^T A p) in the SpMM epilogue or in the streaming dot kernel, the shifted
operator, the split into chunks -- and asserts from the matrix storage and the profiler's per-class call counts that
it was taken.  Options are switched through b200_option_set: the environment is read once, at b200_init."""
import contextlib
import ctypes as C
import functools
from dataclasses import dataclass

import numpy as np
import pytest
import scipy.sparse as sp

from gcge_b200 import problems as P
from oracle import gcg_numpy as G

from test_slots_gpu import _lattice_matrix

X_TOL = 1e-11           # per column: max|x_dev - x_ref| <= X_TOL * max|x_ref|
RES_TOL = 1e-10         # returned residual vs. the reference's largest last_res, relative
MARGIN = 1e-6           # every stop decision of the reference run: |residual / threshold - 1| >= MARGIN
SWEEP = range(13)       # max_iter = 0 ... 12: every stopping point of the deferred x update and the final flush

SETTINGS = {            # (max_iter, rate, tol, tol_type)
    "gcg": (30, 1e-2, 1e-14, "abs"),          # the GCG's inner solve (b200_gcg.c: compW_cg_*)
    "gcg_rel": (30, 1e-2, 1e-14, "rel"),
    "tight_abs": (300, 1e-30, 1e-7, "abs"),
    "tight_rel": (300, 1e-30, 1e-8, "rel"),
}


def _ccs(m):
    m = sp.csc_matrix(m)
    m.sum_duplicates(); m.sort_indices()
    return P.CCS(m.shape[0], m.shape[1], m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data.astype(np.float64))


def _spd_on_pattern(S, seed):
    """An SPD matrix with the sparsity pattern of S: symmetric positive edge weights, the weighted graph Laplacian of
    them plus a positive diagonal (an M-matrix).  Every entry has its own value."""
    rng = np.random.default_rng(seed)
    n = S.shape[0]
    U = sp.triu(sp.csc_matrix(S), 1).tocoo()
    W = sp.coo_matrix((rng.uniform(0.5, 1.5, U.nnz), (U.row, U.col)), shape=(n, n)).tocsc()
    W = W + W.T
    d = np.asarray(W.sum(axis=1)).ravel() + rng.uniform(0.05, 0.5, n)
    return _ccs(sp.diags(d) - W)


def _banded(n=3000, offsets=(1, 7, 40), seed=3):
    """SPD with full bands: a diagonal image, but no lattice (the bands do not stop at lattice faces)."""
    S = sp.diags([np.ones(n - o) for o in offsets], list(offsets), shape=(n, n))
    return _spd_on_pattern(S + S.T, seed)


def _irregular(n=1500, seed=5):
    """SPD with a random pattern: too many diagonals for the diagonal image, so the CSR kernels multiply."""
    S = sp.random(n, n, density=0.004, random_state=seed, format="csc")
    return _spd_on_pattern(S + S.T, seed)


@functools.lru_cache(None)
def matrices(name):
    """(A, B) as problems.CCS"""
    if name == "7pt14":
        return P.laplace3d_7pt(14).A, None
    if name == "7pt12":
        return P.laplace3d_7pt(12).A, None
    if name == "7pt60":
        return P.laplace3d_7pt(60).A, None
    if name == "27pt10":
        pen = P.q1_27pt(10); return pen.A, pen.B
    if name == "p1_12":
        pen = P.p1_fem_kuhn(12); return pen.A, pen.B
    if name == "var7":
        return _spd_on_pattern(_lattice_matrix(13, 9, 7, "7pt").to_scipy(), 1), None
    if name == "varp1":
        return _spd_on_pattern(_lattice_matrix(11, 8, 9, "p1").to_scipy(), 2), None
    if name == "banded":
        return _banded(), None
    if name == "irregular":
        return _irregular(), None
    raise KeyError(name)


class CcsOp:
    """A matrix for oracle/gcg_numpy whose product is the plain-C CCS scatter (oracle/gcge_oracle.c): the bits the
    device SpMM kernels produce."""

    def __init__(self, M):
        self.M, self.shape = M, (M.nrows, M.ncols)

    def __matmul__(self, v):
        v = np.asfortranarray(v)
        n, k = v.shape
        y = np.zeros((n, k), order="F")
        dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))
        G.clib().oracle_ccs_spmm(n, ip(self.M.j_col), ip(self.M.i_row), dp(self.M.data), dp(v), dp(y), k)
        return y


@dataclass(frozen=True)
class Case:
    id: str
    mat: str
    k: int
    arm: str                    # lat_const | lat_var | dia | csr : which SpMM storage multiplies
    fused: bool                 # p^T w in the SpMM epilogue (else the streaming dot kernel)
    setting: str = "gcg"
    b_off: int = 0              # column offsets of b and x inside wider multi-vectors
    x_off: int = 0
    b_pad: int = 0              # extra columns after the solve's range
    x_pad: int = 0
    ws: int = 0                 # workspace columns (0: k, as api.block_pcg makes them)
    mat_opts: tuple = ()        # options read when the device matrix is created
    call_opts: tuple = ()       # options read during the solve
    shift: float = 0.0          # powers of two: shift * v is exact, so A p + shift B p has the reference's bits
    with_B: bool = False
    seed: int = 0

    @property
    def chunks(self):
        wk = min(self.ws or self.k, 128)
        return -(-self.k // wk)


CASES = [
    # lattice SpMM, constant stencil, fused dot (spmm_lat_kernel<.., DOT=true, CONST=true>)
    Case("lat_const_7pt_k8", "7pt14", 8, "lat_const", True, b_off=2, b_pad=2),
    Case("lat_const_27pt_k10", "27pt10", 10, "lat_const", True, "tight_abs", x_off=4, x_pad=1),
    Case("lat_const_p1_k16_rel", "p1_12", 16, "lat_const", True, "gcg_rel", b_off=2, x_off=2),
    Case("lat_const_p1_k16_oddoff", "p1_12", 16, "lat_const", True, b_off=1, x_off=3, x_pad=2, seed=7),
    Case("lat_const_p1_k40_gcg_geometry", "p1_12", 40, "lat_const", True, b_off=3, b_pad=7, ws=40, seed=1),
    Case("lat_const_7pt_k64", "7pt12", 64, "lat_const", True, "tight_rel"),
    Case("lat_const_7pt60_k40", "7pt60", 40, "lat_const", True, seed=2),
    # lattice SpMM, variable coefficients, fused dot (CONST=false)
    Case("lat_var_7pt_k16", "var7", 16, "lat_var", True),
    Case("lat_var_p1_k40", "varp1", 40, "lat_var", True, "tight_abs", b_off=2),
    Case("lat_var_no_const_p1_k10", "p1_12", 10, "lat_var", True, "tight_rel", call_opts=(("lat_no_const", 1),)),
    # 1-D diagonal kernel, fused dot (spmm_dia_ws_kernel<.., DOT=true>)
    Case("dia_7pt_k16", "7pt14", 16, "dia", True, mat_opts=(("no_lat", 1),)),
    Case("dia_p1_k40", "p1_12", 40, "dia", True, "tight_rel", mat_opts=(("no_lat", 1),), x_off=2),
    Case("dia_banded_k10", "banded", 10, "dia", True, "gcg_rel"),
    # SpMM, then the streaming p^T w kernel
    Case("stream_no_fused_p1_k16", "p1_12", 16, "lat_const", False, call_opts=(("no_fused_dot", 1),)),
    Case("stream_7pt_k6", "7pt14", 6, "lat_const", False),
    Case("stream_27pt_k22", "27pt10", 22, "lat_const", False, "tight_abs"),
    Case("stream_p1_k72", "p1_12", 72, "lat_const", False),
    Case("stream_7pt_k128", "7pt12", 128, "lat_const", False, "gcg_rel"),
    Case("stream_p1_k3", "p1_12", 3, "lat_const", False),
    Case("stream_p1_k1", "p1_12", 1, "lat_const", False, "tight_rel"),
    Case("stream_7pt_k9_oddoff", "7pt14", 9, "lat_const", False, b_off=1, x_off=2, x_pad=1),
    # CSR kernels
    Case("csr_no_dia_p1_k16", "p1_12", 16, "csr", False, mat_opts=(("no_dia", 1),)),
    Case("csr_irregular_k10", "irregular", 10, "csr", False, "tight_abs"),
    # (A + shift B) and (A + shift I)
    Case("shift_B_p1_k16", "p1_12", 16, "lat_const", False, shift=2.0, with_B=True),
    Case("shift_I_p1_k10", "p1_12", 10, "lat_const", False, "tight_rel", shift=0.5),
    Case("shift_B_27pt_k40", "27pt10", 40, "lat_const", False, "gcg_rel", b_off=1, shift=0.25, with_B=True),
    # split into chunks: wider than 128, wider than the workspaces
    Case("chunks_7pt_k130", "7pt12", 130, "lat_const", False),
    Case("chunks_p1_k200_ws40", "p1_12", 200, "lat_const", True, ws=40, seed=3),
]
CASE_IDS = [c.id for c in CASES]
BY_ID = {c.id: c for c in CASES}

# column kinds, repeated over the block: they stop at different iterations
KINDS = ["random", "eig", "warm", "solved", "zero", "local", "manufactured", "warm"]


def _op(case):
    A, B = matrices(case.mat)
    Aop = CcsOp(A)
    Bop = CcsOp(B) if case.with_B else None

    def op(v):          # the reference's operator, exactly as G.block_pcg applies it
        y = Aop @ v
        if case.shift != 0.0:
            y += case.shift * (v if Bop is None else Bop @ v)
        return y
    return Aop, Bop, op


def make_problem(case):
    """(b, x0): the right-hand sides and initial guesses of a case, one column kind per column."""
    A, B = matrices(case.mat)
    n, k = A.ncols, case.k
    _, _, op = _op(case)
    rng = np.random.default_rng(100 + case.seed)
    S = A.to_scipy()
    if case.shift != 0.0:
        S = S + case.shift * (B.to_scipy() if case.with_B else sp.identity(n))
    import scipy.sparse.linalg as sla
    V = sla.eigsh(S.tocsc(), k=3, which="LA", tol=1e-12, v0=np.ones(n))[1]
    b = np.zeros((n, k), order="F"); x0 = np.zeros((n, k), order="F")
    for c in range(k):
        kind = KINDS[c % len(KINDS)]
        scale = 10.0 ** rng.uniform(-2, 2)
        if kind in ("random", "warm"):
            b[:, c] = scale * rng.standard_normal(n)
            if kind == "warm":
                x0[:, c] = scale * rng.standard_normal(n)
        elif kind == "eig":             # in a 3-dimensional invariant subspace: stops after a few steps
            b[:, c] = op(V @ rng.standard_normal((3, 1)))[:, 0] * scale
        elif kind == "solved":          # the initial guess already solves it: r = b - A x0 is exactly 0
            x0[:, c] = scale * rng.standard_normal(n)
            b[:, c] = op(x0[:, c:c + 1])[:, 0]
        elif kind == "local":
            lo = int(rng.integers(0, n // 2))
            b[lo:lo + n // 5, c] = scale * rng.standard_normal(len(b[lo:lo + n // 5, c]))
        elif kind == "manufactured":
            b[:, c] = op(scale * rng.random((n, 1)))[:, 0]
    return b, x0


@functools.lru_cache(None)
def problem(case_id):
    return make_problem(BY_ID[case_id])


def reference(case, max_iter):
    """(niter, last_res, info, x) of the reference run truncated at max_iter"""
    _, rate, tol, tol_type = SETTINGS[case.setting]
    Aop, Bop, _ = _op(case)
    b, x0 = problem(case.id)
    x = x0.copy(order="F")
    niter, last, info = G.block_pcg(Aop, b.copy(order="F"), x, max_iter, rate, tol, tol_type, case.shift, Bop,
                                    return_info=True)
    return niter, last, info, x


@functools.lru_cache(None)
def reference_full(case_id):
    case = BY_ID[case_id]
    return reference(case, SETTINGS[case.setting][0])


# ------------------------------------------------------------------------------------------------------ reference side
@pytest.mark.parametrize("case_id", CASE_IDS)
def test_reference_decisions_are_not_marginal(case_id):
    """Every stop decision of the reference run lies at least MARGIN away from its threshold, so the device's
    different summation order cannot flip it: a case that sits on the threshold fails here, on the CPU, instead of
    flaking on the GPU.  The columns also stop at several different iterations, and some stop early."""
    case = BY_ID[case_id]
    niter, last, info, x = reference_full(case_id)
    ratios = info["ratios"]
    assert np.all(np.isfinite(ratios)) and np.abs(ratios - 1.0).min() >= MARGIN, np.abs(ratios - 1.0).min()
    stop = info["stop"]
    assert niter == stop.max() and niter > 0
    if case.k >= 6:
        assert len(set(stop.tolist())) >= 3, stop
        assert stop.min() == 0 and 0 < np.min(stop[stop > 0]) <= 4 < niter, stop        # inactive, early, late


class _SkipOneUpdate(np.ndarray):
    """x whose in-place update is dropped once: the (skip + 1)-th assignment into it is ignored"""

    def __setitem__(self, key, value):
        self.calls = getattr(self, "calls", 0) + 1
        if self.calls != self.skip + 1:
            super().__setitem__(key, value)


class _PerturbedOp(CcsOp):
    """The CCS product, either with one call's rows shifted by one (a kernel bug) or, after the initial residual, with
    every entry moved by up to one ulp (rounding: what a different summation order amounts to)"""

    def __init__(self, M, shift_call=None, ulp_seed=None):
        super().__init__(M)
        self.calls, self.shift_call = 0, shift_call
        self.rng = None if ulp_seed is None else np.random.default_rng(ulp_seed)

    def __matmul__(self, v):
        y = super().__matmul__(v)
        self.calls += 1
        if self.calls == self.shift_call:
            y = np.asfortranarray(np.roll(y, 1, axis=0))
        if self.rng is not None and self.calls > 1:        # the CG steps; r = b - A x0 keeps its bits
            y *= 1.0 + G.EPS * self.rng.choice([-1.0, 0.0, 1.0], size=y.shape)
        return y


def _worst_column_error(x, x_ref):
    scale = np.abs(x_ref).max(axis=0)
    return np.max(np.abs(x - x_ref).max(axis=0) / np.where(scale > 0, scale, 1.0))


@pytest.mark.parametrize("setting", ["gcg", "tight_abs"])
def test_tolerance_tells_a_misstep_from_rounding(setting):
    """The X_TOL bound is sharp: the reference with one x update skipped, or with one SpMM result shifted by one row,
    violates it; the reference with every SpMM result moved by up to one ulp in every call (more rounding than the
    device's summation order brings) stays inside it and stops every column at the same iteration."""
    case = Case("sharp", "p1_12", 16, "lat_const", True, setting)
    max_iter, rate, tol, tol_type = SETTINGS[setting]
    A, _ = matrices(case.mat)
    b, x0 = make_problem(case)
    runs = {}
    for name in ("exact", "skip_x", "shift_w", "ulp"):
        x = x0.copy(order="F")
        Aop = CcsOp(A)
        if name == "skip_x":
            x = x.view(_SkipOneUpdate); x.skip = 4
        elif name == "shift_w":
            Aop = _PerturbedOp(A, shift_call=6)
        elif name == "ulp":
            Aop = _PerturbedOp(A, ulp_seed=1)
        niter, last, info = G.block_pcg(Aop, b.copy(order="F"), x, max_iter, rate, tol, tol_type, return_info=True)
        runs[name] = (niter, info["stop"], np.asarray(x))
    _, stop, x_ref = runs["exact"]
    assert _worst_column_error(runs["skip_x"][2], x_ref) > 100 * X_TOL
    assert _worst_column_error(runs["shift_w"][2], x_ref) > 100 * X_TOL
    assert np.array_equal(runs["ulp"][1], stop)
    err = {name: _worst_column_error(r[2], x_ref) for name, r in runs.items()}
    print(f"sharpness {setting}: worst column max|dx|/max|x|", {k: f"{v:.2e}" for k, v in err.items()})
    assert err["ulp"] < 0.1 * X_TOL


# --------------------------------------------------------------------------------------------------------- device side
@contextlib.contextmanager
def options(opts):
    """b200_option_set for the duration, the previous values restored afterwards"""
    from gcge_b200 import api
    L = api.lib()
    old = []
    try:
        for name, value in opts:
            cur = C.c_int(0)
            api._chk(L.b200_option_get(name.encode(), C.byref(cur)))
            old.append((name, cur.value))
            api._chk(L.b200_option_set(name.encode(), int(value)))
        yield
    finally:
        for name, value in reversed(old):
            L.b200_option_set(name.encode(), value)


def _wide(a, off, pad, seed):
    """a inside a wider block at column offset off, the other columns random"""
    n, k = a.shape
    w = np.asfortranarray(np.random.default_rng(seed).standard_normal((n, off + k + pad)))
    w[:, off:off + k] = a
    return w


class DeviceCase:
    """The device matrices of a case, created under its creation-time options, and one solve at a time"""

    def __init__(self, b200, case):
        self.api, self.case = b200, case
        A, B = matrices(case.mat)
        with options(case.mat_opts):
            self.A = b200.Mat(A)
            self.B = b200.Mat(B) if case.with_B else None
        self.b, self.x0 = problem(case.id)
        self.b_in = _wide(self.b, case.b_off, case.b_pad, 1)
        self.x_in = _wide(self.x0, case.x_off, case.x_pad, 2)
        n = A.ncols
        self.ws = [b200.MultiVec(n, case.ws) for _ in range(3)] if case.ws else None

    def solve(self, max_iter):
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
                                           shift=case.shift, ws=self.ws)
                rep = api.prof_report()
            finally:
                api.prof_enable(False)
        return niter, res, Xv.numpy(), Bv.numpy(), rep


def _path_evidence(dev, case, rep, max_iter):
    """the storage and the per-class call counts that show which path the solve took"""
    st = dev.A.storage()
    if case.arm == "lat_const":
        assert st["lat_s1"] > 0 and st["lat_const"] == 1, st
    elif case.arm == "lat_var":
        assert st["lat_s1"] > 0 and (st["lat_const"] == 0 or dict(case.call_opts).get("lat_no_const") == 1), st
    elif case.arm == "dia":
        assert st["dia_nd"] > 0 and st["lat_s1"] == 0, st
    else:
        assert st["dia_nd"] == 0, st
    # per chunk: r = b - A x0 and the final x update are one bpcg_fused call each; every launched CG step is
    # update_px + update_r, and with the streaming dot the p^T w kernel as well; the fused step books its one-CTA
    # reduction of the SpMM's partial sums as small_dense
    steps = case.chunks * max_iter
    if case.fused:
        assert rep["small_dense"]["calls"] == steps, rep["small_dense"]
        assert rep["bpcg_fused"]["calls"] == 2 * case.chunks + 2 * steps, rep["bpcg_fused"]
    else:
        assert rep["small_dense"]["calls"] == 0, rep["small_dense"]
        assert rep["bpcg_fused"]["calls"] == 2 * case.chunks + 3 * steps, rep["bpcg_fused"]


def _compare(case, dev_out, ref, what):
    """device against the reference run truncated at the same max_iter; returns the worst column error"""
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
@pytest.mark.parametrize("case_id", CASE_IDS)
def test_block_pcg_matches_reference(b200, case_id):
    """One forced path: the device solve and the reference's have the same iteration count, stop every column at the
    same iteration and agree to X_TOL per column; so do the solves truncated at max_iter = 0 ... 12 and on either side
    of every column's stop.  A stopped column's x never moves again (bit for bit), the columns of x outside the range
    and the right-hand side are not touched, and a repeated call gives the same bits."""
    case = BY_ID[case_id]
    max_iter = SETTINGS[case.setting][0]
    dev = DeviceCase(b200, case)
    ref = reference_full(case_id)
    stop = ref[2]["stop"]
    full = dev.solve(max_iter)
    _path_evidence(dev, case, full[4], max_iter)
    worst = _compare(case, full, ref, "full")
    again = dev.solve(max_iter)
    assert again[:2] == full[:2] and np.array_equal(again[2], full[2]) and np.array_equal(again[3], full[3])
    x_full = full[2]
    lo, hi = case.x_off, case.x_off + case.k
    assert np.array_equal(x_full[:, :lo], dev.x_in[:, :lo]) and np.array_equal(x_full[:, hi:], dev.x_in[:, hi:])
    if not (case.shift != 0.0 and case.with_B):          # with B the right-hand side is B p's workspace
        assert np.array_equal(full[3], dev.b_in)
    else:
        bo = case.b_off
        assert np.array_equal(full[3][:, :bo], dev.b_in[:, :bo])
        assert np.array_equal(full[3][:, bo + case.k:], dev.b_in[:, bo + case.k:])
    # truncated solves: the sweep, and both sides of every stop (a column that stops after s steps still moves in
    # step s and never after it)
    ms = set(SWEEP) | {s + d for s in set(stop.tolist()) for d in (-1, 0)}
    if case.mat == "7pt60":                              # the reference takes seconds per run here
        ms = {0, 1, 2} | {s + d for s in set(stop.tolist()) for d in (-1, 0)}
    for m in sorted(v for v in ms if 0 <= v <= max_iter):
        out = dev.solve(m)
        _path_evidence(dev, case, out[4], m)
        worst = max(worst, _compare(case, out, reference(case, m), f"max_iter={m}"))
        xm = out[2][:, lo:hi]
        done = stop <= m
        assert np.array_equal(xm[:, done], x_full[:, lo:hi][:, done]), ("frozen column moved", m, np.nonzero(done)[0])
        moving = (stop == m + 1)
        if moving.any():
            assert not np.any(np.all(xm[:, moving] == x_full[:, lo:hi][:, moving], axis=0)), ("stopped early", m)
    margin = np.abs(ref[2]["ratios"] - 1.0).min()
    print(f"\nBPCG {case_id}: niter {ref[0]}, stops {sorted(set(stop.tolist()))}, "
          f"worst max|dx|/max|x| {worst:.2e}, smallest decision margin {margin:.2e}")


@pytest.mark.gpu
def test_block_pcg_trace_keeps_the_last_x_update(b200):
    """Option bpcg_trace reads the active-column count back every step and leaves the loop once no column is active.
    The x update of the last step is deferred into the next step's launch, so leaving early must still apply it:
    same iteration count and the same bits as the solve without the trace."""
    case = BY_ID["lat_const_p1_k16_rel"]
    dev = DeviceCase(b200, case)
    plain = dev.solve(SETTINGS[case.setting][0])
    with options((("bpcg_trace", 1),)):
        traced = dev.solve(SETTINGS[case.setting][0])
    assert plain[0] < SETTINGS[case.setting][0]                  # the traced loop did stop early
    assert traced[:2] == plain[:2] and np.array_equal(traced[2], plain[2])
