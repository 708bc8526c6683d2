"""TEST INFRASTRUCTURE ONLY -- numpy restatement ("port" oracle) of the GCG hot path.

A CPU restatement of the reference's block GCG eigensolver written from its behaviour,
function by function, each citing the reference file:line it follows.  It is the checker
used where the compiled reference (oracle/_ref) cannot travel, and the test bed on which
algorithmic variants of the device code (panel self-orthogonalisation, masked BlockPCG)
were validated for iteration-count parity BEFORE any CUDA was written.

Pinned in tests/test_oracle.py against oracle/_ref (the unmodified reference built here):
same iteration counts, eigenvalues to 1e-10 relative, on the 1-D pencil of reference
test/test_app_ccs.c:142-184 and on 3-D lattices.  Dense pieces use numpy (LAPACK syevd
in place of the reference's dsyevx call, reference src/ops_eig_sol_gcg.c:1201).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from pathlib import Path

import numpy as np

EPS = np.finfo(float).eps
_HERE = Path(__file__).resolve().parent
_clib = None


def clib():
    """oracle/_ref/libgcge_oracle.so: the plain-C leaf kernels (oracle/gcge_oracle.c)."""
    global _clib
    if _clib is None:
        _clib = C.CDLL(str(_HERE / "_ref" / "libgcge_oracle.so"))
    return _clib


def fill_random(x: np.ndarray, start: int, end: int):
    """reference app/app_lapack.c:322-333 (glibc rand(), column-major order)."""
    assert x.flags.f_contiguous
    n = x.shape[0]
    ptr = x.ctypes.data_as(C.POINTER(C.c_double))
    clib().oracle_fill_random(C.cast(C.addressof(ptr.contents) + 8 * n * start, C.POINTER(C.c_double)),
                              C.c_size_t(n * (end - start)))


def srand(seed: int = 0):
    clib().oracle_srand(C.c_uint(seed))


@dataclass
class OrthParams:
    block_size: int = -1
    max_reorth: int = 2
    orth_zero_tol: float = 2 * EPS
    reorth_tol: float = 50 * EPS


@dataclass
class GCGParams:
    """Defaults of reference test/test_eig_sol_gcg.c:33-115."""
    nev: int = 10
    nev_max: int = 0
    block_size: int = 0
    nev_init: int = 0
    multi_max: int = 1
    gap_min: float = 1e-5
    tol: tuple = (1e-1, 1e-8)
    num_iter_max: int = 500
    check_conv_max_num: int = 50
    initX_orth: OrthParams = field(default_factory=lambda: OrthParams(80, 2, 2 * EPS))
    compP_orth: OrthParams = field(default_factory=lambda: OrthParams(-1, 2, 2 * EPS))
    compW_orth: OrthParams = field(default_factory=lambda: OrthParams(80, 2, 2 * EPS))
    cg_max_iter: int = 30
    cg_rate: float = 1e-2
    cg_tol: float = 1e-14
    cg_tol_type: str = "abs"
    cg_shift: float = 0.0
    cg_auto_shift: int = 0
    cg_order: int = 1                # 2: ComputeW12 (reference src/ops_eig_sol_gcg.c:697-923, -gcge_compW_cg_order 2)
    # variants of the device implementation (False/"column" == the reference's algorithm)
    orth_self: str = "column"        # "column" (reference OrthSelf) | "panel" (Gram + Cholesky recurrence)

    def resolve(self):
        if self.nev_max <= 0:
            self.nev_max = 2 * self.nev
        if self.block_size <= 0:
            self.block_size = (self.nev_max - self.nev) if self.nev < 30 else self.nev // 5
        if self.nev_init <= 0:
            self.nev_init = self.nev_max
        self.nev_init = min(self.nev_init, self.nev_max)
        return self


def _matdot(M, X):
    return X.copy() if M is None else np.asfortranarray(M @ X)


# --------------------------------------------------------------------------- orth
def orth_self_column(x, start, end, B, max_reorth, zero_tol, reorth_tol):
    """OrthSelf, reference src/ops_orth.c:45-118 (column-by-column MGS with drops)."""
    k = start
    while k < end:
        bx = _matdot(B, x[:, k:k + 1])
        r = x[:, k:end].T @ bx[:, 0]                      # QtAP (end-k) x 1, :57
        rk = np.sqrt(r[0])
        if rk < zero_tol:                                   # :64-73 drop: swap in the last column
            if k < end - 1:
                x[:, k] = x[:, end - 1]
            end -= 1
            continue
        x[:, k] *= 1.0 / rk                                 # :77-80
        if k < end - 1:
            coef = r[1:] * (-1.0 / rk)                      # :84-86
            x[:, k + 1:end] += np.outer(x[:, k], coef)      # :90-91
            for _ in range(1, max_reorth - 1):              # :93-115 (empty for max_reorth <= 2)
                bx = _matdot(B, x[:, k:k + 1])
                c2 = -(x[:, k + 1:end].T @ bx[:, 0])
                x[:, k + 1:end] += np.outer(x[:, k], c2)
                if np.max(np.abs(c2)) < reorth_tol:
                    break
        k += 1
    return end


def orth_self_panel(x, start, end, B, max_reorth, zero_tol, reorth_tol):
    """Device variant: the same MGS recurrence carried out on the k x k Gram matrix
    G = X^T B X (a right-looking Cholesky factorisation with the reference's drop rule),
    then one pass X <- X T; done twice so orthogonality is at the level of column MGS.
    Mathematically identical to OrthSelf while no column is numerically dependent."""
    for _pass in range(2):
        k = end - start
        if k <= 0:
            return end
        X = x[:, start:end]
        G = X.T @ _matdot(B, X)
        Tm = np.eye(k)            # current columns == X @ Tm
        pos, n_live = 0, k
        while pos < n_live:
            gkk = G[pos, pos]
            rk = np.sqrt(gkk) if gkk > 0 else 0.0
            if rk < zero_tol:     # reference src/ops_orth.c:64-73: swap the last column in, shrink
                last = n_live - 1
                if pos < last:
                    G[[pos, last], :] = G[[last, pos], :]
                    G[:, [pos, last]] = G[:, [last, pos]]
                    Tm[:, [pos, last]] = Tm[:, [last, pos]]
                n_live -= 1
                continue
            Tm[:, pos] /= rk
            G[pos, :] /= rk
            G[:, pos] /= rk
            c = G[pos, pos + 1:n_live].copy()            # q^T B x_j
            Tm[:, pos + 1:n_live] -= np.outer(Tm[:, pos], c)
            G[pos + 1:n_live, pos + 1:n_live] -= np.outer(c, c)
            G[pos, pos + 1:] = 0.0
            G[pos + 1:, pos] = 0.0
            pos += 1
        x[:, start:start + n_live] = X @ Tm[:, :n_live]
        end = start + n_live
    return end


def _panel_once(x, start, end, B, zero_tol, scale=None):
    """One Gram + Cholesky-with-drops + update pass of orth_self_panel.  ``scale`` carries the
    factors by which earlier passes scaled each column up, so the drop test judges a column
    by its norm in the caller's scaling (gcge_b200/csrc/b200_orth.cu).  Returns (end, scale)."""
    k = end - start
    if k <= 0:
        return end, np.ones(0)
    X = x[:, start:end]
    G = X.T @ _matdot(B, X)
    Tm = np.eye(k)
    sc = np.ones(k) if scale is None else scale.copy()
    pos, n_live = 0, k
    while pos < n_live:
        gkk = G[pos, pos]
        rk = np.sqrt(gkk) if gkk > 0 else 0.0
        if rk * sc[pos] < zero_tol:
            last = n_live - 1
            if pos < last:
                G[[pos, last], :] = G[[last, pos], :]
                G[:, [pos, last]] = G[:, [last, pos]]
                Tm[:, [pos, last]] = Tm[:, [last, pos]]
                sc[[pos, last]] = sc[[last, pos]]
            n_live -= 1
            continue
        sc[pos] *= rk
        Tm[:, pos] /= rk
        G[pos, :] /= rk
        G[:, pos] /= rk
        c = G[pos, pos + 1:n_live].copy()
        Tm[:, pos + 1:n_live] -= np.outer(Tm[:, pos], c)
        G[pos + 1:n_live, pos + 1:n_live] -= np.outer(c, c)
        G[pos, pos + 1:] = 0.0
        G[pos + 1:, pos] = 0.0
        pos += 1
    x[:, start:start + n_live] = X @ Tm[:, :n_live]
    return start + n_live, sc[:n_live]


def orth_bcgs2(x, start_x, end_x, B, prm: OrthParams, rounds=2):
    """Device variant of ModifiedGramSchmidt: block classical Gram-Schmidt with
    re-orthogonalisation ("twice is enough"), the self-orthogonalisation done as a Gram +
    Cholesky panel.  Per block of columns: [project against all earlier columns, panel]
    x rounds.  Same mathematics as reference src/ops_orth.c:203-393 in exact arithmetic;
    differs in floating point by normalising BEFORE the second projection, which removes
    the reference's sensitivity to tiny columns (its re-orthogonalisation test is absolute,
    reference src/ops_orth.c:262-267)."""
    if end_x <= start_x:
        return end_x
    init_start = start_x
    block = prm.block_size
    if block <= 0:
        block = max((end_x - init_start) // 2, 2)
    block = min(block, end_x - init_start)
    while block > 0:
        s1, e1 = init_start, init_start + block
        sc = None
        for _ in range(rounds):
            if s1 > 0 and e1 > s1:
                bx = _matdot(B, x[:, s1:e1])
                x[:, s1:e1] -= x[:, :s1] @ (x[:, :s1].T @ bx)
            e1, sc = _panel_once(x, s1, e1, B, prm.orth_zero_tol, sc)
        init_end = e1
        length = block - (e1 - s1)
        length = min(length, end_x - e1 - length)
        if length > 0:
            x[:, init_end:init_end + length] = x[:, end_x - length:end_x]
        end_x -= block - (init_end - init_start)
        init_start = init_end
        block = min(block, end_x - init_start)
    return end_x


def mgs(x, start_x, end_x, B, prm: OrthParams, orth_self="column"):
    """ModifiedGramSchmidt, reference src/ops_orth.c:203-393."""
    if end_x <= start_x:
        return end_x
    if orth_self == "bcgs2":
        return orth_bcgs2(x, start_x, end_x, B, prm)
    self_fn = orth_self_column if orth_self == "column" else orth_self_panel
    if start_x > 0:                                          # :233-268 X1 -= X0 (X0^T B X1)
        for _ in range(1 + prm.max_reorth):
            bx = _matdot(B, x[:, start_x:end_x])
            coef = -(x[:, :start_x].T @ bx)
            x[:, start_x:end_x] += x[:, :start_x] @ coef
            if np.max(np.abs(coef)) < prm.reorth_tol:
                break
    init_start = start_x
    block = prm.block_size
    if block <= 0:                                           # :275-278
        block = max((end_x - init_start) // 2, 2)
    block = min(block, end_x - init_start)
    while block > 0:
        s1, e1 = init_start, init_start + block
        e1 = self_fn(x, s1, e1, B, prm.max_reorth, prm.orth_zero_tol, prm.reorth_tol)   # :285-287
        if orth_self == "panel2" and s1 > 0 and e1 > s1:
            # device variant: columns that were scaled up by the self-orthogonalisation carry an
            # amplified remainder along the earlier columns; project once more, then re-normalise
            bx = _matdot(B, x[:, s1:e1])
            x[:, s1:e1] -= x[:, :s1] @ (x[:, :s1].T @ bx)
            e1 = self_fn(x, s1, e1, B, prm.max_reorth, prm.orth_zero_tol, prm.reorth_tol)
        init_end = e1
        length = block - (e1 - s1)                           # :293-307 refill from the tail
        length = min(length, end_x - e1 - length)
        if length > 0:
            x[:, init_end:init_end + length] = x[:, end_x - length:end_x]
        end_x -= block - (init_end - init_start)
        if init_end < end_x and init_start < init_end:       # :309-361 project the block out of the rest
            bq = None
            for idx in range(1 + prm.max_reorth):
                if B is not None and idx > 0:
                    coef = -(bq.T @ x[:, init_end:end_x])    # reuse B q left in mv_ws, :315-323
                else:
                    bq = _matdot(B, x[:, init_start:init_end])
                    coef = -(bq.T @ x[:, init_end:end_x])
                x[:, init_end:end_x] += x[:, init_start:init_end] @ coef
                if np.max(np.abs(coef)) < prm.reorth_tol:
                    break
        init_start = init_end
        block = min(block, end_x - init_start)
    return end_x


# ------------------------------------------------------------------------ BlockPCG
def block_pcg(A, b, x, max_iter, rate, tol, tol_type="abs", shift=0.0, B=None, return_info=False):
    """BlockPCG, reference src/ops_lin_sol.c:140-437 (operator A + shift*B as in
    MatDotMultiVecShift, reference src/ops_eig_sol_gcg.c:63-96).  x is updated in place.
    Returns (niter, residual norms); with return_info also a dict with "stop" (per column, the
    number of iterations that updated it) and "ratios" (residual / threshold of every comparison
    behind a stop decision: how close each decision was)."""
    k = b.shape[1]

    def op(v):
        y = _matdot(A, v)
        if shift != 0.0:
            y += shift * (v if B is None else _matdot(B, v))
        return y

    norm_b = np.sqrt(np.sum(b * b, axis=0)) if tol_type == "rel" else np.ones(k)
    r = b - op(x)
    rho2 = np.sum(r * r, axis=0)
    init_res = np.sqrt(rho2)
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
        p[:, u] = r[:, u] + p[:, u] * beta
        w = op(p[:, u])
        ptw = np.sum(p[:, u] * w, axis=0)
        rho1[u] = rho2[u]
        alpha = rho2[u] / ptw
        x[:, u] += p[:, u] * alpha
        r[:, u] -= w * alpha
        rho2[u] = np.sum(r[:, u] * r[:, u], axis=0)
        last_res[u] = np.sqrt(rho2[u])
        if return_info:
            ratios += [last_res[i] / t for i in unconv for t in (rate * init_res[i], tol * norm_b[i]) if t > 0]
        unconv = [i for i in unconv if last_res[i] > rate * init_res[i] and last_res[i] > tol * norm_b[i]]
        niter += 1
    if return_info:
        return niter, last_res, {"stop": stop, "ratios": np.array(ratios)}
    return niter, last_res


# ----------------------------------------------------------------------------- GCG
class GCG:
    """GCG(), reference src/ops_eig_sol_gcg.c:1253-1558, with its phases as methods."""

    def __init__(self, A, B, prm: GCGParams, verbose=False):
        self.A, self.B, self.p = A, B, prm.resolve()
        self.verbose = verbose
        self.n = A.shape[0]

    # -- reference :925-1252
    def rayleigh_ritz(self, nev_conv):
        s = self
        if s.sizeP > 0:                                      # :936-949 P^T (old projected matrix) P
            Pc = s.ss_evec[:, s.sizeX - s.sizeC:s.sizeX - s.sizeC + s.sizeP]
            PtAP = Pc.T @ (s.ss_matA @ Pc)
        s.sizeV = s.sizeX + s.sizeP + s.sizeW
        s.startN += nev_conv - s.sizeC
        s.endN = min(s.endN + (nev_conv - s.sizeC), s.endX)
        s.sizeN = s.endN - s.startN
        s.sizeC = nev_conv
        N = s.sizeV - s.sizeC
        M = np.zeros((N, N))
        V = s.V
        if s.sizeW > 0:                                      # :970-987 one SpMM + Gram
            AW = _matdot(s.A, V[:, s.startW:s.endW])
            blk = V[:, s.startN:s.endW].T @ AW
            c0 = s.sizeX + s.sizeP - s.sizeC
            M[:, c0:c0 + s.sizeW] = blk
            M[c0:c0 + s.sizeW, :c0] = blk[:c0, :].T
        if s.sizeX == s.sizeV:                               # :989-1011 first call: full X^T A X
            AX = _matdot(s.A, V[:, s.sizeC:s.sizeX])
            M[:, :] = V[:, s.sizeC:s.sizeX].T @ AX
        else:
            nx = s.sizeX - s.sizeC
            M[np.arange(nx), np.arange(nx)] = s.ss_eval[s.sizeC:s.sizeX]   # :1020-1024
            if s.sizeP > 0:
                M[nx:nx + s.sizeP, nx:nx + s.sizeP] = PtAP                 # :1025-1032
        M = 0.5 * (M + M.T) if s.sizeX == s.sizeV else M
        Ms = M + s.p.cg_shift * np.eye(N) if s.p.cg_shift != 0.0 else M
        w, Z = np.linalg.eigh(Ms)                            # :1201 dsyevx('V','A','U')
        s.ss_eval[s.sizeC:s.sizeC + N] = w - s.p.cg_shift
        s.ss_evec = np.asfortranarray(Z)
        s.ss_matA = M
        s.ss_eval[s.sizeV:] = s.ss_eval[s.sizeV - 1]         # :1353-1355 / :1488-1490

    # -- reference :159-194
    def ritz_vec_update(self):
        s = self
        s.ritz[:, s.startN:s.endX] = s.V[:, s.startN:s.endW] @ s.ss_evec[:, :s.endX - s.startN]

    # -- reference :195-315
    def check_convergence(self, num_check):
        s = self
        tol = s.p.tol
        lam = s.ss_eval
        X = s.ritz[:, s.startN:s.startN + num_check]
        R = _matdot(s.A, X) - _matdot(s.B, X) * lam[s.startN:s.startN + num_check]
        res = np.sqrt(np.sum(R * R, axis=0)) if num_check > 0 else np.zeros(0)
        s.last_res = res
        idx = 0
        while idx < num_check:
            ev = abs(lam[s.startN + idx])
            if ev > tol[1]:
                if res[idx] > tol[0] or res[idx] > ev * tol[1]:
                    break
            elif res[idx] > tol[0]:
                break
            idx += 1
        while idx > 0:                                       # :253-259 do not split a cluster
            a, b = lam[s.startN + idx - 1], lam[s.startN + idx]
            if abs((a - b) / a) > s.p.gap_min:
                break
            idx -= 1
        nev_conv = s.sizeC + idx
        offset = []                                          # :262-302 unconverged index blocks
        state, num_unconv, cur = 1, 0, None
        done = False
        for i in range(num_check):
            unconverged = res[i] > tol[0] or res[i] > abs(lam[s.startN + i]) * tol[1]
            if unconverged:
                if state:
                    cur = s.startN + i
                    state = 0
                num_unconv += 1
                if num_unconv == s.sizeN:
                    offset.append((cur, s.startN + i + 1))
                    done = True
                    break
            elif not state:
                offset.append((cur, s.startN + i))
                state = 1
        if not done and num_unconv < s.sizeN:
            if state == 1:
                cur = s.startN + num_check
            hi = min(s.startN + num_check + s.sizeN - num_unconv, s.endX)
            assert cur < hi
            offset.append((cur, hi))
        assert offset
        return nev_conv, offset

    # -- reference :316-457
    def compute_p(self, offset):
        s = self
        N = s.sizeV - s.sizeC
        E = s.ss_evec
        cols = []
        for (o1, o2) in offset:
            cols.extend(range(o1 - s.sizeC, o2 - s.sizeC))
        sizeP = len(cols)
        c0 = s.sizeX - s.sizeC
        blockP = E[:, cols].copy()
        blockP[cols, :] = 0.0                                # :345-352 zero the N-part rows
        work = np.asfortranarray(np.zeros((N, c0 + sizeP)))
        work[:, :c0] = E[:, :c0]
        work[:, c0:] = blockP
        endP = mgs(work, c0, c0 + sizeP, None, s.p.compP_orth, "bcgs2" if s.p.orth_self == "bcgs2" else "column")
        sizeP = endP - c0
        s.ss_evec = np.asfortranarray(np.hstack([work[:, :c0 + sizeP], E[:, c0 + sizeP:]]))
        s.startP, s.endP, s.sizeP = s.sizeX, s.sizeX + sizeP, sizeP
        s.V[:, s.startP:s.endP] = s.V[:, s.startN:s.endW] @ work[:, c0:c0 + sizeP]

    # -- reference :472-696
    def compute_w(self, offset):
        s = self
        sigma = 0.0
        if s.p.cg_auto_shift == 1:
            sigma = -s.ss_eval[s.sizeC] + (s.ss_eval[s.sizeC + 1] - s.ss_eval[s.sizeC]) * 0.01
        sigma += s.p.cg_shift
        s.startW = s.endP
        cols = []
        for (o1, o2) in offset:
            cols.extend(range(o1, o2))
        k = len(cols)
        s.endW = s.startW + k
        s.V[:, s.startW:s.endW] = s.ritz[:, cols]                           # initial guess, :500-503
        b = _matdot(s.B, s.V[:, cols]) * (s.ss_eval[cols] + sigma)          # :516-534
        xw = s.V[:, s.startW:s.endW].copy(order="F")
        niter, _ = block_pcg(s.A, b, xw, s.p.cg_max_iter, s.p.cg_rate, s.p.cg_tol, s.p.cg_tol_type,
                             shift=sigma, B=s.B)
        s.cg_iters.append(niter)
        s.V[:, s.startW:s.endW] = xw
        s.endW = mgs(s.V, s.startW, s.endW, s.B, s.p.compW_orth, s.p.orth_self)   # :644-663
        s.sizeW = s.endW - s.startW

    # -- reference :697-923: W = [W1 | W2], the inner solve for the first half of the unconverged columns
    #    and the same systems solved again from W1 as the initial guess
    def compute_w12(self, offset):
        s = self
        ev = s.ss_eval
        sigma = 0.0
        if s.p.cg_auto_shift == 1:                                          # :707-713
            if s.sizeC < 3:
                d = 3 * (ev[1] - ev[0])
            else:
                d = ev[s.sizeC] - ev[s.sizeC - 3]
            sigma = -ev[s.sizeC] + (d if d > 1 else 1)
        sigma += s.p.cg_shift
        cols = []
        for (o1, o2) in offset:
            cols.extend(range(o1, o2))
        cols = cols[:len(cols) // 2]                                        # total_length/2, :740-772
        k = len(cols)
        s.startW = s.endP
        s.V[:, s.startW:s.startW + k] = s.ritz[:, cols]
        b = _matdot(s.B, s.V[:, cols]) * (ev[cols] + sigma)
        xw = s.V[:, s.startW:s.startW + k].copy(order="F")
        n1, _ = block_pcg(s.A, b, xw, s.p.cg_max_iter, s.p.cg_rate, s.p.cg_tol, s.p.cg_tol_type, shift=sigma, B=s.B)
        s.V[:, s.startW:s.startW + k] = xw
        xw2 = xw.copy(order="F")                                            # second solve starts from the first, :800-804
        n2, _ = block_pcg(s.A, b, xw2, s.p.cg_max_iter, s.p.cg_rate, s.p.cg_tol, s.p.cg_tol_type, shift=sigma, B=s.B)
        s.V[:, s.startW + k:s.startW + 2 * k] = xw2
        s.cg_iters.append(n1 + n2)
        s.endW = s.startW + 2 * k
        s.endW = mgs(s.V, s.startW, s.endW, s.B, s.p.compW_orth, s.p.orth_self)
        s.sizeW = s.endW - s.startW

    def solve(self, seed_already_set=False, evec_given=None):
        s, p = self, self.p
        n = s.n
        nev0 = min(p.nev, p.nev_max)
        bs = p.block_size
        s.V = np.zeros((n, p.nev_max + 2 * bs), order="F")
        s.ritz = np.zeros((n, p.nev_max), order="F")
        s.ss_eval = np.ones(p.nev_max + 2 * bs)
        s.cg_iters = []
        s.sizeC, s.sizeN = 0, bs
        s.sizeX, s.sizeP, s.sizeW = p.nev_init, 0, 0
        s.sizeV = s.sizeX
        s.startN, s.endN, s.endX = 0, bs, s.sizeX
        s.startP = s.endP = s.endX
        s.startW = s.endW = s.endP
        # InitializeX, reference :101-158: the given block first (warm start, :107-109,140), then
        # random columns behind whatever survived its orthonormalisation
        ng = 0
        if evec_given is not None and evec_given.shape[1] > 0:
            ng = evec_given.shape[1]
            assert p.nev_init >= ng
            s.V[:, :ng] = evec_given
            ng = mgs(s.V, 0, ng, s.B, p.initX_orth, p.orth_self)
        fill_random(s.V, ng, s.sizeX)
        e = mgs(s.V, ng, s.sizeX, s.B, p.initX_orth, p.orth_self)
        assert e == s.sizeX
        s.ss_matA = None
        s.rayleigh_ritz(0)
        s.ritz_vec_update()
        nev = 2 * bs if p.nev_init < p.nev_max else nev0
        nev = min(nev, nev0)
        num_iter, num_iter_max = 0, p.num_iter_max
        nev_conv = 0
        while True:
            num_check = 0 if num_iter <= 0 else (s.sizeN if s.startN + s.sizeN < s.endX else s.endX - s.startN)
            num_check = min(num_check, p.check_conv_max_num)
            nev_conv, offsetW = s.check_convergence(num_check)
            if s.verbose:
                print(num_iter, nev_conv, s.last_res[:1])
            if nev_conv >= nev:
                if nev_conv >= nev0:
                    break
                # grow X by P and W, reference :1400-1428
                nev = min(nev + s.sizeP + s.sizeW, nev0)
                newX = min(s.sizeX + s.sizeP + s.sizeW, p.nev_max)
                s.ritz[:, s.endX:newX] = s.V[:, s.startN:s.endW] @ s.ss_evec[:, s.endX - s.sizeC:newX - s.sizeC]
                s.sizeX = newX
                s.sizeP = s.sizeW = 0
                s.sizeV = s.sizeX
                s.startP = s.endP = s.endX
                s.startW = s.endW = s.endP
                s.endX = s.sizeX
                s.endN = min(s.startN + bs, s.endX)
                s.sizeN = s.endN - s.startN
                num_iter_max -= num_iter
                num_iter = 0
            if num_iter == 0:
                s.sizeP = 0
                s.startP = s.endP = s.endX
            else:
                s.compute_p(s.offsetP)
            s.V[:, s.startN:s.endX] = s.ritz[:, s.startN:s.endX]          # ComputeX, reference :458-471
            if p.cg_order != 1:
                s.compute_w12(offsetW)                                      # reference :1451-1456
            else:
                s.compute_w(offsetW)
            s.offsetP = offsetW
            s.rayleigh_ritz(nev_conv)
            s.ritz_vec_update()
            num_iter += 1
            if num_iter >= num_iter_max:
                break
        s.num_iter = num_iter + (p.num_iter_max - num_iter_max)
        s.nev_conv = nev_conv
        return {"eval": s.ss_eval[:s.sizeX].copy(), "evec": s.ritz[:, :s.sizeX].copy(),
                "num_iter": s.num_iter, "nev_conv": nev_conv, "cg_iters": s.cg_iters}


def gcg_solve(A, B=None, seed=0, **kw):
    """A, B: scipy sparse (or dense) symmetric matrices.  Seeds glibc rand() like the
    reference driver (srand(0), reference test/test_eig_sol_gcg.c:87)."""
    variant = {k: kw.pop(k) for k in ("orth_self",) if k in kw}
    verbose = kw.pop("verbose", False)
    evec_given = kw.pop("evec_given", None)
    prm = GCGParams(**kw, **variant)
    srand(seed)
    return GCG(A, B, prm, verbose=verbose).solve(evec_given=evec_given)
