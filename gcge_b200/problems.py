"""Synthetic CCS pencils for the GCG hot path (SURVEY.md §8d configs 1-5).

Every generator returns plain CCS arrays in the reference's own layout
(``CCSMAT``: reference app/app_ccs.h:20-24 -- ``data[nnz] f64``, ``i_row[nnz] i32``,
``j_col[ncols+1] i32``, 0-based, rows ascending inside each column), so the SAME
arrays can be handed to the reference (``OPS_CCS_Set``) and to ``OPS_B200_Set``.

Lattice operators are built from their constant stencil directly in CCS order
(no COO round trip): n = m**3 unknowns, lexicographic ``i + m*(j + m*k)``,
homogeneous Dirichlet boundary (boundary nodes are not unknowns).  The P1-FEM
stencils are taken from a genuine element-by-element assembly on the Kuhn
(6 tetrahedra per cube) triangulation -- the triangulation of ``data/cube4.dat``
(reference data/cube4.dat:3-4) -- see :func:`p1_kuhn_assemble`.
"""
from __future__ import annotations

import itertools
from dataclasses import dataclass
from typing import Optional

from pathlib import Path

import numpy as np


@dataclass
class CCS:
    """One CCS matrix (reference app/app_ccs.h:20-24)."""

    nrows: int
    ncols: int
    j_col: np.ndarray  # int32 [ncols+1]
    i_row: np.ndarray  # int32 [nnz]
    data: np.ndarray   # float64 [nnz]

    @property
    def nnz(self) -> int:
        return int(self.j_col[-1])

    def to_scipy(self):
        import scipy.sparse as sp

        return sp.csc_matrix((self.data, self.i_row, self.j_col), shape=(self.nrows, self.ncols))


@dataclass
class Pencil:
    """A x = lambda B x; ``B is None`` is the standard problem."""

    name: str
    A: CCS
    B: Optional[CCS]
    meta: dict


# --------------------------------------------------------------------------- 1-D
def laplace1d_pencil(n: int = 807) -> Pencil:
    """The reference's built-in test pencil (reference test/test_app_ccs.c:142-184):
    A = tridiag(-1,2,-1)/h, B = h*I, h = 1/(n+1); eigenvalues (2-2cos(k pi h))/h**2."""
    h = 1.0 / (n + 1)
    j_col = np.empty(n + 1, np.int32)
    j_col[0] = 0
    cnt = np.full(n, 3, np.int32)
    cnt[0] = 2
    cnt[-1] = 2
    np.cumsum(cnt, out=j_col[1:])
    nnz = 3 * n - 2
    i_row = np.empty(nnz, np.int32)
    data = np.empty(nnz, np.float64)
    i_row[0:2] = (0, 1)
    data[0:2] = (2.0 / h, -1.0 / h)
    cols = np.arange(1, n - 1, dtype=np.int32)
    base = 2 + 3 * (cols - 1)
    for o, (dr, v) in enumerate(((-1, -1.0 / h), (0, 2.0 / h), (1, -1.0 / h))):
        i_row[base + o] = cols + dr
        data[base + o] = v
    i_row[nnz - 2:] = (n - 2, n - 1)
    data[nnz - 2:] = (-1.0 / h, 2.0 / h)
    A = CCS(n, n, j_col, i_row, data)
    B = CCS(n, n, np.arange(n + 1, dtype=np.int32), np.arange(n, dtype=np.int32),
            np.full(n, 1.0 * h, np.float64))
    return Pencil("laplace1d", A, B, {"n": n, "h": h})


def laplace1d_eigenvalues(n: int, k: int) -> np.ndarray:
    h = 1.0 / (n + 1)
    idx = np.arange(1, k + 1)
    return (2.0 - 2.0 * np.cos(idx * np.pi * h)) / h**2


# ------------------------------------------------------------------ lattice stencils
def stencil_to_ccs(m: int, offsets, coefs) -> CCS:
    """CCS of the translation-invariant operator sum_s coefs[s]*shift(offsets[s]) on an
    m**3 Dirichlet lattice.  Built column by column in ascending row order."""
    offsets = np.asarray(offsets, dtype=np.int64).reshape(-1, 3)
    coefs = np.asarray(coefs, dtype=np.float64)
    lin = offsets[:, 0] + m * (offsets[:, 1] + m * offsets[:, 2])
    order = np.argsort(lin, kind="stable")
    offsets, coefs, lin = offsets[order], coefs[order], lin[order]
    n = m**3
    ns = len(lin)
    idx1 = np.arange(m, dtype=np.int64)
    # valid[s, axis, coordinate]
    ok = [((idx1[None, :] + offsets[:, a:a + 1]) >= 0) & ((idx1[None, :] + offsets[:, a:a + 1]) < m)
          for a in range(3)]
    j_col = np.zeros(n + 1, np.int64)
    # count per column: sum_s okx[s,i]*oky[s,j]*okz[s,k]
    cnt = np.einsum("si,sj,sk->kji", ok[0].astype(np.int32), ok[1].astype(np.int32),
                    ok[2].astype(np.int32)).reshape(-1)
    np.cumsum(cnt, out=j_col[1:])
    nnz = int(j_col[-1])
    assert nnz < 2**31, "int32 CCS index overflow"
    i_row = np.empty(nnz, np.int32)
    data = np.empty(nnz, np.float64)
    # process in slabs of k-planes to bound memory
    planes = max(1, int(4_000_000 // (m * m)))
    for k0 in range(0, m, planes):
        k1 = min(m, k0 + planes)
        kk = np.arange(k0, k1, dtype=np.int64)
        cols = (idx1[None, None, :] + m * (idx1[None, :, None] + m * kk[:, None, None])).reshape(-1)
        valid = (ok[0][:, None, None, :] & ok[1][:, None, :, None] & ok[2][:, kk][:, :, None, None])
        valid = valid.reshape(ns, -1).T  # [col, s] -- s ascending == row ascending
        rows = cols[:, None] + lin[None, :]
        lo, hi = int(j_col[cols[0]]), int(j_col[cols[-1] + 1])
        i_row[lo:hi] = rows[valid]
        data[lo:hi] = np.broadcast_to(coefs[None, :], valid.shape)[valid]
    return CCS(n, n, j_col.astype(np.int32), i_row, data)


def stencil_rows(m: int, offsets, coefs, k0: int, k1: int):
    """Rows [k0 m^2, k1 m^2) of the operator stencil_to_ccs builds, as CSR-style arrays (rp, ci, va) with GLOBAL
    column indices ascending inside a row: what one rank of a row-partitioned run owns (planes k0 .. k1-1 of the
    lattice).  Entry (r, c) of sum_s coefs[s] shift(offsets[s]) has c = r - lin(offsets[s]); for the symmetric
    stencils of this module the arrays equal the CCS arrays of the same columns (tests/test_partition.py)."""
    offsets = np.asarray(offsets, dtype=np.int64).reshape(-1, 3)
    coefs = np.asarray(coefs, dtype=np.float64)
    lin = offsets[:, 0] + m * (offsets[:, 1] + m * offsets[:, 2])
    order = np.argsort(-lin, kind="stable")                 # ascending column = descending offset
    offsets, coefs, lin = offsets[order], coefs[order], lin[order]
    ns = len(lin)
    idx1 = np.arange(m, dtype=np.int64)
    ok = [((idx1[None, :] - offsets[:, a:a + 1]) >= 0) & ((idx1[None, :] - offsets[:, a:a + 1]) < m) for a in range(3)]
    nrows = (k1 - k0) * m * m
    rp = np.zeros(nrows + 1, np.int64)
    parts_c, parts_v = [], []
    planes = max(1, int(4_000_000 // (m * m)))
    pos = 0
    for ka in range(k0, k1, planes):
        kb = min(k1, ka + planes)
        kk = np.arange(ka, kb, dtype=np.int64)
        rows = (idx1[None, None, :] + m * (idx1[None, :, None] + m * kk[:, None, None])).reshape(-1)
        valid = (ok[0][:, None, None, :] & ok[1][:, None, :, None] & ok[2][:, kk][:, :, None, None])
        valid = valid.reshape(ns, -1).T                     # [row, s], s in ascending column order
        cols = rows[:, None] - lin[None, :]
        cnt = valid.sum(axis=1)
        r0 = (ka - k0) * m * m
        rp[r0 + 1:r0 + 1 + len(rows)] = pos + np.cumsum(cnt)
        pos += int(cnt.sum())
        parts_c.append(cols[valid].astype(np.int32))
        parts_v.append(np.broadcast_to(coefs[None, :], valid.shape)[valid])
    assert pos < 2**31, "int32 index overflow"
    return rp.astype(np.int32), np.concatenate(parts_c), np.concatenate(parts_v)


def pencil_rows(name: str, m: int, k0: int, k1: int):
    """((rp, ci, va) of A, the same of B or None) for the planes [k0, k1) of one of this module's lattice pencils
    ("laplace3d_7pt", "q1_27pt", "p1_fem_kuhn"): the slab a rank owns, generated without the whole matrix."""
    if name == "laplace3d_7pt":
        offs = [(0, 0, 0), (1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]
        return stencil_rows(m, offs, [6.0] + [-1.0] * 6, k0, k1), None
    if name == "q1_27pt":
        h = 1.0 / (m + 1)
        K1 = (-1.0 / h, 2.0 / h, -1.0 / h)
        M1 = (h / 6.0, 4.0 * h / 6.0, h / 6.0)
        offs, ca, cb = [], [], []
        for dx, dy, dz in itertools.product((-1, 0, 1), repeat=3):
            offs.append((dx, dy, dz))
            ca.append(sum(fx[dx + 1] * fy[dy + 1] * fz[dz + 1] for fx, fy, fz in [(K1, M1, M1), (M1, K1, M1), (M1, M1, K1)]))
            cb.append(M1[dx + 1] * M1[dy + 1] * M1[dz + 1])
        return stencil_rows(m, offs, ca, k0, k1), stencil_rows(m, offs, cb, k0, k1)
    if name == "p1_fem_kuhn":
        ca, cb = _p1_kuhn_coefs(m)
        return stencil_rows(m, _KUHN_OFFS, ca, k0, k1), stencil_rows(m, _KUHN_OFFS, cb, k0, k1)
    raise KeyError(name)


def laplace3d_7pt(m: int) -> Pencil:
    """Config 2 (SURVEY §8d): 7-point Laplacian on an m**3 grid, values 6/-1, B = None.
    Eigenvalues 6 - 2cos(i t) - 2cos(j t) - 2cos(k t), t = pi/(m+1)."""
    offs = [(0, 0, 0), (1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]
    coefs = [6.0] + [-1.0] * 6
    return Pencil("laplace3d_7pt", stencil_to_ccs(m, offs, coefs), None, {"m": m, "n": m**3})


def laplace3d_7pt_eigenvalues(m: int, k: int) -> np.ndarray:
    t = np.pi / (m + 1)
    c = 2.0 - 2.0 * np.cos(np.arange(1, m + 1) * t)
    top = min(m, max(8, int(round(k ** (1 / 3))) * 3 + 4))
    vals = (c[:top, None, None] + c[None, :top, None] + c[None, None, :top]).reshape(-1)
    return np.sort(vals)[:k]


def diffusion7_var(m: int, coef: str = "lognormal", seed: int = 0, sigma: float = 2.0, mass: bool = False) -> Pencil:
    """-div(kappa grad u) on an m**3 cell-centred grid, 7-point, harmonic averages of kappa on the faces, Dirichlet
    faces (2 kappa each), grid spacing 1: heterogeneous coefficients, whose varying diagonal is what a Jacobi
    preconditioner of the inner solve acts on.  coef: "const" (kappa = 1), "jump" (2x2x2 cell blocks, kappa 1 or 1e3
    at random) or "lognormal" (kappa = exp(N(0, sigma^2)) per cell).  mass: B = a random positive diagonal,
    uniform in [0.5, 2]; else B = None.  Lexicographic order i + m (j + m k), like the lattice generators."""
    import scipy.sparse as sp

    n = m ** 3
    rng = np.random.default_rng(seed)
    if coef == "const":
        kap = np.ones(n)
    elif coef == "jump":
        h = m // 2 + 1
        blk = rng.integers(0, 2, size=(h, h, h)).repeat(2, 0).repeat(2, 1).repeat(2, 2)[:m, :m, :m]
        kap = np.where(blk.ravel() == 1, 1e3, 1.0)
    elif coef == "lognormal":
        kap = np.exp(rng.normal(0.0, sigma, n))
    else:
        raise ValueError(f"diffusion7_var: coef {coef!r}")
    K = kap.reshape(m, m, m)                      # K[k, j, i]: cell i + m (j + m k)
    idx = np.arange(n).reshape(m, m, m)
    diag = np.zeros(n)
    rows, cols, vals = [], [], []
    for ax in range(3):
        lo = [slice(None)] * 3; hi = [slice(None)] * 3
        lo[ax] = slice(0, m - 1); hi[ax] = slice(1, m)
        ka, kb = K[tuple(lo)], K[tuple(hi)]
        t = (2.0 * ka * kb / (ka + kb)).ravel()
        ia, ib = idx[tuple(lo)].ravel(), idx[tuple(hi)].ravel()
        rows += [ia, ib]; cols += [ib, ia]; vals += [-t, -t]
        np.add.at(diag, ia, t); np.add.at(diag, ib, t)
        f0 = [slice(None)] * 3; f1 = [slice(None)] * 3
        f0[ax] = 0; f1[ax] = m - 1
        diag[idx[tuple(f0)].ravel()] += 2.0 * K[tuple(f0)].ravel()
        diag[idx[tuple(f1)].ravel()] += 2.0 * K[tuple(f1)].ravel()
    rows.append(np.arange(n)); cols.append(np.arange(n)); vals.append(diag)
    A = sp.csc_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n))
    A.sum_duplicates(); A.sort_indices()

    def ccs(M):
        return CCS(n, n, M.indptr.astype(np.int32), M.indices.astype(np.int32), M.data.astype(np.float64))

    B = None
    if mass:
        B = ccs(sp.diags(np.random.default_rng(seed + 1).uniform(0.5, 2.0, n)).tocsc())
    return Pencil("diffusion7_var", ccs(A), B, {"m": m, "n": n, "coef": coef, "seed": seed, "sigma": sigma, "mass": mass})


def _tensor27(m: int, ax, ay, az, scale_terms):
    """sum over terms of (X (x) Y (x) Z) with 1-D tridiagonal factors given as (lo, di, up)."""
    offs, coefs = [], []
    for dx, dy, dz in itertools.product((-1, 0, 1), repeat=3):
        c = 0.0
        for fx, fy, fz in scale_terms:
            c += fx[dx + 1] * fy[dy + 1] * fz[dz + 1]
        offs.append((dx, dy, dz))
        coefs.append(c)
    return stencil_to_ccs(m, offs, coefs)


def q1_27pt(m: int, with_mass: bool = True) -> Pencil:
    """Config 4 (SURVEY §8d): 27-point tensor-product trilinear (Q1) stiffness (and mass)
    on an m**3 Dirichlet lattice, h = 1/(m+1)."""
    h = 1.0 / (m + 1)
    K1 = (-1.0 / h, 2.0 / h, -1.0 / h)
    M1 = (h / 6.0, 4.0 * h / 6.0, h / 6.0)
    A = _tensor27(m, None, None, None, [(K1, M1, M1), (M1, K1, M1), (M1, M1, K1)])
    B = _tensor27(m, None, None, None, [(M1, M1, M1)]) if with_mass else None
    return Pencil("q1_27pt", A, B, {"m": m, "n": m**3, "h": h})


# ------------------------------------------------------------------------ P1 / Kuhn
_KUHN_PERMS = list(itertools.permutations(range(3)))


def p1_kuhn_assemble(m: int):
    """Element-by-element P1 stiffness and mass on the Kuhn triangulation of the
    (m+2)**3 vertex lattice of [0,1]**3 (h = 1/(m+1)); Dirichlet rows/columns removed,
    leaving m**3 unknowns.  Dense-ish reference assembly for SMALL m (tests and
    stencil extraction); returns scipy CSC matrices with the union pattern kept."""
    import scipy.sparse as sp

    nv = m + 2
    h = 1.0 / (m + 1)

    def vid(i, j, k):
        return i + nv * (j + nv * k)

    rows, cols, va, vb = [], [], [], []
    e = np.eye(3, dtype=np.int64)
    for ci, cj, ck in itertools.product(range(nv - 1), repeat=3):
        base = np.array((ci, cj, ck), dtype=np.int64)
        for perm in _KUHN_PERMS:
            verts = [base.copy()]
            for a in perm:
                verts.append(verts[-1] + e[a])
            X = np.array(verts, dtype=np.float64) * h
            T = np.hstack([np.ones((4, 1)), X])
            vol = abs(np.linalg.det(T)) / 6.0
            grads = np.linalg.inv(T)[1:, :]  # 3 x 4
            Ke = vol * grads.T @ grads
            Me = vol / 20.0 * (np.ones((4, 4)) + np.eye(4))
            ids = [vid(*v) for v in verts]
            for a in range(4):
                for b in range(4):
                    rows.append(ids[a]); cols.append(ids[b])
                    va.append(Ke[a, b]); vb.append(Me[a, b])
    ntot = nv**3
    A = sp.coo_matrix((va, (rows, cols)), shape=(ntot, ntot)).tocsc()
    B = sp.coo_matrix((vb, (rows, cols)), shape=(ntot, ntot)).tocsc()
    g = np.arange(nv)
    inner = (g >= 1) & (g <= m)
    mask = (inner[None, None, :] & inner[None, :, None] & inner[:, None, None]).reshape(-1)
    keep = np.nonzero(mask)[0]
    return A[keep][:, keep].tocsc(), B[keep][:, keep].tocsc(), h


# 15-point Kuhn pattern: self, 6 axis edges, 6 face diagonals (+,+)/(-,-), 2 body diagonals.
_KUHN_OFFS = [(0, 0, 0),
              (1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1),
              (1, 1, 0), (-1, -1, 0), (1, 0, 1), (-1, 0, -1), (0, 1, 1), (0, -1, -1),
              (1, 1, 1), (-1, -1, -1)]


def _p1_kuhn_coefs(m: int):
    """stencil coefficients of the P1 stiffness / mass operators at mesh width 1/(m+1), read off a genuine
    element-by-element assembly at m = 3 (centre row) and scaled: stiffness ~ h, mass ~ h**3"""
    A3, B3, h3 = p1_kuhn_assemble(3)
    centre = 1 + 3 * (1 + 3 * 1)
    h = 1.0 / (m + 1)
    ca, cb = [], []
    for (dx, dy, dz) in _KUHN_OFFS:
        r = centre + dx + 3 * (dy + 3 * dz)
        ca.append(float(A3[r, centre]) * (h / h3))
        cb.append(float(B3[r, centre]) * (h / h3) ** 3)
    # diagonal-edge stiffness entries are exact zeros analytically; snap assembly noise
    ca = [0.0 if abs(c) < 1e-12 * abs(ca[0]) else c for c in ca]
    return ca, cb


def p1_fem_kuhn(m: int) -> Pencil:
    """Config 3 (SURVEY §8d): P1 stiffness / consistent mass pencil on the Kuhn
    triangulation, n = m**3, 15 nnz/row, A and B with identical pattern.  The stencil
    coefficients are read off a genuine assembly at m=3 (centre row) and scaled:
    stiffness ~ h, mass ~ h**3."""
    ca, cb = _p1_kuhn_coefs(m)
    h = 1.0 / (m + 1)
    A = stencil_to_ccs(m, _KUHN_OFFS, ca)
    B = stencil_to_ccs(m, _KUHN_OFFS, cb)
    return Pencil("p1_fem_kuhn", A, B, {"m": m, "n": m**3, "h": h})


# ------------------------------------------------------------------ config 1: the reference's mesh file
_CUBE4_FIXTURE = Path(__file__).resolve().parents[1] / "tests" / "golden" / "cube4_mesh.json"


def read_albert_mesh(path):
    """ALBERT macro-triangulation file (the format of reference data/cube4.dat:1-6,133,519): returns
    (vertices float64 [nv, 3], elements int64 [ne, 4])."""
    import re
    txt = Path(path).read_text()
    nv = int(re.search(r"number of vertices:\s*(\d+)", txt).group(1))
    ne = int(re.search(r"number of elements:\s*(\d+)", txt).group(1))

    def section(name, nxt):
        a = txt.index(name) + len(name)
        return txt[a:txt.index(nxt, a)]

    V = np.array(section("vertex coordinates:", "element vertices:").split(), float).reshape(nv, 3)
    T = np.array(section("element vertices:", "element boundaries:").split(), np.int64).reshape(ne, 4)
    return V, T


def cube4_mesh():
    """The mesh of reference data/cube4.dat from the committed fixture (tests/golden/make_cube4_fixture.py)."""
    import json
    d = json.loads(_CUBE4_FIXTURE.read_text())
    return np.array(d["vertices_quarter_units"], float) * d["unit"], np.array(d["elements"], np.int64)


def refine_uniform(V: np.ndarray, T: np.ndarray):
    """One regular (red) refinement of a tetrahedral mesh: every edge gets its midpoint, every tetrahedron becomes
    4 corner tetrahedra + 4 from the inner octahedron (split along the midpoint pair (01|23) -- any fixed choice gives
    a conforming mesh).  Vertices keep their numbers, midpoints follow in order of first appearance."""
    edges = {}
    Vn = [tuple(v) for v in V]

    def mid(a, b):
        key = (a, b) if a < b else (b, a)
        if key not in edges:
            edges[key] = len(Vn)
            Vn.append(tuple(0.5 * (np.asarray(Vn[a]) + np.asarray(Vn[b]))))
        return edges[key]

    Tn = []
    for (a, b, c, d) in T.tolist():
        ab, ac, ad, bc, bd, cd = mid(a, b), mid(a, c), mid(a, d), mid(b, c), mid(b, d), mid(c, d)
        Tn += [(a, ab, ac, ad), (ab, b, bc, bd), (ac, bc, c, cd), (ad, bd, cd, d),
               (ab, cd, ac, ad), (ab, cd, ad, bd), (ab, cd, bd, bc), (ab, cd, bc, ac)]
    return np.array(Vn, float), np.array(Tn, np.int64)


def p1_assemble_mesh(V: np.ndarray, T: np.ndarray):
    """P1 stiffness and consistent mass matrices on a tetrahedral mesh (all vertices), vectorised over elements;
    scipy CSC with the union pattern kept."""
    import scipy.sparse as sp
    X = V[T]                                                   # [ne, 4, 3]
    M = np.concatenate([np.ones((len(T), 4, 1)), X], axis=2)   # [ne, 4, 4]
    vol = np.abs(np.linalg.det(M)) / 6.0
    grads = np.linalg.inv(M)[:, 1:, :]                         # [ne, 3, 4]
    Ke = vol[:, None, None] * np.einsum("eda,edb->eab", grads, grads)
    Me = vol[:, None, None] / 20.0 * (np.ones((4, 4)) + np.eye(4))[None]
    r = np.repeat(T, 4, axis=1).reshape(-1)
    c = np.tile(T, (1, 4)).reshape(-1)
    nv = len(V)
    A = sp.coo_matrix((Ke.reshape(-1), (r, c)), shape=(nv, nv)).tocsc()
    B = sp.coo_matrix((Me.reshape(-1), (r, c)), shape=(nv, nv)).tocsc()
    return A, B


def cube4_p1(refine: int = 2, order: str = "lattice") -> Pencil:
    """Config 1 restated (SURVEY.md 8d): P1 stiffness / mass pencil on the mesh of reference data/cube4.dat after
    `refine` regular refinements, homogeneous Dirichlet vertices (on the faces of [0,1]^3) removed.  refine = 2:
    17^3 vertices, 15^3 = 3375 unknowns.  order = "lattice": unknowns in natural lattice order x + m (y + m z) (a
    27-neighbour pattern with element-dependent coefficients: the device takes it for a lattice operator);
    order = "mesh": in the mesh's own hierarchical vertex order (an unstructured matrix: the CSR kernels)."""
    V, T = cube4_mesh()
    for _ in range(refine):
        V, T = refine_uniform(V, T)
    A, B = p1_assemble_mesh(V, T)
    inner = np.all((V > 1e-12) & (V < 1 - 1e-12), axis=1)
    keep = np.nonzero(inner)[0]
    if order == "lattice":
        h = 0.25 / 2 ** refine
        q = np.rint(V[keep] / h).astype(np.int64) - 1
        m = int(round(1.0 / h)) - 1
        keep = keep[np.argsort(q[:, 0] + m * (q[:, 1] + m * q[:, 2]), kind="stable")]

    def ccs(M):
        M = M[keep][:, keep].tocsc()
        M.sort_indices()
        return CCS(M.shape[0], M.shape[1], M.indptr.astype(np.int32), M.indices.astype(np.int32), M.data.astype(np.float64))

    return Pencil("cube4_p1", ccs(A), ccs(B), {"refine": refine, "order": order, "n": len(keep)})


def cube4_p1_mesh(refine: int = 2) -> Pencil:
    """cube4_p1 in the mesh's own hierarchical vertex order: an unstructured matrix (no diagonal image; the CSR kernels)."""
    return cube4_p1(refine, "mesh")


def ccs_to_dense(M: CCS) -> np.ndarray:
    out = np.zeros((M.nrows, M.ncols))
    for j in range(M.ncols):
        sl = slice(M.j_col[j], M.j_col[j + 1])
        out[M.i_row[sl], j] += M.data[sl]
    return out
