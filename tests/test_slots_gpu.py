"""GPU parity of the OPS slot kernels, through the C ABI, against the reference
(oracle/_ref when it travelled) and the plain-C oracle.  The call sequences follow the
reference's own drivers TestMultiVec (reference test/test_multi_vec.c:19-228) turned into
assertions.  Bit-exact where the reference's arithmetic order is reproducible (SpMM, copies,
RNG, CCS round trip); 1e-13 relative for BLAS-ordered reductions (tolerance stated per test)."""
import ctypes as C

import numpy as np
import pytest

from gcge_b200 import problems as P
from oracle import gcg_numpy as G

pytestmark = pytest.mark.gpu
dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))


def rel(a, b):
    return np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)


def oracle_spmm(M, x):
    n, k = x.shape
    y = np.zeros((n, k), order="F")
    xx = np.asfortranarray(x)
    G.clib().oracle_ccs_spmm(n, ip(M.j_col), ip(M.i_row), dp(M.data), dp(xx), dp(y), k)
    return y


@pytest.fixture(scope="module")
def pencil():
    return P.p1_fem_kuhn(9)      # n = 729, 15 nnz/row, A and B


def test_ccs_round_trip_bitexact(b200):
    rng = np.random.default_rng(0)
    for pen in (P.laplace1d_pencil(57), P.p1_fem_kuhn(5)):
        for M in (pen.A, pen.B):
            d = b200.Mat(M)
            j, i, v = d.to_ccs()
            assert np.array_equal(j, M.j_col) and np.array_equal(i, M.i_row) and np.array_equal(v, M.data)
    # non-symmetric, unsorted rows inside a column, an empty column, an empty row
    j_col = np.array([0, 3, 3, 5, 6], np.int32)
    i_row = np.array([2, 0, 3, 1, 0, 2], np.int32)
    data = rng.standard_normal(6)
    M = P.CCS(4, 4, j_col, i_row, data)
    d = b200.Mat(M)
    j, i, v = d.to_ccs()
    assert np.array_equal(j, j_col) and np.array_equal(i, i_row) and np.array_equal(v, data)
    x = np.asfortranarray(rng.standard_normal((4, 3)))
    X = b200.MultiVec.from_numpy(x); Y = b200.MultiVec(4, 3)
    from gcge_b200 import api
    api.mat_dot_multivec(d, X, Y, (0, 0), (3, 3))
    assert np.array_equal(Y.numpy(), oracle_spmm(M, x))
    api.mat_dot_multivec(d, X, Y, (0, 0), (3, 3), trans=True)
    assert np.allclose(Y.numpy(), P.ccs_to_dense(M).T @ x, rtol=1e-14, atol=1e-14)


@pytest.mark.parametrize("name", ["p1", "p1_mass", "7pt", "27pt", "1d", "unsym_random", "long_row", "rect"])
def test_device_matrix_build_matches_host_build(b200, name):
    """b200_matbuild.cu (CCS -> CSR slab, symmetry flag, diagonal image, all on the device) against
    the host construction (b200_partition_build + dia_build): the CSR image bit for bit, the CCS
    round trip, and the SpMM result (which goes through the diagonal image where there is one)."""
    from gcge_b200 import api
    L = api.lib()
    if name == "p1":
        M = P.p1_fem_kuhn(11).A
    elif name == "p1_mass":
        M = P.p1_fem_kuhn(8).B
    elif name == "7pt":
        M = P.laplace3d_7pt(9).A
    elif name == "27pt":
        M = P.q1_27pt(7).A
    elif name == "1d":
        M = P.laplace1d_pencil(300).B
    elif name == "unsym_random":
        M = _random_unsymmetric(n=257)
    elif name == "long_row":          # one dense row: longer than the device sort handles -> host path
        import scipy.sparse as sp
        m = sp.identity(200, format="lil"); m[7, :] = 1.5; m[:, 7] = 2.5
        m = m.tocsc(); m.sort_indices()
        M = P.CCS(200, 200, m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data.astype(np.float64))
    else:                             # rectangular 30 x 20
        import scipy.sparse as sp
        m = sp.random(30, 20, density=0.2, random_state=np.random.default_rng(3), format="csc"); m.sort_indices()
        M = P.CCS(30, 20, m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data.astype(np.float64))
    rng = np.random.default_rng(1)
    x = np.asfortranarray(rng.standard_normal((M.ncols, 8)))
    res, launches = [], []
    for host in (0, 1):
        old = C.c_int(0)
        assert L.b200_option_get(b"host_build", C.byref(old)) == 0
        assert L.b200_option_set(b"host_build", host) == 0
        try:
            l0 = L.b200_kernel_launches()
            A = b200.Mat(M)
            launches.append(L.b200_kernel_launches() - l0)
        finally:
            L.b200_option_set(b"host_build", old.value)
        nnz = int(M.j_col[-1])
        rp = np.zeros(M.nrows + 1, np.int32); ci = np.zeros(max(nnz, 1), np.int32); va = np.zeros(max(nnz, 1))
        api._chk(api.lib().b200_mat_local_csr(A.h, ip(rp), ip(ci), dp(va)))
        X = b200.MultiVec.from_numpy(x); Y = b200.MultiVec(M.nrows, 8)
        api.mat_dot_multivec(A, X, Y, (0, 0), (8, 8))
        res.append((rp, ci[:nnz], va[:nnz], A.to_ccs(), Y.numpy()))
    d, h = res
    # the device build launches its mb_* kernels (even where it hands over to the host build, as for the long row);
    # the host build launches none of them
    print(f"\nmatrix build {name}: kernel launches device {launches[0]}, host {launches[1]}")
    assert launches[0] > launches[1], launches
    assert np.array_equal(d[0], h[0]) and np.array_equal(d[1], h[1]) and np.array_equal(d[2], h[2])
    for a, b in zip(d[3], h[3]):
        assert np.array_equal(a, b)
    assert np.array_equal(d[4], h[4])
    if M.nrows == M.ncols:
        assert np.array_equal(d[4], oracle_spmm(M, x))


def test_upload_download_and_views(b200):
    rng = np.random.default_rng(1)
    for n, k in ((1, 1), (33, 2), (1000, 7), (257, 40)):
        a = np.asfortranarray(rng.standard_normal((n, k)))
        mv = b200.MultiVec.from_numpy(a)
        assert np.array_equal(mv.numpy(), a)
        assert np.array_equal(mv.numpy(1 if k > 1 else 0, k), a[:, (1 if k > 1 else 0):])
    empty = b200.MultiVec(0, 3)
    assert empty.numpy().shape == (0, 3)


def test_set_random_is_glibc_stream(b200, refmod):
    n, k = 501, 6
    mv = b200.MultiVec(n, k)
    b200.libc_srand(0)
    mv.set_random(1, 5)
    got = mv.numpy()
    want = np.zeros((n, k), order="F")
    G.srand(0); G.fill_random(want, 1, 5)
    assert np.array_equal(got, want)
    assert got[0, 1] == 1804289383 / 2147483648.0
    if refmod is not None:
        r = np.zeros((n, k), order="F")
        refmod.srand(0); refmod.multivec_set_random(r, 1, 5)
        assert np.array_equal(got, r)


@pytest.mark.parametrize("n,k,seed", [(1, 3, 0), (31, 1, 5), (1984, 2, 0), (70001, 9, 0), (300007, 5, 42)])
def test_set_random_device_jump_ahead(b200, n, k, seed):
    """The device generator (jump-ahead of glibc's lagged-Fibonacci recurrence, one chunk of 1984
    stream positions per thread, 128 chunks per CTA) must reproduce the rand() stream bit for bit
    across chunk, CTA and column boundaries, and must leave the PROCESS generator advanced by
    n*k calls, so a later rand() -- e.g. the next MultiVecSetRandomValue -- continues the stream."""
    import ctypes as C
    libc = C.CDLL("libc.so.6")
    mv = b200.MultiVec(n, k + 2)
    b200.libc_srand(seed)
    mv.set_random(1, 1 + k)
    after = [libc.rand() for _ in range(5)]
    want = np.zeros((n, k + 2), order="F")
    G.srand(seed); G.fill_random(want, 1, 1 + k)
    got = mv.numpy()
    assert np.array_equal(got, want)
    assert np.all(got[:, 0] == 0) and np.all(got[:, k + 1] == 0)
    b200.libc_srand(seed)
    skip = np.zeros((n, k), order="F")
    G.fill_random(skip, 0, k)                 # n*k real rand() calls on the host
    assert after == [libc.rand() for _ in range(5)]


@pytest.mark.parametrize("k", [1, 2, 3, 8, 10, 16, 31, 40, 70])
def test_spmm_bitexact(b200, refmod, pencil, k):
    """MatDotMultiVec (reference app/app_ccs.c:50-139): identical bits, any block width."""
    from gcge_b200 import api
    rng = np.random.default_rng(k)
    n = pencil.A.ncols
    x = np.asfortranarray(rng.standard_normal((n, k + 3)))
    A = b200.Mat(pencil.A)
    X = b200.MultiVec.from_numpy(x); Y = b200.MultiVec(n, k + 5)
    api.mat_dot_multivec(A, X, Y, (2, 4), (2 + k, 4 + k))
    got = Y.numpy()
    want = oracle_spmm(pencil.A, x[:, 2:2 + k])
    assert np.array_equal(got[:, 4:4 + k], want)
    assert not got[:, :4].any() and not got[:, 4 + k:].any()      # neighbours untouched
    if refmod is not None:
        yr = np.zeros((n, k + 5), order="F")
        refmod.mat_dot_multivec(pencil.A, x, yr, (2, 4), (2 + k, 4 + k))
        assert np.array_equal(got, yr)
    # NULL matrix == copy (reference app/app_ccs.c:134-137)
    api.mat_dot_multivec(None, X, Y, (0, 0), (k, k))
    assert np.array_equal(Y.numpy()[:, :k], x[:, :k])


def _random_unsymmetric(n=413, density=0.03, seed=5):
    import scipy.sparse as sp
    m = sp.random(n, n, density=density, random_state=np.random.default_rng(seed), format="csc") + 3.0 * sp.identity(n, format="csc")
    m = m.tocsc(); m.sort_indices()
    return P.CCS(n, n, m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data.astype(np.float64))


@pytest.mark.parametrize("name", ["7pt", "27pt", "p1_mass", "1d", "unsym_random", "ragged_banded"])
@pytest.mark.parametrize("k", [5, 6, 16, 22, 40, 64, 80, 130])
def test_spmm_bitexact_both_storage_paths(b200, name, k):
    """The diagonal-image kernel (lattice operators: 7/15/27 diagonals, Dirichlet rows with missing
    neighbours) and the CSR kernels (irregular matrices) must both reproduce the reference's CCS
    scatter bit for bit, at aligned and unaligned column offsets."""
    from gcge_b200 import api
    if name == "7pt":
        M = P.laplace3d_7pt(11).A
    elif name == "27pt":
        M = P.q1_27pt(9).A
    elif name == "p1_mass":
        M = P.p1_fem_kuhn(10).B
    elif name == "1d":
        M = P.laplace1d_pencil(1001).A
    elif name == "unsym_random":
        M = _random_unsymmetric()
    else:   # banded, but every third row lacks some of its diagonals and a few rows are empty
        import scipy.sparse as sp
        n = 700
        rng = np.random.default_rng(2)
        d = {o: rng.standard_normal(n - abs(o)) for o in (-30, -29, -1, 0, 1, 2, 29, 31)}
        m = sp.diags(list(d.values()), list(d.keys()), shape=(n, n), format="lil")
        m[3::3, :] = m[3::3, :].multiply(sp.random(1, n, density=0.5, random_state=rng, format="csr") != 0)
        m[10, :] = 0; m[500, :] = 0
        m = m.tocsc(); m.eliminate_zeros(); m.sort_indices()
        M = P.CCS(n, n, m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data.astype(np.float64))
    n = M.ncols
    x = np.asfortranarray(np.random.default_rng(k).standard_normal((n, k + 3)))
    A = b200.Mat(M)
    X = b200.MultiVec.from_numpy(x)
    for xo, yo in ((0, 0), (1, 2), (2, 1), (3, 4)):
        if xo + k > k + 3:
            continue
        Y = b200.MultiVec(n, k + 5)
        api.mat_dot_multivec(A, X, Y, (xo, yo), (xo + k, yo + k))
        got = Y.numpy()
        want = oracle_spmm(M, np.asfortranarray(x[:, xo:xo + k]))
        assert np.array_equal(got[:, yo:yo + k], want), (name, k, xo, yo)
        assert not got[:, :yo].any() and not got[:, yo + k:].any()


def _lattice_matrix(mx, my, mz, kind, seed=0, periodic=False):
    """Variable-coefficient operator on an mx x my x mz lattice (row = i + mx (j + my k)): the pattern of a
    7-point, 27-point or P1-Kuhn (15-point) stencil, every entry its own random value -- unlike the constant
    stencils of gcge_b200.problems this catches a value that lands on the wrong row or diagonal."""
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    if kind == "7pt":
        offs = [(0, 0, 0), (1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]
    elif kind == "27pt":
        offs = [(a, b, c) for a in (-1, 0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1)]
    else:
        offs = P._KUHN_OFFS
    i, j, k = np.meshgrid(np.arange(mx), np.arange(my), np.arange(mz), indexing="ij")
    i, j, k = (a.transpose(2, 1, 0).reshape(-1) for a in (i, j, k))          # row-major in (k, j, i)
    row = i + mx * (j + my * k)
    rows, cols = [], []
    for (di, dj, dk) in offs:
        ii, jj2, kk = i + di, j + dj, k + dk
        if periodic:
            ok = np.ones(len(row), bool); ii %= mx; jj2 %= my; kk %= mz
        else:
            ok = (ii >= 0) & (ii < mx) & (jj2 >= 0) & (jj2 < my) & (kk >= 0) & (kk < mz)
        rows.append(row[ok]); cols.append((ii + mx * (jj2 + my * kk))[ok])
    rows = np.concatenate(rows); cols = np.concatenate(cols)
    m = sp.csc_matrix((rng.standard_normal(len(rows)), (rows, cols)), shape=(mx * my * mz,) * 2)
    m.sum_duplicates(); m.sort_indices()
    return P.CCS(m.shape[0], m.shape[1], m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data.astype(np.float64))


@pytest.mark.parametrize("kind,dims", [("7pt", (13, 7, 5)), ("27pt", (12, 9, 4)), ("p1", (21, 6, 7)), ("p1", (40, 40, 6)),
                                       ("27pt", (8, 8, 3)), ("7pt", (50, 11, 9))])
@pytest.mark.parametrize("k", [8, 10, 20, 40, 64])
def test_spmm_lattice_kernel_bitexact(b200, kind, dims, k, monkeypatch):
    """The plane-marching lattice kernel (b200_spmm_lat.cu) on non-cubic lattices with variable coefficients,
    partial tiles in i and j, short k extents: recognised as a lattice, identical bits to the reference's CCS
    scatter (plain-C oracle), at aligned and unaligned column offsets of a wider block."""
    from gcge_b200 import api
    M = _lattice_matrix(*dims, kind, seed=k)
    A = b200.Mat(M)
    st = A.storage()
    assert st["lat_s1"] == dims[0] and st["lat_s2"] == dims[0] * dims[1], st
    n = M.ncols
    x = np.asfortranarray(np.random.default_rng(k + 1).standard_normal((n, k + 4)))
    X = b200.MultiVec.from_numpy(x)
    for xo, yo in ((0, 0), (2, 4), (1, 2)):
        Y = b200.MultiVec(n, k + 6)
        api.mat_dot_multivec(A, X, Y, (xo, yo), (xo + k, yo + k))
        got = Y.numpy()
        want = oracle_spmm(M, np.asfortranarray(x[:, xo:xo + k]))
        assert np.array_equal(got[:, yo:yo + k], want), (kind, dims, k, xo, yo)
        assert not got[:, :yo].any() and not got[:, yo + k:].any()


@pytest.mark.parametrize("name,m", [("p1_fem_kuhn", 9), ("q1_27pt", 8), ("laplace3d_7pt", 10)])
def test_matrix_from_local_rows_matches_whole_ccs(b200, name, m):
    """b200_mat_create_from_local_rows (a rank hands over only its rows; here one rank = all rows) builds the same
    device matrix as b200_mat_create_from_ccs: same storage decisions, bit-identical SpMM, bit-identical solve."""
    from gcge_b200 import api
    pen = getattr(P, name)(m)
    rowsA, rowsB = P.pencil_rows(name, m, 0, m)
    n = pen.A.ncols
    A1 = b200.Mat(pen.A); A2 = api.Mat.from_local_rows(n, 0, *rowsA)
    assert A1.storage() == A2.storage() and A2.storage()["lat_s1"] == m
    x = np.asfortranarray(np.random.default_rng(1).standard_normal((n, 20)))
    X = b200.MultiVec.from_numpy(x); Y1 = b200.MultiVec(n, 20); Y2 = b200.MultiVec(n, 20)
    api.mat_dot_multivec(A1, X, Y1, (0, 0), (20, 20)); api.mat_dot_multivec(A2, X, Y2, (0, 0), (20, 20))
    assert np.array_equal(Y1.numpy(), Y2.numpy()) and np.array_equal(Y1.numpy(), oracle_spmm(pen.A, x))
    B1 = None if pen.B is None else b200.Mat(pen.B)
    B2 = None if rowsB is None else api.Mat.from_local_rows(n, 0, *rowsB)
    o1 = b200.gcg_solve(A1, B1, nev=6); o2 = b200.gcg_solve(A2, B2, nev=6)
    assert o1["num_iter"] == o2["num_iter"] and np.array_equal(o1["eval"], o2["eval"])


def test_matrix_from_local_rows_rejects_malformed_rows(b200):
    """The arrays are checked on the device after the upload: a row whose columns do not ascend, a column outside the
    matrix and decreasing row pointers are errors, not silently different matrices.  An irregular (non-banded) matrix
    handed over by rows keeps its CSR storage and multiplies exactly."""
    from gcge_b200 import api
    import scipy.sparse as sp
    rng = np.random.default_rng(5)
    n = 300
    S = sp.random(n, n, density=0.03, random_state=7, format="csr"); S = (S + S.T + sp.eye(n)).tocsr(); S.sort_indices()
    rp = S.indptr.astype(np.int32); ci = S.indices.astype(np.int32); va = S.data.astype(np.float64)
    A = api.Mat.from_local_rows(n, 0, rp, ci, va)
    assert A.storage()["dia_nd"] == 0
    x = np.asfortranarray(rng.standard_normal((n, 7)))
    X = b200.MultiVec.from_numpy(x); Y = b200.MultiVec(n, 7)
    api.mat_dot_multivec(A, X, Y, (0, 0), (7, 7))
    Sc = S.tocsc(); Sc.sort_indices()
    M = P.CCS(n, n, Sc.indptr.astype(np.int32), Sc.indices.astype(np.int32), Sc.data.astype(np.float64))
    assert np.array_equal(Y.numpy(), oracle_spmm(M, x))
    r = int(np.argmax(np.diff(rp) >= 2))
    bad = ci.copy(); bad[rp[r]], bad[rp[r] + 1] = ci[rp[r] + 1], ci[rp[r]]
    with pytest.raises(RuntimeError, match="ascending"):
        api.Mat.from_local_rows(n, 0, rp, bad, va)
    bad = ci.copy(); bad[rp[r + 1] - 1] = n
    with pytest.raises(RuntimeError, match="out of range"):
        api.Mat.from_local_rows(n, 0, rp, bad, va)
    badrp = rp.copy(); badrp[r + 1] = rp[r] - 1 if rp[r] > 0 else rp[r + 2] + 1
    with pytest.raises(RuntimeError, match="monotone"):
        api.Mat.from_local_rows(n, 0, badrp, ci, va)


@pytest.mark.parametrize("name,m", [("p1_fem_kuhn", 11), ("q1_27pt", 9), ("laplace3d_7pt", 12)])
def test_spmm_constant_stencil_path(b200, name, m):
    """Constant stencils (every row the same coefficients, entries exactly where the neighbour is inside the lattice:
    all of BASELINE's lattice pencils) are recognised and multiplied WITHOUT streaming matrix values; the result is
    bit-identical to the general lattice kernel (option lat_no_const) and to the reference's CCS scatter.  One
    perturbed entry makes the matrix non-constant: the general kernel takes over, still exact."""
    import ctypes as C
    from gcge_b200 import api
    L = b200.lib()
    pen = getattr(P, name)(m)
    n = pen.A.ncols
    for M in (pen.A, pen.B):
        if M is None:
            continue
        A = b200.Mat(M)
        assert A.storage()["lat_const"] == 1 and A.storage()["lat_s1"] == m
        for k in (10, 40):
            x = np.asfortranarray(np.random.default_rng(k).standard_normal((n, k)))
            X = b200.MultiVec.from_numpy(x); Y1 = b200.MultiVec(n, k); Y2 = b200.MultiVec(n, k)
            api.mat_dot_multivec(A, X, Y1, (0, 0), (k, k))
            try:
                L.b200_option_set(b"lat_no_const", 1)
                api.mat_dot_multivec(A, X, Y2, (0, 0), (k, k))
            finally:
                L.b200_option_set(b"lat_no_const", 0)
            want = oracle_spmm(M, x)
            assert np.array_equal(Y1.numpy(), want) and np.array_equal(Y2.numpy(), want)
    data = pen.A.data.copy(); data[len(data) // 2] *= 1.0 + 2.0 ** -40
    Mp = P.CCS(pen.A.nrows, pen.A.ncols, pen.A.j_col, pen.A.i_row, data)
    Ap = b200.Mat(Mp)
    assert Ap.storage()["lat_const"] == 0 and Ap.storage()["lat_s1"] == m
    x = np.asfortranarray(np.random.default_rng(5).standard_normal((n, 16)))
    Y = b200.MultiVec(n, 16)
    api.mat_dot_multivec(Ap, b200.MultiVec.from_numpy(x), Y, (0, 0), (16, 16))
    assert np.array_equal(Y.numpy(), oracle_spmm(Mp, x))


def test_mat_axpby_keeps_the_stencil_flags_right(b200):
    """A + sigma B of two constant stencils is one again (the in-place shift of the inner solve); adding a diagonal
    with varying entries ends it -- the flag follows the values."""
    import scipy.sparse as sp
    from gcge_b200 import api
    pen = P.p1_fem_kuhn(9)
    n = pen.A.ncols
    Y = b200.Mat(pen.A); X = b200.Mat(pen.B)
    Y.axpby(2.5, X, 1.0)
    assert Y.storage()["lat_const"] == 1
    x = np.asfortranarray(np.random.default_rng(2).standard_normal((n, 10)))
    Xv = b200.MultiVec.from_numpy(x); Yv = b200.MultiVec(n, 10)
    api.mat_dot_multivec(Y, Xv, Yv, (0, 0), (10, 10))
    want = (pen.A.to_scipy() + 2.5 * pen.B.to_scipy()) @ x
    assert rel(Yv.numpy(), want) < 1e-14
    D = _ccs_from_scipy(sp.diags(np.linspace(1.0, 2.0, n)))
    Y.axpby(1.0, b200.Mat(D), 1.0)
    assert Y.storage()["lat_const"] == 0
    api.mat_dot_multivec(Y, Xv, Yv, (0, 0), (10, 10))
    assert rel(Yv.numpy(), want + np.linspace(1.0, 2.0, n)[:, None] * x) < 1e-14


def test_spmm_lattice_recognition_rejects_wrap_around(b200):
    """A periodic operator has the same diagonals (plus the wrap diagonals) but couples across the lattice faces:
    it must NOT be taken for a Dirichlet lattice (the tiles would read zero-filled rows outside the lattice),
    and the result through the other kernels is still the reference's."""
    from gcge_b200 import api
    M = _lattice_matrix(10, 8, 6, "7pt", periodic=True)
    A = b200.Mat(M)
    assert A.storage()["lat_s1"] == 0
    n = M.ncols
    x = np.asfortranarray(np.random.default_rng(3).standard_normal((n, 16)))
    Y = b200.MultiVec(n, 16)
    api.mat_dot_multivec(A, b200.MultiVec.from_numpy(x), Y, (0, 0), (16, 16))
    assert np.array_equal(Y.numpy(), oracle_spmm(M, x))


def test_axpby_semantics(b200, refmod):
    """MultiVecAxpby (reference app/app_lapack.c:334-395; call shapes of
    reference test/test_multi_vec.c:103-116)."""
    from gcge_b200 import api
    rng = np.random.default_rng(3)
    n = 777
    x = np.asfortranarray(rng.standard_normal((n, 6))); y = np.asfortranarray(rng.standard_normal((n, 9)))
    for alpha, beta, s, e in ((1.0, 0.0, (1, 2), (4, 5)), (0.5, 1.0, (0, 0), (6, 6)), (-2.0, 3.0, (2, 7), (4, 9)),
                              (1.0, -1.0, (0, 3), (1, 4))):
        X = b200.MultiVec.from_numpy(x); Y = b200.MultiVec.from_numpy(y)
        api.multivec_axpby(alpha, X, beta, Y, s, e)
        want = y.copy(order="F")
        k = e[0] - s[0]
        blk = np.ascontiguousarray(want[:, s[1]:s[1] + k].T).T
        want[:, s[1]:s[1] + k] = alpha * x[:, s[0]:e[0]] + (0.0 if beta == 0.0 else beta * blk)
        got = Y.numpy()
        assert rel(got, want) < 1e-15
        if beta == 0.0 and alpha == 1.0:
            assert np.array_equal(got[:, s[1]:e[1]], x[:, s[0]:e[0]])       # copies are exact
        if refmod is not None:
            yr = y.copy(order="F")
            refmod.multivec_axpby(alpha, x, beta, yr, s, e)
            assert rel(got, yr) < 1e-15
    # x == NULL: scale only; beta == 0 overwrites NaNs (memset in the reference)
    ynan = y.copy(order="F"); ynan[3, 2] = np.nan
    Y = b200.MultiVec.from_numpy(ynan)
    api.multivec_axpby(0.0, None, 2.0, Y, (0, 0), (2, 2))
    assert np.array_equal(Y.numpy()[:, :2], 2.0 * y[:, :2])
    api.multivec_axpby(1.0, b200.MultiVec.from_numpy(x), 0.0, Y, (0, 2), (1, 3))
    assert np.array_equal(Y.numpy()[:, 2], x[:, 0])
    # same multi-vector, disjoint ranges: column copy (reference src/ops_orth.c:70,302)
    Y = b200.MultiVec.from_numpy(y)
    api.multivec_axpby(1.0, Y, 0.0, Y, (7, 1), (9, 3))
    assert np.array_equal(Y.numpy()[:, 1:3], y[:, 7:9])


def test_axpby_single_column_calls_are_batched_bit_exactly(b200):
    """The reference's BlockPCG calls MultiVecAxpby one column at a time with per-column alpha / beta
    (src/ops_lin_sol.c:256-405).  The slot defers such calls and launches runs of adjacent columns as one kernel:
    same bits as the call-by-call path (option no_axpby_batch), in every order of calls -- adjacent runs, gaps, more
    columns than a batch holds, beta = 0 over NaNs, a view of the same storage, other calls in between."""
    from gcge_b200 import api
    L = b200.lib()
    rng = np.random.default_rng(3)
    n, kx, ky = 4099, 90, 96
    x = np.asfortranarray(rng.standard_normal((n, kx))); y0 = np.asfortranarray(rng.standard_normal((n, ky)))
    y0[5, 7] = np.nan                                             # overwritten by a beta = 0 call below
    alphas = rng.standard_normal(200); betas = rng.standard_normal(200)
    betas[3] = 0.0; betas[11] = 1.0; alphas[4] = 0.0

    def sequence(X, Y):
        calls = 0
        launches0 = L.b200_kernel_launches()
        for j in range(80):                                       # one adjacent run, longer than a batch
            api.multivec_axpby(alphas[j], X, betas[j] if j != 7 else 0.0, Y, (j + 2, j), (j + 3, j + 1)); calls += 1
        for j in (0, 1, 2, 5, 6, 9, 20, 21, 22, 23):              # gaps: several short batches
            api.multivec_axpby(alphas[100 + j], X, betas[100 + j], Y, (j, 80 + j // 2), (j + 1, 81 + j // 2)); calls += 1
        api.multivec_axpby(0.5, X, 2.0, Y, (0, 90), (3, 93)); calls += 1           # a 3-column call joins ...
        api.multivec_axpby(0.25, X, 1.0, Y, (3, 93), (4, 94)); calls += 1          # ... and is extended
        d = np.zeros(2)
        api.multivec_inner_prod("D", Y, Y, (92, 92), (94, 94), d, 1)               # any other call sees the result
        Yv = Y.view(10, 20)                                                          # same storage through a view
        api.multivec_axpby(1.5, Y, 0.5, Yv, (12, 1), (13, 2)); calls += 1           # reads column 12, writes column 11
        api.multivec_axpby(1.5, Y, 0.5, Yv, (13, 2), (14, 3)); calls += 1           # reads column 13, writes column 12
        api.multivec_axpby(-1.0, Yv, 0.0, Y, (2, 13), (3, 14)); calls += 1          # reads column 12 (just written)
        out = Y.numpy()
        return out, d, calls, L.b200_kernel_launches() - launches0

    X = b200.MultiVec.from_numpy(x)
    got, dg, calls, launched = sequence(X, b200.MultiVec.from_numpy(y0))
    try:
        L.b200_option_set(b"no_axpby_batch", 1)
        want, dw, _, launched_plain = sequence(X, b200.MultiVec.from_numpy(y0))
    finally:
        L.b200_option_set(b"no_axpby_batch", 0)
    assert np.array_equal(got, want, equal_nan=True) and np.array_equal(dg, dw)
    assert not np.isnan(got[5, 7])
    assert launched < launched_plain - 60, (launched, launched_plain, calls)       # the run of 80 went in two launches
    # numpy restatement of the first run (same formula: beta*y rounded, then one fma -- checked to a few ulps)
    for j in (0, 3, 11, 40, 79):
        b = betas[j] if j != 7 else 0.0
        ref = alphas[j] * x[:, j + 2] + (b * y0[:, j] if b != 0.0 else 0.0)
        if j not in range(11, 14) and j != 7:
            assert np.allclose(got[:, j], ref, rtol=1e-14, atol=1e-14)


def test_axpby_interleaved_streams_are_batched(b200):
    """BlockPCG's update loop alternates x[:, c] += alpha_c p[:, c] and r[:, c] -= alpha_c w[:, c] column by column
    (reference src/ops_lin_sol.c:330-345): two independent batches stay open side by side; a call that depends on an
    open batch (reads what it writes) launches everything first.  Same bits as call by call."""
    from gcge_b200 import api
    L = b200.lib()
    rng = np.random.default_rng(8)
    n, k = 3001, 24
    p = np.asfortranarray(rng.standard_normal((n, k))); w = np.asfortranarray(rng.standard_normal((n, k)))
    x0 = np.asfortranarray(rng.standard_normal((n, k + 6))); r0 = np.asfortranarray(rng.standard_normal((n, k)))
    al = rng.standard_normal(k)

    def run():
        Pm = b200.MultiVec.from_numpy(p); Wm = b200.MultiVec.from_numpy(w)
        Xm = b200.MultiVec.from_numpy(x0); Rm = b200.MultiVec.from_numpy(r0)
        l0 = L.b200_kernel_launches()
        for c in range(k):
            api.multivec_axpby(al[c], Pm, 1.0, Xm, (c, 3 + c), (c + 1, 4 + c))
            api.multivec_axpby(-al[c], Wm, 1.0, Rm, (c, c), (c + 1, c + 1))
        # depends on the open r batch: r[:, 0] is read
        api.multivec_axpby(2.0, Rm, 0.0, Xm, (0, 0), (1, 1))
        # p = r + beta p, column by column (src/ops_lin_sol.c:270-282)
        for c in range(k):
            api.multivec_axpby(1.0, Rm, al[c], Pm, (c, c), (c + 1, c + 1))
        nl = L.b200_kernel_launches() - l0
        return Xm.numpy(), Rm.numpy(), Pm.numpy(), nl

    xg, rg, pg, nl = run()
    try:
        L.b200_option_set(b"no_axpby_batch", 1)
        xw, rw, pw, nl_plain = run()
    finally:
        L.b200_option_set(b"no_axpby_batch", 0)
    assert np.array_equal(xg, xw) and np.array_equal(rg, rw) and np.array_equal(pg, pw)
    assert nl <= 6 and nl_plain == 3 * k + 1, (nl, nl_plain)
    assert np.allclose(xg[:, 3:3 + k], x0[:, 3:3 + k] + p * al, rtol=1e-14, atol=1e-14)
    assert np.allclose(xg[:, 0], 2.0 * (r0[:, 0] - al[0] * w[:, 0]), rtol=1e-14, atol=1e-14)


@pytest.mark.parametrize("shape", [(2, 5), (1, 1), (17, 3), (40, 40), (100, 37), (70, 130)])
def test_inner_prod_modes(b200, refmod, shape):
    """MultiVecInnerProd N / S / D (reference app/app_lapack.c:24-183 via :299-321;
    reference test/test_multi_vec.c:40-102).  Tolerance 1e-13 relative to the block's
    largest entry: summation order differs from BLAS."""
    from gcge_b200 import api
    p, q = shape
    rng = np.random.default_rng(p * 131 + q)
    n = 2311
    x = np.asfortranarray(rng.standard_normal((n, p + 2))); y = np.asfortranarray(rng.standard_normal((n, q + 1)))
    X = b200.MultiVec.from_numpy(x); Y = b200.MultiVec.from_numpy(y)
    ld = p + 3
    got = np.full((ld, q), 7.0, order="F")
    api.multivec_inner_prod("N", X, Y, (1, 1), (1 + p, 1 + q), got, ld)
    want = x[:, 1:1 + p].T @ y[:, 1:1 + q]
    assert rel(got[:p], want) < 1e-13
    assert np.all(got[p:] == 7.0)                    # rows beyond the block untouched (ldIP)
    if refmod is not None:
        r = np.zeros((ld, q), order="F")
        refmod.multivec_inner_prod("N", x, y, (1, 1), (1 + p, 1 + q), r, ld)
        assert rel(got[:p], r[:p]) < 1e-13
    m = min(p, q)
    d = np.zeros(m)
    api.multivec_inner_prod("D", X, Y, (0, 0), (m, m), d, 1)
    assert rel(d, np.einsum("ij,ij->j", x[:, :m], y[:, :m])) < 1e-13
    s = np.zeros((p, p), order="F")
    api.multivec_inner_prod("S", X, X, (0, 0), (p, p), s, p)
    assert rel(s, x[:, :p].T @ x[:, :p]) < 1e-13
    assert np.array_equal(s, s.T)


@pytest.mark.parametrize("k,xo,yo", [(1, 0, 0), (7, 1, 0), (40, 0, 2), (41, 3, 3), (128, 0, 0), (129, 1, 2), (300, 2, 5)])
def test_inner_prod_column_dots(b200, refmod, k, xo, yo):
    """'D' on the streaming geometry: any width (more than 128 columns go in several launches), odd column offsets
    (8-byte path), a strided destination (ldIP: reference app/app_lapack.c:67-115), run-to-run identical bits."""
    from gcge_b200 import api
    rng = np.random.default_rng(k)
    n = 5003
    x = np.asfortranarray(rng.standard_normal((n, k + 4))); y = np.asfortranarray(rng.standard_normal((n, k + 6)))
    X = b200.MultiVec.from_numpy(x); Y = b200.MultiVec.from_numpy(y)
    want = np.einsum("ij,ij->j", x[:, xo:xo + k], y[:, yo:yo + k])
    d = np.zeros(k); d2 = np.zeros(k)
    api.multivec_inner_prod("D", X, Y, (xo, yo), (xo + k, yo + k), d, 1)
    api.multivec_inner_prod("D", X, Y, (xo, yo), (xo + k, yo + k), d2, 1)
    assert rel(d, want) < 1e-13 and np.array_equal(d, d2)
    ds = np.full(3 * k, 7.0)
    api.multivec_inner_prod("D", X, Y, (xo, yo), (xo + k, yo + k), ds, 3)
    assert np.array_equal(ds[::3], d) and np.all(ds[1::3] == 7.0) and np.all(ds[2::3] == 7.0)
    if refmod is not None:
        r = np.zeros(k)
        refmod.multivec_inner_prod("D", x, y, (xo, yo), (xo + k, yo + k), r, 1)
        assert rel(d, r) < 1e-13


def test_inner_prod_deterministic(b200):
    from gcge_b200 import api
    rng = np.random.default_rng(9)
    x = np.asfortranarray(rng.standard_normal((50000, 24)))
    X = b200.MultiVec.from_numpy(x)
    a = np.zeros((24, 24), order="F"); b = np.zeros((24, 24), order="F")
    api.multivec_inner_prod("N", X, X, (0, 0), (24, 24), a, 24)
    api.multivec_inner_prod("N", X, X, (0, 0), (24, 24), b, 24)
    assert np.array_equal(a, b)


@pytest.mark.parametrize("modes", [("S", "S"), ("S", "D"), ("S", "N"), ("N", "N"), ("S", "T")])
def test_qtap_modes_and_workspace_side_effect(b200, refmod, pencil, modes):
    """MultiVecQtAP (reference src/ops_multi_vec.c:351-411; reference
    test/test_multi_vec.c:139-197), including A*P left in mv_ws, which ops_orth.c relies on
    (reference src/ops_orth.c:315-323)."""
    from gcge_b200 import api
    ntsA, out = modes
    rng = np.random.default_rng(11)
    n = pencil.A.ncols
    q = np.asfortranarray(rng.standard_normal((n, 6))); p = np.asfortranarray(rng.standard_normal((n, 5)))
    A = b200.Mat(pencil.A)
    Q = b200.MultiVec.from_numpy(q); Pm = b200.MultiVec.from_numpy(p); W = b200.MultiVec(n, 5)
    Ad = pencil.A.to_scipy()
    if out in ("S", "D"):
        s, e = (1, 1), (4, 4)
        Pm = Q; pp = q
    else:
        s, e = (1, 0), (6, 4)
        pp = p
    nr, nc = e[0] - s[0], e[1] - s[1]
    AP = Ad @ pp[:, s[1]:e[1]]
    full = q[:, s[0]:e[0]].T @ AP
    if out == "D":
        got = np.zeros(nr)
        api.multivec_qtap(ntsA, out, Q, A, Pm, s, e, got, 1, W)
        assert rel(got, np.diag(full)) < 1e-13
    elif out == "T":
        got = np.zeros((nc, nr), order="F")
        api.multivec_qtap(ntsA, out, Q, A, Pm, s, e, got, nc, W)
        assert rel(got, full.T) < 1e-13
    else:
        got = np.zeros((nr, nc), order="F")
        api.multivec_qtap(ntsA, out, Q, A, Pm, s, e, got, nr, W)
        assert rel(got, full) < 1e-13
    assert np.array_equal(W.numpy()[:, :nc], oracle_spmm(pencil.A, pp[:, s[1]:e[1]]))
    # A == NULL: plain inner product
    g2 = np.zeros((nr, nc), order="F")
    if out in ("N",):
        api.multivec_qtap("N", "N", Q, None, Pm, s, e, g2, nr, None)
        assert rel(g2, q[:, s[0]:e[0]].T @ pp[:, s[1]:e[1]]) < 1e-13


@pytest.mark.parametrize("shape", [(1, 4), (5, 2), (16, 16), (33, 70), (120, 40), (7, 129)])
def test_linear_comb(b200, refmod, shape):
    """MultiVecLinearComb (reference app/app_lapack.c:463-534; reference
    test/test_multi_vec.c:199-222): beta NULL / scalar / per column, scaling-only forms and the
    same-multi-vector update used by OrthSelf."""
    from gcge_b200 import api
    p, q = shape
    rng = np.random.default_rng(p + 1000 * q)
    n = 1234
    x = np.asfortranarray(rng.standard_normal((n, p + 1))); y = np.asfortranarray(rng.standard_normal((n, q + 2)))
    ldc = p + 2
    coef = np.asfortranarray(rng.standard_normal((ldc, q)))
    X = b200.MultiVec.from_numpy(x)
    base = x[:, 1:1 + p] @ coef[:p]
    # beta == NULL: overwrite, even over NaNs
    ynan = y.copy(order="F"); ynan[0, 1] = np.nan
    Y = b200.MultiVec.from_numpy(ynan)
    api.multivec_linear_comb(X, Y, (1, 1), (1 + p, 1 + q), coef, ldc, None, 0)
    got = Y.numpy()
    assert rel(got[:, 1:1 + q], base) < 1e-13
    assert np.array_equal(got[:, 0], y[:, 0]) and np.array_equal(got[:, 1 + q:], y[:, 1 + q:])
    # one scalar beta (incb == 0)
    Y = b200.MultiVec.from_numpy(y)
    b1 = np.array([0.75])
    api.multivec_linear_comb(X, Y, (1, 1), (1 + p, 1 + q), coef, ldc, b1, 0)
    assert rel(Y.numpy()[:, 1:1 + q], base + 0.75 * y[:, 1:1 + q]) < 1e-13
    # per-column beta with stride
    Y = b200.MultiVec.from_numpy(y)
    bv = rng.standard_normal(2 * q)
    api.multivec_linear_comb(X, Y, (1, 1), (1 + p, 1 + q), coef, ldc, bv, 2)
    want = base + y[:, 1:1 + q] * bv[::2]
    assert rel(Y.numpy()[:, 1:1 + q], want) < 1e-13
    if refmod is not None:
        yr = y.copy(order="F")
        refmod.multivec_linear_comb(x, yr, (1, 1), (1 + p, 1 + q), coef, ldc, bv, 2)
        assert rel(Y.numpy(), yr) < 1e-13
    # scaling only (x == NULL), as CheckConvergence does (reference src/ops_eig_sol_gcg.c:217-218)
    Y = b200.MultiVec.from_numpy(y)
    api.multivec_linear_comb(None, Y, (0, 1), (q, 1 + q), None, 0, bv, 2)
    assert rel(Y.numpy()[:, 1:1 + q], y[:, 1:1 + q] * bv[::2]) < 1e-15
    # x == NULL and beta == NULL: nothing happens (reference app/app_lapack.c:476-505)
    api.multivec_linear_comb(None, Y, (0, 1), (q, 1 + q), None, 0, None, 0)
    assert rel(Y.numpy()[:, 1:1 + q], y[:, 1:1 + q] * bv[::2]) < 1e-15


@pytest.mark.parametrize("shape", [(16, 16), (40, 40), (64, 8), (120, 40), (33, 70), (200, 130), (480, 400), (441, 40)])
@pytest.mark.parametrize("n", [128, 1234, 5001])
def test_linear_comb_aligned_blocks_tma_kernel(b200, shape, n):
    """The TMA-fed LinearComb kernel (b200_dense.cu: lincomb_tma_kernel) takes 16-byte aligned blocks
    with an even number of output columns: contraction lengths beyond the 4-deep tile ring, several
    column tiles, ragged last tiles in every dimension, with and without beta."""
    from gcge_b200 import api
    p, q = shape
    rng = np.random.default_rng(p + 1000 * q + n)
    x = np.asfortranarray(rng.standard_normal((n, p + 2))); y = np.asfortranarray(rng.standard_normal((n, q + 6)))
    coef = np.asfortranarray(rng.standard_normal((p, q)))
    X = b200.MultiVec.from_numpy(x)
    base = x[:, 2:2 + p] @ coef
    scale = np.abs(x[:, 2:2 + p]) @ np.abs(coef)
    Y = b200.MultiVec.from_numpy(y)
    api.multivec_linear_comb(X, Y, (2, 4), (2 + p, 4 + q), coef, p, None, 0)
    got = Y.numpy()
    assert np.max(np.abs(got[:, 4:4 + q] - base) / scale) < 1e-14
    assert np.array_equal(got[:, :4], y[:, :4]) and np.array_equal(got[:, 4 + q:], y[:, 4 + q:])
    bv = rng.standard_normal(q)
    Y = b200.MultiVec.from_numpy(y)
    api.multivec_linear_comb(X, Y, (2, 4), (2 + p, 4 + q), coef, p, bv, 1)
    want = base + y[:, 4:4 + q] * bv
    assert np.max(np.abs(Y.numpy()[:, 4:4 + q] - want) / (scale + np.abs(y[:, 4:4 + q] * bv))) < 1e-14


@pytest.mark.parametrize("n", [440, 3000])
@pytest.mark.parametrize("s1,kb", [(400, 40), (40, 40), (120, 20), (6, 10)])
def test_linear_comb_in_place_update_like_orth(b200, n, s1, kb):
    """The update of the block orthogonalisation (host/b200_orth.c: X1 += X0 C with X0, X1 column
    ranges of ONE multi-vector, beta a single scalar, incb == 0) at the sizes the solver uses,
    including the coefficient-space call with n = sizeV rows."""
    from gcge_b200 import api
    rng = np.random.default_rng(n + s1 + kb)
    v = np.asfortranarray(rng.standard_normal((n, 480)))
    V = b200.MultiVec.from_numpy(v)
    coef = np.asfortranarray(rng.standard_normal((s1, kb)))
    one = np.array([1.0])
    api.multivec_linear_comb(V, V, (0, s1), (s1, s1 + kb), coef, s1, one, 0)
    want = v.copy()
    want[:, s1:s1 + kb] += v[:, :s1] @ coef
    got = V.numpy()
    scale = np.abs(v[:, :s1]) @ np.abs(coef) + np.abs(v[:, s1:s1 + kb])
    assert np.max(np.abs(got[:, s1:s1 + kb] - want[:, s1:s1 + kb]) / scale) < 1e-14
    assert np.array_equal(got[:, :s1], v[:, :s1]) and np.array_equal(got[:, s1 + kb:], v[:, s1 + kb:])


def test_linear_comb_in_place_disjoint_columns(b200):
    from gcge_b200 import api
    rng = np.random.default_rng(21)
    n = 999
    v = np.asfortranarray(rng.standard_normal((n, 12)))
    V = b200.MultiVec.from_numpy(v)
    coef = np.asfortranarray(rng.standard_normal((4, 8)))
    one = np.array([1.0])
    api.multivec_linear_comb(V, V, (0, 4), (4, 12), coef, 4, one, 0)
    want = v.copy()
    want[:, 4:] += v[:, :4] @ coef
    assert rel(V.numpy(), want) < 1e-13


def test_mat_axpby(b200, pencil):
    from gcge_b200 import api
    A = b200.Mat(pencil.A); B = b200.Mat(pencil.B)
    A.axpby(0.25, B, 1.0)        # A += 0.25 B, the in-place shift of reference src/ops_eig_sol_gcg.c:594-602
    _, _, v = A.to_ccs()
    assert rel(v, pencil.A.data + 0.25 * pencil.B.data) < 1e-15
    A.axpby(-0.25, B, 1.0)
    _, _, v = A.to_ccs()
    assert rel(v, pencil.A.data) < 1e-15


def _ccs_from_scipy(M):
    M = M.tocsc(); M.sort_indices()
    return P.CCS(M.shape[0], M.shape[1], M.indptr.astype(np.int32), M.indices.astype(np.int32), M.data.astype(np.float64))


def test_mat_axpby_subset_pattern_and_validation(b200):
    """ADVICE r1: Y = alpha X + beta Y where X's pattern is a strict SUBSET of Y's (A = stiffness, B = lumped
    diagonal mass -- what the reference's SLEPc back end passes as SUBSET_NONZERO_PATTERN), checked through
    SpMM (diagonal image), the CCS round trip (transpose image) and beta != 1; a pattern that is NOT a subset
    fails before Y is touched."""
    import scipy.sparse as sp
    from gcge_b200 import api
    pen = P.p1_fem_kuhn(9)
    n = pen.A.ncols
    lumped = np.asarray(pen.B.to_scipy().sum(axis=1)).ravel()
    D = _ccs_from_scipy(sp.diags(lumped))
    Y = b200.Mat(pen.A); X = b200.Mat(D)
    Y.axpby(0.75, X, 1.0)
    want = (pen.A.to_scipy() + 0.75 * sp.diags(lumped)).tocsc(); want.sort_indices()
    jc, ir, v = Y.to_ccs()
    assert np.array_equal(jc, pen.A.j_col) and np.array_equal(ir, pen.A.i_row)      # Y keeps its own pattern
    cols = np.repeat(np.arange(n), np.diff(pen.A.j_col))
    on_diag = pen.A.i_row == cols
    want_v = pen.A.data.copy(); want_v[on_diag] += 0.75 * lumped
    assert rel(v, want_v) < 1e-15
    x = np.asfortranarray(np.random.default_rng(0).standard_normal((n, 10)))
    Xv = b200.MultiVec.from_numpy(x); Yv = b200.MultiVec(n, 10)
    api.mat_dot_multivec(Y, Xv, Yv, (0, 0), (10, 10))
    assert rel(Yv.numpy(), want @ x) < 1e-14
    Y.axpby(-1.5, X, 2.0)                                    # beta != 1
    want2 = (2.0 * want - 1.5 * sp.diags(lumped)).tocsc(); want2.sort_indices()
    _, _, v = Y.to_ccs()
    want_v = 2.0 * want_v; want_v[on_diag] -= 1.5 * lumped
    assert rel(v, want_v) < 1e-15
    api.mat_dot_multivec(Y, Xv, Yv, (0, 0), (10, 10))
    assert rel(Yv.numpy(), want2 @ x) < 1e-14
    # not a subset: same nnz as X would have passed the old shape/nnz check
    off = sp.diags([lumped[:-7]], [7], shape=(n, n))         # a diagonal the P1 pattern does not have
    Z = b200.Mat(_ccs_from_scipy(off))
    before = Y.to_ccs()[2].copy()
    with pytest.raises(api.B200Error, match="subset"):
        Y.axpby(1.0, Z, 3.0)
    assert np.array_equal(Y.to_ccs()[2], before)             # nothing was modified
    api.mat_dot_multivec(Y, Xv, Yv, (0, 0), (10, 10))
    assert rel(Yv.numpy(), want2 @ x) < 1e-14


def test_tierA_shifted_solve_with_diagonal_B(b200, refmod, drive_b200):
    """The route ADVICE r1 names: the reference's GCG over OPS_B200_Set with sigma != 0 and B != NULL takes
    MatAxpby(sigma, B, 1, A) (src/ops_eig_sol_gcg.c:594-602); with B = lumped (diagonal) mass its pattern
    differs from A's.  Same run on the reference's CCS back end (whose MatAxpby slot is NULL: shifted
    operator route): same eigenvalues, iteration count within 1."""
    if drive_b200 is None:
        pytest.skip("oracle/_ref (reference + driver) not present on this box")
    import scipy.sparse as sp
    pen = P.p1_fem_kuhn(10)
    lumped = np.asarray(pen.B.to_scipy().sum(axis=1)).ravel()
    D = _ccs_from_scipy(sp.diags(lumped))
    argv = ("-gcge_compW_cg_shift", 2.0)
    r = refmod.gcg_solve(pen.A, D, nev=8, want_evec=False, argv=argv)
    a = drive_b200(0, pen.A, D, nev=8, argv=argv)
    assert a["nev_conv"] >= 8 and r["nev_conv"] >= 8
    assert abs(a["num_iter"] - r["num_iter"]) <= 1, (a["num_iter"], r["num_iter"])
    assert rel(a["eval"][:8], r["eval"][:8]) < 1e-10


def test_argument_errors_are_loud(b200):
    from gcge_b200 import api
    X = b200.MultiVec(10, 3); Y = b200.MultiVec(11, 3)
    with pytest.raises(api.B200Error):
        api.multivec_axpby(1.0, X, 0.0, Y, (0, 0), (2, 2))       # row counts differ
    with pytest.raises(api.B200Error):
        api.multivec_axpby(1.0, X, 0.0, X, (0, 1), (2, 3))       # overlapping ranges
    with pytest.raises(api.B200Error):
        api.multivec_axpby(1.0, X, 0.0, X, (0, 0), (2, 5))       # out of range
