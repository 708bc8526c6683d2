"""On-disk matrix input (SURVEY.md 8f row 4): the library's MatrixMarket reader against scipy's, on
general / symmetric / pattern files; CPU only."""
import numpy as np
import pytest
import scipy.io
import scipy.sparse as sp

from gcge_b200 import api, problems as P


def _same(ccs, m):
    m = sp.csc_matrix(m); m.sort_indices()
    assert (ccs.nrows, ccs.ncols) == m.shape
    assert np.array_equal(ccs.j_col, m.indptr) and np.array_equal(ccs.i_row, m.indices)
    assert np.array_equal(ccs.data, m.data)


def test_matrix_market_general_and_symmetric(tmp_path):
    rng = np.random.default_rng(0)
    g = sp.random(37, 23, density=0.15, random_state=rng, format="coo")
    scipy.io.mmwrite(str(tmp_path / "g.mtx"), g, precision=17)
    _same(api.read_matrix_market(tmp_path / "g.mtx"), g)
    pen = P.p1_fem_kuhn(6)
    a = pen.A.to_scipy()
    scipy.io.mmwrite(str(tmp_path / "a.mtx"), sp.coo_matrix(a), symmetry="symmetric", precision=17)
    got = api.read_matrix_market(tmp_path / "a.mtx")
    _same(got, a)
    assert np.array_equal(got.j_col, pen.A.j_col) and np.array_equal(got.i_row, pen.A.i_row)
    assert np.array_equal(got.data, pen.A.data)        # 17 digits round-trip the doubles bit for bit


def test_matrix_market_pattern_and_errors(tmp_path):
    (tmp_path / "p.mtx").write_text("%%MatrixMarket matrix coordinate pattern general\n% c\n3 4 3\n1 1\n3 2\n2 4\n")
    got = api.read_matrix_market(tmp_path / "p.mtx")
    want = sp.coo_matrix((np.ones(3), ([0, 2, 1], [0, 1, 3])), shape=(3, 4))
    _same(got, want)
    (tmp_path / "bad.mtx").write_text("%%MatrixMarket matrix array real general\n2 2\n1\n2\n3\n4\n")
    with pytest.raises(RuntimeError):
        api.read_matrix_market(tmp_path / "bad.mtx")
    with pytest.raises(RuntimeError):
        api.read_matrix_market(tmp_path / "missing.mtx")
    (tmp_path / "oob.mtx").write_text("%%MatrixMarket matrix coordinate real general\n2 2 1\n3 1 1.0\n")
    with pytest.raises(RuntimeError):
        api.read_matrix_market(tmp_path / "oob.mtx")


def _write_petsc(path, m):
    """PETSc binary AIJ as MatView writes it: big-endian header, row lengths, column indices, values."""
    m = sp.csr_matrix(m); m.sort_indices()
    with open(path, "wb") as f:
        np.array([1211216, m.shape[0], m.shape[1], m.nnz], dtype=">i4").tofile(f)
        np.diff(m.indptr).astype(">i4").tofile(f)
        m.indices.astype(">i4").tofile(f)
        m.data.astype(">f8").tofile(f)


def test_petsc_binary(tmp_path):
    rng = np.random.default_rng(4)
    g = sp.random(29, 41, density=0.2, random_state=rng, format="csr")
    _write_petsc(tmp_path / "g.petsc", g)
    _same(api.read_petsc_binary(tmp_path / "g.petsc"), g)
    pen = P.p1_fem_kuhn(6)
    _write_petsc(tmp_path / "b.petsc", pen.B.to_scipy())
    got = api.read_petsc_binary(tmp_path / "b.petsc")
    assert np.array_equal(got.j_col, pen.B.j_col) and np.array_equal(got.i_row, pen.B.i_row)
    assert np.array_equal(got.data, pen.B.data)
    (tmp_path / "bad.petsc").write_bytes(b"\x00" * 32)
    with pytest.raises(RuntimeError):
        api.read_petsc_binary(tmp_path / "bad.petsc")
    with open(tmp_path / "trunc.petsc", "wb") as f:
        np.array([1211216, 3, 3, 5], dtype=">i4").tofile(f)
        np.array([2, 2, 1], dtype=">i4").tofile(f)
    with pytest.raises(RuntimeError):
        api.read_petsc_binary(tmp_path / "trunc.petsc")


# ---- BASELINE config 1: the reference's mesh file data/cube4.dat ---------------------------------------------
def test_cube4_fixture_is_the_reference_file(tmp_path):
    """tests/golden/cube4_mesh.json (made by tests/golden/make_cube4_fixture.py from the reference's data/cube4.dat)
    holds what that file says -- 125 vertices, exactly the 5^3 lattice of [0,1]^3, 384 tetrahedra over them -- and
    goes through the ALBERT reader unchanged when written back in the file's format.  The digest pins the vertex
    and element lists to the ones make_cube4_fixture.py parsed from that file when the fixture was made."""
    import hashlib
    V, T = P.cube4_mesh()
    assert V.shape == (125, 3) and T.shape == (384, 4)
    q = np.rint(V * 4).astype(np.int64)
    assert hashlib.sha256(q.tobytes() + T.astype(np.int64).tobytes()).hexdigest() == \
        "17f73130985d1518b5cdc9ed62f4d6c0769e847b90caaf5d1ecf2117366c0127"
    assert np.array_equal(q / 4.0, V) and len(np.unique(q, axis=0)) == 125 and q.min() == 0 and q.max() == 4
    assert T.min() == 0 and T.max() == 124 and all(len(set(t)) == 4 for t in T.tolist())
    fmt = lambda rows: "\n".join(" ".join(repr(v) for v in r) for r in rows)
    (tmp_path / "cube4.dat").write_text(
        "DIM: 3\nDIM_OF_WORLD: 3\n\nnumber of elements: 384\nnumber of vertices: 125\n\n"
        f"vertex coordinates:\n{fmt(V.tolist())}\n\nelement vertices:\n{fmt(T.tolist())}\n\n"
        f"element boundaries:\n{fmt(np.zeros_like(T).tolist())}\n")
    V2, T2 = P.read_albert_mesh(tmp_path / "cube4.dat")
    assert np.array_equal(V, V2) and np.array_equal(T, T2)


def test_cube4_mesh_is_a_conforming_triangulation_of_the_unit_cube():
    """volumes add up to 1 before and after the regular refinements; after r refinements the vertices are the
    (4 * 2^r + 1)^3 lattice; the P1 matrices are symmetric, the mass matrix sums to the volume of the cube."""
    V, T = P.cube4_mesh()
    for r in range(3):
        M = np.concatenate([np.ones((len(T), 4, 1)), V[T]], axis=2)
        vol = np.abs(np.linalg.det(M)) / 6.0
        assert abs(vol.sum() - 1.0) < 1e-12 and vol.min() > 0
        nl = 4 * 2 ** r + 1
        assert len(V) == nl ** 3 and len(np.unique(np.rint(V * (nl - 1)).astype(int), axis=0)) == nl ** 3
        if r < 2:
            V, T = P.refine_uniform(V, T)
    A, B = P.p1_assemble_mesh(V, T)
    assert abs(A - A.T).max() < 1e-13 and abs(B - B.T).max() < 1e-15
    assert abs(B.sum() - 1.0) < 1e-12 and abs(A.sum()) < 1e-9          # constants are in the kernel of the stiffness matrix


def test_cube4_pencil_golden_is_mesh_order_independent(golden=None):
    """the reference's recorded eigenvalues for config 1 (tests/golden/gcg_reference.json) agree between the two
    orderings of the unknowns, and with a sparse eigensolver on the assembled pencil"""
    import json
    from pathlib import Path
    import scipy.sparse.linalg as sla
    cases = json.loads((Path(__file__).parent / "golden" / "gcg_reference.json").read_text())["cases"]
    c4 = [c for c in cases if c["generator"] == "cube4_p1"]
    assert len(c4) == 2 and c4[0]["nev_conv"] >= 10
    ev = [np.array(c["eval"][:10]) for c in c4]
    assert np.max(np.abs(ev[0] - ev[1]) / ev[0]) < 1e-10
    pen = P.cube4_p1(2)
    assert pen.A.ncols == 15 ** 3
    w = np.sort(sla.eigsh(pen.A.to_scipy(), k=10, M=pen.B.to_scipy(), sigma=0.0, which="LM")[0])
    assert np.max(np.abs(w - ev[0]) / ev[0]) < 1e-9
