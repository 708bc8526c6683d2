"""Whole-solve parity on the GPU (BASELINE.md §4): eigenvalues within 1e-10 relative of the
reference's CCS+OpenMP GCG on the same matrix, every returned pair meets the reference's
residual test, outer iteration counts agree, eigenvectors agree by subspace angle per
eigenvalue cluster.  Three arms: the reference (oracle/_ref, or its committed golden output),
tier A = the reference's own GCG/orth/BlockPCG driving OPS_B200_Set unchanged, tier B = the
device-resident GCG (b200_gcg_solve)."""
import os
import numpy as np
import pytest

from conftest import pencil_eigenvalues, recorded_reference_runs, reference_runs_over_threads
from gcge_b200 import problems as P

pytestmark = pytest.mark.gpu

# outer-iteration parity of the device GCG (tier B) with the reference: the north_star contract
# (BASELINE.md section 4) is +-1; scripts/parity_deltas.py prints the per-case differences
# (profiles/parity_deltas_r2.log)
ITER_TOL = 1


def rel(a, b):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


def gen(case):
    return getattr(P, case["generator"])(**case["args"])


def residual_test(pen, ev, vec, tol=(1e-1, 1e-8)):
    """reference src/ops_eig_sol_gcg.c:229-252."""
    A = pen.A.to_scipy(); Bx = vec if pen.B is None else pen.B.to_scipy() @ vec
    r = np.linalg.norm(A @ vec - Bx * ev, axis=0)
    return np.all(r <= tol[0]) and np.all(r <= np.abs(ev) * tol[1] * 1.0000001), r


def cluster_angles(pen, ev, v1, v2, gap=1e-5):
    """largest principal angle between the two eigenvector sets, cluster by cluster (clusters
    split where the relative gap exceeds gapMin, reference src/ops_eig_sol_gcg.c:253-259)."""
    Bd = None if pen.B is None else pen.B.to_scipy()
    worst = 0.0
    k = len(ev)
    i = 0
    while i < k:
        j = i + 1
        while j < k and abs((ev[j - 1] - ev[j]) / ev[j - 1]) <= gap * 100:
            j += 1
        if j < k or True:
            a, b = v1[:, i:j], v2[:, i:j]
            m = a.T @ (b if Bd is None else Bd @ b)
            s = np.linalg.svd(m, compute_uv=False)
            worst = max(worst, float(np.sqrt(max(0.0, 1.0 - min(1.0, s.min()) ** 2))))
        i = j
    return worst


@pytest.mark.parametrize("idx", [0, 1, 2, 4, 3, 5, 6, 7, 8])
def test_device_gcg_vs_golden(b200, golden, idx):
    case = golden["cases"][idx]
    pen = gen(case)
    A = b200.Mat(pen.A); B = None if pen.B is None else b200.Mat(pen.B)
    o = b200.gcg_solve(A, B, nev=case["nev"])
    assert o["nev_conv"] >= case["nev"]
    assert abs(o["num_iter"] - case["num_iter"]) <= ITER_TOL, (o["num_iter"], case["num_iter"])
    k = min(o["nev_conv"], case["nev_conv"])
    assert rel(o["eval"][:k], np.array(case["eval"][:k])) < 1e-10
    vec = o["evec_mv"].numpy(0, k)
    ok, r = residual_test(pen, o["eval"][:k], vec)
    assert ok, r
    assert o["stats"]["launches"] > 0


@pytest.mark.parametrize("order", ["lattice", "mesh"])
def test_device_gcg_config1_cube4_mesh(b200, golden, drive_b200, order):
    """BASELINE config 1 restated (SURVEY 8d): P1 pencil on the reference's own mesh data/cube4.dat after two regular
    refinements (15^3 unknowns), nev = 10 (nevMax 20, block_size 10) -- device GCG and the reference's GCG over
    OPS_B200_Set against the reference's recorded CCS+OpenMP run.  In lattice order the matrix has a 27-neighbour
    pattern with element-dependent coefficients (lattice SpMM kernel); in the mesh's own order it is unstructured."""
    case = [c for c in golden["cases"] if c["generator"] == "cube4_p1" and c["args"].get("order", "lattice") == order][0]
    pen = gen(case)
    A = b200.Mat(pen.A); B = b200.Mat(pen.B)
    assert (A.storage()["lat_s1"] == 15) == (order == "lattice"), A.storage()     # 49.8 % fill of 27 diagonals: still a diagonal image
    o = b200.gcg_solve(A, B, nev=10)
    assert o["nev_conv"] >= 10
    assert abs(o["num_iter"] - case["num_iter"]) <= ITER_TOL, (o["num_iter"], case["num_iter"])
    assert rel(o["eval"][:10], np.array(case["eval"][:10])) < 1e-10
    ok, r = residual_test(pen, o["eval"][:10], o["evec_mv"].numpy(0, 10))
    assert ok, r
    if drive_b200 is not None:
        a = drive_b200(0, pen.A, pen.B, nev=10)
        assert abs(a["num_iter"] - case["num_iter"]) <= 1 and rel(a["eval"][:10], np.array(case["eval"][:10])) < 1e-10


def test_device_gcg_analytic_7pt(b200):
    m, nev = 24, 12
    pen = P.laplace3d_7pt(m)
    o = b200.gcg_solve(b200.Mat(pen.A), None, nev=nev)
    k = o["nev_conv"]
    assert k >= nev
    assert rel(o["eval"][:k], P.laplace3d_7pt_eigenvalues(m, k)) < 1e-10


def test_tierA_reference_gcg_over_ops_b200(b200, refmod, drive_b200, golden):
    """The drop-in claim: the reference's GCG, ops_orth.c and ops_lin_sol.c run UNCHANGED over
    OPS_B200_Set.  Iteration count within 1 of the reference on CCS, eigenvalues 1e-10."""
    if drive_b200 is None:
        pytest.skip("oracle/_ref (reference + driver) not present on this box")
    for idx in (0, 4):
        case = golden["cases"][idx]
        pen = gen(case)
        a = drive_b200(0, pen.A, pen.B, nev=case["nev"])
        assert a["nev_conv"] >= case["nev"]
        assert abs(a["num_iter"] - case["num_iter"]) <= 1, (a["num_iter"], case["num_iter"])
        k = min(a["nev_conv"], case["nev_conv"])
        assert rel(a["eval"][:k], np.array(case["eval"][:k])) < 1e-10


@pytest.mark.skipif(not os.environ.get("GCGE_TIERS_AT"), reason="opt-in measurement: GCGE_TIERS_AT=<m>[,<nev>]")
def test_tiers_side_by_side_at_size(b200, refmod, drive_b200):
    """Measurement, not a gate (run with -s): the same P1 pencil at lattice size m solved (1) by the reference on
    CCS + OpenMP, (2) by the reference's UNCHANGED GCG / ops_orth.c / ops_lin_sol.c over OPS_B200_Set (tier A: what a
    user gets by swapping the one Set call) and (3) by the device GCG installed through the OPS table (tier B);
    same iteration counts within 1, eigenvalues 1e-10; prints one JSON line with the three times."""
    import json
    if drive_b200 is None:
        pytest.skip("oracle/_ref (reference + driver) not present on this box")
    parts = os.environ["GCGE_TIERS_AT"].split(",")
    m = int(parts[0]); nev = int(parts[1]) if len(parts) > 1 else 50
    pen = P.p1_fem_kuhn(m)
    out = {"m": m, "n": pen.A.ncols, "nev": nev}
    a = drive_b200(0, pen.A, pen.B, nev=nev)
    b = drive_b200(1, pen.A, pen.B, nev=nev)
    b2 = drive_b200(1, pen.A, pen.B, nev=nev)                     # second solve: buffers cached, kernels loaded
    out["tierA"] = {"seconds": a["seconds"], "num_iter": a["num_iter"], "nev_conv": a["nev_conv"]}
    if os.environ.get("GCGE_TIERS_PROF"):
        # where tier A's device time goes, per kernel class (events around every call: the solve itself gets slower)
        from gcge_b200 import api
        api.prof_enable(True)
        ap = drive_b200(0, pen.A, pen.B, nev=nev)
        rep = api.prof_report(); api.prof_enable(False)
        out["tierA_profiled"] = {"seconds": ap["seconds"],
                                 "classes": {k: {"ms": round(v["ms"], 1), "calls": v["calls"], "gap_before_ms": round(v.get("gap_before_ms", 0.0), 1)}
                                             for k, v in rep.items() if v["calls"]}}
    out["tierB"] = {"seconds": b2["seconds"], "first_call_seconds": b["seconds"], "num_iter": b["num_iter"], "nev_conv": b["nev_conv"]}
    if os.environ.get("GCGE_TIERS_REF", "1") != "0":
        refmod.set_threads(refmod.max_threads())
        r = refmod.gcg_solve(pen.A, pen.B, nev=nev)
        out["reference"] = {"seconds": r["seconds"], "num_iter": r["num_iter"], "nev_conv": r["nev_conv"], "threads": refmod.max_threads()}
        assert abs(a["num_iter"] - r["num_iter"]) <= 1 and abs(b["num_iter"] - r["num_iter"]) <= 1, out
        assert rel(a["eval"][:nev], r["eval"][:nev]) < 1e-10 and rel(b["eval"][:nev], r["eval"][:nev]) < 1e-10
    else:
        assert abs(a["num_iter"] - b["num_iter"]) <= 1, out
        assert rel(a["eval"][:nev], b["eval"][:nev]) < 1e-10
    print("TIERS " + json.dumps(out))


def test_tierB_through_ops_table_and_live_reference(b200, refmod, drive_b200):
    """EigenSolverSetup_GCG_B200 installed in ops->EigenSolver, driven through the reference's
    own parameter plumbing; compared with the live reference incl. subspace angles."""
    if drive_b200 is None:
        pytest.skip("oracle/_ref (reference + driver) not present on this box")
    pen = P.p1_fem_kuhn(14)
    nev = 12
    r = refmod.gcg_solve(pen.A, pen.B, nev=nev)
    b = drive_b200(1, pen.A, pen.B, nev=nev, want_evec=True)
    assert b["nev_conv"] >= nev
    assert abs(b["num_iter"] - r["num_iter"]) <= ITER_TOL, (b["num_iter"], r["num_iter"])
    k = min(b["nev_conv"], r["nev_conv"])
    assert rel(b["eval"][:k], r["eval"][:k]) < 1e-10
    ok, res = residual_test(pen, b["eval"][:k], b["evec"][:, :k])
    assert ok, res
    assert cluster_angles(pen, r["eval"][:k], r["evec"][:, :k], b["evec"][:, :k]) < 1e-5


@pytest.mark.parametrize("argv", [
    ("-gcge_compW_cg_order", 2),                                                   # ComputeW12
    ("-gcge_initX_orth_method", "bgs", "-gcge_compP_orth_method", "bgs", "-gcge_compW_orth_method", "bgs"),
    ("-gcge_compW_cg_auto_shift", 1),                                              # A + sigma B through MatAxpby
    ("-gcge_compW_cg_shift", 3.0),
])
def test_tierA_reference_options_over_ops_b200(b200, refmod, drive_b200, argv, golden):
    """SURVEY 8f rows 1-2 at tier A: the reference's ComputeW12 (order-2 Krylov W,
    src/ops_eig_sol_gcg.c:697-923), BinaryGramSchmidt / OrthSelfEVP (src/ops_orth.c:122-201,415-640)
    and the shifted inner solve (MatAxpby slot, :594-625) run UNCHANGED over OPS_B200_Set; same
    options to the reference on CCS: iteration count within 1, eigenvalues 1e-10."""
    if drive_b200 is None:
        pytest.skip("oracle/_ref (reference + driver) not present on this box")
    pen = P.p1_fem_kuhn(12)
    r = refmod.gcg_solve(pen.A, pen.B, nev=10, want_evec=False, argv=argv)
    a = drive_b200(0, pen.A, pen.B, nev=10, argv=argv)
    assert a["nev_conv"] >= 10
    assert abs(a["num_iter"] - r["num_iter"]) <= 1, (a["num_iter"], r["num_iter"])
    k = min(a["nev_conv"], r["nev_conv"])
    assert rel(a["eval"][:k], r["eval"][:k]) < 1e-10
    case = _golden_case(golden, 12, 10, argv)            # and the recorded run (tests/golden)
    assert abs(a["num_iter"] - case["num_iter"]) <= 1
    assert rel(a["eval"][:10], np.array(case["eval"][:10])) < 1e-10


def test_device_gcg_order2_krylov_W(b200, refmod, golden):
    """Tier B ComputeW12 (b200_gcg.c: compute_w12) against the live reference with
    -gcge_compW_cg_order 2: eigenvalues 1e-10, iteration count within 1."""
    pen = P.p1_fem_kuhn(12)
    A = b200.Mat(pen.A); B = b200.Mat(pen.B)
    o = b200.gcg_solve(A, B, nev=10, compW_cg_order=2)
    base = b200.gcg_solve(A, B, nev=10)
    assert o["nev_conv"] >= 10
    assert rel(o["eval"][:10], base["eval"][:10]) < 1e-9
    case = _golden_case(golden, 12, 10, ("-gcge_compW_cg_order", 2))
    assert abs(o["num_iter"] - case["num_iter"]) <= ITER_TOL, (o["num_iter"], case["num_iter"])
    assert rel(o["eval"][:10], np.array(case["eval"][:10])) < 1e-10
    if refmod is not None:
        r = refmod.gcg_solve(pen.A, pen.B, nev=10, want_evec=False, argv=("-gcge_compW_cg_order", 2))
        assert abs(o["num_iter"] - r["num_iter"]) <= ITER_TOL, (o["num_iter"], r["num_iter"])
        k = min(o["nev_conv"], r["nev_conv"])
        assert rel(o["eval"][:k], r["eval"][:k]) < 1e-10


def test_device_gcg_binary_gram_schmidt(b200, refmod, golden):
    """Tier B with -gcge_*_orth_method bgs (SURVEY 8f row 2): the device BinaryGramSchmidt / OrthSelfEVP in all three
    places against the reference's recorded run with the same options and the live reference."""
    pen = P.p1_fem_kuhn(12)
    A = b200.Mat(pen.A); B = b200.Mat(pen.B)
    o = b200.gcg_solve(A, B, nev=10, initX_orth_method=1, compP_orth_method=1, compW_orth_method=1)
    argv = ("-gcge_initX_orth_method", "bgs", "-gcge_compP_orth_method", "bgs", "-gcge_compW_orth_method", "bgs")
    case = _golden_case(golden, 12, 10, argv)
    assert o["nev_conv"] >= 10
    assert abs(o["num_iter"] - case["num_iter"]) <= ITER_TOL, (o["num_iter"], case["num_iter"])
    assert rel(o["eval"][:10], np.array(case["eval"][:10])) < 1e-10
    ok, res = residual_test(pen, o["eval"][:10], o["evec_mv"].numpy(0, 10))
    assert ok, res
    if refmod is not None:
        pen2 = P.p1_fem_kuhn(16)
        r = refmod.gcg_solve(pen2.A, pen2.B, nev=30, want_evec=False, argv=argv)
        o2 = b200.gcg_solve(b200.Mat(pen2.A), b200.Mat(pen2.B), nev=30, initX_orth_method=1, compP_orth_method=1, compW_orth_method=1)
        assert abs(o2["num_iter"] - r["num_iter"]) <= ITER_TOL, (o2["num_iter"], r["num_iter"])
        k = min(o2["nev_conv"], r["nev_conv"])
        assert rel(o2["eval"][:k], r["eval"][:k]) < 1e-10


def test_device_gcg_block_size_200(b200, refmod):
    """block_size = 200 -- the value the reference's large runs use (test/test_eig_sol_PHG_MAT.c:38-39,
    test/submit.sh:30-34) and beyond the 128 of round 1: nev = 50, nevMax = 300, projected problems of order up to 700.
    Against the live reference with the same -nevMax / -blockSize."""
    pen = P.p1_fem_kuhn(13)
    A = b200.Mat(pen.A); B = b200.Mat(pen.B)
    o = b200.gcg_solve(A, B, nev=50, nev_max=300, block_size=200)
    assert o["nev_conv"] >= 50
    ok, res = residual_test(pen, o["eval"][:50], o["evec_mv"].numpy(0, 50))
    assert ok, res
    if refmod is not None:
        r = refmod.gcg_solve(pen.A, pen.B, nev=50, nev_max=300, block_size=200, want_evec=False)
        assert abs(o["num_iter"] - r["num_iter"]) <= ITER_TOL, (o["num_iter"], r["num_iter"])
        k = min(o["nev_conv"], r["nev_conv"])
        assert rel(o["eval"][:k], r["eval"][:k]) < 1e-10


def test_runtime_options_from_command_line(b200, drive_b200):
    """-b200_<name> <int> reaches the library through the OPS table's GetOptionFromCommandLine
    (B200_SetOptionsFromCommandLine in the adaptor), like the reference's own -gcge_* options."""
    if drive_b200 is None:
        pytest.skip("oracle/_ref (reference + driver) not present on this box")
    import ctypes as C
    L = b200.lib()
    pen = P.p1_fem_kuhn(8)
    v = C.c_int(-1)
    try:
        a = drive_b200(0, pen.A, pen.B, nev=4, argv=("-b200_no_fused_dot", 1, "-b200_lat_no_const", 1))
        assert a["nev_conv"] >= 4
        assert L.b200_option_get(b"no_fused_dot", C.byref(v)) == 0 and v.value == 1
        assert L.b200_option_get(b"lat_no_const", C.byref(v)) == 0 and v.value == 1
    finally:
        L.b200_option_set(b"no_fused_dot", 0); L.b200_option_set(b"lat_no_const", 0)


def test_runtime_options_table(b200):
    """-b200_* switches: one table, read once from the environment, changeable at run time (include/gcge_b200.h)."""
    import ctypes as C
    L = b200.lib()
    L.b200_option_name.restype = C.c_char_p
    names = [L.b200_option_name(i).decode() for i in range(L.b200_option_count())]
    # the exact set, each once: a switch is added or retired with its entry in DESIGN.md §10
    assert sorted(names) == sorted(["no_dia", "no_lat", "no_fused_dot", "host_build", "no_overlap", "no_p2p",
                                    "no_kernel_allreduce", "syev_prof", "bpcg_trace", "lat_no_const", "orth_trace",
                                    "no_axpby_batch"]), names
    v = C.c_int(-1)
    assert L.b200_option_get(b"no_lat", C.byref(v)) == 0 and v.value == 0
    pen = P.p1_fem_kuhn(8)
    try:
        assert L.b200_option_set(b"no_lat", 1) == 0
        assert b200.Mat(pen.A).storage()["lat_s1"] == 0            # the switch is honoured without a restart
    finally:
        assert L.b200_option_set(b"no_lat", 0) == 0
    assert b200.Mat(pen.A).storage()["lat_s1"] == 8
    assert L.b200_option_set(b"no_such_option", 1) != 0


def test_device_gcg_from_matrix_market_files(b200, tmp_path):
    """On-disk input (SURVEY 8f row 4): pencil written as MatrixMarket, read by the library's reader,
    solved on device: the same bits in, so the same eigenvalues out."""
    import scipy.io, scipy.sparse as sp
    pen = P.p1_fem_kuhn(10)
    for name, M in (("A", pen.A), ("B", pen.B)):
        scipy.io.mmwrite(str(tmp_path / f"{name}.mtx"), sp.coo_matrix(M.to_scipy()), symmetry="symmetric", precision=17)
    Af = b200.read_matrix_market(tmp_path / "A.mtx"); Bf = b200.read_matrix_market(tmp_path / "B.mtx")
    assert np.array_equal(Af.data, pen.A.data) and np.array_equal(Bf.i_row, pen.B.i_row)
    o1 = b200.gcg_solve(b200.Mat(Af), b200.Mat(Bf), nev=8)
    o2 = b200.gcg_solve(b200.Mat(pen.A), b200.Mat(pen.B), nev=8)
    assert o1["num_iter"] == o2["num_iter"] and np.array_equal(o1["eval"][:8], o2["eval"][:8])


def _golden_case(golden, m, nev, argv=()):
    want = [str(a) for a in argv]
    for c in golden["cases"]:
        if c["generator"] == "p1_fem_kuhn" and c["args"] == {"m": m} and c["nev"] == nev and c.get("argv", []) == want:
            return c
    raise KeyError((m, nev, argv))


def test_device_gcg_headline_block_structure(b200, refmod, golden):
    """nev = 200 (nevMax 400, block_size 40, projected problems of order up to 480) on a small lattice:
    the shapes of the headline run -- contraction lengths far beyond the kernels' tile rings, several
    column tiles, locked columns shifting the block offsets -- which the nev = 10 cases never reach.
    Against the live reference: iteration count within 1, eigenvalues 1e-10."""
    pen = P.p1_fem_kuhn(24)
    A = b200.Mat(pen.A); B = b200.Mat(pen.B)
    o = b200.gcg_solve(A, B, nev=200)
    assert o["nev_conv"] >= 200 and o["num_iter"] < 60, (o["nev_conv"], o["num_iter"])
    ev = o["eval"][:200]
    assert np.all(np.diff(ev) > -1e-9 * ev[-1]) and ev[0] > 25.0
    case = _golden_case(golden, 24, 200)                 # the reference's recorded run of the same pencil
    assert abs(o["num_iter"] - case["num_iter"]) <= ITER_TOL, (o["num_iter"], case["num_iter"])
    k = min(o["nev_conv"], case["nev_conv"])
    assert rel(o["eval"][:k], np.array(case["eval"][:k])) < 1e-10
    if refmod is not None:
        r = refmod.gcg_solve(pen.A, pen.B, nev=200, want_evec=False)
        assert abs(o["num_iter"] - r["num_iter"]) <= ITER_TOL, (o["num_iter"], r["num_iter"])
        k = min(o["nev_conv"], r["nev_conv"])
        assert rel(o["eval"][:k], r["eval"][:k]) < 1e-10


def test_device_gcg_moving_window_and_shift(b200, refmod):
    """nevInit < nevMax (reference src/ops_eig_sol_gcg.c:1400-1428) and the shifted inner
    solve (compW_cg_shift, reference :482-492): same eigenvalues as the plain run, and -- with the
    live reference on the box -- as the reference run with the same -nevMax / -nevInit."""
    pen = P.p1_fem_kuhn(12)
    A = b200.Mat(pen.A); B = b200.Mat(pen.B)
    base = b200.gcg_solve(A, B, nev=30)
    win = b200.gcg_solve(A, B, nev=30, nev_max=48, nev_init=18)
    assert win["nev_conv"] >= 30
    assert rel(win["eval"][:30], base["eval"][:30]) < 1e-9
    sh = b200.gcg_solve(A, B, nev=10, compW_cg_shift=5.0)
    assert sh["nev_conv"] >= 10
    assert rel(sh["eval"][:10], base["eval"][:10]) < 1e-9
    if refmod is not None:
        r = refmod.gcg_solve(pen.A, pen.B, nev=10, want_evec=False, argv=("-gcge_compW_cg_shift", 5.0))
        assert abs(sh["num_iter"] - r["num_iter"]) <= ITER_TOL, (sh["num_iter"], r["num_iter"])
        assert rel(sh["eval"][:10], r["eval"][:10]) < 1e-10


@pytest.mark.parametrize("gen_args,nev,nev_max,nev_init", [
    (("p1_fem_kuhn", {"m": 14}), 40, 64, 24),       # block_size 8: several growth steps of the window
    (("p1_fem_kuhn", {"m": 12}), 30, 48, 18),       # block_size 6
])
def test_device_gcg_moving_window_vs_live_reference(b200, refmod, gen_args, nev, nev_max, nev_init):
    """Moving window (SURVEY 8f row 3, reference src/ops_eig_sol_gcg.c:1281-1283,1400-1428): X starts with
    nevInit < nevMax columns and grows by P and W every time the window has converged.  Same
    -nevMax / -nevInit to the live reference: eigenvalues 1e-10, residual test, and the iteration count
    within 1 of the reference's own spread over OpenMP thread counts (its reductions reorder; these long
    runs move by up to 3 iterations between 1, 2, 4 and 8 threads).  Without oracle/_ref: the spread of the
    reference's recorded runs (tests/golden/reference_iteration_spread.json), eigenvalues against the pencil's own."""
    pen = getattr(P, gen_args[0])(**gen_args[1])
    if refmod is not None:
        runs = reference_runs_over_threads(
            refmod, lambda: refmod.gcg_solve(pen.A, pen.B, nev=nev, nev_max=nev_max, nev_init=nev_init, want_evec=False))
    else:
        runs = recorded_reference_runs(gen_args[0], gen_args[1], nev, nev_max, nev_init)
    its = [r["num_iter"] for r in runs]
    r = runs[0]
    A = b200.Mat(pen.A); B = None if pen.B is None else b200.Mat(pen.B)
    o = b200.gcg_solve(A, B, nev=nev, nev_max=nev_max, nev_init=nev_init)
    assert o["nev_conv"] >= nev and r["nev_conv"] >= nev
    assert min(its) - ITER_TOL <= o["num_iter"] <= max(its) + ITER_TOL, (o["num_iter"], its)
    k = min(o["nev_conv"], r["nev_conv"])
    want = r["eval"][:k] if refmod is not None else pencil_eigenvalues(pen, k)
    assert rel(o["eval"][:k], want) < 1e-10
    ok, res = residual_test(pen, o["eval"][:k], o["evec_mv"].numpy(0, k))
    assert ok, res


def _warm_start_block(pen, nev, noise, seed=3):
    """approximate eigenvectors: the reference's converged ones plus relative noise"""
    import scipy.sparse.linalg as sla
    A = pen.A.to_scipy().tocsc(); Bm = None if pen.B is None else pen.B.to_scipy().tocsc()
    w, v = sla.eigsh(A, k=nev, M=Bm, sigma=0.0, which="LM")
    order = np.argsort(w)
    v = v[:, order]
    rng = np.random.default_rng(seed)
    v = v + noise * np.abs(v).max() * rng.standard_normal(v.shape)
    return np.asfortranarray(v)


@pytest.mark.parametrize("nev_given,noise", [(10, 1e-3), (6, 1e-6), (14, 1e-2)])
def test_device_gcg_warm_start_vs_live_reference(b200, refmod, drive_b200, golden, nev_given, noise):
    """Warm start (SURVEY 8f row 3, reference src/ops_eig_sol_gcg.c:107-109,140): the first nevGiven
    columns of evec hold approximate eigenvectors; InitializeX copies them into V, B-orthonormalises
    them and fills the rest of X with random columns.  Same given block to the live reference, to the
    device GCG (tier B) and to the reference's GCG over OPS_B200_Set (tier A): iteration counts
    within 1, eigenvalues 1e-10, and fewer iterations than the cold start.  Without oracle/_ref: the reference's
    recorded cold solve of this pencil (golden case 4) -- its eigenvalues, and the warm start no slower (+1)."""
    pen = P.p1_fem_kuhn(12)
    nev = 10
    given = _warm_start_block(pen, nev_given, noise)
    if refmod is not None:
        cold = refmod.gcg_solve(pen.A, pen.B, nev=nev, want_evec=False)
        r = refmod.gcg_solve(pen.A, pen.B, nev=nev, want_evec=False, evec_given=given)
        assert r["nev_conv"] >= nev and r["num_iter"] <= cold["num_iter"]
    else:
        cold = r = golden["cases"][4]
        assert (r["generator"], r["args"], r["nev"]) == ("p1_fem_kuhn", {"m": 12}, nev)
    A = b200.Mat(pen.A); B = b200.Mat(pen.B)
    prm = b200.default_params(nev)
    evec = b200.MultiVec(pen.A.ncols, prm.nevMax)
    evec.upload(given, 0)
    o = b200.gcg_solve(A, B, nev=nev, evec=evec, nev_given=nev_given)
    assert o["nev_conv"] >= nev
    if refmod is not None:
        assert abs(o["num_iter"] - r["num_iter"]) <= ITER_TOL, (o["num_iter"], r["num_iter"])
    else:
        assert o["num_iter"] <= cold["num_iter"] + ITER_TOL, (o["num_iter"], cold["num_iter"])
    k = min(o["nev_conv"], r["nev_conv"])
    assert rel(o["eval"][:k], np.asarray(r["eval"][:k])) < 1e-10
    ok, res = residual_test(pen, o["eval"][:k], evec.numpy(0, k))
    assert ok, res
    if drive_b200 is not None:
        for tier in (0, 1):
            a = drive_b200(tier, pen.A, pen.B, nev=nev, evec_given=given)
            assert a["nev_conv"] >= nev
            assert abs(a["num_iter"] - r["num_iter"]) <= ITER_TOL, (tier, a["num_iter"], r["num_iter"])
            assert rel(a["eval"][:k], r["eval"][:k]) < 1e-10
