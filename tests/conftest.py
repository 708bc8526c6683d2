import ctypes as C
import json
import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


def _cuda_device_present() -> bool:
    try:
        from gcge_b200 import api
        return api.device_count() > 0
    except Exception:
        return False


@pytest.fixture(scope="session")
def b200():
    """The product library through its ctypes harness.  GPU tests FAIL (not skip) when the
    library or the device is missing: there is no fallback path to fall back to."""
    from gcge_b200 import api
    api.init(0)
    return api


@pytest.fixture(scope="session")
def refmod():
    """oracle/_ref (the unmodified reference).  Test infrastructure; None when the prebuilt
    library did not travel, in which case tests use the plain-C / numpy oracle and the
    committed golden vectors."""
    from oracle import ref
    if not ref.available():
        return None
    ref.set_threads(min(8, os.cpu_count() or 1))
    return ref


def reference_runs_over_threads(refmod, solve, threads=(1, 2, 4, 8)):
    """The reference's OpenMP reductions make its own outer-iteration count move with the thread count
    (profiles/reference_iteration_spread_r2.log: 69..72 on one moving-window case, 101..122 on another):
    run it at several thread counts and return the runs, so a test can hold the device solver to
    [min - 1, max + 1] of the reference's own spread instead of to one arbitrary member of it."""
    runs = []
    for t in threads:
        refmod.set_threads(t)
        runs.append(solve())
    refmod.set_threads(min(8, os.cpu_count() or 1))
    return runs


def recorded_reference_runs(generator, args, nev, nev_max, nev_init):
    """The reference's own runs of one solve at 1, 2, 4 and 8 OpenMP threads as recorded in
    tests/golden/reference_iteration_spread.json: what reference_runs_over_threads returns, for a checkout without
    oracle/_ref.  Dicts with num_iter and nev_conv; the record keeps no eigenvalues."""
    d = json.loads((ROOT / "tests" / "golden" / "reference_iteration_spread.json").read_text())
    key = (generator, args, nev, nev_max, nev_init)
    for r in d["runs"]:
        if (r["generator"], r["args"], r["nev"], r["nev_max"], r["nev_init"]) == key:
            return r["by_threads"]
    raise KeyError(f"no recorded reference run for {key}")


def pencil_eigenvalues(pen, k):
    """The k smallest eigenvalues of A x = lambda B x by shift-invert Lanczos (scipy): the eigenvalues a golden path
    compares with where the recorded reference runs kept none."""
    import scipy.sparse.linalg as sla
    A = pen.A.to_scipy().tocsc()
    B = None if pen.B is None else pen.B.to_scipy().tocsc()
    return np.sort(sla.eigsh(A, k=k, M=B, sigma=0.0, which="LM", tol=0)[0])


@pytest.fixture(scope="session")
def golden():
    return json.loads((ROOT / "tests" / "golden" / "gcg_reference.json").read_text())


@pytest.fixture(scope="session")
def drive_b200(refmod):
    """Loads the reference (global symbols), the OPS adaptor and the test driver that runs
    the reference's own GCG over OPS_B200_Set (oracle/drive_b200.c)."""
    if refmod is None:
        return None
    refmod.lib()
    ref_path = ROOT / "oracle" / "_ref" / "libgcge_ref.so"
    ops_path = ROOT / "gcge_b200" / "lib" / "libgcge_b200_ops.so"
    drv_path = ROOT / "oracle" / "_ref" / "libdrive_b200.so"
    if not (ops_path.exists() and drv_path.exists()):
        return None
    C.CDLL(str(ref_path), mode=C.RTLD_GLOBAL)
    C.CDLL(str(ROOT / "gcge_b200" / "lib" / "libgcge_b200.so"), mode=C.RTLD_GLOBAL)
    C.CDLL(str(ops_path), mode=C.RTLD_GLOBAL)
    drv = C.CDLL(str(drv_path))

    def run(tier, A, B=None, nev=10, nev_max=0, block_size=0, nev_init=0, tol=(1e-1, 1e-8), max_iter=500,
            argv=(), want_evec=False, evec_given=None):
        n = A.ncols
        nm = nev_max if nev_max > 0 else 2 * nev
        ev = np.zeros(nm)
        evec = np.zeros((n, nm), order="F") if want_evec else None
        it = C.c_int(0); nc = C.c_int(0); secs = C.c_double(0)
        args = [b"drv"] + [str(a).encode() for a in argv]
        argv_c = (C.c_char_p * len(args))(*args)
        ip = lambda a: None if a is None else a.ctypes.data_as(C.POINTER(C.c_int))
        dp = lambda a: None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))
        drv.drive_gcg_b200(int(tier), n, ip(A.j_col), ip(A.i_row), dp(A.data),
                           ip(None if B is None else B.j_col), ip(None if B is None else B.i_row),
                           dp(None if B is None else B.data),
                           int(nev), int(nev_max), int(block_size), int(nev_init),
                           C.c_double(tol[0]), C.c_double(tol[1]), int(max_iter),
                           len(args), argv_c, 1, dp(ev), dp(evec), C.byref(it), C.byref(nc), C.byref(secs),
                           0 if evec_given is None else int(evec_given.shape[1]),
                           dp(None if evec_given is None else np.asfortranarray(evec_given, dtype=np.float64)))
        return {"eval": ev, "evec": evec, "num_iter": it.value, "nev_conv": nc.value, "seconds": secs.value}

    def block_amg(A_levels, P_levels, b, x, max_iter, rate, tol):
        """the reference's BlockAMG unchanged over OPS_B200_Set (oracle/drive_b200.c: drive_block_amg_b200);
        A_levels / P_levels: problems.CCS per level (P rectangular n_l x n_{l+1}); x updated in place"""
        L = len(A_levels)
        ipp, dpp = C.POINTER(C.c_int), C.POINTER(C.c_double)
        n_l = (C.c_int * L)(*[a.ncols for a in A_levels])
        mk = lambda typ, arrs: (typ * L)(*arrs)
        Aj = mk(ipp, [a.j_col.ctypes.data_as(ipp) for a in A_levels]); Ai = mk(ipp, [a.i_row.ctypes.data_as(ipp) for a in A_levels])
        Ad = mk(dpp, [a.data.ctypes.data_as(dpp) for a in A_levels])
        Pj = mk(ipp, [p.j_col.ctypes.data_as(ipp) for p in P_levels] + [None]); Pi = mk(ipp, [p.i_row.ctypes.data_as(ipp) for p in P_levels] + [None])
        Pd = mk(dpp, [p.data.ctypes.data_as(dpp) for p in P_levels] + [None])
        mi = (C.c_int * len(max_iter))(*max_iter); ra = (C.c_double * len(rate))(*rate); to = (C.c_double * len(tol))(*tol)
        drv.drive_block_amg_b200(L, n_l, Aj, Ai, Ad, Pj, Pi, Pd, int(x.shape[1]), b.ctypes.data_as(dpp), x.ctypes.data_as(dpp), mi, ra, to)
        return x

    run.block_amg = block_amg
    return run
