"""ctypes harness over include/gcge_b200.h (tests and bench only; no numerical code here).

Names and argument meaning follow the reference's OPS slots (reference src/ops.h:43-152):
``start``/``end`` are the 2-element column-range arrays, host results are column-major.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_LIB = None

c_int_p = C.POINTER(C.c_int)
c_dbl_p = C.POINTER(C.c_double)


class B200Error(RuntimeError):
    pass


def lib_path() -> Path:
    return _HERE / "lib" / "libgcge_b200.so"


class _OrthParams(C.Structure):
    _fields_ = [("block_size", C.c_int), ("max_reorth", C.c_int),
                ("orth_zero_tol", C.c_double), ("reorth_tol", C.c_double)]


class _BpcgParams(C.Structure):
    _fields_ = [("max_iter", C.c_int), ("rate", C.c_double), ("tol", C.c_double),
                ("tol_type", C.c_int), ("shift", C.c_double)]


class GCGParams(C.Structure):
    """b200_gcg_params (include/gcge_b200.h); mirrors GCGSolver, reference src/ops_eig_sol_gcg.h:26-52."""
    _fields_ = [("nevMax", C.c_int), ("multiMax", C.c_int), ("nevInit", C.c_int), ("block_size", C.c_int),
                ("numIterMax", C.c_int), ("gapMin", C.c_double), ("tol", C.c_double * 2),
                ("check_conv_max_num", C.c_int),
                ("initX_orth_block_size", C.c_int), ("initX_orth_max_reorth", C.c_int),
                ("initX_orth_zero_tol", C.c_double),
                ("compP_orth_block_size", C.c_int), ("compP_orth_max_reorth", C.c_int),
                ("compP_orth_zero_tol", C.c_double),
                ("compW_orth_block_size", C.c_int), ("compW_orth_max_reorth", C.c_int),
                ("compW_orth_zero_tol", C.c_double),
                ("compW_cg_max_iter", C.c_int), ("compW_cg_rate", C.c_double), ("compW_cg_tol", C.c_double),
                ("compW_cg_tol_type", C.c_int), ("compW_cg_auto_shift", C.c_int), ("compW_cg_shift", C.c_double),
                ("compRR_tol", C.c_double), ("compW_cg_order", C.c_int), ("verbose", C.c_int),
                ("initX_orth_method", C.c_int), ("compP_orth_method", C.c_int), ("compW_orth_method", C.c_int),
                ("compW_cg_pc", C.c_int)]


class _GCGStats(C.Structure):
    _fields_ = [("numIter", C.c_int), ("nevConv", C.c_int)] + \
               [(k, C.c_double) for k in ("time_total", "initX", "checkconv", "compP", "compRR", "rr_eig",
                                          "compRV", "compW", "linsol", "compX")] + \
               [("launches", C.c_longlong)]


def lib():
    """Load libgcge_b200.so; raises if it has not been built (no fallback)."""
    global _LIB
    if _LIB is None:
        p = lib_path()
        if not p.exists():
            raise B200Error(f"{p} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(there is no CPU fallback)")
        L = C.CDLL(str(p))
        L.b200_last_error.restype = C.c_char_p
        L.b200_wtime.restype = C.c_double
        L.b200_kernel_launches.restype = C.c_longlong
        L.b200_mv_axpby.argtypes = [C.c_double, C.c_void_p, C.c_double, C.c_void_p, c_int_p, c_int_p]
        L.b200_mat_axpby.argtypes = [C.c_double, C.c_void_p, C.c_double, C.c_void_p]
        L.b200_mv_linear_comb.argtypes = [C.c_void_p, C.c_void_p, c_int_p, c_int_p, c_dbl_p, C.c_int, c_dbl_p, C.c_int]
        L.b200_mv_inner_prod.argtypes = [C.c_char, C.c_void_p, C.c_void_p, c_int_p, c_int_p, c_dbl_p, C.c_int]
        L.b200_mv_qtap.argtypes = [C.c_char, C.c_char, C.c_void_p, C.c_void_p, C.c_void_p, c_int_p, c_int_p,
                                   c_dbl_p, C.c_int, C.c_void_p]
        L.b200_mat_dot_multivec.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, c_int_p, c_int_p]
        L.b200_mv_upload.argtypes = [C.c_void_p, C.c_int, C.c_int, c_dbl_p, C.c_int]
        L.b200_mv_download.argtypes = [C.c_void_p, C.c_int, C.c_int, c_dbl_p, C.c_int]
        L.b200_mv_upload_local.argtypes = [C.c_void_p, C.c_int, C.c_int, c_dbl_p, C.c_int]
        L.b200_mv_download_local.argtypes = [C.c_void_p, C.c_int, C.c_int, c_dbl_p, C.c_int]
        L.b200_mv_local_range.argtypes = [C.c_void_p, c_int_p, c_int_p]
        L.b200_mv_set_random.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.b200_mv_create.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.b200_mv_destroy.argtypes = [C.c_void_p]
        L.b200_mat_create_from_ccs.argtypes = [C.c_int, C.c_int, c_int_p, c_int_p, c_dbl_p, C.POINTER(C.c_void_p)]
        L.b200_mat_destroy.argtypes = [C.c_void_p]
        L.b200_mat_to_ccs.argtypes = [C.c_void_p, c_int_p, c_int_p, c_dbl_p]
        L.b200_mat_shape.argtypes = [C.c_void_p, c_int_p, c_int_p, c_int_p]
        L.b200_mv_orth.argtypes = [C.c_void_p, C.c_int, c_int_p, C.c_void_p, C.POINTER(_OrthParams), C.c_void_p]
        L.b200_block_pcg.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, c_int_p, c_int_p,
                                     C.POINTER(_BpcgParams), C.c_void_p, C.c_void_p, C.c_void_p, c_int_p, c_dbl_p]
        L.b200_block_pcg_pc.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, c_int_p, c_int_p,
                                        C.POINTER(_BpcgParams), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, c_int_p, c_dbl_p]
        L.b200_dense_syev.argtypes = [C.c_int, c_dbl_p, C.c_int, c_dbl_p, c_dbl_p, C.c_int, c_int_p]
        L.b200_prof_get.argtypes = [C.c_int, C.POINTER(C.c_char_p), c_dbl_p, C.POINTER(C.c_longlong), c_dbl_p, c_dbl_p]
        L.b200_host_register.argtypes = [C.c_void_p, C.c_ulonglong]
        L.b200_host_unregister.argtypes = [C.c_void_p]
        L.b200_measure_dmma_peak.argtypes = [c_dbl_p]
        L.b200_gcg_default_params.argtypes = [C.c_int, C.POINTER(GCGParams)]
        L.b200_gcg_default_params.restype = None
        L.b200_gcg_solve.argtypes = [C.c_void_p, C.c_void_p, c_dbl_p, C.c_void_p, C.c_int, c_int_p,
                                     C.POINTER(GCGParams), C.POINTER(C.c_void_p), C.POINTER(_GCGStats)]
        _LIB = L
    return _LIB


def _chk(rc: int):
    if rc != 0:
        raise B200Error(lib().b200_last_error().decode())


def init(device: int = -1):
    _chk(lib().b200_init(int(device)))


def device_count() -> int:
    return lib().b200_device_count()


def sync():
    _chk(lib().b200_sync())


def wtime() -> float:
    return lib().b200_wtime()


def kernel_launches() -> int:
    return lib().b200_kernel_launches()


def timer_start():
    _chk(lib().b200_timer_start())


def timer_stop() -> float:
    ms = C.c_double(0)
    _chk(lib().b200_timer_stop(C.byref(ms)))
    return ms.value


def flush_l2():
    _chk(lib().b200_flush_l2())


def prof_enable(on: bool = True):
    _chk(lib().b200_prof_enable(1 if on else 0))


def prof_report() -> dict:
    """{class: {ms, calls, bytes, flops}} since prof_enable(True) (device time from CUDA events
    on the library stream, algorithmic bytes/flops of SURVEY.md 8d)."""
    out = {}
    for c in range(lib().b200_prof_classes()):
        name = C.c_char_p(); ms = C.c_double(); calls = C.c_longlong(); by = C.c_double(); fl = C.c_double()
        _chk(lib().b200_prof_get(c, C.byref(name), C.byref(ms), C.byref(calls), C.byref(by), C.byref(fl)))
        gap = C.c_double()
        _chk(lib().b200_prof_get_gap(c, C.byref(gap)))
        out[name.value.decode()] = {"ms": ms.value, "calls": calls.value, "bytes": by.value, "flops": fl.value,
                                    "gap_before_ms": gap.value}
    return out


def gcg_free_cache():
    """Release the [X P W] buffer the solver keeps between solves (b200_gcg_free_cache)."""
    lib().b200_gcg_free_cache.restype = None
    lib().b200_gcg_free_cache()


def host_register(a: np.ndarray):
    _chk(lib().b200_host_register(a.ctypes.data, a.nbytes))


def host_unregister(a: np.ndarray):
    _chk(lib().b200_host_unregister(a.ctypes.data))


def measure_dmma_peak() -> float:
    t = C.c_double(0)
    _chk(lib().b200_measure_dmma_peak(C.byref(t)))
    return t.value


def _read_ccs_file(fn_name: str, path):
    from . import problems as P
    L = lib()
    fn = getattr(L, fn_name)
    fn.argtypes = [C.c_char_p, c_int_p, c_int_p, C.POINTER(c_int_p), C.POINTER(c_int_p), C.POINTER(c_dbl_p)]
    L.b200_ccs_free.argtypes = [c_int_p, c_int_p, c_dbl_p]
    L.b200_ccs_free.restype = None
    m, n = C.c_int(0), C.c_int(0)
    jc, ir, da = c_int_p(), c_int_p(), c_dbl_p()
    _chk(fn(str(path).encode(), C.byref(m), C.byref(n), C.byref(jc), C.byref(ir), C.byref(da)))
    try:
        j_col = np.ctypeslib.as_array(jc, shape=(n.value + 1,)).copy()
        nnz = int(j_col[-1])
        i_row = np.ctypeslib.as_array(ir, shape=(max(nnz, 1),)).copy()[:nnz]
        data = np.ctypeslib.as_array(da, shape=(max(nnz, 1),)).copy()[:nnz]
    finally:
        L.b200_ccs_free(jc, ir, da)
    return P.CCS(m.value, n.value, j_col.astype(np.int32), i_row.astype(np.int32), data.astype(np.float64))


def read_matrix_market(path):
    """On-disk matrix (MatrixMarket coordinate file) -> problems.CCS, through the library's own reader."""
    return _read_ccs_file("b200_ccs_read_matrix_market", path)


def read_petsc_binary(path):
    """On-disk matrix (PETSc binary AIJ, MatView/MatLoad format) -> problems.CCS."""
    return _read_ccs_file("b200_ccs_read_petsc_binary", path)


def partition_plan(ccs, rank: int, nranks: int) -> dict:
    """Host-only (no device): the row-block partition plan rank `rank` of `nranks` builds for a CCS
    matrix -- the same code path b200_mat_create_from_ccs runs on every rank (b200_plan_*)."""
    L = lib()
    j_col = np.ascontiguousarray(ccs.j_col, dtype=np.int32); i_row = np.ascontiguousarray(ccs.i_row, dtype=np.int32)
    data = np.ascontiguousarray(ccs.data, dtype=np.float64)
    h = C.c_void_p()
    L.b200_plan_create.argtypes = [C.c_int, C.c_int, c_int_p, c_int_p, c_dbl_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    L.b200_plan_sizes.argtypes = [C.c_void_p] + [c_int_p] * 9
    L.b200_plan_copy.argtypes = [C.c_void_p, c_int_p, c_int_p, c_dbl_p, c_int_p, c_int_p, c_int_p, c_int_p, c_int_p]
    L.b200_plan_destroy.argtypes = [C.c_void_p]
    _chk(L.b200_plan_create(ccs.nrows, ccs.ncols, _ip(j_col), _ip(i_row), _dp(data), rank, nranks, C.byref(h)))
    v = [C.c_int(0) for _ in range(9)]
    _chk(L.b200_plan_sizes(h, *[C.byref(x) for x in v]))
    row0, nloc, nnz, nhalo, nnbr, nsend, sym, contig, hbelow = [x.value for x in v]
    out = {"row0": row0, "nloc": nloc, "nnz": nnz, "nhalo": nhalo, "symmetric": bool(sym),
           "halo_contiguous": bool(contig), "halo_below": hbelow,
           "rp": np.zeros(nloc + 1, np.int32), "ci": np.zeros(max(nnz, 1), np.int32), "va": np.zeros(max(nnz, 1)),
           "halo_cols": np.zeros(max(nhalo, 1), np.int32), "nbr": np.zeros(max(nnbr, 1), np.int32),
           "recv_off": np.zeros(nnbr + 1, np.int32), "send_off": np.zeros(nnbr + 1, np.int32),
           "send_rows": np.zeros(max(nsend, 1), np.int32)}
    _chk(L.b200_plan_copy(h, _ip(out["rp"]), _ip(out["ci"]), _dp(out["va"]), _ip(out["halo_cols"]), _ip(out["nbr"]),
                          _ip(out["recv_off"]), _ip(out["send_off"]), _ip(out["send_rows"])))
    L.b200_plan_destroy(h)
    out["ci"] = out["ci"][:nnz]; out["va"] = out["va"][:nnz]; out["halo_cols"] = out["halo_cols"][:nhalo]
    out["nbr"] = out["nbr"][:nnbr]; out["send_rows"] = out["send_rows"][:nsend]
    return out


def comm_init_from_torch():
    """Bootstrap the library's NCCL communicator from an initialised torch.distributed group:
    rank 0 creates the unique id, broadcast_object_list ships it, every rank joins."""
    import torch.distributed as dist
    rank, world = dist.get_rank(), dist.get_world_size()
    buf = C.create_string_buffer(128)
    if rank == 0:
        _chk(lib().b200_comm_unique_id(buf))
    box = [bytes(buf.raw)]
    dist.broadcast_object_list(box, src=0)
    _chk(lib().b200_comm_init(rank, world, C.create_string_buffer(box[0], 128)))
    return rank, world


def comm_finalize():
    lib().b200_comm_finalize()


def libc_srand(seed: int = 0):
    """srand() of the process's glibc -- the generator b200_mv_set_random consumes, exactly as
    the reference's drivers do (reference test/test_eig_sol_gcg.c:87)."""
    C.CDLL("libc.so.6").srand(C.c_uint(seed))


def _ip(a):
    return None if a is None else a.ctypes.data_as(c_int_p)


def _dp(a):
    return None if a is None else a.ctypes.data_as(c_dbl_p)


def _se(start, end):
    return (C.c_int * 2)(*start), (C.c_int * 2)(*end)


class Mat:
    """Device image of a CCSMAT (reference app/app_ccs.h:20-24)."""

    def __init__(self, ccs):
        self.h = C.c_void_p()
        self.nrows, self.ncols = ccs.nrows, ccs.ncols
        j_col = np.ascontiguousarray(ccs.j_col, dtype=np.int32)
        i_row = np.ascontiguousarray(ccs.i_row, dtype=np.int32)
        data = np.ascontiguousarray(ccs.data, dtype=np.float64)
        _chk(lib().b200_mat_create_from_ccs(ccs.nrows, ccs.ncols, _ip(j_col), _ip(i_row), _dp(data), C.byref(self.h)))
        self.nnz = int(j_col[-1])

    @classmethod
    def from_local_rows(cls, nrows_global: int, row0: int, rp, ci, va):
        """This rank's row block only (b200_mat_create_from_local_rows): CSR-style arrays with global, ascending
        column indices -- for symmetric matrices the CCS arrays of the columns [row0, row0 + nrows_local)."""
        self = cls.__new__(cls)
        self.h = C.c_void_p()
        self.nrows = self.ncols = int(nrows_global)
        rp = np.ascontiguousarray(rp, dtype=np.int32); ci = np.ascontiguousarray(ci, dtype=np.int32)
        va = np.ascontiguousarray(va, dtype=np.float64)
        L = lib()
        L.b200_mat_create_from_local_rows.argtypes = [C.c_int, C.c_int, C.c_int, c_int_p, c_int_p, c_dbl_p, C.POINTER(C.c_void_p)]
        _chk(L.b200_mat_create_from_local_rows(int(nrows_global), int(row0), len(rp) - 1, _ip(rp), _ip(ci), _dp(va), C.byref(self.h)))
        self.nnz = int(rp[-1] - rp[0])
        return self

    def to_ccs(self):
        j_col = np.empty(self.ncols + 1, np.int32)
        i_row = np.empty(max(self.nnz, 1), np.int32)
        data = np.empty(max(self.nnz, 1), np.float64)
        _chk(lib().b200_mat_to_ccs(self.h, _ip(j_col), _ip(i_row), _dp(data)))
        return j_col, i_row[:self.nnz], data[:self.nnz]

    def storage(self) -> dict:
        """{'dia_nd', 'lat_s1', 'lat_s2', 'lat_const'}: which SpMM storage the matrix got (b200_mat_storage)."""
        v = [C.c_int(0) for _ in range(4)]
        lib().b200_mat_storage.argtypes = [C.c_void_p, c_int_p, c_int_p, c_int_p, c_int_p]
        _chk(lib().b200_mat_storage(self.h, *[C.byref(x) for x in v]))
        return {"dia_nd": v[0].value, "lat_s1": v[1].value, "lat_s2": v[2].value, "lat_const": v[3].value}

    def axpby(self, alpha, X, beta):
        """self = alpha*X + beta*self (slot MatAxpby)."""
        _chk(lib().b200_mat_axpby(alpha, X.h, beta, self.h))

    def close(self):
        if self.h:
            lib().b200_mat_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiVec:
    """Device multi-vector (replaces LAPACKVEC, reference app/app_lapack.h:17-20)."""

    def __init__(self, nrows: int, ncols: int):
        self.h = C.c_void_p()
        self.nrows, self.ncols = int(nrows), int(ncols)
        _chk(lib().b200_mv_create(self.nrows, self.ncols, C.byref(self.h)))

    @classmethod
    def from_numpy(cls, a: np.ndarray):
        mv = cls(a.shape[0], a.shape[1])
        mv.upload(a)
        return mv

    def upload(self, a: np.ndarray, start: int = 0):
        a = np.asfortranarray(a, dtype=np.float64)
        _chk(lib().b200_mv_upload(self.h, start, start + a.shape[1], _dp(a), max(a.shape[0], 1)))

    def numpy(self, start: int = 0, end: int | None = None) -> np.ndarray:
        end = self.ncols if end is None else end
        out = np.zeros((self.nrows, end - start), order="F")
        if out.size:
            _chk(lib().b200_mv_download(self.h, start, end, _dp(out), max(self.nrows, 1)))
        return out

    def local_range(self):
        """(row0, nrows_local): this rank's row block (the whole vector on one GPU)."""
        r0, nl = C.c_int(0), C.c_int(0)
        _chk(lib().b200_mv_local_range(self.h, C.byref(r0), C.byref(nl)))
        return r0.value, nl.value

    def numpy_local(self, start: int = 0, end: int | None = None, out: np.ndarray | None = None) -> np.ndarray:
        end = self.ncols if end is None else end
        _, nl = self.local_range()
        if out is None:
            out = np.zeros((nl, end - start), order="F")
        if out.size:
            _chk(lib().b200_mv_download_local(self.h, start, end, _dp(out), max(nl, 1)))
        return out

    def set_random(self, start: int, end: int):
        _chk(lib().b200_mv_set_random(self.h, start, end))

    def view(self, start: int, end: int) -> "MultiVec":
        """The columns [start, end) as a multi-vector of their own on the same storage (b200_mv_view; the reference's
        GetVecFromMultiVec, app/app_lapack.c:270-286).  The view must not outlive self."""
        v = MultiVec.__new__(MultiVec)
        v.h = C.c_void_p()
        v.nrows, v.ncols = self.nrows, int(end - start)
        _chk(lib().b200_mv_view(self.h, int(start), int(end), C.byref(v.h)))
        return v

    def close(self):
        if self.h:
            lib().b200_mv_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- slots (names follow the reference's OPS table) ------------------------------------------
def mat_dot_multivec(A, x, y, start, end, trans=False):
    s, e = _se(start, end)
    _chk(lib().b200_mat_dot_multivec(None if A is None else A.h, 1 if trans else 0, x.h, y.h, s, e))


def multivec_axpby(alpha, x, beta, y, start, end):
    s, e = _se(start, end)
    _chk(lib().b200_mv_axpby(alpha, None if x is None else x.h, beta, y.h, s, e))


def multivec_linear_comb(x, y, start, end, coef, ldc, beta, incb):
    s, e = _se(start, end)
    _chk(lib().b200_mv_linear_comb(None if x is None else x.h, y.h, s, e, _dp(coef), int(ldc), _dp(beta), int(incb)))


def multivec_inner_prod(nsd, x, y, start, end, ip, ld):
    s, e = _se(start, end)
    _chk(lib().b200_mv_inner_prod(nsd.encode(), x.h, y.h, s, e, _dp(ip), int(ld)))


def multivec_qtap(ntsA, ntsdQAP, Q, A, P, start, end, qAp, ld, ws):
    s, e = _se(start, end)
    _chk(lib().b200_mv_qtap(ntsA.encode(), ntsdQAP.encode(), Q.h, None if A is None else A.h, P.h, s, e,
                            _dp(qAp), int(ld), None if ws is None else ws.h))


def orth(x, start_x, end_x, B=None, ws=None, block_size=-1, max_reorth=2,
         orth_zero_tol=2 * np.finfo(float).eps, reorth_tol=50 * np.finfo(float).eps):
    """slot MultiVecOrth (reference src/ops.h:125-126); returns the new end."""
    prm = _OrthParams(block_size, max_reorth, orth_zero_tol, reorth_tol)
    own = ws is None
    if own:
        ws = MultiVec(x.nrows, min(max(end_x - start_x, 1), 128))
    e = C.c_int(end_x)
    _chk(lib().b200_mv_orth(x.h, start_x, C.byref(e), None if B is None else B.h, C.byref(prm), ws.h))
    if own:
        ws.close()
    return e.value


def orth_bgs(x, start_x, end_x, B=None, ws=None, block_size=-1, max_reorth=2,
             orth_zero_tol=2 * np.finfo(float).eps, reorth_tol=50 * np.finfo(float).eps):
    """slot MultiVecOrth with BinaryGramSchmidt / OrthSelfEVP (reference src/ops_orth.c:122-201,415-640); returns the new end."""
    prm = _OrthParams(block_size, max_reorth, orth_zero_tol, reorth_tol)
    own = ws is None
    if own:
        ws = MultiVec(x.nrows, max(end_x - start_x, 1))
    e = C.c_int(end_x)
    lib().b200_mv_orth_bgs.argtypes = lib().b200_mv_orth.argtypes
    _chk(lib().b200_mv_orth_bgs(x.h, start_x, C.byref(e), None if B is None else B.h, C.byref(prm), ws.h))
    if own:
        ws.close()
    return e.value


PRECONDITIONERS = {"none": 0, "jacobi": 1}


def block_pcg(A, b, x, start, end, B=None, max_iter=30, rate=1e-2, tol=1e-14, tol_type="abs", shift=0.0, ws=None,
              precond="none"):
    """slot MultiLinearSolver (reference src/ops.h:121-122); returns (niter, residual).  precond "jacobi": point
    Jacobi with D = diag(A + shift B) (b200_block_pcg_pc); "none" calls b200_block_pcg, the reference's BlockPCG."""
    if precond not in PRECONDITIONERS:
        raise B200Error(f"block_pcg: precond {precond!r} (one of {', '.join(PRECONDITIONERS)})")
    prm = _BpcgParams(max_iter, rate, tol, 1 if tol_type == "rel" else 0, shift)
    s, e = _se(start, end)
    k = end[0] - start[0]
    own = ws is None
    if own:
        ws = [MultiVec(x.nrows, max(k, 1)) for _ in range(3)]
    niter = C.c_int(0)
    res = C.c_double(0)
    try:
        if precond == "none":
            _chk(lib().b200_block_pcg(A.h, None if B is None else B.h, b.h, x.h, s, e, C.byref(prm),
                                      ws[0].h, ws[1].h, ws[2].h, C.byref(niter), C.byref(res)))
        else:
            _chk(lib().b200_block_pcg_pc(A.h, None if B is None else B.h, b.h, x.h, s, e, C.byref(prm),
                                         PRECONDITIONERS[precond], ws[0].h, ws[1].h, ws[2].h, C.byref(niter), C.byref(res)))
    finally:
        if own:
            for w in ws:
                w.close()
    return niter.value, res.value


def dense_syev(a: np.ndarray):
    """All eigenpairs of a symmetric matrix on device (replaces dsyevx, reference
    src/ops_eig_sol_gcg.c:1201).  Returns (w, z, sweeps)."""
    a = np.asfortranarray(a, dtype=np.float64)
    n = a.shape[0]
    w = np.zeros(n)
    z = np.zeros((n, n), order="F")
    sw = C.c_int(0)
    _chk(lib().b200_dense_syev(n, _dp(a), n, _dp(w), _dp(z), n, C.byref(sw)))
    return w, z, sw.value


def default_params(nev: int) -> GCGParams:
    p = GCGParams()
    lib().b200_gcg_default_params(int(nev), C.byref(p))
    return p


def gcg_workspace(n: int, p) -> list:
    """The four multi-vector workspaces of EigenSolverSetup_GCG (reference
    test/test_eig_sol_gcg.c:57-68: nevMax + 2 block_size, block_size, block_size, block_size
    columns), created by the caller before the solve like the reference's driver does."""
    return [MultiVec(n, p.nevMax + 2 * p.block_size)] + [MultiVec(n, p.block_size) for _ in range(3)]


def gcg_solve(A, B=None, nev=10, nev_max=0, block_size=0, nev_init=0, tol=None, max_iter=0, verbose=False,
              evec=None, seed=0, ws=None, nev_given=0, **overrides):
    """slot EigenSolver (reference src/ops.h:146-147) through b200_gcg_solve, with the driver
    defaults of reference test/test_eig_sol_gcg.c:33-115.  ``A``/``B`` are :class:`Mat`.
    Seeds glibc rand() like the reference driver unless seed is None.  ``nev_given`` > 0: warm start
    from the first nev_given columns of ``evec`` (reference src/ops_eig_sol_gcg.c:107-109)."""
    p = default_params(nev)
    if nev_max > 0:
        p.nevMax = nev_max
        p.block_size = (p.nevMax - nev) if nev < 30 else nev // 5
        p.nevInit = p.nevMax
    if block_size > 0:
        p.block_size = block_size
    if nev_init > 0:
        p.nevInit = min(nev_init, p.nevMax)
    if tol is not None:
        p.tol[0], p.tol[1] = tol
    if max_iter > 0:
        p.numIterMax = max_iter
    p.verbose = 1 if verbose else 0
    for k, v in overrides.items():
        setattr(p, k, v)
    own = evec is None
    if own:
        evec = MultiVec(A.nrows, p.nevMax)
    if seed is not None:
        libc_srand(seed)
    ev = np.zeros(p.nevMax)
    nconv = C.c_int(nev)
    st = _GCGStats()
    ws_c = None
    if ws is not None:
        ws_c = (C.c_void_p * 4)(*[w.h for w in ws])
    if nev_given > 0 and own:
        raise B200Error("gcg_solve: nev_given needs the caller's evec multi-vector")
    _chk(lib().b200_gcg_solve(A.h, None if B is None else B.h, _dp(ev), evec.h, int(nev_given), C.byref(nconv), C.byref(p),
                              ws_c, C.byref(st)))
    out = {"eval": ev, "num_iter": st.numIter, "nev_conv": nconv.value, "evec_mv": evec,
           "stats": {k: getattr(st, k) for k, _ in _GCGStats._fields_}}
    return out
