/* gcge_b200.h -- C ABI of the B200-native GCG hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b): plain pointers and sizes, no
 * C++ or torch types.  Every entry point names the reference interface it
 * replaces (file:line under the reference tree).  The OPS adaptor
 * gcge_b200/app/app_b200.c fills the reference's `struct OPS_`
 * (reference src/ops.h:43-152) with thin wrappers over these functions, so the
 * reference's GCG, ops_orth.c and ops_lin_sol.c can drive them unchanged
 * (INTEGRATION.md).
 *
 * Conventions (same as the reference's slots, reference src/ops.h:78-103):
 *   - start[0],end[0] index columns of the first multi-vector argument,
 *     start[1],end[1] of the second; half-open ranges.
 *   - inner_prod / qAp / coef / beta / eval are HOST pointers, column-major,
 *     owned by the caller; they are valid on return (the call synchronises).
 *   - matrices are borrowed, multi-vectors are created/destroyed by the caller.
 *   - all arithmetic is FP64, all indices are 32-bit int.
 * Multi-vectors live in HBM row-major (n x ld doubles, ld >= ncols); the
 * layout is never exposed: hosts see column-major through upload/download.
 *
 * Return value: 0 on success, non-zero on failure with a message available
 * from b200_last_error().  The reference's slots return void and abort() on
 * failure (reference app/app_ccs.c:53-55); the OPS adaptor reproduces that.
 * There is NO CPU fallback: without a CUDA device every call fails loudly.
 */
#ifndef GCGE_B200_H_
#define GCGE_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200_mat_ b200_mat; /* device CSR image of a CCSMAT (reference app/app_ccs.h:20-24) */
typedef struct b200_mv_  b200_mv;  /* device multi-vector; replaces LAPACKVEC (reference app/app_lapack.h:17-20) */

/* ---- runtime ------------------------------------------------------------ */
int  b200_init(int device);            /* select device, create streams/workspaces; idempotent */
void b200_finalize(void);
const char *b200_last_error(void);
int  b200_device_count(void);
int  b200_sync(void);                  /* cudaStreamSynchronize on the library stream */
double b200_wtime(void);               /* synchronising wall clock; replaces DefaultGetWtime, reference src/ops_multi_vec.c:45-56 */
long long b200_kernel_launches(void);  /* number of kernels this library launched since init */
/* CUDA-event stopwatch on the library stream (the stream every kernel is launched on):
 * start records an event, stop records a second one, synchronises and returns milliseconds */
int  b200_timer_start(void);
int  b200_timer_stop(double *ms);
/* measured FP64 tensor-core (DMMA m8n8k4) issue ceiling of this GPU, TFLOP/s: the roofline
 * denominator of the Gram / LinearComb kernels */
int  b200_measure_dmma_peak(double *tflops);
/* out[0..4] TFLOP/s: DMMA with one shared operand pair; DMMA with the 2 A x 8 B fragment pattern of the
 * Gram / LinearComb inner loops in two issue orders; the plain DFMA pipe; DMMA and DFMA interleaved. */
int  b200_measure_fp64_peaks(double *out5);
/* overwrite a buffer larger than L2 so the next timed kernel starts cold */
int  b200_flush_l2(void);
/* Per-kernel-class device timing for bench.py's roofline: while enabled, every kernel call of
 * the library is bracketed by two CUDA events on the library stream and booked, with its
 * ALGORITHMIC bytes and flops (SURVEY.md 8d), to one of b200_prof_classes() classes ("spmm",
 * "gram", "lincomb", "axpby", "dots", "bpcg_fused", "orth_panel", "syev_jacobi", "small_dense").
 * enable(1) resets the counters; get() synchronises and returns the totals since then. */
/* page-lock / unlock a caller-owned host buffer so uploads from it run at full PCIe speed */
int  b200_host_register(void *host, unsigned long long bytes);
int  b200_host_unregister(void *host);
int  b200_prof_enable(int on);
int  b200_prof_classes(void);
int  b200_prof_get(int cls, const char **name, double *ms, long long *calls, double *bytes, double *flops);
/* stream time between the end of the previous profiled call and the start of the calls of class cls
 * (unclassified kernels, copies, collectives, idle time): where the step's time outside the classes goes */
int  b200_prof_get_gap(int cls, double *ms);

/* Run-time switches (diagnosis and A/B measurements; DESIGN.md lists them).  Each one is read ONCE from the
 * environment variable B200_<NAME> when the library initialises; afterwards b200_option_set changes it.  The OPS
 * adaptor maps the command-line options -b200_<name> <int> onto them through the reference's
 * GetOptionFromCommandLine (reference src/ops_multi_vec.c:58-95): B200_SetOptionsFromCommandLine, app_b200.h. */
int  b200_option_count(void);
const char *b200_option_name(int i);
int  b200_option_set(const char *name, int value);
int  b200_option_get(const char *name, int *value);

/* ---- on-disk matrices (SURVEY.md 8f) ---------------------------------------------------------
 * MatrixMarket "matrix coordinate real|integer|pattern general|symmetric|skew-symmetric" into CCS
 * arrays (malloc'ed; release with b200_ccs_free): rows ascending inside every column, symmetric
 * files expanded to both triangles.  Host only. */
int  b200_ccs_read_matrix_market(const char *path, int *nrows, int *ncols, int **j_col, int **i_row, double **data);
/* PETSc binary matrix (MatView/MatLoad format, big-endian AIJ): the files the reference's SLEPc driver reads */
int  b200_ccs_read_petsc_binary(const char *path, int *nrows, int *ncols, int **j_col, int **i_row, double **data);
void b200_ccs_free(int *j_col, int *i_row, double *data);

/* ---- several GPUs: one process per GPU, 1-D contiguous row blocks (SURVEY.md 8e) -----------
 * The scheme of the reference's MPI back ends (every rank owns a row slab of A, B and of
 * every multi-vector; reference app/app_slepc.c:610-634, app/app_phg.c:292-357,
 * src/ops_multi_vec.c:214): rank g owns rows [floor(g n/G), floor((g+1) n/G)).  After
 * b200_comm_init every call below keeps its GLOBAL meaning -- matrices are created from the
 * global CCS arrays, multi-vectors are created / uploaded / downloaded with global shapes, Gram
 * blocks and dots come back globally reduced and identical on every rank -- while each process
 * stores and computes its slab only.  SpMM halo rows travel by ncclSend/ncclRecv over NVLink,
 * reductions by ncclAllReduce; the small projected problem is replicated.  All ranks must make
 * the same calls in the same order (they do: the host control flow is replicated, exactly like
 * the reference under MPI).  Bootstrap: rank 0 obtains the 128-byte id, the host program ships
 * it to the other ranks (bench.py: torch.distributed), every rank calls b200_comm_init. */
int  b200_comm_unique_id(char *id128);
int  b200_comm_init(int rank, int nranks, const char *id128);
int  b200_comm_finalize(void);
int  b200_comm_rank(void);
int  b200_comm_size(void);
void b200_partition_range(long long n, int rank, int nranks, long long *lo, long long *hi);
/* host-only: lay out as rank `rank` of `nranks` without a communicator (partition tests) */
int  b200_comm_set_layout(int rank, int nranks);
/* host-only view of one rank's partition plan: local CSR slab with remapped columns (banded
 * matrices, halo_contiguous: column = global - row0, the halo being the halo_below rows in front
 * of and the rest behind the local rows; otherwise local column = global - row0 and halo column
 * = nrows_local + slot), the sorted halo list, the neighbour
 * ranks and, per neighbour, the halo slots received from it and the local rows sent to it */
typedef struct b200_plan_ b200_plan;
int  b200_plan_create(int nrows, int ncols, const int *j_col, const int *i_row, const double *data,
                      int rank, int nranks, b200_plan **out);
int  b200_plan_sizes(const b200_plan *p, int *row0, int *nrows_local, int *nnz_local, int *nhalo, int *nnbr,
                     int *nsend, int *symmetric, int *halo_contiguous, int *halo_below);
int  b200_plan_copy(const b200_plan *p, int *rp, int *ci, double *va, int *halo_cols, int *nbr,
                    int *recv_off, int *send_off, int *send_rows);
int  b200_plan_destroy(b200_plan *p);

/* ---- matrix: replaces the host CCSMAT the reference's drivers build directly
 *      (reference test/test_app_ccs.c:99-102, :142-184) ------------------------ */
int b200_mat_create_from_ccs(int nrows, int ncols, const int *j_col, const int *i_row,
                             const double *data, b200_mat **out);
/* Several ranks, large matrices: every rank hands over ONLY its own row block [row0, row0 + nrows_local) =
 * b200_partition_range(nrows_global, rank, nranks) as CSR-style arrays (rp[nrows_local + 1], global column indices
 * ascending inside a row) -- for the symmetric matrices of the eigenproblem exactly the CCS arrays of those columns.
 * What the reference's distributed back ends do (every rank owns its rows only, app/app_phg.c:292-357); collective.
 * Banded matrices only; the matrix is taken to be symmetric (the reference assumes that for every matrix,
 * app/app_ccs.c:140-150).  Works on one rank too (the block is then the whole matrix). */
int b200_mat_create_from_local_rows(int nrows_global, int row0, int nrows_local, const int *rp, const int *ci,
                                    const double *va, b200_mat **out);
int b200_mat_destroy(b200_mat *A);
int b200_mat_shape(const b200_mat *A, int *nrows, int *ncols, int *nnz);
/* gather the device matrix back to CCS arrays; bit-exact round trip (SURVEY §8c) */
int b200_mat_to_ccs(const b200_mat *A, int *j_col, int *i_row, double *data);
/* several ranks: this rank's row block and its CSR slab read back from the device with GLOBAL
 * column indices; the slabs of all ranks, concatenated in rank order, are the CSR image of the
 * whole matrix (== the CCS arrays of its transpose) bit for bit */
int b200_mat_local_range(const b200_mat *A, int *row0, int *nrows_local, int *nnz_local, int *nhalo);
int b200_mat_local_csr(const b200_mat *A, int *rp, int *ci, double *va);
/* Y = alpha X + beta Y; the pattern of X must be a subset of Y's (checked before Y is touched); slot MatAxpby,
 * reference src/ops.h:52, used for the in-place shift A + sigma B, src/ops_eig_sol_gcg.c:594-602 */
int b200_mat_axpby(double alpha, const b200_mat *X, double beta, b200_mat *Y);
/* which SpMM storage the matrix got (diagnosis / tests): number of diagonals of its diagonal image (0: CSR
 * kernels only), the lattice strides recognised in it (0, 0: none; else row = i + s1 (j + (s2/s1) k)), and whether
 * it is a constant stencil on that lattice (the same coefficients in every row: no matrix values are streamed) */
int b200_mat_storage(const b200_mat *A, int *dia_nd, int *lat_s1, int *lat_s2, int *lat_const);

/* ---- multi-vector life cycle: reference app/app_ccs.c:40-49 (MultiVecCreateByMat),
 *      app/app_lapack.c:230-286 (create/destroy) ------------------------------ */
int b200_mv_create(int nrows, int ncols, b200_mv **out);   /* zero-filled */
int b200_mv_destroy(b200_mv *x);
int b200_mv_shape(const b200_mv *x, int *nrows, int *ncols);   /* global shape */
int b200_mv_local_range(const b200_mv *x, int *row0, int *nrows_local);
/* non-owning view of columns [start,end); destroy with b200_mv_destroy.  Replaces
 * GetVecFromMultiVec / RestoreVecForMultiVec, reference app/app_lapack.c:262-286 */
int b200_mv_view(const b200_mv *x, int start, int end, b200_mv **view);
/* host column-major (ld >= nrows, GLOBAL shape) <-> device columns [start,end); on several ranks
 * each process moves its own rows [row0, row0 + nrows_local) of the host block only */
int b200_mv_upload(b200_mv *x, int start, int end, const double *host, int ld);
int b200_mv_download(const b200_mv *x, int start, int end, double *host, int ld);
/* same, but `host` holds this rank's row block only (nrows_local rows, ld >= nrows_local) */
int b200_mv_upload_local(b200_mv *x, int start, int end, const double *host, int ld);
int b200_mv_download_local(const b200_mv *x, int start, int end, double *host, int ld);
/* x[row,col] = rand()/(RAND_MAX+1.0), column-major fill order, consuming the process's
 * glibc rand() stream exactly like reference app/app_lapack.c:322-333.  The values are
 * generated ON DEVICE by jump-ahead of glibc's lagged-Fibonacci recurrence from the live
 * generator state; on return the process's generator has advanced by nrows*(end-start) calls. */
int b200_mv_set_random(b200_mv *x, int start, int end);
/* host-only self check of that jump-ahead against glibc's rand() itself (needs no device) */
int b200_rand_selfcheck(unsigned long long steps);

/* ---- slots --------------------------------------------------------------- */
/* y[:,s1:e1] = A x[:,s0:e0]; A == NULL => copy.  Replaces MatDotMultiVec,
 * reference app/app_ccs.c:50-139 (kernel :116-131); also serves MatTransDotMultiVec
 * (reference app/app_ccs.c:140-150, symmetry assumed there; here `trans` != 0
 * multiplies by the true transpose). */
int b200_mat_dot_multivec(const b200_mat *A, int trans, const b200_mv *x, b200_mv *y,
                          const int *start, const int *end);
/* y[:,s1:e1] = alpha x[:,s0:e0] + beta y[:,s1:e1]; x == NULL => scale; beta == 0 =>
 * overwrite.  Replaces MultiVecAxpby, reference app/app_lapack.c:334-395 */
int b200_mv_axpby(double alpha, const b200_mv *x, double beta, b200_mv *y,
                  const int *start, const int *end);
/* y[:,s1:e1] = x[:,s0:e0] coef + y diag(beta).  coef host col-major (e0-s0)x(e1-s1), ldc;
 * beta == NULL => 0, incb == 0 => one scalar, else beta[incb*col]; x == NULL or
 * coef == NULL => scaling only.  Replaces MultiVecLinearComb, reference app/app_lapack.c:463-534 */
int b200_mv_linear_comb(const b200_mv *x, b200_mv *y, const int *start, const int *end,
                        const double *coef, int ldc, const double *beta, int incb);
/* inner_prod = x[:,s0:e0]^T y[:,s1:e1]; nsd: 'N' full, 'S' symmetric (computed once,
 * mirrored), 'D' diagonal only into inner_prod[ld*idx].  Replaces
 * MultiVecLocalInnerProd / MultiVecInnerProd, reference app/app_lapack.c:299-321 (via
 * DenseMatQtAP :24-183) and src/ops_multi_vec.c:202-230. */
int b200_mv_inner_prod(char nsd, const b200_mv *x, const b200_mv *y,
                       const int *start, const int *end, double *inner_prod, int ld);
/* qAp = Q[:,s0:e0]^T A P[:,s1:e1]; leaves A P[:,s1:e1] in ws[:,0:e1-s1] (callers rely on
 * it, reference src/ops_orth.c:315-323); ntsdQAP 'T' stores the transpose.  A == NULL =>
 * plain inner product, ws untouched.  Replaces DefaultMultiVecQtAP, reference
 * src/ops_multi_vec.c:351-411. */
int b200_mv_qtap(char ntsA, char ntsdQAP, const b200_mv *Q, const b200_mat *A, const b200_mv *P,
                 const int *start, const int *end, double *qAp, int ldQAP, b200_mv *ws);

/* ---- fused L3 providers (SURVEY §7 tier B) -------------------------------- */
/* B-orthonormalise x[:,start_x:*end_x] against x[:,0:start_x] and itself, dropping
 * dependent columns (shrinks *end_x).  Replaces ModifiedGramSchmidt, reference
 * src/ops_orth.c:203-393 (+ OrthSelf :45-118).  ws: at least min(block,*end_x-start_x)
 * columns of workspace. */
typedef struct b200_orth_params_ {
	int    block_size;     /* <=0: half of the block, reference src/ops_orth.c:275-278 */
	int    max_reorth;
	double orth_zero_tol;
	double reorth_tol;     /* reference default 50*DBL_EPSILON, src/ops_orth.c:401-404 */
} b200_orth_params;
int b200_mv_orth(b200_mv *x, int start_x, int *end_x, const b200_mat *B,
                 const b200_orth_params *prm, b200_mv *ws);

/* The same through BinaryGramSchmidt with OrthSelfEVP leaves (recursive halving; a leaf is orthonormalised through the
 * eigen-decomposition of its Gram matrix, on the device Jacobi kernel).  Replaces BinaryGramSchmidt / OrthBinary /
 * OrthSelfEVP, reference src/ops_orth.c:518-600, :415-516, :122-201 (-gcge_*_orth_method bgs).  ws: as many columns as
 * the widest block it has to hold (the reference's rule: end_x - start_x). */
int b200_mv_orth_bgs(b200_mv *x, int start_x, int *end_x, const b200_mat *B,
                     const b200_orth_params *prm, b200_mv *ws);

/* Block CG on A x = b for columns b[:,s0:e0], x[:,s1:e1], per-column convergence
 * masks, device-resident scalars.  shift != 0 solves (A + shift*B) x = b (B may be
 * NULL => identity).  Replaces BlockPCG, reference src/ops_lin_sol.c:140-437, and the
 * shifted operator MatDotMultiVecShift, reference src/ops_eig_sol_gcg.c:63-96. */
typedef struct b200_bpcg_params_ {
	int    max_iter;
	double rate;
	double tol;
	int    tol_type;       /* 0 "abs", 1 "rel" (reference src/ops_lin_sol.c:175-200) */
	double shift;
} b200_bpcg_params;
/* NOTE: with shift != 0 and B != NULL the right-hand side columns b[:,s0:e0] are used as workspace once the
 * initial residual has been formed (they hold B p afterwards) -- exactly what the reference's shifted operator
 * does with the block GCG hands it (src/ops_eig_sol_gcg.c:63-96); callers that need b afterwards keep a copy. */
int b200_block_pcg(const b200_mat *A, const b200_mat *B, b200_mv *b, b200_mv *x,
                   const int *start, const int *end, const b200_bpcg_params *prm,
                   b200_mv *ws_r, b200_mv *ws_p, b200_mv *ws_w, int *niter, double *residual);
/* The same with a preconditioner: pc = 0 none (== b200_block_pcg), 1 point Jacobi with D = diag(A + shift B)
 * (B NULL: diag(A) + shift).  rho = r^T D^-1 r drives alpha and beta, p = D^-1 r + beta p; the residual norms, the
 * stop test and *residual stay on ||r||_2, so rate / tol mean what they mean without it.  Fails, with x untouched,
 * when a row of A (or B) stores no diagonal entry or the diagonal of A + shift B is not > 0. */
int b200_block_pcg_pc(const b200_mat *A, const b200_mat *B, b200_mv *b, b200_mv *x,
                      const int *start, const int *end, const b200_bpcg_params *prm, int pc,
                      b200_mv *ws_r, b200_mv *ws_p, b200_mv *ws_w, int *niter, double *residual);

/* All eigenpairs of the symmetric n x n host matrix a (column-major, lda; upper or lower
 * triangle both read), ascending; on-device parallel-order Jacobi.  Replaces the dsyevx
 * call of the projected problem, reference src/ops_eig_sol_gcg.c:1201-1204. */
int b200_dense_syev(int n, const double *a, int lda, double *w, double *z, int ldz,
                    int *sweeps);

/* Whole GCG solve (reference src/ops_eig_sol_gcg.c:1253-1558) with the parameters of
 * GCGSolver (reference src/ops_eig_sol_gcg.h:26-52).  evec: n x nevMax multi-vector. */
typedef struct b200_gcg_params_ {
	int    nevMax, multiMax, nevInit, block_size, numIterMax;
	double gapMin;
	double tol[2];
	int    check_conv_max_num;
	int    initX_orth_block_size, initX_orth_max_reorth; double initX_orth_zero_tol;
	int    compP_orth_block_size, compP_orth_max_reorth; double compP_orth_zero_tol;
	int    compW_orth_block_size, compW_orth_max_reorth; double compW_orth_zero_tol;
	int    compW_cg_max_iter; double compW_cg_rate, compW_cg_tol; int compW_cg_tol_type;
	int    compW_cg_auto_shift; double compW_cg_shift;
	double compRR_tol;
	int    compW_cg_order;      /* 1: ComputeW; 2: ComputeW12 (W = [W1 W2], reference src/ops_eig_sol_gcg.c:697-923) */
	int    verbose;
	/* 0 "mgs" (b200_mv_orth), 1 "bgs" (b200_mv_orth_bgs): -gcge_{initX,compP,compW}_orth_method,
	 * reference src/ops_eig_sol_gcg.c:1757-1785 */
	int    initX_orth_method, compP_orth_method, compW_orth_method;
	/* preconditioner of the inner BlockPCG (b200_block_pcg_pc): 0 none (the reference's), 1 Jacobi with the sigma
	 * of each ComputeW / ComputeW12 call */
	int    compW_cg_pc;
} b200_gcg_params;
typedef struct b200_gcg_stats_ {
	int    numIter, nevConv;
	double time_total, initX, checkconv, compP, compRR, rr_eig, compRV, compW, linsol, compX;
	long long launches;
} b200_gcg_stats;
void b200_gcg_default_params(int nevConv, b200_gcg_params *prm); /* defaults of reference test/test_eig_sol_gcg.c:33-115 */
/* mv_ws: NULL, or the four workspaces of EigenSolverSetup_GCG (reference
 * src/ops_eig_sol_gcg.c:1561: [0] nevMax+2*block_size columns, [1..3] block_size columns).
 * nevGiven > 0: warm start from the first nevGiven columns of evec (reference :107-109).
 * The library keeps one more buffer of the shape of mv_ws[0] between solves ([X P W] is double-buffered so
 * that ComputeX, reference :458-471, is a pointer swap) and a block_size-wide block for the unknowns of the inner
 * solve; b200_finalize or b200_gcg_free_cache releases them. */
void b200_gcg_free_cache(void);
int  b200_gcg_solve(const b200_mat *A, const b200_mat *B, double *eval, b200_mv *evec,
                    int nevGiven, int *nevConv, const b200_gcg_params *prm, b200_mv **mv_ws,
                    b200_gcg_stats *stats);

#ifdef __cplusplus
}
#endif
#endif /* GCGE_B200_H_ */
