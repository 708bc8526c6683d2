/* b200_dev.h -- the thin C layer between the host-side C drivers (b200_orth.c,
 * b200_bpcg.c, b200_gcg.c) and the CUDA kernels.  Everything here takes raw DEVICE
 * pointers to row-major blocks (pointer to the first element, leading dimension) and
 * only enqueues work on the library stream; nothing synchronises unless it says so.
 * Public, reference-facing surface: include/gcge_b200.h.
 */
#ifndef B200_DEV_H_
#define B200_DEV_H_

#include <stddef.h>
#include "gcge_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Multi-GPU (b200_comm.cu): every rank owns the row block [row0, row0 + nrows) of a matrix
 * with nrows_global rows.  nrows / ncols / nnz below are LOCAL; column indices of the local
 * CSR are remapped.  Banded matrices (halo_contiguous): column c becomes c - row0, so the halo
 * is the two row ranges [-halo_below, 0) and [nrows, nrows + nhalo - halo_below) around the
 * local rows -- the x block is ONE contiguous window of the global vector.  Otherwise a column
 * owned by this rank becomes (column - row0) and any other column nrows + (its position in the
 * sorted halo list).  Every multi-vector keeps room for the halo rows in front of and behind its
 * local rows.  Single GPU: row0 = 0, nhalo = 0, local == global. */
struct b200_mat_ {
	int nrows, ncols, nnz;
	/* CSR of A: row r holds entries rp[r]..rp[r+1] in ascending column order -- the order
	 * in which the reference's CCS scatter loop (app/app_ccs.c:116-131) adds into y[r]. */
	int *rp; int *ci; double *va;
	/* the caller's CCS arrays verbatim (== CSR of A^T): A^T x and the bit-exact round
	 * trip; shares storage with the CSR image when the two coincide (t_shared). */
	int *t_rp; int *t_ci; double *t_va;
	int t_shared;
	int row0;
	int max_row_nnz, t_max_row_nnz;   /* longest row of the CSR image / of the transpose image */
	int nrows_global, ncols_global, nnz_global;
	int symmetric;                    /* CSR image == CCS image (A == A^T bit for bit) */
	/* halo exchange plan (nranks > 1) */
	int nhalo;                        /* halo rows of x this matrix needs */
	int halo_contiguous;              /* halo = [row0 - halo_below, row0) U [row0 + nrows, ...): two contiguous column ranges */
	int halo_below;
	int nnbr;                         /* ranks exchanged with, ascending */
	int *nbr;                         /* [nnbr] */
	int *halo_cols;                   /* host, [nhalo] global column of each halo slot, ascending */
	int *recv_off;                    /* host, [nnbr+1] halo slots received from nbr[i]: [recv_off[i], recv_off[i+1]) */
	int *send_off;                    /* host, [nnbr+1] */
	int *send_rows;                   /* host, [send_off[nnbr]] LOCAL row sent to nbr[i], ascending per neighbour */
	int *send_rows_dev;               /* device copy */
	long long t_col0;                 /* first CCS column kept in the t_ arrays (== row0) */
	int p2p_ok;                       /* every rank can exchange this matrix's halos through the copy-engine mailboxes */
	/* Diagonal image (b200_mat.cu: dia_build), present when the matrix is a sum of at most 32
	 * diagonals -- stencils and FEM operators on lattices in natural ordering.  The offsets are
	 * grouped into runs of consecutive values (at most 3 wide); run g starts at the even slot
	 * dia_grp_h[2g] of a row of the image, has width dia_grp_h[2g+1] and first offset dia_off_h[g];
	 * entry (r, r + off_g + j) is dia_val[r*dia_ndp + start_g + j], +0.0 where the CCS input has no
	 * such entry.  Rows are padded to a multiple of B200_DIA_PAD. */
	int dia_nd;                       /* distinct offsets; 0: no image */
	int dia_ndp;                      /* slots per row of the image (runs padded to even widths) */
	int dia_ng;                       /* runs */
	int dia_off_h[32], dia_grp_h[64];
	int *dia_off, *dia_grp;           /* device copies */
	double *dia_val;                  /* device [rows padded][dia_ndp] */
	/* Lattice structure read off the diagonal image (b200_spmm_lat.cu: b200k_lat_detect): row = i + lat_s1 (j +
	 * (lat_s2 / lat_s1) k), every entry couples lattice neighbours (|di|, |dj|, |dk| <= 1), nothing crosses a
	 * lattice face, slabs are whole planes.  0: not a lattice (the 1-D diagonal kernel or the CSR kernels run). */
	int lat_s1, lat_s2;
	/* ... and, when every row carries the same coefficients (a constant stencil: entries exist exactly where the
	 * neighbour is inside the lattice), those coefficients by value slot: the lattice kernel then loads no values */
	int lat_const;
	double lat_coef[40];
};

/* host-side partition plan, usable without a device (tests): fills a zeroed b200_mat with
 * the LOCAL CSR (host arrays rp_h/ci_h/va_h malloc'ed, to be freed by the caller), the halo
 * and send lists.  rank/nranks explicit. */
int b200_partition_build(int nrows, int ncols, const int *j_col, const int *i_row, const double *data,
                         int rank, int nranks, struct b200_mat_ *A, int **rp_h, int **ci_h, double **va_h);

struct b200_mv_ {
	int nrows, ncols, ld;       /* nrows: LOCAL rows */
	double *d;
	int owner;          /* 0: view into another multi-vector's storage */
	int nrows_global;
	int halo_cap;       /* rows allocated in FRONT of and BEHIND the local ones for SpMM halos */
	double *alloc;      /* start of the allocation (d = alloc + halo_cap*ld); NULL for views */
	int dist;           /* rows are a slab of a distributed object (Gram blocks need an allreduce) */
	long long row0;
};

int  b200_fail(const char *fmt, ...);
void b200_gcg_free_cache(void);               /* b200_gcg.c: the solver's cached second [X P W] buffer */
void *b200_scratch(int slot, size_t bytes);   /* growable device scratch; NULL on failure */
void *b200_pinned(int slot, size_t bytes);    /* growable pinned host staging */
int  b200k_num_sms(void);
/* Run-time switches (b200_runtime.cu, DESIGN.md §10), X(ID, name) each: the ids B200_OPT_<ID> and the names of
 * b200_option_name both come from this one list.  b200k_opt: the cached value, for the host-side C drivers. */
#define B200_OPTIONS(X)                                                                                            \
	X(NO_DIA, no_dia) X(NO_LAT, no_lat) X(NO_FUSED_DOT, no_fused_dot) X(HOST_BUILD, host_build)                    \
	X(NO_OVERLAP, no_overlap) X(NO_P2P, no_p2p) X(NO_KERNEL_ALLREDUCE, no_kernel_allreduce) X(SYEV_PROF, syev_prof) \
	X(BPCG_TRACE, bpcg_trace) X(LAT_NO_CONST, lat_no_const) X(ORTH_TRACE, orth_trace) X(NO_AXPBY_BATCH, no_axpby_batch)
#define B200_OPT_ID_(id, name) B200_OPT_##id,
enum { B200_OPTIONS(B200_OPT_ID_) B200_OPT_COUNT };
#undef B200_OPT_ID_
int  b200k_opt(int id);

/* synchronising small transfers */
int b200k_d2h(void *host, const void *dev, size_t bytes);
/* launch what b200_mv_axpby deferred (a batch of narrow calls on adjacent columns); every entry point calls it first */
int b200k_pending_flush(void);
int b200k_h2d(void *dev, const void *host, size_t bytes);
int b200k_memset(void *dev, int value, size_t bytes);
int b200k_malloc(void **dev, size_t bytes);
int b200k_free(void *dev);

/* y = A x for k columns; separate multiply and add in CSR column order (bit-exact with
 * the reference's scatter loop).  x, y may live in one multi-vector (disjoint columns). */
/* trans != 0 multiplies by the true transpose (the caller's CCS arrays read as CSR).
 * gate_dev != NULL: the kernel returns at once when *gate_dev == 0 (device-side loop control) */
int b200k_spmm(const b200_mat *M, int trans, const double *x, int ldx, double *y, int ldy, int k,
               const int *gate_dev);
/* Several ranks: the x block must belong to a multi-vector with room for M's halo rows behind its
 * local rows (b200_mv.halo_cap >= M->nhalo); b200k_spmm fills them from the slab neighbours
 * before multiplying.  Callers check with this helper. */
int b200k_spmm_check_halo(const b200_mat *M, const b200_mv *x);
/* y = alpha x + beta y over n x k; x may be NULL (scale); beta == 0 overwrites. */
int b200k_axpby(long long n, int k, double alpha, const double *x, int ldx,
                double beta, double *y, int ldy);
/* C(p x q, device, element (i,j) at c[i*c_rs + j*c_cs]) = alpha X^T Y over n rows;
 * mode 'N', 'S' (lower triangle mirrored) or 'D' (dots: c[i*(c_rs+c_cs)]... see .cu). */
/* dist != 0: the n rows are this rank's slab of a distributed block; the result is summed over
 * all ranks (NCCL allreduce on the library stream) and identical on every rank. */
int b200k_gram(char mode, long long n, int p, int q, double alpha, const double *x, int ldx,
               const double *y, int ldy, double *c_dev, int c_rs, int c_cs, int dist);
int b200k_multi(void);          /* number of ranks (1 = single GPU) */
/* Y(n x q) = X(n x p) C + Y diag(beta); C device, element (k,j) at c[k*c_rs + j*c_cs];
 * beta_dev NULL => 0 (overwrite) else beta_dev[incb*col]; x or c NULL => scaling only. */
int b200k_lincomb(long long n, int p, int q, const double *x, int ldx,
                  const double *c_dev, int c_rs, int c_cs,
                  const double *beta_dev, int incb, double *y, int ldy);
/* column scaling y[:,j] *= s_dev[j] (or by 1/s_dev[j] when invert != 0) */
int b200k_colscale(long long n, int q, const double *s_dev, int invert, double *y, int ldy);
/* column-major (ld_cm) <-> row-major (ld_rm) transposes of an n x k block, on device */
int b200k_cm_to_rm(long long n, int k, const double *cm, long long ld_cm, double *rm, int ld_rm);
int b200k_rm_to_cm(long long n, int k, const double *rm, int ld_rm, double *cm, long long ld_cm);

/* ---- orthogonalisation panel (b200_orth.cu) ----------------------------------------
 * Right-looking Cholesky of the k x k Gram matrix g (row-major, ld k, destroyed) with the
 * reference's drop rule (r_k < zero_tol: swap the last live column in, shrink; reference
 * src/ops_orth.c:64-73).  Writes T (k x k, element (i,j) at t[i*k+j]) with
 * X_new[:, 0:n_live] = X T[:, 0:n_live], and n_live to *n_live_dev.
 * scale_in (NULL = ones): factors by which earlier passes scaled each column up; the drop
 * test is r_k*scale_in[k] < zero_tol, so a second pass still judges a column by its norm
 * in the caller's scaling (the Cholesky pivot alone cannot resolve r_k below ~1e-8 |x_k|).
 * scale_out (NULL ok): the accumulated factors of the surviving columns, in final order. */
int b200k_chol_drop(int k, double *g_dev, double zero_tol, double *t_dev, int *n_live_dev,
                    const double *scale_in, double *scale_out);

/* t (n x (n - lin_dep), row-major) = z[:, lin_dep:n] diag(w[lin_dep:n])^(-1/2): the update block of OrthSelfEVP */
int b200k_evp_coef(int n, int lin_dep, const double *w_dev, const double *z_dev, double *t_dev);
/* *out_dev = max |c[i][j]| * scale[j] over a row-major rows x cols coefficient block (scale NULL: 1); one CTA */
int b200k_absmax(int rows, int cols, const double *c_dev, const double *scale_dev, double *out_dev);

/* ---- BlockPCG (b200_bpcg.cu): device-resident scalars and masks ----------------------- */
typedef struct b200_bpcg_state_ {
	int k;
	double *norm_b, *rho1, *rho2, *ptw, *init_res, *last_res;   /* k doubles each (device) */
	int *active;        /* k ints (device): 1 while the column is unconverged */
	int *counters;      /* [0] number of active columns, [1] iterations done, [2] 1 + iteration of the pending alpha (device) */
	double *totals;     /* 3k doubles: per-column sums of the current reduction (allreduced across ranks) */
	double *alpha;      /* k doubles: step length of the x update deferred into the next p update */
	double *partials;   /* reduction scratch */
	unsigned *tickets;  /* last-block election counters */
	const double *dinv; /* n doubles (device): Jacobi preconditioner D^-1, NULL: none (b200k_bpcg_state leaves it NULL) */
} b200_bpcg_state;
int b200k_bpcg_state(int k, b200_bpcg_state *st);               /* carve state out of scratch */
/* Jacobi preconditioner of A + shift B (B NULL: A + shift I): *dinv_dev = 1 / diagonal, one double per local row, in a
 * scratch slot of its own.  Reads the device CSR; fails (synchronises once) when a row has no diagonal entry or a
 * diagonal <= 0, on any rank. */
int b200k_bpcg_jacobi(const b200_mat *A, const b200_mat *B, double shift, const double **dinv_dev);
/* several ranks: 0, or an error if an in-kernel allreduce timed out since the communicator was made (synchronises) */
int b200k_ar_check(void);
/* r = b - r (r holds A x on entry); rho2 = diag(r^T r); norm_b = 1 or ||b||; then decide the
 * initial active set: init_res > tol*norm_b (reference src/ops_lin_sol.c:221-247).
 * With st->dinv set (Jacobi), here and in update_r / update_px: z = D^-1 r is formed in registers, rho = diag(r^T z)
 * drives alpha and beta, p = z + beta p; the residual norms and the stop test stay on sqrt(r^T r). */
int b200k_bpcg_begin(long long n, const b200_bpcg_state *st, const double *b, int ldb,
                     double *r, int ldr, double tol, int rel);
/* w += shift * z (optional), ptw = diag(p^T w) */
int b200k_bpcg_ptw(long long n, const b200_bpcg_state *st, const double *p, int ldp,
                   double *w, int ldw, double shift, const double *z, int ldz);
/* w = A p and ptw = diag(p^T w): one fused pass when A has a diagonal image (b200_spmm.cu),
 * otherwise SpMM + b200k_bpcg_ptw */
int b200k_bpcg_spmm_ptw(const b200_mat *A, long long n, const b200_bpcg_state *st, const double *p, int ldp,
                        double *w, int ldw);
/* update_r: alpha = rho2/ptw; r -= alpha w; rho1 = rho2; rho2 = diag(r^T r); the per-column stop test
 * (reference src/ops_lin_sol.c:383-394) and ++iterations; alpha is left behind, and
 * update_px: applies x += alpha p of the previous iteration, then p = r + (rho2/rho1) p on the active
 * columns (it == 0: p = r) -- p is read once for both: bit-identical iterates, 8 streams instead of 9 */
int b200k_bpcg_update_r(long long n, const b200_bpcg_state *st, const double *w, int ldw, double *r, int ldr,
                        double rate, double tol, int it);
int b200k_bpcg_update_px(long long n, const b200_bpcg_state *st, const double *r, int ldr, double *p, int ldp,
                         double *x, int ldx, int it, int flush);

/* ---- projected eigenproblem (b200_syev.cu) --------------------------------------------
 * All eigenpairs of the symmetric n x n device matrix a (element (i,j) at a[i*lda+j]; both
 * triangles must be filled), ascending in w_dev; eigenvector j in column j of z (element
 * (i,j) at z[i*ldz+j]).  a is destroyed.  Parallel-order cyclic Jacobi, cooperative grid. */
int b200k_syev_jacobi(int n, double *a_dev, int lda, double *w_dev, double *z_dev, int ldz,
                      int *sweeps_host);
/* non-zero (with a message) when the most recent eigen-solve ran out of sweeps; synchronises */
int b200k_syev_check(void);

/* ---- GCG helpers (b200_gcgk.cu) --------------------------------------------------------- */
/* res[j] = || ax[:,j] - lam[j] * bx[:,j] ||_2 ; ax is overwritten with the residual */
int b200k_residual_norms(long long n, int k, double *ax, int ldax, const double *bx, int ldbx,
                         const double *lam_dev, double *res_dev);
/* generic small elementwise helpers on device matrices */
int b200k_copy2d(int rows, int cols, const double *src, int s_rs, int s_cs, double *dst, int d_rs, int d_cs);
int b200k_set_diag(int n, double *a, int lda, const double *d, double shift);   /* a[i,i] = d[i]+shift (d NULL: += shift) */
int b200k_symmetrize_upper(int n, double *a, int lda);                          /* a[i,j] = a[j,i] for i > j */
int b200k_zero_rows(int nidx, const int *idx_dev, int cols, double *a, int rs, int cs); /* a[idx[i], 0:cols] = 0 */
int b200k_gather_cols(int rows, int nidx, const int *idx_dev, const double *src, int s_rs, int s_cs,
                      double *dst, int d_rs, int d_cs);                         /* dst[:, i] = src[:, idx[i]] */

#ifdef __cplusplus
}
#endif
#endif
