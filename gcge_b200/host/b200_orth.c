/* b200_orth.c -- host driver of the device block orthogonalisation (C-ABI b200_mv_orth).
 *
 * Replaces ModifiedGramSchmidt + OrthSelf (reference src/ops_orth.c:203-393, :45-118).
 * Same block structure as the reference (blocks of block_size columns, each block
 * B-orthonormalised against everything before it and against itself, dependent columns
 * dropped and refilled from the tail, *end_x shrunk), but each block is processed as
 *
 *     twice:  X1 -= X0 (X0^T B X1)          one Gram (s1 x k) + one update, tensor-core tiles
 *             G = X1^T B X1 ; X1 <- X1 T     panel: k x k Gram, Cholesky recurrence with the
 *                                            reference's drop rule on device, one update
 *
 * i.e. block classical Gram-Schmidt with re-orthogonalisation and a Gram/Cholesky panel in
 * place of the column-by-column OrthSelf.  In exact arithmetic the result is the reference's
 * (QR factorisation is unique); in floating point it differs by normalising BEFORE the second
 * projection.  The reference stops re-projecting on an ABSOLUTE test, max|coef| < 50 eps
 * (src/ops_orth.c:262-267), which lets tiny columns (norm ~1e-12, routine for P and W near
 * convergence) keep an O(1e-2) relative component along X0 once they are normalised; the
 * test-suite reproduces that loss of orthogonality with the reference's own ops_orth.c on
 * identical input (DESIGN.md "Orthogonalisation").  The panel costs two reads
 * of the n x k block instead of OrthSelf's k reads.
 */
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <float.h>
#include <stdio.h>
#include "b200_dev.h"

#define ORTH_MAX_BLOCK 112      /* the k x k panel kernel keeps G and T in shared memory: 2 k (k+1) doubles */
#define LINCOMB_INPLACE_MAX 64      /* LC_BN of b200_dense.cu: output columns of one LinearComb CTA */

static int orth_panel(long long n, double *x1, int ldx, int kb, const b200_mat *B, double *ws, int ldws,
                      double zero_tol, double *g_dev, double *t_dev, int *nlive_dev, int *n_live,
                      const double *scale_in, double *scale_out, int dist)
{
	const double *y = x1; int ldy = ldx;
	if (B) {
		if (b200k_spmm(B, 0, x1, ldx, ws, ldws, kb, NULL)) return 1;
		y = ws; ldy = ldws;
	}
	if (b200k_gram('S', n, kb, kb, 1.0, x1, ldx, y, ldy, g_dev, kb, 1, dist)) return 1;
	if (b200k_chol_drop(kb, g_dev, zero_tol, t_dev, nlive_dev, scale_in, scale_out)) return 1;
	/* X1 <- X1 T (T: element (i,j) at t[i*kb+j]).  A block of at most LINCOMB_INPLACE_MAX columns is one
	 * column tile of the LinearComb kernels: a CTA owns whole rows of X1, reads them completely through its
	 * tile ring and stores them afterwards, so the update runs in place; wider blocks go through the
	 * workspace like the reference's (src/ops_orth.c:108-114) */
	if (kb <= LINCOMB_INPLACE_MAX) {
		if (b200k_lincomb(n, kb, kb, x1, ldx, t_dev, kb, 1, NULL, 0, x1, ldx)) return 1;
	} else {
		if (b200k_lincomb(n, kb, kb, x1, ldx, t_dev, kb, 1, NULL, 0, ws, ldws)) return 1;
		if (b200k_axpby(n, kb, 1.0, ws, ldws, 0.0, x1, ldx)) return 1;
	}
	if (b200k_d2h(n_live, nlive_dev, sizeof(int))) return 1;
	return 0;
}

int b200_mv_orth(b200_mv *x, int start_x, int *end_x, const b200_mat *B,
                 const b200_orth_params *prm, b200_mv *ws)
{
	if (!x || !end_x || !prm || !ws) return b200_fail("b200_mv_orth: bad arguments");
	if (b200k_pending_flush()) return 1;
	if (*end_x <= start_x) return 0;
	if (start_x < 0 || *end_x > x->ncols) return b200_fail("b200_mv_orth: range [%d,%d) outside %d columns", start_x, *end_x, x->ncols);
	if (ws->nrows != x->nrows) return b200_fail("b200_mv_orth: workspace row count differs");
	if (B && (B->nrows != x->nrows || B->ncols != x->nrows)) return b200_fail("b200_mv_orth: B is not n x n");
	if (B && b200k_spmm_check_halo(B, x)) return 1;
	const long long n = x->nrows;
	int end = *end_x;
	int init_start = start_x;
	int block = prm->block_size;
	if (block <= 0) {                                       /* reference src/ops_orth.c:275-278 */
		block = (end - init_start) / 2 > 2 ? (end - init_start) / 2 : 2;
	}
	if (block > ORTH_MAX_BLOCK) block = ORTH_MAX_BLOCK;
	if (block > ws->ncols) block = ws->ncols;
	if (block < 1) return b200_fail("b200_mv_orth: workspace has no columns");
	if (block > end - init_start) block = end - init_start;

	/* device scratch: coefficient block (<= ncols x block), G, T, ones, n_live */
	const size_t ncoef = (size_t)x->ncols * ORTH_MAX_BLOCK;
	const size_t npan = (size_t)ORTH_MAX_BLOCK * ORTH_MAX_BLOCK;
	double *base = (double *)b200_scratch(1, sizeof(double) * (ncoef + 2 * npan + 2 * ORTH_MAX_BLOCK + 12) + 64);
	if (!base) return 1;
	double *c_dev = base, *g_dev = base + ncoef, *t_dev = g_dev + npan, *one_dev = t_dev + npan;
	double *sc0_dev = one_dev + 4, *sc1_dev = sc0_dev + ORTH_MAX_BLOCK;
	double *cmax_dev = sc1_dev + ORTH_MAX_BLOCK;
	int *nlive_dev = (int *)(cmax_dev + 2);
	const double one = 1.0;
	if (b200k_h2d(one_dev, &one, sizeof(double))) return 1;

	while (block > 0) {
		const int s1 = init_start;
		int e1 = s1 + block;
		/* Rounds of (project out X0, orthonormalise the panel).  Two always: block classical Gram-Schmidt needs its
		 * second pass.  Further ones, up to 1 + max_reorth in all (the reference's loop, src/ops_orth.c:233-268),
		 * only when the second pass did NOT confirm the first.  The columns entering a pass >= 1 have unit B-norm (the
		 * previous panel normalised them), so the coefficients c of that pass are what the pass before left behind:
		 * kappa eps for a block of condition kappa against X0.  "Twice is enough" (Giraud, Langou, Rozloznik) holds
		 * while kappa eps << 1, and the error after the pass is the rounding level of the inner products, eps sqrt(n),
		 * whatever c was -- a further pass would subtract noise.  So another pass is made only for c >= 1e-3 (or the
		 * caller's reorth_tol if that is larger).  The reference tests max |coef| < 50 eps on columns it never
		 * normalises; taken over literally (relative or rescaled) that costs every W block of the headline solve a
		 * third pass -- second-pass coefficients are 1e-8 .. 1e-6 there -- +1.2 s of 17 for an unchanged result
		 * (profiles/orth_reorth_trace_r2.log). */
		const int max_rounds = prm->max_reorth + 1 > 2 ? prm->max_reorth + 1 : 2;
		const double again_tol = prm->reorth_tol > 1e-3 ? prm->reorth_tol : 1e-3;
		double cmax = 0.0;
		for (int round = 0; round < max_rounds && e1 > s1; ++round) {
			if (round >= 2 && !(s1 > 0 && cmax >= again_tol)) break;
			const int kb = e1 - s1;
			double *x1 = x->d + s1;
			if (s1 > 0) {
				const double *y = x1; int ldy = x->ld;
				if (B) {
					if (b200k_spmm(B, 0, x1, x->ld, ws->d, ws->ld, kb, NULL)) return 1;
					y = ws->d; ldy = ws->ld;
				}
				/* C = -(X0^T B X1), row-major s1 x kb; X1 += X0 C */
				if (b200k_gram('N', n, s1, kb, -1.0, x->d, x->ld, y, ldy, c_dev, kb, 1, x->dist)) return 1;
				if (round >= 1 && round + 1 < max_rounds && b200k_absmax(s1, kb, c_dev, NULL, cmax_dev)) return 1;
				if (b200k_lincomb(n, s1, kb, x->d, x->ld, c_dev, kb, 1, one_dev, 0, x1, x->ld)) return 1;
			}
			int n_live = kb;
			double *sc_in = (round == 0) ? NULL : ((round & 1) ? sc0_dev : sc1_dev);
			double *sc_out = (round & 1) ? sc1_dev : sc0_dev;
			if (orth_panel(n, x1, x->ld, kb, B, ws->d, ws->ld, prm->orth_zero_tol, g_dev, t_dev, nlive_dev, &n_live,
			               sc_in, sc_out, x->dist))
				return 1;
			if (s1 > 0 && round >= 1 && round + 1 < max_rounds && b200k_d2h(&cmax, cmax_dev, sizeof(double))) return 1;
			if (b200k_opt(B200_OPT_ORTH_TRACE) && s1 > 0 && round >= 1)
				fprintf(stderr, "orth: block at %d of %d columns, round %d: max |coef| on unit columns %.3e (another pass from %.3e)\n",
				        s1, kb, round, cmax, again_tol);
			e1 = s1 + n_live;
		}
		const int init_end = e1;
		/* refill the dropped slots from the tail, reference src/ops_orth.c:293-307 */
		int length = block - (init_end - s1);
		if (length > end - init_end - length) length = end - init_end - length;
		if (length > 0) {
			if (b200k_axpby(n, length, 1.0, x->d + (end - length), x->ld, 0.0, x->d + init_end, x->ld)) return 1;
		}
		end -= block - (init_end - init_start);
		init_start = init_end;
		if (block > end - init_start) block = end - init_start;
	}
	*end_x = end;
	return 0;
}


/* ==== BinaryGramSchmidt + OrthSelfEVP on the device (SURVEY 8f row 2) ===================================
 * Replaces BinaryGramSchmidt / OrthBinary / OrthSelfEVP, reference src/ops_orth.c:518-600, :415-516, :122-201
 * (selected there by -gcge_*_orth_method bgs, src/ops_eig_sol_gcg.c:1757-1785).  Same recursion and the same
 * numerical scheme -- the block is first projected against x[:,0:start_x], then halved recursively: orthonormalise
 * the left half, project the right half against it, orthonormalise the right half, fill the slots of dropped
 * columns from the right; a leaf of at most block_size columns is orthonormalised through the eigen-decomposition
 * of its Gram matrix, X <- X V diag(lambda)^(-1/2), eigenvalues <= orth_zero_tol dropped, repeated until the
 * scaling factors sum to N within reorth_tol -- with the Gram blocks and updates on tensor-core tiles and the
 * small symmetric eigenproblem on the device Jacobi kernel (reference: dsyev on the host).  A block of fewer than
 * 16 columns goes to the panel path of b200_mv_orth (the reference uses the column-wise OrthSelf there, :575-581). */
typedef struct {
	b200_mv *x, *ws;
	const b200_mat *B;
	int max_reorth;
	double zero_tol, reorth_tol;
	double again_tol;           /* max(reorth_tol, eps sqrt(n)): projections are not repeated over rounding noise */
	double *c_dev, *g_dev, *z_dev, *t_dev, *w_dev, *cmax_dev, *one_dev;
	int chunk;                  /* columns of X1 handled per pass: min(workspace columns, ORTH_MAX_BLOCK) */
} bgs_t;

/* X1 = x[:, b0:b1) minus its components along X0 = x[:, a0:a1), reference :455-493 / :538-567 */
static int bgs_project(bgs_t *g, int a0, int a1, int b0, int b1)
{
	b200_mv *x = g->x;
	const long long n = x->nrows;
	const int s0 = a1 - a0;
	if (s0 <= 0 || b1 <= b0) return 0;
	for (int idx = 0; idx < 1 + g->max_reorth; ++idx) {
		double cmax_all = 0.0;
		for (int c0 = b0; c0 < b1; c0 += g->chunk) {
			const int kc = b1 - c0 < g->chunk ? b1 - c0 : g->chunk;
			double *x1 = x->d + c0;
			const double *y = x1; int ldy = x->ld;
			if (g->B) {
				if (b200k_spmm(g->B, 0, x1, x->ld, g->ws->d, g->ws->ld, kc, NULL)) return 1;
				y = g->ws->d; ldy = g->ws->ld;
			}
			if (b200k_gram('N', n, s0, kc, -1.0, x->d + a0, x->ld, y, ldy, g->c_dev, kc, 1, x->dist)) return 1;
			if (b200k_absmax(s0, kc, g->c_dev, NULL, g->cmax_dev)) return 1;
			if (b200k_lincomb(n, s0, kc, x->d + a0, x->ld, g->c_dev, kc, 1, g->one_dev, 0, x1, x->ld)) return 1;
			double cmax = 0.0;
			if (b200k_d2h(&cmax, g->cmax_dev, sizeof(double))) return 1;
			if (cmax > cmax_all) cmax_all = cmax;
		}
		if (cmax_all < g->again_tol) break;
	}
	return 0;
}

/* OrthSelfEVP, reference :122-201 */
static int bgs_self_evp(bgs_t *g, int start, int *end)
{
	b200_mv *x = g->x;
	const long long n = x->nrows;
	for (int idx = 0; idx < 1 + g->max_reorth; ++idx) {
		const int N = *end - start;
		if (N <= 0) return 0;
		double *x1 = x->d + start;
		const double *y = x1; int ldy = x->ld;
		if (g->B) {
			if (b200k_spmm(g->B, 0, x1, x->ld, g->ws->d, g->ws->ld, N, NULL)) return 1;
			y = g->ws->d; ldy = g->ws->ld;
		}
		if (b200k_gram('S', n, N, N, 1.0, x1, x->ld, y, ldy, g->g_dev, N, 1, x->dist)) return 1;
		if (b200k_syev_jacobi(N, g->g_dev, N, g->w_dev, g->z_dev, N, NULL)) return 1;
		double w[ORTH_MAX_BLOCK];
		if (b200k_d2h(w, g->w_dev, sizeof(double) * (size_t)N)) return 1;
		if (b200k_syev_check()) return 1;
		int lin_dep = 0; double sum = 0.0;
		for (int k = 0; k < N; ++k) {
			if (!(w[k] > -g->zero_tol)) return b200_fail("orth (bgs): Gram matrix has the eigenvalue %g (reference assert src/ops_orth.c:172)", w[k]);
			if (w[k] > g->zero_tol || -w[k] > g->zero_tol) sum += 1.0 / sqrt(w[k]);
			else ++lin_dep;                            /* ascending: the dependent directions come first */
		}
		const int nk = N - lin_dep;
		if (nk > 0) {
			/* T = V[:, lin_dep:N] diag(lambda)^(-1/2); X1[:, 0:nk) = X1 T (reference :183-192) */
			if (b200k_evp_coef(N, lin_dep, g->w_dev, g->z_dev, g->t_dev)) return 1;
			if (N <= LINCOMB_INPLACE_MAX) {
				if (b200k_lincomb(n, N, nk, x1, x->ld, g->t_dev, nk, 1, NULL, 0, x1, x->ld)) return 1;
			} else {
				if (b200k_lincomb(n, N, nk, x1, x->ld, g->t_dev, nk, 1, NULL, 0, g->ws->d, g->ws->ld)) return 1;
				if (b200k_axpby(n, nk, 1.0, g->ws->d, g->ws->ld, 0.0, x1, x->ld)) return 1;
			}
		}
		*end -= lin_dep;
		if (lin_dep == 0 && fabs(sum - N) < g->reorth_tol) break;
	}
	return 0;
}

/* OrthBinary, reference :415-516 */
static int bgs_binary(bgs_t *g, int start_x, int *end_x, int block_size)
{
	const int ncols = *end_x - start_x;
	if (ncols <= 0) return 0;
	if (ncols <= block_size) return bgs_self_evp(g, start_x, end_x);
	int s0 = start_x, e0 = start_x + ncols / 2, s1 = e0, e1 = *end_x;
	if (bgs_binary(g, s0, &e0, block_size)) return 1;          /* X0; e0 may shrink */
	if (bgs_project(g, s0, e0, s1, e1)) return 1;                /* X1 -= X0 (X0^T B X1) */
	if (bgs_binary(g, s1, &e1, block_size)) return 1;          /* X1 */
	/* the slots of X0's dropped columns are filled with orthonormal columns from the end of X1, :494-513 */
	int length = start_x + ncols / 2 - e0;
	*end_x = e1 - length;
	if (length > e1 - s1) length = e1 - s1;
	if (length > 0 &&
	    b200k_axpby(g->x->nrows, length, 1.0, g->x->d + (e1 - length), g->x->ld, 0.0, g->x->d + e0, g->x->ld))
		return 1;
	return 0;
}

int b200_mv_orth_bgs(b200_mv *x, int start_x, int *end_x, const b200_mat *B,
                     const b200_orth_params *prm, b200_mv *ws)
{
	if (!x || !end_x || !prm || !ws) return b200_fail("b200_mv_orth_bgs: bad arguments");
	if (b200k_pending_flush()) return 1;
	if (*end_x <= start_x) return 0;
	if (start_x < 0 || *end_x > x->ncols) return b200_fail("b200_mv_orth_bgs: range [%d,%d) outside %d columns", start_x, *end_x, x->ncols);
	if (ws->nrows != x->nrows || ws->ncols < 1) return b200_fail("b200_mv_orth_bgs: workspace shape");
	if (B && (B->nrows != x->nrows || B->ncols != x->nrows)) return b200_fail("b200_mv_orth_bgs: B is not n x n");
	if (B && b200k_spmm_check_halo(B, x)) return 1;
	const int ncols = *end_x - start_x;
	if (ncols < 16) return b200_mv_orth(x, start_x, end_x, B, prm, ws);      /* reference :575-581 uses OrthSelf here */
	bgs_t g; memset(&g, 0, sizeof(g));
	g.x = x; g.ws = ws; g.B = B; g.max_reorth = prm->max_reorth;
	g.zero_tol = prm->orth_zero_tol; g.reorth_tol = prm->reorth_tol;
	{
		/* never below the rounding level of an n-term inner product: the reference's 50 eps lies under eps sqrt(n)
		 * from n ~ 2500 on, where its own loop simply runs to max_reorth */
		const double noise = DBL_EPSILON * sqrt((double)(x->nrows_global > 0 ? x->nrows_global : x->nrows));
		g.again_tol = prm->reorth_tol > noise ? prm->reorth_tol : noise;
	}
	g.chunk = ws->ncols < ORTH_MAX_BLOCK ? ws->ncols : ORTH_MAX_BLOCK;
	int block = prm->block_size;                                          /* reference :583-586 */
	if (block <= 0 || block > ncols / 4) block = ncols / 4;
	if (block > g.chunk) block = g.chunk;
	if (block < 1) block = 1;
	const size_t ncoef = (size_t)x->ncols * ORTH_MAX_BLOCK, npan = (size_t)ORTH_MAX_BLOCK * ORTH_MAX_BLOCK;
	double *base = (double *)b200_scratch(1, sizeof(double) * (ncoef + 3 * npan + ORTH_MAX_BLOCK + 16) + 64);
	if (!base) return 1;
	g.c_dev = base; g.g_dev = base + ncoef; g.z_dev = g.g_dev + npan; g.t_dev = g.z_dev + npan;
	g.w_dev = g.t_dev + npan; g.cmax_dev = g.w_dev + ORTH_MAX_BLOCK; g.one_dev = g.cmax_dev + 2;
	const double one = 1.0;
	if (b200k_h2d(g.one_dev, &one, sizeof(double))) return 1;
	if (start_x > 0 && bgs_project(&g, 0, start_x, start_x, *end_x)) return 1;   /* reference :538-567 */
	return bgs_binary(&g, start_x, end_x, block);
}
