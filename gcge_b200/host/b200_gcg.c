/* b200_gcg.c -- host driver of the device-resident block GCG eigensolver (C-ABI b200_gcg_solve).
 *
 * Follows GCG() of the reference (src/ops_eig_sol_gcg.c:1253-1558) phase by phase --
 * InitializeX :101, ComputeRayleighRitz :925, ComputeRitzVec :159, CheckConvergence :195,
 * ComputeP :316, ComputeX :458, ComputeW :472 -- with the same state variables
 * (V = [X | P | W], sizeC/sizeN/sizeX/sizeP/sizeW, startN/endN ...), the same parameters
 * (GCGSolver, src/ops_eig_sol_gcg.h:26-52) and the same stopping logic.  What changes is
 * where the data lives: the projected matrix ss_matA, the Ritz coefficients ss_evec, the
 * P coefficients and every Gram block stay in HBM; the projected eigenproblem is solved by
 * the device Jacobi kernel; BlockPCG and the orthogonalisation are the fused device
 * providers.  Per outer iteration the host reads back only the Ritz values (N doubles), the
 * residual norms of the checked columns and a few block sizes -- it needs them to steer the
 * loop exactly like the reference does.
 *
 * [X | P | W] is double-buffered (V, V2): ComputeRitzVec writes the new X and ComputeP the new P straight
 * into the other buffer and ComputeX (reference :458-471, a copy of up to nevMax columns per iteration) is
 * a pointer swap; columns are copied across once, when they are locked.  The caller's evec block serves
 * as workspace (right-hand sides of the inner solve, like the reference) and receives the eigenvectors
 * once at the end.
 *
 * Small dense objects are ROW-major on device with a fixed leading dimension ldE
 * (element (i,j) at base[i*ldE + j]), so an N x N coefficient matrix is at the same time a
 * row-major "multi-vector" with N rows: the projected-space orthogonalisation of ComputeP
 * (reference :371-414, done there on the host through lapack_ops) reuses b200_mv_orth.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <float.h>
#include "b200_dev.h"

#define TRY(call) do { if ((call) != 0) return 1; } while (0)
#define GCG_MAX_BLOCK 512      /* the reference is run at block_size = 200 (test/test_eig_sol_PHG_MAT.c:38-39) */

typedef struct {
	const b200_mat *A, *B;
	const b200_gcg_params *p;
	b200_mv *V, *V2, *ritz, *ws[3];     /* V: the current [X | P | W]; V2: where the next X and P are built */
	b200_mv *V_alloc;                   /* the buffer this solve allocated (V and V2 trade places) */
	b200_mv *xw;                        /* the inner solve's unknowns as a block of their own (compute_w) */
	int own_ws;
	long long n;
	/* reference file-scope state, src/ops_eig_sol_gcg.c:44-54 */
	int sizeN, startN, endN, sizeP, startP, endP, sizeW, startW, endW, sizeC, sizeX, sizeV, endX;
	/* device small dense */
	int ldE, Nmax;
	double *eval_d;      /* nevMax + 2 bs */
	double *matA_d;      /* Nmax x ldE, symmetric, both triangles */
	double *evec_d;      /* Nmax x ldE */
	double *t1_d;        /* Nmax x bsp   (matA * Pc) */
	double *ptap_d;      /* bs x bs */
	double *wsE_d;       /* Nmax x bsp   (orth workspace in coefficient space) */
	double *res_d;       /* bs */
	double *scal_d;      /* bs  (lambda + sigma) */
	int    *idx_d;       /* bs */
	int bsp;
	/* host mirrors */
	double *eval_h, *res_h;
	int *offP, *offW;    /* [0] = count, then pairs; reference offsetP/offsetW */
	b200_gcg_stats st;
	int timing;
} gcg_t;

static int orth_by(int method, b200_mv *x, int start_x, int *end_x, const b200_mat *B, const b200_orth_params *op, b200_mv *ws)
{
	return method == 1 ? b200_mv_orth_bgs(x, start_x, end_x, B, op, ws) : b200_mv_orth(x, start_x, end_x, B, op, ws);
}

static double tick(gcg_t *g) { return g->timing ? b200_wtime() : 0.0; }

static int spmm_mv(const b200_mat *M, const double *x, int ldx, double *y, int ldy, long long n, int k)
{
	if (M) return b200k_spmm(M, 0, x, ldx, y, ldy, k, NULL);
	return b200k_axpby(n, k, 1.0, x, ldx, 0.0, y, ldy);      /* NULL matrix == identity, reference app/app_ccs.c:134-137 */
}

/* ---- ComputeRayleighRitz, reference :925-1252 ------------------------------------------- */
static int rayleigh_ritz(gcg_t *g, int nevConv)
{
	const b200_gcg_params *p = g->p;
	const int ldE = g->ldE, bs = p->block_size;
	double t0 = tick(g);
	if (g->sizeP > 0) {
		/* P^T (old projected matrix) P, reference :936-949 */
		const int Nold = g->sizeV - g->sizeC, c0 = g->sizeX - g->sizeC;
		TRY(b200k_lincomb(Nold, Nold, g->sizeP, g->matA_d, ldE, g->evec_d + c0, ldE, 1, NULL, 0, g->t1_d, g->bsp));
		TRY(b200k_gram('N', Nold, g->sizeP, g->sizeP, 1.0, g->evec_d + c0, ldE, g->t1_d, g->bsp, g->ptap_d, bs, 1, 0));
	}
	g->sizeV  = g->sizeX + g->sizeP + g->sizeW;
	if (nevConv > g->sizeC)      /* newly locked columns: the other buffer still holds their previous iterate */
		TRY(b200k_axpby(g->n, nevConv - g->sizeC, 1.0, g->V->d + g->sizeC, g->V->ld, 0.0, g->V2->d + g->sizeC, g->V2->ld));
	g->startN = g->startN + (nevConv - g->sizeC);
	g->endN   = g->endN + (nevConv - g->sizeC);
	if (g->endN > g->endX) g->endN = g->endX;
	g->sizeN  = g->endN - g->startN;
	g->sizeC  = nevConv;
	const int N = g->sizeV - g->sizeC;
	TRY(b200k_memset(g->matA_d, 0, sizeof(double) * (size_t)N * ldE));
	if (g->sizeW > 0) {
		/* V[:,startN:endW]^T A V[:,startW:endW]: one SpMM + one Gram, reference :970-987 */
		const int c0 = g->sizeX + g->sizeP - g->sizeC;
		TRY(spmm_mv(g->A, g->V->d + g->startW, g->V->ld, g->ws[0]->d, g->ws[0]->ld, g->n, g->sizeW));
		TRY(b200k_gram('N', g->n, N, g->sizeW, 1.0, g->V->d + g->startN, g->V->ld, g->ws[0]->d, g->ws[0]->ld,
		               g->matA_d + c0, ldE, 1, 1));
	}
	if (g->sizeX == g->sizeV) {
		/* first call: full X^T A X by block_size-wide panels, reference :989-1011 */
		int length = g->sizeX - g->sizeC, c = g->sizeC;
		while (length > 0) {
			const int w = bs < length ? bs : length;
			TRY(spmm_mv(g->A, g->V->d + c, g->V->ld, g->ws[0]->d, g->ws[0]->ld, g->n, w));
			TRY(b200k_gram('N', g->n, g->sizeX - g->sizeC, w, 1.0, g->V->d + g->sizeC, g->V->ld,
			               g->ws[0]->d, g->ws[0]->ld, g->matA_d + (c - g->sizeC), ldE, 1, 1));
			c += w; length -= w;
		}
	} else {
		/* diag(X part) = Ritz values, P^T A P block, reference :1013-1033 */
		const int nx = g->sizeX - g->sizeC;
		TRY(b200k_set_diag(nx, g->matA_d, ldE, g->eval_d + g->sizeC, 0.0));
		if (g->sizeP > 0)
			TRY(b200k_copy2d(g->sizeP, g->sizeP, g->ptap_d, bs, 1, g->matA_d + (size_t)nx * ldE + nx, ldE, 1));
	}
	/* the reference hands dsyevx the UPPER triangle (UPLO='U', :1186): make both triangles agree */
	TRY(b200k_symmetrize_upper(N, g->matA_d, ldE));
	double t2 = tick(g);
	/* projected eigenproblem on device (replaces dsyevx, reference :1201); optional shift :1043-1050 */
	if (p->compW_cg_shift != 0.0) TRY(b200k_set_diag(N, g->matA_d, ldE, NULL, p->compW_cg_shift));
	TRY(b200k_syev_jacobi(N, g->matA_d, ldE, g->eval_d + g->sizeC, g->evec_d, ldE, NULL));
	if (p->compW_cg_shift != 0.0) TRY(b200k_set_diag(N, g->matA_d, ldE, NULL, -p->compW_cg_shift));
	TRY(b200k_d2h(g->eval_h + g->sizeC, g->eval_d + g->sizeC, sizeof(double) * (size_t)N));
	TRY(b200k_syev_check());     /* the reference asserts on dsyevx's INFO, :1204 */
	if (p->compW_cg_shift != 0.0)
		for (int i = 0; i < N; ++i) g->eval_h[g->sizeC + i] -= p->compW_cg_shift;
	/* reference :1353-1355 / :1488-1490 */
	for (int i = g->sizeV; i < p->nevMax + 2 * bs; ++i) g->eval_h[i] = g->eval_h[g->sizeV - 1];
	TRY(b200k_h2d(g->eval_d, g->eval_h, sizeof(double) * (size_t)(p->nevMax + 2 * bs)));
	double t3 = tick(g);
	g->st.compRR += t3 - t0; g->st.rr_eig += t3 - t2;
	return 0;
}

/* ---- ComputeRitzVec, reference :159-194 ------------------------------------------------------ */
static int compute_ritz_vec(gcg_t *g)
{
	double t0 = tick(g);
	const int N = g->sizeV - g->sizeC;
	TRY(b200k_lincomb(g->n, N, g->endX - g->startN, g->V->d + g->startN, g->V->ld, g->evec_d, g->ldE, 1,
	                  NULL, 0, g->V2->d + g->startN, g->V2->ld));
	g->st.compRV += tick(g) - t0;
	return 0;
}

/* ---- CheckConvergence, reference :195-315 ------------------------------------------------------ */
static int check_convergence(gcg_t *g, int numCheck, int *offset, int *nevConv_out)
{
	const b200_gcg_params *p = g->p;
	const double *tol = p->tol, *ev = g->eval_h;
	double *res = g->res_h;
	double t0 = tick(g);
	if (numCheck > 0) {
		const double *x = g->V2->d + g->startN;      /* the Ritz vectors of ComputeRitzVec */
		const int ldx = g->V2->ld;
		TRY(spmm_mv(g->A, x, ldx, g->ws[0]->d, g->ws[0]->ld, g->n, numCheck));
		const double *bx = x; int ldbx = ldx;
		if (g->B) {
			TRY(spmm_mv(g->B, x, ldx, g->ws[1]->d, g->ws[1]->ld, g->n, numCheck));
			bx = g->ws[1]->d; ldbx = g->ws[1]->ld;
		}
		TRY(b200k_residual_norms(g->n, numCheck, g->ws[0]->d, g->ws[0]->ld, bx, ldbx, g->eval_d + g->startN, g->res_d));
		TRY(b200k_d2h(res, g->res_d, sizeof(double) * (size_t)numCheck));
	}
	int idx;
	for (idx = 0; idx < numCheck; ++idx) {
		const double lam = fabs(ev[g->startN + idx]);
		if (lam > tol[1]) {
			if (res[idx] > tol[0] || res[idx] > lam * tol[1]) break;
		} else if (res[idx] > tol[0]) break;
	}
	if (p->verbose && idx < numCheck)
		printf("GCG: [%d] %6.14e (%6.4e, %6.4e)\n", g->startN + idx, ev[g->startN + idx], res[idx],
		       res[idx] / fabs(ev[g->startN + idx]));
	for (; idx > 0; --idx) {      /* never split a cluster, reference :253-259 */
		if (fabs((ev[g->startN + idx - 1] - ev[g->startN + idx]) / ev[g->startN + idx - 1]) > p->gapMin) break;
	}
	const int nevConv = g->sizeC + idx;
	/* blocks of unconverged indices, reference :262-302 */
	int state = 1, num_unconv = 0;
	offset[0] = 0;
	for (idx = 0; idx < numCheck; ++idx) {
		if (res[idx] > tol[0] || res[idx] > fabs(ev[g->startN + idx]) * tol[1]) {
			if (state) { offset[offset[0] * 2 + 1] = g->startN + idx; state = 0; }
			++num_unconv;
			if (num_unconv == g->sizeN) { offset[offset[0] * 2 + 2] = g->startN + idx + 1; ++offset[0]; break; }
		} else if (!state) {
			offset[offset[0] * 2 + 2] = g->startN + idx; ++offset[0]; state = 1;
		}
	}
	if (num_unconv < g->sizeN) {
		if (state == 1) offset[offset[0] * 2 + 1] = g->startN + numCheck;
		int hi = g->startN + numCheck + g->sizeN - num_unconv;
		if (hi > g->endX) hi = g->endX;
		offset[offset[0] * 2 + 2] = hi;
		if (!(offset[offset[0] * 2 + 1] < hi)) return b200_fail("gcg: empty unconverged block (reference assert :297)");
		++offset[0];
	}
	if (offset[0] <= 0) return b200_fail("gcg: no unconverged block (reference assert :313)");
	*nevConv_out = nevConv;
	g->st.checkconv += tick(g) - t0;
	return 0;
}

/* ---- ComputeP, reference :316-457 ------------------------------------------------------------------ */
static int compute_p(gcg_t *g, const int *offset)
{
	const b200_gcg_params *p = g->p;
	const int ldE = g->ldE;
	double t0 = tick(g);
	const int N = g->sizeV - g->sizeC, c0 = g->sizeX - g->sizeC;
	int idx_h[GCG_MAX_BLOCK], np = 0;
	for (int b = 0; b < offset[0]; ++b)
		for (int o = offset[b * 2 + 1]; o < offset[b * 2 + 2]; ++o) idx_h[np++] = o - g->sizeC;
	TRY(b200k_h2d(g->idx_d, idx_h, sizeof(int) * (size_t)np));
	/* copy the Ritz coefficient columns of the unconverged block behind the X part and zero
	 * their N-part rows, reference :329-352 */
	TRY(b200k_gather_cols(N, np, g->idx_d, g->evec_d, ldE, 1, g->evec_d + c0, ldE, 1));
	TRY(b200k_zero_rows(np, g->idx_d, np, g->evec_d + c0, ldE, 1));
	/* orthonormalise them against the X coefficient columns and themselves (B = I) in
	 * coefficient space, reference :371-414 */
	b200_mv E, W;
	/* replicated coefficient-space objects: not distributed, no allreduce in their Gram blocks */
	memset(&E, 0, sizeof(E)); memset(&W, 0, sizeof(W));
	E.nrows = N; E.nrows_global = N; E.ncols = c0 + np; E.ld = ldE; E.d = g->evec_d; E.owner = 0;
	W.nrows = N; W.nrows_global = N; W.ncols = g->bsp; W.ld = g->bsp; W.d = g->wsE_d; W.owner = 0;
	b200_orth_params op;
	op.block_size = p->compP_orth_block_size; op.max_reorth = p->compP_orth_max_reorth;
	op.orth_zero_tol = p->compP_orth_zero_tol; op.reorth_tol = 50 * DBL_EPSILON;
	int endP = c0 + np;
	TRY(orth_by(p->compP_orth_method, &E, c0, &endP, NULL, &op, &W));
	g->sizeP = endP - c0;
	g->startP = g->sizeX; g->endP = g->startP + g->sizeP;
	/* P = V[:,startN:endW] * coef (:425-436; there through a workspace because V is source and
	 * destination): straight into the P columns of the other buffer */
	if (g->sizeP > 0)
		TRY(b200k_lincomb(g->n, N, g->sizeP, g->V->d + g->startN, g->V->ld, g->evec_d + c0, ldE, 1, NULL, 0,
		                  g->V2->d + g->startP, g->V2->ld));
	g->st.compP += tick(g) - t0;
	return 0;
}

/* ---- ComputeW, reference :472-696 -------------------------------------------------------------------- */
static int compute_w(gcg_t *g, const int *offset)
{
	const b200_gcg_params *p = g->p;
	double t0 = tick(g);
	double sigma = 0.0;
	if (p->compW_cg_auto_shift == 1)
		sigma = -g->eval_h[g->sizeC] + (g->eval_h[g->sizeC + 1] - g->eval_h[g->sizeC]) * 0.01;
	sigma += p->compW_cg_shift;
	g->startW = g->endP;
	double scal_h[GCG_MAX_BLOCK];
	int acc = 0;
	for (int b = 0; b < offset[0]; ++b)
		for (int o = offset[b * 2 + 1]; o < offset[b * 2 + 2]; ++o) scal_h[acc++] = g->eval_h[o] + sigma;
	TRY(b200k_h2d(g->scal_d, scal_h, sizeof(double) * (size_t)acc));
	acc = 0;
	const int b0 = offset[1];
	for (int b = 0; b < offset[0]; ++b) {
		const int o1 = offset[b * 2 + 1], len = offset[b * 2 + 2] - o1;
		/* initial guess: the Ritz vectors (X part of V since ComputeX), :500-503 -- into the solve's own block */
		TRY(b200k_axpby(g->n, len, 1.0, g->V->d + o1, g->V->ld, 0.0, g->xw->d + acc, g->xw->ld));
		/* right-hand side (lambda+sigma) B x, stored in the Ritz-vector block like the reference, :516-534 */
		TRY(spmm_mv(g->B, g->V->d + o1, g->V->ld, g->ritz->d + b0 + acc, g->ritz->ld, g->n, len));
		TRY(b200k_colscale(g->n, len, g->scal_d + acc, 0, g->ritz->d + b0 + acc, g->ritz->ld));
		acc += len;
	}
	g->endW = g->startW + acc;
	double t1 = tick(g);
	b200_bpcg_params bp;
	bp.max_iter = p->compW_cg_max_iter; bp.rate = p->compW_cg_rate; bp.tol = p->compW_cg_tol;
	bp.tol_type = p->compW_cg_tol_type; bp.shift = sigma;
	int s[2], e[2];
	s[0] = b0; e[0] = b0 + acc; s[1] = 0; e[1] = acc;
	TRY(b200_block_pcg_pc(g->A, g->B, g->ritz, g->xw, s, e, &bp, p->compW_cg_pc, g->ws[0], g->ws[1], g->ws[2], NULL, NULL));
	/* W block of [X P W] <- the solutions (one pass; the 30 CG steps had x to themselves) */
	TRY(b200k_axpby(g->n, acc, 1.0, g->xw->d, g->xw->ld, 0.0, g->V->d + g->startW, g->V->ld));
	double t2 = tick(g);
	b200_orth_params op;
	op.block_size = p->compW_orth_block_size; op.max_reorth = p->compW_orth_max_reorth;
	op.orth_zero_tol = p->compW_orth_zero_tol; op.reorth_tol = 50 * DBL_EPSILON;
	TRY(orth_by(p->compW_orth_method, g->V, g->startW, &g->endW, g->B, &op, g->ws[0]));
	g->sizeW = g->endW - g->startW;
	double t3 = tick(g);
	g->st.compW += t3 - t0; g->st.linsol += t2 - t1;
	return 0;
}

/* ---- ComputeW12, reference :697-923 (-gcge_compW_cg_order 2) ----------------------------------------
 * W = [W1 | W2]: the inner solve for the first half of the unconverged columns (W1), then the
 * same systems solved again from W1 as the initial guess (W2 = max_iter more CG steps), both kept
 * in the search space. */
static int compute_w12(gcg_t *g, const int *offset)
{
	const b200_gcg_params *p = g->p;
	double t0 = tick(g);
	const double *ev = g->eval_h;
	double sigma = 0.0;
	if (p->compW_cg_auto_shift == 1) {          /* reference :707-713 */
		if (g->sizeC < 3) { const double d = 3 * (ev[1] - ev[0]); sigma = -ev[g->sizeC] + (d > 1 ? d : 1); }
		else { const double d = ev[g->sizeC] - ev[g->sizeC - 3]; sigma = -ev[g->sizeC] + (d > 1 ? d : 1); }
	}
	sigma += p->compW_cg_shift;
	int total = 0;
	for (int b = 0; b < offset[0]; ++b) total += offset[b * 2 + 2] - offset[b * 2 + 1];
	const int half = total / 2;
	g->startW = g->endP;
	const int b0 = offset[1];
	double scal_h[GCG_MAX_BLOCK];
	/* x = Ritz vectors, b = (lambda + sigma) B x for the first `half` unconverged columns, :744-772 */
	int acc = 0;
	for (int b = 0; b < offset[0] && acc < half; ++b) {
		int len = offset[b * 2 + 2] - offset[b * 2 + 1];
		if (acc + len >= half) len = half - acc;
		const int o1 = offset[b * 2 + 1];
		TRY(b200k_axpby(g->n, len, 1.0, g->V->d + o1, g->V->ld, 0.0, g->V->d + g->startW + acc, g->V->ld));
		for (int i = 0; i < len; ++i) scal_h[acc + i] = ev[o1 + i] + sigma;
		acc += len;
	}
	TRY(b200k_h2d(g->scal_d, scal_h, sizeof(double) * (size_t)(acc > 0 ? acc : 1)));
	for (int pass = 0; pass < 2; ++pass) {
		/* right-hand side from the Ritz vectors in V (X part), stored in the Ritz-vector block; the
		 * shifted solve uses it as scratch, so it is rebuilt for the second solve (reference :836-858) */
		if (pass == 0 || (sigma != 0.0 && g->B)) {
			int a2 = 0;
			for (int b = 0; b < offset[0] && a2 < half; ++b) {
				int len = offset[b * 2 + 2] - offset[b * 2 + 1];
				if (a2 + len >= half) len = half - a2;
				const int o1 = offset[b * 2 + 1];
				TRY(spmm_mv(g->B, g->V->d + o1, g->V->ld, g->ritz->d + b0 + a2, g->ritz->ld, g->n, len));
				TRY(b200k_colscale(g->n, len, g->scal_d + a2, 0, g->ritz->d + b0 + a2, g->ritz->ld));
				a2 += len;
			}
		}
		if (pass == 1)      /* initial guess of the second solve = the first solution, :800-804 */
			TRY(b200k_axpby(g->n, acc, 1.0, g->V->d + g->startW, g->V->ld, 0.0, g->V->d + g->startW + acc, g->V->ld));
		double t1 = tick(g);
		b200_bpcg_params bp;
		bp.max_iter = p->compW_cg_max_iter; bp.rate = p->compW_cg_rate; bp.tol = p->compW_cg_tol;
		bp.tol_type = p->compW_cg_tol_type; bp.shift = sigma;
		int s[2], e[2];
		s[0] = b0; e[0] = b0 + acc; s[1] = g->startW + pass * acc; e[1] = s[1] + acc;
		if (acc > 0) TRY(b200_block_pcg_pc(g->A, g->B, g->ritz, g->V, s, e, &bp, p->compW_cg_pc, g->ws[0], g->ws[1], g->ws[2], NULL, NULL));
		g->st.linsol += tick(g) - t1;
	}
	g->endW = g->startW + 2 * acc;
	b200_orth_params op;
	op.block_size = p->compW_orth_block_size; op.max_reorth = p->compW_orth_max_reorth;
	op.orth_zero_tol = p->compW_orth_zero_tol; op.reorth_tol = 50 * DBL_EPSILON;
	TRY(orth_by(p->compW_orth_method, g->V, g->startW, &g->endW, g->B, &op, g->ws[0]));
	g->sizeW = g->endW - g->startW;
	g->st.compW += tick(g) - t0;
	return 0;
}

void b200_gcg_default_params(int nevConv, b200_gcg_params *p)
{
	/* reference test/test_eig_sol_gcg.c:33-115 */
	memset(p, 0, sizeof(*p));
	p->nevMax = 2 * nevConv;
	p->multiMax = 1; p->gapMin = 1e-5;
	p->block_size = nevConv < 30 ? (p->nevMax - nevConv) : nevConv / 5;
	p->nevInit = p->nevMax;
	p->numIterMax = 500; p->tol[0] = 1e-1; p->tol[1] = 1e-8;
	p->check_conv_max_num = 50;
	p->initX_orth_block_size = 80; p->initX_orth_max_reorth = 2; p->initX_orth_zero_tol = 2 * DBL_EPSILON;
	p->compP_orth_block_size = -1; p->compP_orth_max_reorth = 2; p->compP_orth_zero_tol = 2 * DBL_EPSILON;
	p->compW_orth_block_size = 80; p->compW_orth_max_reorth = 2; p->compW_orth_zero_tol = 2 * DBL_EPSILON;
	p->compW_cg_max_iter = 30; p->compW_cg_rate = 1e-2; p->compW_cg_tol = 1e-14; p->compW_cg_tol_type = 0;
	p->compW_cg_auto_shift = 0; p->compW_cg_shift = 0.0;
	p->compRR_tol = 2 * DBL_EPSILON;
	p->compW_cg_order = 1;
	p->verbose = 0;
	p->compW_cg_pc = 0;
}

/* The second [X | P | W] buffer is kept between solves (a solver object would own it; the reference's
 * EigenSolverSetup_GCG receives its workspaces from the caller, and its four do not include this one):
 * allocating ~n x (nevMax + 2 block_size) doubles inside every solve would sit in the timed region. */
static b200_mv *g_v2_cache;
/* ... and a block_size-wide block for the unknowns of the inner solve: BlockPCG reads and writes x in every step,
 * and as a block of [X P W] that is k*8-byte row segments at a (nevMax + 2 block_size)*8-byte pitch -- its two
 * streaming kernels run at 5.6 TB/s on that against 6.2 TB/s on a block of its own (profiles/bpcg_layout_r2i.log) */
static b200_mv *g_xw_cache;

void b200_gcg_free_cache(void)
{
	if (g_v2_cache) { b200_mv_destroy(g_v2_cache); g_v2_cache = NULL; }
	if (g_xw_cache) { b200_mv_destroy(g_xw_cache); g_xw_cache = NULL; }
}

static b200_mv *gcg_solve_buffer(const b200_mv *V, int ncols)
{
	if (g_xw_cache && (g_xw_cache->nrows_global != V->nrows_global || g_xw_cache->nrows != V->nrows ||
	                   g_xw_cache->ncols < ncols || g_xw_cache->ncols > ncols + 64 ||
	                   g_xw_cache->halo_cap < V->halo_cap || g_xw_cache->dist != V->dist)) {
		b200_mv_destroy(g_xw_cache); g_xw_cache = NULL;
	}
	if (!g_xw_cache && b200_mv_create(V->nrows_global, ncols, &g_xw_cache)) return NULL;
	return g_xw_cache;
}

static b200_mv *gcg_second_buffer(const b200_mv *V)
{
	if (g_v2_cache && (g_v2_cache->nrows_global != V->nrows_global || g_v2_cache->nrows != V->nrows ||
	                   g_v2_cache->ncols < V->ncols || g_v2_cache->ncols > V->ncols + 64 ||
	                   g_v2_cache->halo_cap < V->halo_cap || g_v2_cache->dist != V->dist))
		b200_gcg_free_cache();
	if (!g_v2_cache && b200_mv_create(V->nrows_global, V->ncols, &g_v2_cache)) return NULL;
	return g_v2_cache;
}

static void gcg_release(gcg_t *g)
{
	/* (the device work arrays live in scratch slot 9: nothing to free) */
	free(g->eval_h); free(g->res_h); free(g->offP); free(g->offW);
	if (g->own_ws) {
		b200_mv_destroy(g->V_alloc);
		for (int i = 0; i < 3; ++i) b200_mv_destroy(g->ws[i]);
	}
}

static int gcg_run(gcg_t *g, double *eval, int nevGiven, int *nevConv)
{
	const b200_gcg_params *p = g->p;
	const int bs = p->block_size, nevMax = p->nevMax, nevInit = p->nevInit;
	/* reference asserts :1275-1280 */
	if (!(nevInit >= nevGiven && nevInit <= nevMax && (nevInit >= 3 * bs || nevInit == nevMax) &&
	      nevMax >= *nevConv + bs && nevMax <= *nevConv + nevInit && p->multiMax <= bs))
		return b200_fail("gcg: inconsistent sizes nevConv=%d nevMax=%d nevInit=%d block_size=%d (reference asserts src/ops_eig_sol_gcg.c:1275-1280)",
		                 *nevConv, nevMax, nevInit, bs);
	int numIterMax = p->numIterMax;
	g->sizeC = 0; g->sizeN = bs; g->sizeX = nevInit; g->sizeP = 0; g->sizeW = 0;
	g->sizeV = g->sizeX; g->startN = 0; g->endN = bs; g->endX = g->sizeX;
	g->startP = g->endX; g->endP = g->startP; g->startW = g->endP; g->endW = g->startW;
	for (int i = 0; i < nevMax + 2 * bs; ++i) g->eval_h[i] = 1.0;
	TRY(b200k_h2d(g->eval_d, g->eval_h, sizeof(double) * (size_t)(nevMax + 2 * bs)));

	/* InitializeX, reference :101-158 */
	double t0 = tick(g);
	{
		b200_orth_params op;
		op.block_size = p->initX_orth_block_size; op.max_reorth = p->initX_orth_max_reorth;
		op.orth_zero_tol = p->initX_orth_zero_tol; op.reorth_tol = 50 * DBL_EPSILON;
		int ng = nevGiven;
		if (ng > 0) {
			TRY(b200k_axpby(g->n, ng, 1.0, g->ritz->d, g->ritz->ld, 0.0, g->V->d, g->V->ld));
			TRY(orth_by(p->initX_orth_method, g->V, 0, &ng, g->B, &op, g->ritz));
		}
		TRY(b200_mv_set_random(g->V, ng, g->sizeX));
		TRY(orth_by(p->initX_orth_method, g->V, ng, &g->endX, g->B, &op, g->ritz));
		if (g->endX != g->sizeX) return b200_fail("gcg: initial block is rank deficient (%d of %d), reference assert :143", g->endX, g->sizeX);
	}
	g->st.initX += tick(g) - t0;

	TRY(rayleigh_ritz(g, 0));
	TRY(compute_ritz_vec(g));

	if (*nevConv > nevMax) *nevConv = nevMax;
	const int nev0 = *nevConv; *nevConv = 0;
	int nev = nevInit < nevMax ? 2 * bs : nev0;
	if (nev > nev0) nev = nev0;
	int numIter = 0, numCheck;
	int *offsetP = g->offP, *offsetW = g->offW;
	if (p->verbose) printf("------------------------------\nnumIter\tnevConv\n");
	do {
		if (numIter <= 0) numCheck = 0;
		else numCheck = (g->startN + g->sizeN < g->endX) ? g->sizeN : (g->endX - g->startN);
		if (numCheck > p->check_conv_max_num) numCheck = p->check_conv_max_num;
		TRY(check_convergence(g, numCheck, offsetW, nevConv));
		if (p->verbose) printf("%d\t%d\n", numIter, *nevConv);
		if (*nevConv >= nev) {
			if (*nevConv >= nev0) break;
			/* grow X by P and W, reference :1400-1428 */
			nev += g->sizeP + g->sizeW; if (nev > nev0) nev = nev0;
			int newX = g->sizeX + g->sizeP + g->sizeW; if (newX > nevMax) newX = nevMax;
			const int N = g->sizeV - g->sizeC;
			TRY(b200k_lincomb(g->n, N, newX - g->endX, g->V->d + g->startN, g->V->ld,
			                  g->evec_d + (g->endX - g->sizeC), g->ldE, 1, NULL, 0,
			                  g->V2->d + g->endX, g->V2->ld));
			g->sizeX = newX;
			g->sizeP = 0; g->sizeW = 0; g->sizeV = g->sizeX;
			g->startP = g->endX; g->endP = g->startP; g->startW = g->endP; g->endW = g->startW;
			g->endX = g->sizeX;
			g->endN = g->startN + bs; if (g->endN > g->endX) g->endN = g->endX;
			g->sizeN = g->endN - g->startN;
			numIterMax -= numIter; numIter = 0;
		}
		if (numIter == 0) { g->sizeP = 0; g->startP = g->endX; g->endP = g->startP; }
		else TRY(compute_p(g, offsetP));
		/* ComputeX, reference :458-471 (V[:,startN:endX] = ritz_vec[:,startN:endX]): the buffer that holds
		 * the new X (and P) becomes V */
		{ b200_mv *tmp = g->V; g->V = g->V2; g->V2 = tmp; }
		if (p->compW_cg_order != 1) TRY(compute_w12(g, offsetW));      /* reference :1451-1456 */
		else TRY(compute_w(g, offsetW));
		{ int *tmp = offsetP; offsetP = offsetW; offsetW = tmp; }
		TRY(rayleigh_ritz(g, *nevConv));
		TRY(compute_ritz_vec(g));
		++numIter;
	} while (numIter < numIterMax);
	/* the eigenvectors: locked columns and the last Ritz vectors, reference ritz_vec == evec */
	TRY(b200k_axpby(g->n, g->sizeX, 1.0, g->V2->d, g->V2->ld, 0.0, g->ritz->d, g->ritz->ld));
	TRY(b200k_ar_check());
	g->st.numIter = numIter + (p->numIterMax - numIterMax);
	g->st.nevConv = *nevConv;
	memcpy(eval, g->eval_h, sizeof(double) * (size_t)g->sizeX);      /* reference :1508 */
	return 0;
}

int b200_gcg_solve(const b200_mat *A, const b200_mat *B, double *eval, b200_mv *evec,
                   int nevGiven, int *nevConv, const b200_gcg_params *prm, b200_mv **mv_ws,
                   b200_gcg_stats *stats)
{
	if (!A || !eval || !evec || !nevConv || !prm) return b200_fail("b200_gcg_solve: bad arguments");
	if (b200k_pending_flush()) return 1;
	if (A->nrows != A->ncols || evec->nrows != A->nrows) return b200_fail("b200_gcg_solve: shape mismatch");
	if (B && (B->nrows != A->nrows || B->ncols != A->ncols)) return b200_fail("b200_gcg_solve: B shape mismatch");
	const int bs = prm->block_size, nevMax = prm->nevMax;
	if (bs < 1 || bs > GCG_MAX_BLOCK) return b200_fail("b200_gcg_solve: block_size %d (1..%d supported)", bs, GCG_MAX_BLOCK);
	if (evec->ncols < nevMax) return b200_fail("b200_gcg_solve: evec has %d columns, nevMax = %d", evec->ncols, nevMax);
	gcg_t g; memset(&g, 0, sizeof(g));
	g.A = A; g.B = B; g.p = prm; g.n = A->nrows; g.ritz = evec; g.timing = 1;
	const int sizeVmax = nevMax + 2 * bs;
	int rc = 1;
	if (mv_ws) {
		g.V = mv_ws[0]; g.ws[0] = mv_ws[1]; g.ws[1] = mv_ws[2]; g.ws[2] = mv_ws[3];
		if (!g.V || g.V->ncols < sizeVmax || g.V->nrows != A->nrows) return b200_fail("b200_gcg_solve: mv_ws[0] needs %d columns", sizeVmax);
		for (int i = 0; i < 3; ++i)
			if (!g.ws[i] || g.ws[i]->ncols < bs || g.ws[i]->nrows != A->nrows) return b200_fail("b200_gcg_solve: mv_ws[%d] needs %d columns", i + 1, bs);
	} else {
		g.own_ws = 1;
		if (b200_mv_create(A->nrows_global, sizeVmax, &g.V)) return 1;
		g.V_alloc = g.V;
		for (int i = 0; i < 3; ++i) if (b200_mv_create(A->nrows_global, bs, &g.ws[i])) goto done;
	}
	g.V2 = gcg_second_buffer(g.V);
	if (!g.V2) goto done;
	g.xw = gcg_solve_buffer(g.V, prm->block_size);
	if (!g.xw) goto done;
	if (b200k_spmm_check_halo(A, g.xw) || (B && b200k_spmm_check_halo(B, g.xw))) goto done;
	if (b200k_spmm_check_halo(A, g.V2) || (B && b200k_spmm_check_halo(B, g.V2))) goto done;
	if (b200k_spmm_check_halo(A, g.V) || b200k_spmm_check_halo(A, evec) || b200k_spmm_check_halo(A, g.ws[1]) ||
	    (B && (b200k_spmm_check_halo(B, g.V) || b200k_spmm_check_halo(B, evec) || b200k_spmm_check_halo(B, g.ws[1]))))
		goto done;
	g.Nmax = prm->nevInit + 2 * bs; if (g.Nmax < sizeVmax) g.Nmax = sizeVmax;
	g.ldE = (g.Nmax + 3) & ~3;
	g.bsp = (bs + 3) & ~3;
	{
		/* the solver's small device arrays come out of one persistent scratch slot: cudaMalloc / cudaFree of nine
		 * buffers per solve is milliseconds on one GPU and up to seconds in a multi-GPU process (peer mappings, IPC) */
		const size_t cnt[9] = {(size_t)(sizeVmax + 8), (size_t)g.Nmax * g.ldE, (size_t)g.Nmax * g.ldE, (size_t)g.Nmax * g.bsp,
		                       (size_t)g.Nmax * g.bsp, (size_t)bs * bs, (size_t)(bs + 64), (size_t)(bs + 64), (size_t)(bs + 64)};
		size_t off[10]; off[0] = 0;
		for (int i = 0; i < 9; ++i) off[i + 1] = off[i] + ((cnt[i] * sizeof(double) + 255) & ~(size_t)255);
		char *slab = (char *)b200_scratch(9, off[9]);
		if (!slab || b200k_memset(slab, 0, off[9])) goto done;
		g.eval_d = (double *)(slab + off[0]); g.matA_d = (double *)(slab + off[1]); g.evec_d = (double *)(slab + off[2]);
		g.t1_d = (double *)(slab + off[3]); g.wsE_d = (double *)(slab + off[4]); g.ptap_d = (double *)(slab + off[5]);
		g.res_d = (double *)(slab + off[6]); g.scal_d = (double *)(slab + off[7]); g.idx_d = (int *)(slab + off[8]);
	}
	g.eval_h = (double *)calloc((size_t)sizeVmax + 8, sizeof(double));
	g.res_h = (double *)calloc((size_t)bs + 64, sizeof(double));
	g.offP = (int *)calloc(2 * (size_t)bs + 16, sizeof(int));
	g.offW = (int *)calloc(2 * (size_t)bs + 16, sizeof(int));
	{
		const double t0 = b200_wtime();
		const long long l0 = b200_kernel_launches();
		rc = gcg_run(&g, eval, nevGiven, nevConv);
		g.st.time_total = b200_wtime() - t0;
		g.st.launches = b200_kernel_launches() - l0;
	}
	if (rc == 0 && prm->verbose) {
		const b200_gcg_stats *s = &g.st;
		printf("|--GCG (B200)---------------------\n|Total Time = %.3f, Avg Time per Iteration = %.4f, kernel launches = %lld\n",
		       s->time_total, s->time_total / (s->numIter > 0 ? s->numIter : 1), s->launches);
		printf("|checkconv   compP   compRR   (eig)   compRV   compW   (linsol)   compX   initX\n");
		printf("|%.3f\t%.3f\t%.3f\t(%.3f)\t%.3f\t%.3f\t(%.3f)\t%.3f\t%.3f\n", s->checkconv, s->compP, s->compRR,
		       s->rr_eig, s->compRV, s->compW, s->linsol, s->compX, s->initX);
	}
	if (stats) *stats = g.st;
done:
	gcg_release(&g);
	return rc;
}
