/* b200_bpcg.c -- host driver of the fused device BlockPCG (C-ABI b200_block_pcg).
 *
 * Replaces BlockPCG (reference src/ops_lin_sol.c:140-437).  The reference's loop makes, per
 * CG iteration, one single-column MultiVecAxpby per column for p, one SpMM and one 'D'
 * inner product per contiguous index block, two more single-column axpbys per column, and
 * decides convergence on the host from scalars it pulled back.  Here one iteration is a
 * fixed sequence of launches on the whole block (update_px, SpMM with p^T w in its epilogue,
 * update_r; with a shift: update_px, SpMM, SpMM, ptw, update_r);
 * rho/alpha/beta, the residual norms, the active-column masks and the iteration counter
 * stay in HBM, and every launch returns at once when no column is active any more, so the
 * host never reads anything back inside the loop.  Converged columns are frozen exactly as
 * in the reference (their x, r, p are no longer updated).
 *
 * pc = 1 (b200_block_pcg_pc): point Jacobi, D = diag(A + shift B).  D^-1 is formed once per call by one
 * kernel over the device CSR (the only synchronisation it adds: a bad diagonal fails the call before
 * anything is written), and z = D^-1 r lives in registers of the streaming kernels only.
 */
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <stdio.h>
#include "b200_dev.h"

#define BPCG_MAX_K 128

static int bpcg_chunk(const b200_mat *A, const b200_mat *B, long long n,
                      double *b, int ldb, double *x, int ldx, int k, const b200_bpcg_params *prm,
                      double *r, int ldr, double *p, int ldp, double *w, int ldw, const double *dinv,
                      int *niter, double *residual)
{
	b200_bpcg_state st;
	if (b200k_bpcg_state(k, &st)) return 1;
	st.dinv = dinv;
	const double shift = prm->shift;
	/* r = (A + shift B) x, then r = b - r and the initial masks */
	if (b200k_spmm(A, 0, x, ldx, r, ldr, k, NULL)) return 1;
	if (shift != 0.0) {
		if (B) {
			if (b200k_spmm(B, 0, x, ldx, p, ldp, k, NULL)) return 1;
			if (b200k_axpby(n, k, shift, p, ldp, 1.0, r, ldr)) return 1;
		} else {
			if (b200k_axpby(n, k, shift, x, ldx, 1.0, r, ldr)) return 1;
		}
	}
	if (b200k_bpcg_begin(n, &st, b, ldb, r, ldr, prm->tol, prm->tol_type == 1)) return 1;
	/* B200_BPCG_TRACE=1 (diagnostic, synchronises every iteration): column-iterations really needed
	 * vs. launched -- how much a compaction of the active columns could save */
	const int trace = b200k_opt(B200K_OPT_BPCG_TRACE);
	long long act_sum = 0, iters_run = 0;
	int it = 0;
	for (; it < prm->max_iter; ++it) {
		if (trace) {
			int c2[2];
			if (b200k_d2h(c2, st.counters, sizeof(c2))) return 1;
			if (c2[0] == 0) break;
			act_sum += c2[0]; ++iters_run;
		}
		/* x += alpha_{it-1} p_{it-1} (deferred), p_it = r + beta p_{it-1} */
		if (b200k_bpcg_update_px(n, &st, r, ldr, p, ldp, x, ldx, it, 0)) return 1;
		if (shift == 0.0) {
			/* w = A p with p^T w in the SpMM epilogue */
			if (b200k_bpcg_spmm_ptw(A, n, &st, p, ldp, w, ldw)) return 1;
		} else {
			if (b200k_spmm(A, 0, p, ldp, w, ldw, k, st.counters)) return 1;
			if (B) {
				/* the right-hand side is dead after the initial residual: use it as B p, like the
				 * reference's MatDotMultiVecShift does (src/ops_eig_sol_gcg.c:63-96) */
				if (b200k_spmm(B, 0, p, ldp, b, ldb, k, st.counters)) return 1;
				if (b200k_bpcg_ptw(n, &st, p, ldp, w, ldw, shift, b, ldb)) return 1;
			} else {
				if (b200k_bpcg_ptw(n, &st, p, ldp, w, ldw, shift, p, ldp)) return 1;
			}
		}
		if (b200k_bpcg_update_r(n, &st, w, ldw, r, ldr, prm->rate, prm->tol, it)) return 1;
	}
	/* the x update of the last iteration that ran; `it`, not max_iter: the trace leaves the loop early */
	if (b200k_bpcg_update_px(n, &st, r, ldr, p, ldp, x, ldx, it, 1)) return 1;
	if (trace) fprintf(stderr, "bpcg k=%d: %lld iterations, active column-iterations %lld of %lld (%.0f %%)\n", k, iters_run,
	                   act_sum, iters_run * k, iters_run ? 100.0 * act_sum / (iters_run * k) : 0.0);
	if (niter || residual) {
		int counters[2];
		if (b200k_ar_check()) return 1;
		double res[BPCG_MAX_K];
		if (b200k_d2h(counters, st.counters, sizeof(counters))) return 1;
		if (b200k_d2h(res, st.last_res, sizeof(double) * (size_t)k)) return 1;
		if (niter && counters[1] > *niter) *niter = counters[1];
		if (residual) for (int i = 0; i < k; ++i) if (res[i] > *residual) *residual = res[i];
	}
	return 0;
}

int b200_block_pcg_pc(const b200_mat *A, const b200_mat *B, b200_mv *b, b200_mv *x,
                      const int *start, const int *end, const b200_bpcg_params *prm, int pc,
                      b200_mv *ws_r, b200_mv *ws_p, b200_mv *ws_w, int *niter, double *residual)
{
	if (!A || !b || !x || !start || !end || !prm || !ws_r || !ws_p || !ws_w)
		return b200_fail("b200_block_pcg: bad arguments");
	if (pc != 0 && pc != 1) return b200_fail("b200_block_pcg: preconditioner %d (0 none, 1 Jacobi)", pc);
	if (b200k_pending_flush()) return 1;
	const int k = end[0] - start[0];
	if (k != end[1] - start[1]) return b200_fail("b200_block_pcg: column counts differ");
	if (k <= 0) return 0;
	if (start[0] < 0 || end[0] > b->ncols || start[1] < 0 || end[1] > x->ncols)
		return b200_fail("b200_block_pcg: column range out of bounds");
	const long long n = x->nrows;
	if (A->nrows != n || A->ncols != n || b->nrows != n || ws_r->nrows != n || ws_p->nrows != n || ws_w->nrows != n)
		return b200_fail("b200_block_pcg: shape mismatch");
	if (b200k_spmm_check_halo(A, x) || b200k_spmm_check_halo(A, ws_p)) return 1;
	if (B && prm->shift != 0.0 && (b200k_spmm_check_halo(B, x) || b200k_spmm_check_halo(B, ws_p))) return 1;
	if (niter) *niter = 0;
	if (residual) *residual = 0.0;
	int wk = ws_r->ncols;
	if (ws_p->ncols < wk) wk = ws_p->ncols;
	if (ws_w->ncols < wk) wk = ws_w->ncols;
	if (wk > BPCG_MAX_K) wk = BPCG_MAX_K;
	if (wk < 1) return b200_fail("b200_block_pcg: workspaces have no columns");
	const double *dinv = NULL;
	if (pc == 1 && b200k_bpcg_jacobi(A, B, prm->shift, &dinv)) return 1;      /* D^-1 of the whole call, before x is touched */
	for (int c0 = 0; c0 < k; c0 += wk) {
		const int kc = (k - c0 < wk) ? k - c0 : wk;
		if (bpcg_chunk(A, B, n, b->d + start[0] + c0, b->ld, x->d + start[1] + c0, x->ld, kc, prm,
		               ws_r->d, ws_r->ld, ws_p->d, ws_p->ld, ws_w->d, ws_w->ld, dinv, niter, residual))
			return 1;
	}
	return 0;
}

int b200_block_pcg(const b200_mat *A, const b200_mat *B, b200_mv *b, b200_mv *x,
                   const int *start, const int *end, const b200_bpcg_params *prm,
                   b200_mv *ws_r, b200_mv *ws_p, b200_mv *ws_w, int *niter, double *residual)
{
	return b200_block_pcg_pc(A, B, b, x, start, end, prm, 0, ws_r, ws_p, ws_w, niter, residual);
}
