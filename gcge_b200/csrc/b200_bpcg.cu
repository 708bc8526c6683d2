// K5: fused BlockPCG step kernels.  Replaces the per-column MultiVecAxpby / 'D' inner-product
// chain of the reference's BlockPCG (src/ops_lin_sol.c:256-405: ~6 single-column BLAS-1
// calls per column per iteration, every scalar on the host) by three streaming kernels per
// CG iteration that work on the whole column block at once, keep rho/alpha/beta, the residual
// norms, the per-column convergence masks and the iteration counter in HBM, and fold the
// global reductions into the streaming kernels (last-CTA reduction, b200_reduce.cuh).
// Nothing crosses to the host inside the CG loop.
//
// Per iteration, per column block k (algorithmic HBM traffic, SURVEY §8d):
//   update_px: read r,p,x    write p,x        5 * 8nk     x += alpha_prev p ; p = r + beta p
//   SpMM     : matrix + read p, write w       nnz*12 + 2 * 8nk   (+ p^T w in its epilogue, b200_spmm.cu)
//   ptw      : read p,w                       2 * 8nk     (only with a shift: read z, write w)
//   update_r : read w,r      write r          3 * 8nk     r -= alpha w ; rho = r^T r ; stop test
// The x update of iteration i is deferred into the p update of iteration i+1: x does not feed back
// into the iteration, so the iterates are bit-identical to the textbook order (x += alpha p next to
// r -= alpha w, 6 + 3 streams), and p is read once for both -- 8 streams instead of 9.
//
// Jacobi preconditioner (template flag JAC, st.dinv != NULL): z = D^-1 r is never stored.  begin and
// update_r form it in registers from the r they hold and add r^T z as one more accumulator; update_px
// forms it again from the r it reads, p = z + beta p.  D^-1 is one double per row shared by the k
// columns: +8n bytes per launch.  p^T A p is unchanged, so every SpMM path serves as it is.  The JAC =
// false instantiations are the unpreconditioned kernels unchanged.
#include "b200_stream.cuh"

constexpr int BPCG_CTAS_MAX = 8;                 // buffers are sized for this many CTAs per SM
// CTAs per SM the streaming kernels of the CG step are cut into (option bpcg_ctas, 1 ... 8; measured: profiles/)
static inline int bpcg_ctas() { const int v = b200_opt(B200_OPT_BPCG_CTAS); return (v >= 1 && v <= BPCG_CTAS_MAX) ? v : 6; }
#define BPCG_CTAS_PER_SM bpcg_ctas()

extern "C" int b200k_bpcg_state(int k, b200_bpcg_state *st)
{
	const int chunks_max = g_b200.num_sms * BPCG_CTAS_MAX + 8;
	const size_t dbl = (size_t)10 * k + (size_t)chunks_max * 3 * k;
	const size_t bytes = sizeof(double) * dbl + sizeof(int) * ((size_t)k + 8) + 64;
	char *base = (char *)b200_scratch(4, bytes);
	if (!base) return 1;
	double *d = (double *)base;
	st->k = k;
	st->norm_b = d; st->rho1 = d + k; st->rho2 = d + 2 * k; st->ptw = d + 3 * k;
	st->init_res = d + 4 * k; st->last_res = d + 5 * k;
	st->totals = d + 6 * k;                       /* 3k: per-column sums of the current reduction */
	st->alpha = d + 9 * k;                        /* k: step length of the x update still to be applied */
	st->partials = d + 10 * k;                    /* chunks x 3 accumulators x k */
	st->dinv = nullptr;
	int *ip = (int *)(d + dbl);
	st->active = ip; st->counters = ip + k; st->tickets = (unsigned *)(ip + k + 4);
	B200_CUDA(cudaMemsetAsync(st->counters, 0, sizeof(int) * 8, g_b200.stream));
	return 0;
}

// The tiny per-column scalar step that follows each reduction.  Single GPU: run by the last
// CTA of the streaming kernel itself.  Several ranks: the streaming kernel only leaves the
// per-column sums in st.totals, the host enqueues one ncclAllReduce on them (reference:
// MPI_Allreduce at src/ops_lin_sol.c:317,365) and then this runs as a one-CTA kernel -- every
// rank computes the same alpha / beta / masks from the same bits.
//   phase 0: after r = b - A x     phase 1: after p^T w     phase 2: after r -= alpha w
// totals: phase 0 [r^T r | b^T b | r^T z], phase 2 [r^T r | r^T z]; rho is r^T z with JAC, else r^T r
template <bool JAC>
__device__ __forceinline__ void bpcg_scalar_phase(int phase, int k, const b200_bpcg_state &st, double tol, int rel,
                                                  double rate)
{
	__shared__ int n_active;
	if (threadIdx.x == 0) n_active = 0;
	__syncthreads();
	for (int c = threadIdx.x; c < k; c += blockDim.x) {
		if (phase == 0) {
			const double rr = st.totals[c], bb = st.totals[k + c];
			const double rho = JAC ? st.totals[2 * k + c] : rr;
			const double nb = rel ? sqrt(bb) : 1.0;
			const double res = sqrt(rr);
			st.norm_b[c] = nb; st.rho2[c] = rho; st.rho1[c] = rho;
			st.init_res[c] = res; st.last_res[c] = res;
			const int act = (res > tol * nb) ? 1 : 0;      // reference src/ops_lin_sol.c:239-247
			st.active[c] = act;
			if (act) atomicAdd(&n_active, 1);
		} else if (phase == 1) {
			if (st.active[c]) st.ptw[c] = st.totals[c];
		} else if (st.active[c]) {
			const double rr = st.totals[c];
			st.rho1[c] = st.rho2[c];
			st.rho2[c] = JAC ? st.totals[k + c] : rr;
			const double res = sqrt(rr);
			st.last_res[c] = res;
			// reference src/ops_lin_sol.c:383-394: stay active while res > rate*res0 AND res > tol*||b||
			const int still = (res > rate * st.init_res[c]) && (res > tol * st.norm_b[c]);
			st.active[c] = still;
			if (still) atomicAdd(&n_active, 1);
		}
	}
	__syncthreads();
	if (threadIdx.x == 0) {
		if (phase == 0) { st.counters[0] = n_active; st.counters[1] = 0; }
		else if (phase == 2) { st.counters[0] = n_active; st.counters[1] += 1; }
	}
}

// last CTA: per-column totals of NACC accumulators into st.totals[a*k + c]
template <int NACC>
__device__ __forceinline__ void bpcg_store_totals(int k, const b200_bpcg_state &st)
{
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	for (int c = warp; c < k; c += ST_THREADS / 32) {
#pragma unroll
		for (int a = 0; a < NACC; ++a) {
			const double s = stream_total<NACC>(st.partials, gridDim.x, k, a, c);
			if (lane == 0) st.totals[a * k + c] = s;
		}
	}
	__syncthreads();
}

template <bool JAC>
__global__ void bpcg_finish_kernel(int phase, int k, b200_bpcg_state st, double tol, int rel, double rate)
{
	if (phase != 0 && st.counters[0] == 0) return;
	bpcg_scalar_phase<JAC>(phase, k, st, tol, rel, rate);
}

// ---------------------------------------------------------------------------- begin
// r <- b - r ; acc0 = r.r ; acc1 = b.b (rel only) ; JAC: acc2 = r.z, z = D^-1 r
template <int VEC, bool JAC>
__global__ void __launch_bounds__(ST_THREADS)
bpcg_begin_kernel(long long n, int k, StreamGeom g, const double *__restrict__ b, int ldb, double *__restrict__ r, int ldr,
                  double tol, int rel, int defer, b200_bpcg_state st, B200ArCtx ar)
{
	const StreamThread t = stream_thread<VEC>(g);
	const long long r_begin = (long long)blockIdx.x * g.rows_per_chunk;
	long long r_end = r_begin + g.rows_per_chunk; if (r_end > n) r_end = n;
	constexpr int NACC = JAC ? 3 : 2;
	double acc[NACC][VEC];
#pragma unroll
	for (int a = 0; a < NACC; ++a)
#pragma unroll
		for (int i = 0; i < VEC; ++i) acc[a][i] = 0.0;
	if (t.active) {
		for (long long row0 = r_begin + t.rl; row0 < r_end; row0 += (long long)ST_UNROLL * g.rp) {
			StV<VEC> bv[ST_UNROLL], rv[ST_UNROLL];
			double dv[ST_UNROLL];
#pragma unroll
			for (int u = 0; u < ST_UNROLL; ++u) {
				const long long row = row0 + (long long)u * g.rp;
				if (row < r_end) {
					bv[u] = st_ld<VEC>(b + (size_t)row * ldb + t.c); rv[u] = st_ld<VEC>(r + (size_t)row * ldr + t.c);
					if constexpr (JAC) dv[u] = st.dinv[row];
				}
			}
#pragma unroll
			for (int u = 0; u < ST_UNROLL; ++u) {
				const long long row = row0 + (long long)u * g.rp;
				if (row < r_end) {
#pragma unroll
					for (int i = 0; i < VEC; ++i) {
						const double x = bv[u].v[i] - rv[u].v[i];
						rv[u].v[i] = x;
						acc[0][i] = fma(x, x, acc[0][i]);
						acc[1][i] = fma(bv[u].v[i], bv[u].v[i], acc[1][i]);
						if constexpr (JAC) acc[NACC - 1][i] = fma(x, dv[u] * x, acc[NACC - 1][i]);
					}
					st_st<VEC>(r + (size_t)row * ldr + t.c, rv[u]);
				}
			}
		}
	}
	if (!stream_reduce_and_elect<VEC, NACC>(acc, k, g, t, st.partials, st.tickets)) return;
	bpcg_store_totals<NACC>(k, st);
	if (ar.nranks > 1) stream_allreduce_cta(ar, st.totals, NACC * k);
	if (!defer) bpcg_scalar_phase<JAC>(0, k, st, tol, rel, 0.0);
}

// ------------------------------------------------------------------------------ ptw
// w += shift z (optional) ; ptw = diag(p^T w)
template <int VEC>
__global__ void __launch_bounds__(ST_THREADS)
bpcg_ptw_kernel(long long n, int k, StreamGeom g, const double *p, int ldp, double *__restrict__ w, int ldw,
                double shift, const double *z, int ldz, int defer, b200_bpcg_state st, B200ArCtx ar)
{
	if (st.counters[0] == 0) return;
	const StreamThread t = stream_thread<VEC>(g);
	const long long r_begin = (long long)blockIdx.x * g.rows_per_chunk;
	long long r_end = r_begin + g.rows_per_chunk; if (r_end > n) r_end = n;
	double acc[1][VEC];
#pragma unroll
	for (int i = 0; i < VEC; ++i) acc[0][i] = 0.0;
	if (t.active) {
		for (long long row0 = r_begin + t.rl; row0 < r_end; row0 += (long long)ST_UNROLL * g.rp) {
			StV<VEC> pv[ST_UNROLL], wv[ST_UNROLL], zv[ST_UNROLL];
#pragma unroll
			for (int u = 0; u < ST_UNROLL; ++u) {
				const long long row = row0 + (long long)u * g.rp;
				if (row < r_end) {
					pv[u] = st_ld<VEC>(p + (size_t)row * ldp + t.c);
					wv[u] = st_ld<VEC>(w + (size_t)row * ldw + t.c);
					if (z) zv[u] = st_ld<VEC>(z + (size_t)row * ldz + t.c);
				}
			}
#pragma unroll
			for (int u = 0; u < ST_UNROLL; ++u) {
				const long long row = row0 + (long long)u * g.rp;
				if (row < r_end) {
					if (z) {       // w = (A + shift B) p, reference src/ops_eig_sol_gcg.c:63-96
#pragma unroll
						for (int i = 0; i < VEC; ++i) wv[u].v[i] = fma(shift, zv[u].v[i], wv[u].v[i]);
						st_st<VEC>(w + (size_t)row * ldw + t.c, wv[u]);
					}
#pragma unroll
					for (int i = 0; i < VEC; ++i) acc[0][i] = fma(pv[u].v[i], wv[u].v[i], acc[0][i]);
				}
			}
		}
	}
	if (!stream_reduce_and_elect<VEC, 1>(acc, k, g, t, st.partials, st.tickets)) return;
	bpcg_store_totals<1>(k, st);
	if (ar.nranks > 1) stream_allreduce_cta(ar, st.totals, k);
	if (!defer) bpcg_scalar_phase<false>(1, k, st, 0.0, 0, 0.0);
}

// ------------------------------------------------------------------------- update_r
// alpha = rho2/ptw ; r -= alpha w ; rho1 = rho2 ; rho2 = diag(r^T r) (JAC: diag(r^T z)) ; stop test on
// sqrt(r^T r).  alpha is left in st.alpha for the deferred x update; counters[2] = it + 1 says which
// iteration it belongs to.
template <int VEC, bool JAC>
__global__ void __launch_bounds__(ST_THREADS)
bpcg_update_r_kernel(long long n, int k, StreamGeom g, const double *__restrict__ w, int ldw, double *__restrict__ r, int ldr,
                     double rate, double tol, int it, int defer, b200_bpcg_state st, B200ArCtx ar)
{
	if (st.counters[0] == 0) return;
	const StreamThread t = stream_thread<VEC>(g);
	const long long r_begin = (long long)blockIdx.x * g.rows_per_chunk;
	long long r_end = r_begin + g.rows_per_chunk; if (r_end > n) r_end = n;
	constexpr int NACC = JAC ? 2 : 1;
	double acc[NACC][VEC], alpha[VEC];
	bool act[VEC]; bool any = false;
#pragma unroll
	for (int i = 0; i < VEC; ++i) {
#pragma unroll
		for (int a = 0; a < NACC; ++a) acc[a][i] = 0.0;
		act[i] = t.active && st.active[t.c + i];
		alpha[i] = act[i] ? st.rho2[t.c + i] / st.ptw[t.c + i] : 0.0;       // reference src/ops_lin_sol.c:328
		any = any || act[i];
	}
	if (blockIdx.x == 0 && t.active && t.rl == 0) {
#pragma unroll
		for (int i = 0; i < VEC; ++i) st.alpha[t.c + i] = alpha[i];
		if (t.cg == 0) st.counters[2] = it + 1;
	}
	if (any) {
		for (long long row0 = r_begin + t.rl; row0 < r_end; row0 += (long long)ST_UNROLL * g.rp) {
			StV<VEC> wv[ST_UNROLL], rv[ST_UNROLL];
			double dv[ST_UNROLL];
#pragma unroll
			for (int u = 0; u < ST_UNROLL; ++u) {
				const long long row = row0 + (long long)u * g.rp;
				if (row < r_end) {
					wv[u] = st_ld<VEC>(w + (size_t)row * ldw + t.c);
					rv[u] = st_ld<VEC>(r + (size_t)row * ldr + t.c);
					if constexpr (JAC) dv[u] = st.dinv[row];
				}
			}
#pragma unroll
			for (int u = 0; u < ST_UNROLL; ++u) {
				const long long row = row0 + (long long)u * g.rp;
				if (row < r_end) {
#pragma unroll
					for (int i = 0; i < VEC; ++i) {
						if (act[i]) {
							const double nr = fma(-alpha[i], wv[u].v[i], rv[u].v[i]);
							rv[u].v[i] = nr;
							acc[0][i] = fma(nr, nr, acc[0][i]);
							if constexpr (JAC) acc[NACC - 1][i] = fma(nr, dv[u] * nr, acc[NACC - 1][i]);
						}
					}
					st_st<VEC>(r + (size_t)row * ldr + t.c, rv[u]);
				}
			}
		}
	}
	if (!stream_reduce_and_elect<VEC, NACC>(acc, k, g, t, st.partials, st.tickets)) return;
	bpcg_store_totals<NACC>(k, st);
	if (ar.nranks > 1) stream_allreduce_cta(ar, st.totals, NACC * k);
	if (!defer) bpcg_scalar_phase<JAC>(2, k, st, tol, 0, rate);
}

// ------------------------------------------------------------------------ update_px
// x += alpha p for the step length left by update_r of iteration `expect - 1` (if any), then
// p = r + (rho2/rho1) p on the columns still active (reference src/ops_lin_sol.c:271-284, :330-340);
// JAC: p = D^-1 r + (rho2/rho1) p.  flush: only the x update (after the last iteration).
template <int VEC, bool JAC>
__global__ void __launch_bounds__(ST_THREADS)
bpcg_update_px_kernel(long long n, int k, StreamGeom g, const double *__restrict__ r, int ldr, double *__restrict__ p,
                      int ldp, double *__restrict__ x, int ldx, int first, int expect, int flush, b200_bpcg_state st)
{
	const bool pending = !first && st.counters[2] == expect;
	const bool running = !flush && st.counters[0] != 0;
	if (!pending && !running) return;
	const StreamThread t = stream_thread<VEC>(g);
	if (!t.active) return;
	bool act[VEC]; double beta[VEC], al[VEC]; bool any_p = false, any_x = false;
#pragma unroll
	for (int i = 0; i < VEC; ++i) {
		act[i] = running && st.active[t.c + i] != 0;
		beta[i] = (act[i] && !first) ? st.rho2[t.c + i] / st.rho1[t.c + i] : 0.0;
		al[i] = pending ? st.alpha[t.c + i] : 0.0;
		any_p = any_p || act[i];
		any_x = any_x || (al[i] != 0.0);
	}
	if (!any_p && !any_x) return;
	const long long r_begin = (long long)blockIdx.x * g.rows_per_chunk;
	long long r_end = r_begin + g.rows_per_chunk; if (r_end > n) r_end = n;
	for (long long row0 = r_begin + t.rl; row0 < r_end; row0 += (long long)ST_UNROLL * g.rp) {
		StV<VEC> rv[ST_UNROLL], pv[ST_UNROLL], xv[ST_UNROLL];
		double dv[ST_UNROLL];
#pragma unroll
		for (int u = 0; u < ST_UNROLL; ++u) {
			const long long row = row0 + (long long)u * g.rp;
			if (row < r_end) {
				if (any_p) rv[u] = st_ld<VEC>(r + (size_t)row * ldr + t.c);
				if constexpr (JAC) { if (any_p) dv[u] = st.dinv[row]; }
				pv[u] = st_ld<VEC>(p + (size_t)row * ldp + t.c);
				if (any_x) xv[u] = st_ld<VEC>(x + (size_t)row * ldx + t.c);
			}
		}
#pragma unroll
		for (int u = 0; u < ST_UNROLL; ++u) {
			const long long row = row0 + (long long)u * g.rp;
			if (row < r_end) {
				if (any_x) {
#pragma unroll
					for (int i = 0; i < VEC; ++i)
						if (al[i] != 0.0) xv[u].v[i] = fma(al[i], pv[u].v[i], xv[u].v[i]);
					st_st<VEC>(x + (size_t)row * ldx + t.c, xv[u]);
				}
				if (any_p) {
					if constexpr (JAC) {
#pragma unroll
						for (int i = 0; i < VEC; ++i) rv[u].v[i] *= dv[u];
					}
#pragma unroll
					for (int i = 0; i < VEC; ++i)
						if (act[i]) pv[u].v[i] = first ? rv[u].v[i] : fma(beta[i], pv[u].v[i], rv[u].v[i]);
					st_st<VEC>(p + (size_t)row * ldp + t.c, pv[u]);
				}
			}
		}
	}
}

// ------------------------------------------------------------------------- launchers
// in-kernel allreduce context when the reduction fits it (several ranks, <= B200_AR_MAX_COUNT values)
static B200ArCtx bpcg_ar(int count)
{
	B200ArCtx ar = b200k_ar_ctx();
	if (count > B200_AR_MAX_COUNT) ar.nranks = 0;
	return ar;
}

// several ranks: sum the per-column totals over the ranks, then the scalar step
static int bpcg_finish(int phase, int nacc, const b200_bpcg_state *st, double tol, int rel, double rate)
{
	if (b200k_allreduce_sum(st->totals, (size_t)nacc * st->k)) return 1;
	if (st->dinv && phase != 1) bpcg_finish_kernel<true><<<1, 128, 0, g_b200.stream>>>(phase, st->k, *st, tol, rel, rate);
	else bpcg_finish_kernel<false><<<1, 128, 0, g_b200.stream>>>(phase, st->k, *st, tol, rel, rate);
	B200_KERNEL_CHECK();
	return 0;
}

extern "C" int b200k_bpcg_begin(long long n, const b200_bpcg_state *st, const double *b, int ldb,
                                double *r, int ldr, double tol, int rel)
{
	const int k = st->k;
	const bool jac = st->dinv != nullptr;
	const int nacc = jac ? 3 : 2;
	const B200ArCtx ar = bpcg_ar(nacc * k);
	const int defer = (b200_multi() && ar.nranks == 0) ? 1 : 0;
	B200_CHECK(k >= 1 && k <= 128, "BlockPCG: %d columns (1..128 supported per block)", k);
	B200Prof prof(B200_PROF_BPCG, 24.0 * n * k + (jac ? 8.0 * n : 0.0), (jac ? 8.0 : 5.0) * n * k);
	const StreamGeom g = stream_geometry(n, k, stream_aligned16(b, ldb) && stream_aligned16(r, ldr), BPCG_CTAS_PER_SM);
	if (jac)
		ST_DISPATCH_VEC(g, (bpcg_begin_kernel<VEC, true><<<g.chunks, ST_THREADS, 0, g_b200.stream>>>(n, k, g, b, ldb, r, ldr, tol, rel, defer, *st, ar)));
	else
		ST_DISPATCH_VEC(g, (bpcg_begin_kernel<VEC, false><<<g.chunks, ST_THREADS, 0, g_b200.stream>>>(n, k, g, b, ldb, r, ldr, tol, rel, defer, *st, ar)));
	B200_KERNEL_CHECK();
	if (defer) return bpcg_finish(0, nacc, st, tol, rel, 0.0);
	return 0;
}

extern "C" int b200k_bpcg_ptw(long long n, const b200_bpcg_state *st, const double *p, int ldp,
                              double *w, int ldw, double shift, const double *z, int ldz)
{
	const int k = st->k;
	const B200ArCtx ar = bpcg_ar(k);
	const int defer = (b200_multi() && ar.nranks == 0) ? 1 : 0;
	B200Prof prof(B200_PROF_BPCG, (z ? 32.0 : 16.0) * n * k, (z ? 4.0 : 2.0) * n * k);
	const StreamGeom g = stream_geometry(n, k, stream_aligned16(p, ldp) && stream_aligned16(w, ldw) &&
	                                     (!z || stream_aligned16(z, ldz)), BPCG_CTAS_PER_SM);
	ST_DISPATCH_VEC(g, (bpcg_ptw_kernel<VEC><<<g.chunks, ST_THREADS, 0, g_b200.stream>>>(n, k, g, p, ldp, w, ldw, shift, z, ldz, defer, *st, ar)));
	B200_KERNEL_CHECK();
	if (defer) return bpcg_finish(1, 1, st, 0.0, 0, 0.0);
	return 0;
}

// p^T w from the per-CTA partials the fused SpMM left in st.partials[part][k]
__global__ void __launch_bounds__(ST_THREADS)
bpcg_ptw_parts_kernel(int nparts, int k, int defer, b200_bpcg_state st, B200ArCtx ar)
{
	if (st.counters[0] == 0) return;
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	for (int c = warp; c < k; c += ST_THREADS / 32) {
		const double s = stream_total<1>(st.partials, nparts, k, 0, c);
		if (lane == 0) st.totals[c] = s;
	}
	__syncthreads();
	if (ar.nranks > 1) stream_allreduce_cta(ar, st.totals, k);
	if (!defer) bpcg_scalar_phase<false>(1, k, st, 0.0, 0, 0.0);
}

int b200k_spmm_dot(const b200_mat *M, const double *x, int ldx, double *y, int ldy, int k, const int *gate,
                   double *dot_part, int dot_cap, int *nparts);

// w = A p and ptw = diag(p^T w) in one pass over p (SpMM with the dot in its epilogue) when the
// matrix has a diagonal image; otherwise the SpMM followed by the streaming dot kernel.
extern "C" int b200k_bpcg_spmm_ptw(const b200_mat *A, long long n, const b200_bpcg_state *st, const double *p, int ldp,
                                   double *w, int ldw)
{
	const int k = st->k;
	const B200ArCtx ar = bpcg_ar(k);
	const int defer = (b200_multi() && ar.nranks == 0) ? 1 : 0;
	const int cap = g_b200.num_sms * BPCG_CTAS_PER_SM;       // rows of k doubles available in st->partials (x2)
	int nparts = 0;
	const int rc = b200k_spmm_dot(A, p, ldp, w, ldw, k, st->counters, st->partials, cap, &nparts);
	if (rc == 1) return 1;
	if (rc == 2) {
		if (b200k_spmm(A, 0, p, ldp, w, ldw, k, st->counters)) return 1;
		return b200k_bpcg_ptw(n, st, p, ldp, w, ldw, 0.0, nullptr, 0);
	}
	{
		// booked with the small dense work: a one-CTA reduction of nparts x k partials -- counting it as a launch of
		// the streaming class would halve that class's algorithmic bytes per launch for no traffic of its own
		B200Prof prof(B200_PROF_SMALL, 8.0 * nparts * k, 1.0 * nparts * k);
		bpcg_ptw_parts_kernel<<<1, ST_THREADS, 0, g_b200.stream>>>(nparts, k, defer, *st, ar);
		B200_KERNEL_CHECK();
	}
	if (defer) return bpcg_finish(1, 1, st, 0.0, 0, 0.0);
	return 0;
}

extern "C" int b200k_bpcg_update_r(long long n, const b200_bpcg_state *st, const double *w, int ldw, double *r, int ldr,
                                   double rate, double tol, int it)
{
	const int k = st->k;
	const bool jac = st->dinv != nullptr;
	const int nacc = jac ? 2 : 1;
	const B200ArCtx ar = bpcg_ar(nacc * k);
	const int defer = (b200_multi() && ar.nranks == 0) ? 1 : 0;
	B200Prof prof(B200_PROF_BPCG, 24.0 * n * k + (jac ? 8.0 * n : 0.0), (jac ? 7.0 : 4.0) * n * k);
	const StreamGeom g = stream_geometry(n, k, stream_aligned16(w, ldw) && stream_aligned16(r, ldr), BPCG_CTAS_PER_SM);
	if (jac)
		ST_DISPATCH_VEC(g, (bpcg_update_r_kernel<VEC, true><<<g.chunks, ST_THREADS, 0, g_b200.stream>>>(n, k, g, w, ldw, r, ldr, rate, tol, it, defer, *st, ar)));
	else
		ST_DISPATCH_VEC(g, (bpcg_update_r_kernel<VEC, false><<<g.chunks, ST_THREADS, 0, g_b200.stream>>>(n, k, g, w, ldw, r, ldr, rate, tol, it, defer, *st, ar)));
	B200_KERNEL_CHECK();
	if (defer) return bpcg_finish(2, nacc, st, tol, 0, rate);
	return 0;
}

// it: the iteration whose p is being formed (0 = first: p = r, nothing pending); flush != 0: only the
// pending x update of iteration it - 1
extern "C" int b200k_bpcg_update_px(long long n, const b200_bpcg_state *st, const double *r, int ldr, double *p, int ldp,
                                    double *x, int ldx, int it, int flush)
{
	const int k = st->k;
	const bool jac = st->dinv != nullptr && !flush;       // the flush updates x only
	B200Prof prof(B200_PROF_BPCG, (flush ? 24.0 : (it == 0 ? 24.0 : 40.0)) * n * k + (jac ? 8.0 * n : 0.0),
	              (jac ? 5.0 : 4.0) * n * k);
	const StreamGeom g = stream_geometry(n, k, stream_aligned16(r, ldr) && stream_aligned16(p, ldp) && stream_aligned16(x, ldx),
	                                     BPCG_CTAS_PER_SM);
	if (jac)
		ST_DISPATCH_VEC(g, (bpcg_update_px_kernel<VEC, true><<<g.chunks, ST_THREADS, 0, g_b200.stream>>>(n, k, g, r, ldr, p, ldp, x, ldx,
		                                                                                               it == 0, it, flush, *st)));
	else
		ST_DISPATCH_VEC(g, (bpcg_update_px_kernel<VEC, false><<<g.chunks, ST_THREADS, 0, g_b200.stream>>>(n, k, g, r, ldr, p, ldp, x, ldx,
		                                                                                                it == 0, it, flush, *st)));
	B200_KERNEL_CHECK();
	return 0;
}

// ------------------------------------------------------------------------- Jacobi diagonal
// the entry (row, row) of a CSR; found = false when it is not stored.  On a row slab the diagonal of local row r has
// local column r in both halo layouts (b200_dev.h, struct b200_mat_).  A linear scan: the remapped columns of a slab
// with a scattered halo are not ascending, and the rows are short.
__device__ __forceinline__ double csr_diag(const int *__restrict__ rp, const int *__restrict__ ci, const double *__restrict__ va,
                                           int row, bool &found)
{
	const int e1 = rp[row + 1];
	for (int e = rp[row]; e < e1; ++e)
		if (ci[e] == row) { found = true; return va[e]; }
	found = false;
	return 0.0;
}

// dinv[row] = 1 / (a_rr + shift b_rr)  (bmode 1),  1 / (a_rr + shift)  (bmode 2),  1 / a_rr  (bmode 0).
// bad[0] counts the rows without a stored diagonal or with one that is not > 0 (NaN included); ibad[0] = the smallest
// such row (memset to 0x7f7f7f7f before).
__global__ void __launch_bounds__(256)
bpcg_jacobi_diag_kernel(int n, const int *__restrict__ arp, const int *__restrict__ aci, const double *__restrict__ ava,
                        const int *__restrict__ brp, const int *__restrict__ bci, const double *__restrict__ bva,
                        double shift, int bmode, double *__restrict__ dinv, double *__restrict__ bad, int *__restrict__ ibad)
{
	for (int row = blockIdx.x * blockDim.x + threadIdx.x; row < n; row += gridDim.x * blockDim.x) {
		bool fa = false, fb = true;
		double d = csr_diag(arp, aci, ava, row, fa);
		if (bmode == 1) d += shift * csr_diag(brp, bci, bva, row, fb);
		else if (bmode == 2) d += shift;
		if (!fa || !fb || !(d > 0.0)) {
			atomicAdd(bad, 1.0);
			atomicMin(ibad, row);
			d = 1.0;                      // the solve does not run; keep the buffer finite
		}
		dinv[row] = 1.0 / d;
	}
}

extern "C" int b200k_bpcg_jacobi(const b200_mat *A, const b200_mat *B, double shift, const double **dinv_dev)
{
	const int n = A->nrows;
	B200_CHECK(A->rp && A->ci && A->va, "BlockPCG Jacobi: the matrix has no device CSR image");
	const int bmode = (shift == 0.0) ? 0 : (B ? 1 : 2);
	if (bmode == 1) B200_CHECK(B->nrows == n && B->rp && B->ci && B->va, "BlockPCG Jacobi: B does not match A's rows");
	char *base = (char *)b200_scratch(10, sizeof(double) * ((size_t)n + 4) + 64);
	if (!base) return 1;
	double *dinv = (double *)base, *bad = dinv + n;
	int *ibad = (int *)(bad + 2);
	B200_CUDA(cudaMemsetAsync(bad, 0, sizeof(double), g_b200.stream));
	B200_CUDA(cudaMemsetAsync(ibad, 0x7f, sizeof(int), g_b200.stream));
	{
		B200Prof prof(B200_PROF_BPCG, 4.0 * n + 12.0 * A->nnz + (bmode == 1 ? 4.0 * n + 12.0 * B->nnz : 0.0) + 8.0 * n,
		              (bmode == 1 ? 3.0 : 2.0) * n);
		const int blocks = n > 0 ? b200_ceil_div(n, 256) : 1;
		bpcg_jacobi_diag_kernel<<<blocks < 65535 * 16 ? blocks : 65535 * 16, 256, 0, g_b200.stream>>>(
		    n, A->rp, A->ci, A->va, bmode == 1 ? B->rp : nullptr, bmode == 1 ? B->ci : nullptr, bmode == 1 ? B->va : nullptr,
		    shift, bmode, dinv, bad, ibad);
		B200_KERNEL_CHECK();
	}
	// every rank has to take the same branch: the count of bad rows is summed over the ranks
	if (b200_multi() && b200k_allreduce_sum(bad, 1)) return 1;
	double nbad = 0.0; int first = 0;
	if (b200k_d2h(&nbad, bad, sizeof(double)) || b200k_d2h(&first, ibad, sizeof(int))) return 1;
	if (nbad != 0.0) {
		if (first < n)
			return b200_fail("BlockPCG Jacobi: %.0f rows of A + shift*B (shift %g) have no diagonal entry or one <= 0 "
			                 "(first: row %lld)", nbad, shift, (long long)A->row0 + first);
		return b200_fail("BlockPCG Jacobi: %.0f rows of A + shift*B (shift %g) have no diagonal entry or one <= 0 "
		                 "(on another rank)", nbad, shift);
	}
	*dinv_dev = dinv;
	return 0;
}
