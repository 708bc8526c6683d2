// K7: on-device eigen-solve of the projected Rayleigh-Ritz problem (N <= 3*nev, a few hundred).
// Replaces the host dsyevx call of the reference (src/ops_eig_sol_gcg.c:1201-1204) so the
// projected matrix and the Ritz coefficients never leave HBM.
//
// Two-sided cyclic Jacobi, organised so that the number of GRID-WIDE steps per sweep is N/16
// instead of N.  The first version of this kernel rotated element pairs directly on the N x N
// matrix: N-1 rounds per sweep, one grid barrier and one pass over A and V each -- 31 ms at
// N = 480 (11 sweeps x 479 rounds x ~6 us), all of it barrier latency.  Here the indices are
// grouped in blocks of 16 and the blocks meet pairwise in a round-robin tournament (circle
// method, NB-1 block rounds per sweep):
//
//   phase 1  one CTA per block pair (P, Q): the 32 x 32 pivot matrix is pulled into shared
//            memory and every index pair (p in P, q in Q) is rotated once -- 16 inner rounds of
//            16 disjoint rotations, __syncthreads only; in block round 0 of a sweep the inner
//            tournament is the full one over all 32 indices, so pairs inside a block are
//            rotated once per sweep as well.  The product of the rotations is kept as a
//            32 x 32 orthogonal block J.
//   phase 2  every other 32 x 32 tile of A gets J_I^T T J_J, every 32-row tile of V gets T J_J:
//            small dense products spread over the whole grid.
//
// Mathematically this is still an element-wise cyclic Jacobi method -- every index pair is
// rotated exactly once per sweep, in a parallel ordering -- so accuracy and sweep counts are
// those of the plain method (measured: 10 sweeps on a projected matrix of order 480, 11 with
// the element ordering), but a sweep costs 2 (NB-1) grid barriers instead of N-1 and the bulk
// of the arithmetic runs as 32 x 32 x 32 products out of shared memory.
// Rotations are skipped under the relative criterion |a_pq| <= eps*sqrt(|a_pp a_qq|); a sweep
// that applies no rotation ends the iteration.  All decisions are integer counts, so the
// result is run-to-run deterministic and identical on every rank of a multi-GPU run.
#include "b200_internal.h"
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

constexpr int BJ_B = 16;            // indices per block
constexpr int BJ_T = 2 * BJ_B;      // order of a pivot matrix
constexpr int BJ_LD = BJ_T + 4;     // shared-memory row stride == 4 (mod 16) doubles: two-wavefront DMMA fragment loads
constexpr int BJ_TILE = BJ_T * BJ_LD;

// circle method: the two members of pair k in round r of a tournament of N players (N even)
__device__ __forceinline__ int jac_player(int pos, int r, int N)
{
	if (pos == 0) return N - 1;
	if (pos == 1) return r;
	const int k = pos >> 1, M = N - 1;       // r in [0,M), k in [1,N/2)
	int v = (pos & 1) ? r - k : r + k;
	if (v < 0) v += M;
	if (v >= M) v -= M;
	return v;
}

// |a_pq| <= eps sqrt(|a_pp a_qq|), compared in squares (no square root on the critical path)
__device__ __forceinline__ bool jac_small(double app, double aqq, double apq)
{
	const double eps2 = 2.220446049250313e-16 * 2.220446049250313e-16;
	return apq * apq <= eps2 * fabs(app * aqq) || fabs(apq) < 1e-150;      // (squares underflow below ~1e-154)
}

// Rotation that annihilates a_pq: t = tan(theta) is the smaller root of t^2 + 2 tau t - 1 = 0,
// tau = (a_qq - a_pp) / (2 a_pq), written as t = sgn(d) 2 a_pq / (|d| + sqrt(d^2 + 4 a_pq^2)) so
// that the dependent chain is one square root, one division and one reciprocal square root
// (the textbook form through tau has two of each; the chain latency is what a round costs).
__device__ __forceinline__ bool jac_rotation(double app, double aqq, double apq, double &c, double &s)
{
	if (jac_small(app, aqq, apq)) { c = 1.0; s = 0.0; return false; }
	const double d = aqq - app, num = 2.0 * apq;
	const double h = fma(d, d, num * num);
	const double t = (d >= 0.0 ? num : -num) / (fabs(d) + sqrt(h));
	c = rsqrt(fma(t, t, 1.0));
	s = t * c;
	return true;
}

// members (p, q) of inner pair a in inner round r.  full: tournament over all 32 local indices;
// otherwise only the cross pairs (p in the first block, q in the second)
__device__ __forceinline__ void bj_pair(int a, int r, bool full, int &p, int &q)
{
	if (full) { p = jac_player(2 * a, r, BJ_T); q = jac_player(2 * a + 1, r, BJ_T); }
	else { p = a; q = BJ_B + ((a + r) & (BJ_B - 1)); }
}

// global index of local index l of the pair (P, Q)
__device__ __forceinline__ int bj_glob(int l, int P, int Q) { return (l < BJ_B ? P : Q) * BJ_B + (l & (BJ_B - 1)); }

// Phase 1 on one pivot matrix held in S0 (32 x 32, stride BJ_LD): rotate every pair of the
// inner ordering once.  Thread (a, b) of the 16 x 16 thread grid owns the 2 x 2 block (rows of
// inner pair a) x (columns of inner pair b) and rows a, a + 16 of J for the columns of pair b;
// it computes the rotation of its column pair from that pair's diagonal 2 x 2 block and gets the
// rotation of its row pair by a shuffle (the first version had every thread compute both:
// 2 x ~250 dependent FP64 instructions per round, 1 us per round with 8 warps on an SM).
// S is double buffered (one barrier per inner round); J is
// updated in place (every thread owns its entries).  Returns the number of rotations applied
// (the same value in every thread); the result is in S0.
__device__ int bj_pivot_sweep(double *S0, double *S1, double *Jm, bool full)
{
	const int tid = threadIdx.x, a = tid >> 4, b = tid & 15;
	// anything to do at all?
	int need = 0;
	for (int i = tid; i < BJ_T * BJ_T; i += 256) {
		const int r = i >> 5, c = i & 31;
		if (r < c && (full || (r < BJ_B && c >= BJ_B)) &&
		    !jac_small(S0[r * BJ_LD + r], S0[c * BJ_LD + c], S0[r * BJ_LD + c]))
			need = 1;
	}
	if (!__syncthreads_or(need)) return 0;
	for (int i = tid; i < BJ_T * BJ_T; i += 256) Jm[(i >> 5) * BJ_LD + (i & 31)] = ((i >> 5) == (i & 31)) ? 1.0 : 0.0;
	__syncthreads();
	double *cur = S0, *nxt = S1;
	int rotated = 0;
	const int rounds = full ? BJ_T - 1 : BJ_B;
	for (int r = 0; r < rounds; ++r) {
		int pa, qa, pb, qb;
		bj_pair(a, r, full, pa, qa);
		bj_pair(b, r, full, pb, qb);
		// one rotation per thread (its column pair b); the row pair's comes from lane a of the warp
		// (lane = 16 (a & 1) + b, so lanes 0..15 hold the pairs 0..15)
		double ca, sa, cb, sb;
		const bool rotb = jac_rotation(cur[pb * BJ_LD + pb], cur[qb * BJ_LD + qb], cur[pb * BJ_LD + qb], cb, sb);
		ca = __shfl_sync(0xffffffffu, cb, a);
		sa = __shfl_sync(0xffffffffu, sb, a);
		const bool rot = rotb;                                 // used only where a == b
		if (a == b && rot) ++rotated;
		const double b00 = cur[pa * BJ_LD + pb], b01 = cur[pa * BJ_LD + qb];
		const double b10 = cur[qa * BJ_LD + pb], b11 = cur[qa * BJ_LD + qb];
		// left: rows (p,q) <- (c p - s q, s p + c q); right: the same on the columns
		const double l00 = ca * b00 - sa * b10, l01 = ca * b01 - sa * b11;
		const double l10 = sa * b00 + ca * b10, l11 = sa * b01 + ca * b11;
		double n00 = cb * l00 - sb * l01, n01 = sb * l00 + cb * l01;
		double n10 = cb * l10 - sb * l11, n11 = sb * l10 + cb * l11;
		if (a == b && rot) { n01 = 0.0; n10 = 0.0; }          // annihilated exactly
		nxt[pa * BJ_LD + pb] = n00; nxt[pa * BJ_LD + qb] = n01;
		nxt[qa * BJ_LD + pb] = n10; nxt[qa * BJ_LD + qb] = n11;
#pragma unroll
		for (int h = 0; h < 2; ++h) {
			double *jr = Jm + (a + h * BJ_B) * BJ_LD;
			const double x0 = jr[pb], x1 = jr[qb];
			jr[pb] = cb * x0 - sb * x1;
			jr[qb] = sb * x0 + cb * x1;
		}
		__syncthreads();
		double *tp = cur; cur = nxt; nxt = tp;
	}
	const int total = __syncthreads_count(rotated);       // threads (a == a) that rotated at least once
	if (cur != S0) {
		for (int i = tid; i < BJ_T * BJ_T; i += 256) S0[(i >> 5) * BJ_LD + (i & 31)] = cur[(i >> 5) * BJ_LD + (i & 31)];
		__syncthreads();
	}
	return total;                                         // > 0 iff any rotation was applied
}

// D(32 x 32) = op(X) Y with X, Y, D in shared memory (stride BJ_LD); TRANS_X: X^T Y.  On the FP64
// tensor pipe: 16 output tiles of 8 x 8, two per warp, 8 k-steps of mma.m8n8k4 each (fragment
// layout as in b200_dense.cu: lane = 4 g + t; a = A[g][t], b = B[t][g], c0/c1 = C[g][2t], C[g][2t+1]).
// The first version ran these products on the FMA pipe with scalar shared-memory loads: ~2.3 k
// cycles each, bound by bank conflicts; here a product is ~48 DMMA issue slots per SM sub-partition.
template <bool TRANS_X>
__device__ __forceinline__ void bj_mm(const double *X, const double *Y, double *D)
{
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int g = lane >> 2, t = lane & 3;
	const int tr = warp >> 1, tc = 2 * (warp & 1);
	double c[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
#pragma unroll
	for (int ks = 0; ks < BJ_T / 4; ++ks) {
		const int kk = 4 * ks + t;
		const double a = TRANS_X ? X[kk * BJ_LD + 8 * tr + g] : X[(8 * tr + g) * BJ_LD + kk];
#pragma unroll
		for (int j = 0; j < 2; ++j) {
			const double b = Y[kk * BJ_LD + 8 * (tc + j) + g];
			asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
			             : "+d"(c[j][0]), "+d"(c[j][1]) : "d"(a), "d"(b));
		}
	}
#pragma unroll
	for (int j = 0; j < 2; ++j) {
		D[(8 * tr + g) * BJ_LD + 8 * (tc + j) + 2 * t] = c[j][0];
		D[(8 * tr + g) * BJ_LD + 8 * (tc + j) + 2 * t + 1] = c[j][1];
	}
}

// Mg: Np x Np symmetric matrix, Vg: Np x Np accumulated transformations (both row-major, ld Np,
// Np = 16 NB, NB even; indices >= n are padding: zero rows and columns that never rotate).
// On exit w ascending, z[i*ldz + j] = component i of eigenvector j, *sweeps_out = sweeps done.
__global__ void __launch_bounds__(256)
syev_block_jacobi_kernel(int n, int NB, double *Mg, double *Vg, double *jbuf, int *nrot, double *w, double *z, int ldz,
                         int max_sweeps, int *rot_count, int *rank_of, int *sweeps_out, long long *cycles)
{
	cg::grid_group grid = cg::this_grid();
	__shared__ double sm[4 * BJ_TILE];
	double *T0 = sm, *T1 = sm + BJ_TILE, *T2 = sm + 2 * BJ_TILE, *T3 = sm + 3 * BJ_TILE;
	const int tid = threadIdx.x;
	const int Np = NB * BJ_B, m = NB / 2;
	const int vrb = (Np / BJ_T + 1) / 2;                   // V jobs take two 32-row tiles each
	const int a_jobs = m * (m - 1) / 2, v_jobs = vrb * m;
	// where the time goes (block 0's view, clock64 ticks): [0] phase 1, [1] barrier, [2] phase 2, [3] barrier.
	// Kept on every call: without these clock reads ptxas schedules the kernel differently and it runs 0.4 - 1.2 %
	// slower at N = 400 - 480 (B200, 1000 W power limit), same bits.
	long long cyc[6] = {0, 0, 0, 0, 0, 0}, t_prev = clock64();     // [4], [5]: tile load / rotations inside phase 1
	auto lap = [&](int slot) { const long long t = clock64(); cyc[slot] += t - t_prev; t_prev = t; };
	int sweep = 0, converged = 0;
	for (; sweep < max_sweeps; ++sweep) {
		for (int R = 0; R < NB - 1; ++R) {
			// ---- phase 1: pivot matrices
			for (int k = blockIdx.x; k < m; k += gridDim.x) {
				const int P = jac_player(2 * k, R, NB), Q = jac_player(2 * k + 1, R, NB);
				for (int i = tid; i < BJ_T * BJ_T; i += 256) {
					const int r = i >> 5, c = i & 31;
					T0[r * BJ_LD + c] = Mg[(size_t)bj_glob(r, P, Q) * Np + bj_glob(c, P, Q)];
				}
				__syncthreads();
				const long long t_a = clock64();
				const int cnt = bj_pivot_sweep(T0, T1, T2, R == 0);
				cyc[4] += t_a - t_prev; cyc[5] += clock64() - t_a;
				if (cnt > 0) {
					for (int i = tid; i < BJ_T * BJ_T; i += 256) {
						const int r = i >> 5, c = i & 31;
						Mg[(size_t)bj_glob(r, P, Q) * Np + bj_glob(c, P, Q)] = T0[r * BJ_LD + c];
						jbuf[(size_t)k * BJ_T * BJ_T + i] = T2[r * BJ_LD + c];
					}
				}
				if (tid == 0) {
					nrot[k] = cnt;
					if (cnt > 0) atomicAdd(rot_count, 1);
				}
				__syncthreads();
			}
			lap(0);
			grid.sync();
			lap(1);
			// ---- phase 2: the rest of A (upper tiles, mirrored) and V
			for (int job = blockIdx.x; job < a_jobs + v_jobs; job += gridDim.x) {
				if (job < a_jobs) {
					// job -> (I, J), I < J
					int I = 0, rem = job;
					while (rem >= m - 1 - I) { rem -= m - 1 - I; ++I; }
					const int J = I + 1 + rem;
					const int nI = nrot[I], nJ = nrot[J];
					if (nI == 0 && nJ == 0) continue;
					const int PI = jac_player(2 * I, R, NB), QI = jac_player(2 * I + 1, R, NB);
					const int PJ = jac_player(2 * J, R, NB), QJ = jac_player(2 * J + 1, R, NB);
					{   // all twelve loads of a thread in flight at once: one L2 round trip, not three
						double tv[4], ji[4], jj[4];
#pragma unroll
						for (int u = 0; u < 4; ++u) {
							const int i = tid + u * 256, r = i >> 5, c = i & 31;
							tv[u] = Mg[(size_t)bj_glob(r, PI, QI) * Np + bj_glob(c, PJ, QJ)];
							ji[u] = nI ? jbuf[(size_t)I * BJ_T * BJ_T + i] : (r == c ? 1.0 : 0.0);
							jj[u] = nJ ? jbuf[(size_t)J * BJ_T * BJ_T + i] : (r == c ? 1.0 : 0.0);
						}
#pragma unroll
						for (int u = 0; u < 4; ++u) {
							const int i = tid + u * 256, r = i >> 5, c = i & 31;
							T0[r * BJ_LD + c] = tv[u]; T1[r * BJ_LD + c] = ji[u]; T2[r * BJ_LD + c] = jj[u];
						}
					}
					__syncthreads();
					bj_mm<true>(T1, T0, T3);               // U = J_I^T T
					__syncthreads();
					bj_mm<false>(T3, T2, T0);              // T' = U J_J
					__syncthreads();
					for (int i = tid; i < BJ_T * BJ_T; i += 256) {
						const int r = i >> 5, c = i & 31;
						const double v = T0[r * BJ_LD + c];
						const int gr = bj_glob(r, PI, QI), gc = bj_glob(c, PJ, QJ);
						Mg[(size_t)gr * Np + gc] = v;
						Mg[(size_t)gc * Np + gr] = v;
					}
					__syncthreads();
				} else {
					const int vj = job - a_jobs, rb2 = vj / m, J = vj - rb2 * m;
					const int nJ = nrot[J];
					if (nJ == 0) continue;
					const int PJ = jac_player(2 * J, R, NB), QJ = jac_player(2 * J + 1, R, NB);
					const int nt = (2 * rb2 + 1 < Np / BJ_T) ? 2 : 1;
					{
						double tv[2][4], jj[4];
#pragma unroll
						for (int u = 0; u < 4; ++u) {
							const int i = tid + u * 256, r = i >> 5, c = i & 31;
							tv[0][u] = Vg[(size_t)((2 * rb2) * BJ_T + r) * Np + bj_glob(c, PJ, QJ)];
							tv[1][u] = (nt == 2) ? Vg[(size_t)((2 * rb2 + 1) * BJ_T + r) * Np + bj_glob(c, PJ, QJ)] : 0.0;
							jj[u] = jbuf[(size_t)J * BJ_T * BJ_T + i];
						}
#pragma unroll
						for (int u = 0; u < 4; ++u) {
							const int i = tid + u * 256, r = i >> 5, c = i & 31;
							T0[r * BJ_LD + c] = tv[0][u]; T1[r * BJ_LD + c] = tv[1][u]; T2[r * BJ_LD + c] = jj[u];
						}
					}
					__syncthreads();
					for (int h = 0; h < nt; ++h) {
						bj_mm<false>(h ? T1 : T0, T2, T3);      // T' = T J_J
						__syncthreads();
						for (int i = tid; i < BJ_T * BJ_T; i += 256) {
							const int r = i >> 5, c = i & 31;
							Vg[(size_t)((2 * rb2 + h) * BJ_T + r) * Np + bj_glob(c, PJ, QJ)] = T3[r * BJ_LD + c];
						}
						__syncthreads();
					}
				}
			}
			lap(2);
			grid.sync();
			lap(3);
		}
		// end of sweep: did anything rotate?
		const int rotated = *((volatile int *)rot_count);
		grid.sync();
		if (blockIdx.x == 0 && tid == 0) *rot_count = 0;
		grid.sync();
		if (rotated == 0) { ++sweep; converged = 1; break; }
	}
	// rank the diagonal (padding excluded) and emit
	const int gtid = blockIdx.x * blockDim.x + tid, gsz = gridDim.x * blockDim.x;
	for (int i = gtid; i < n; i += gsz) {
		const double d = Mg[(size_t)i * Np + i];
		int rank = 0;
		for (int q = 0; q < n; ++q) {
			const double dq = Mg[(size_t)q * Np + q];
			if (dq < d || (dq == d && q < i)) ++rank;
		}
		w[rank] = d;
		rank_of[i] = rank;
	}
	grid.sync();
	for (int idx = gtid; idx < n * n; idx += gsz) {
		const int i = idx / n, j = idx - i * n;
		z[(size_t)i * ldz + rank_of[j]] = Vg[(size_t)i * Np + j];
	}
	if (gtid == 0) {
		sweeps_out[0] = sweep;
		sweeps_out[1] = converged;                        // the last sweep applied no rotation
		for (int i = 0; i < 6; ++i) cycles[i] = cyc[i];
	}
}

// padded copies: Mg = A (zero padded), Vg = I
__global__ void syev_init_kernel(int n, int Np, const double *a, int lda, double *Mg, double *Vg)
{
	const long long gsz = (long long)gridDim.x * blockDim.x;
	for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < (long long)Np * Np; idx += gsz) {
		const int i = (int)(idx / Np), j = (int)(idx - (long long)i * Np);
		Mg[idx] = (i < n && j < n) ? a[(size_t)i * lda + j] : 0.0;
		Vg[idx] = (i == j) ? 1.0 : 0.0;
	}
}

// device address of {sweeps, converged} of the most recent eigen-solve (callers that do not want a synchronisation
// inside b200k_syev_jacobi read it together with the eigenvalues: b200k_syev_check)
static int *g_syev_status;

// 0 when the most recent b200k_syev_jacobi converged (the reference checks dsyevx's INFO, src/ops_eig_sol_gcg.c:1204);
// synchronises.  The Ritz pairs of a non-converged projected problem must not steer the outer loop silently.
extern "C" int b200k_syev_check(void)
{
	if (!g_syev_status) return 0;
	int h[2] = {0, 1};
	if (b200k_d2h(h, g_syev_status, sizeof(h))) return 1;
	B200_CHECK(h[1] == 1, "syev: the Jacobi iteration of the projected eigenproblem did not converge (%d sweeps)", h[0]);
	return 0;
}

extern "C" int b200k_syev_jacobi(int n, double *a_dev, int lda, double *w_dev, double *z_dev, int ldz,
                                 int *sweeps_host)
{
	B200_CHECK(n >= 1, "syev: n = %d", n);
	B200Prof prof(B200_PROF_SYEV, 24.0 * n * n, 0.0);
	cudaStream_t st = g_b200.stream;
	int NB = (n + BJ_B - 1) / BJ_B; NB += NB & 1; if (NB < 2) NB = 2;
	const int Np = NB * BJ_B, m = NB / 2;
	const size_t nn = (size_t)Np * Np;
	const size_t dbl = 2 * nn + (size_t)m * BJ_T * BJ_T;
	char *base = (char *)b200_scratch(5, sizeof(double) * (dbl + 8) + sizeof(int) * ((size_t)m + Np + 8));
	if (!base) return 1;
	double *Mg = (double *)base, *Vg = Mg + nn, *jbuf = Vg + nn;
	long long *cycles = (long long *)(jbuf + (size_t)m * BJ_T * BJ_T);
	int *nrot = (int *)(cycles + 8), *rank_of = nrot + m, *ctr = rank_of + Np;
	B200_CUDA(cudaMemsetAsync(ctr, 0, 3 * sizeof(int), st));
	syev_init_kernel<<<b200_ceil_div((long long)Np * Np, 256), 256, 0, st>>>(n, Np, a_dev, lda, Mg, Vg);
	B200_KERNEL_CHECK();
	int per_sm = 0;
	B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, syev_block_jacobi_kernel, 256, 0));
	B200_CHECK(per_sm >= 1, "syev: kernel does not fit on an SM");
	if (per_sm > 2) per_sm = 2;
	const long long jobs = (long long)m * (m - 1) / 2 + (long long)((Np / BJ_T + 1) / 2) * m;
	long long want = jobs > m ? jobs : m;
	const long long cap = (long long)per_sm * g_b200.num_sms;
	int blocks = (int)(want < cap ? want : cap);
	if (blocks < 1) blocks = 1;
	int max_sweeps = 40;
	int *rot = ctr, *sw = ctr + 1;
	void *args[] = {&n, &NB, &Mg, &Vg, &jbuf, &nrot, &w_dev, &z_dev, &ldz, &max_sweeps, &rot, &rank_of, &sw, &cycles};
	B200_CUDA(cudaLaunchCooperativeKernel((void *)syev_block_jacobi_kernel, dim3(blocks), dim3(256), args, 0, st));
	B200_LAUNCHED();
	g_syev_status = sw;
	if (sweeps_host) {
		int h[2];
		if (b200k_d2h(h, sw, sizeof(h))) return 1;
		*sweeps_host = h[0];
		B200_CHECK(h[1] == 1, "syev: the Jacobi iteration did not converge in %d sweeps (n = %d)", max_sweeps, n);
	}
	if (b200_opt(B200_OPT_SYEV_PROF)) {
		long long cyc[6];
		if (b200k_d2h(cyc, cycles, sizeof(cyc))) return 1;
		fprintf(stderr, "syev n=%d grid=%d clock64 ticks: phase1 %lld (tile load %lld, rotations %lld) barrier %lld phase2 %lld barrier %lld\n",
		        n, blocks, cyc[0], cyc[4], cyc[5], cyc[1], cyc[2], cyc[3]);
	}
	return 0;
}

// host-matrix convenience entry (tests, tier A users): see include/gcge_b200.h
extern "C" int b200_dense_syev(int n, const double *a, int lda, double *w, double *z, int ldz, int *sweeps)
{
	B200_REQUIRE_INIT();
	B200_CHECK(n >= 1 && a && w && z && lda >= n && ldz >= n, "b200_dense_syev: bad arguments");
	const size_t nn = (size_t)n * n;
	double *dev = (double *)b200_scratch(3, sizeof(double) * (2 * nn + n));
	if (!dev) return 1;
	double *da = dev, *dz = dev + nn, *dw = dz + nn;
	double *pin = (double *)b200_pinned(1, sizeof(double) * nn);
	if (!pin) return 1;
	B200_CUDA(cudaStreamSynchronize(g_b200.stream));
	// symmetrise from the caller's upper triangle (dsyevx UPLO='U' semantics)
	for (int j = 0; j < n; ++j)
		for (int i = 0; i < n; ++i)
			pin[(size_t)i * n + j] = (i <= j) ? a[(size_t)j * lda + i] : a[(size_t)i * lda + j];
	B200_CUDA(cudaMemcpyAsync(da, pin, sizeof(double) * nn, cudaMemcpyHostToDevice, g_b200.stream));
	if (b200k_syev_jacobi(n, da, n, dw, dz, n, sweeps)) return 1;
	if (b200k_d2h(w, dw, sizeof(double) * n)) return 1;
	if (b200k_d2h(pin, dz, sizeof(double) * nn)) return 1;   // dz row-major (i,j) -> host col-major
	for (int j = 0; j < n; ++j)
		for (int i = 0; i < n; ++i) z[(size_t)j * ldz + i] = pin[(size_t)i * n + j];
	return 0;
}
