// SpMM for lattice operators: tiles of a plane marching through the planes.
//
// Replaces MatDotMultiVec (reference app/app_ccs.c:50-139) for matrices whose diagonal image
// (b200_mat.cu: dia_build) is that of an operator on an s1 x my x nz lattice in natural ordering,
// row = i + s1 (j + my k), every entry coupling (i, j, k) with (i + di, j + dj, k + dk),
// |di|, |dj|, |dk| <= 1, and nothing across the lattice faces -- the 7-point, 27-point and P1-Kuhn
// operators of BASELINE.json's configs.
//
// The 1-D kernel (b200_spmm.cu: spmm_dia_ws_kernel) stages one (ROWS + 2)-row box of x PER RUN of
// consecutive offsets: 7 boxes per row block for the 15-point operator, so every x row enters shared
// memory 7.3 times, and shared-memory bandwidth (TMA writes + fragment reads + matrix values) is what
// binds it at 0.47-0.50 of HBM inside the solve (profiles/ncu_r1h_spmm_*: l1tex 82 %).  Here a CTA owns a
// TJ x TI tile of a plane and marches along k: the (TJ + 2) x (TI + 2) patches of planes k - 1, k, k + 1
// sit in a ring of shared-memory slices (one 4-D tensor-map copy per plane, rows outside the lattice
// zero-filled by the TMA unit), every patch serves three consecutive output planes, and each x row
// enters shared memory (TJ + 2)(TI + 2) / (TJ TI) ~ 1.5 times.  The matrix values of the tile's rows come
// by one 4-D tensor-map copy of the image per plane.  Row groups (KP consecutive threads, one column
// pair per lane), register accumulators over RB consecutive rows, sliding reads along i, per-warp
// mbarrier hand-back and the fused p^T w epilogue are those of the 1-D kernel; so is the arithmetic: per
// matrix row the runs, and the offsets inside a run, are visited in ascending column order with separate
// multiply and add -- bit-identical to the reference's scatter loop for every finite x.
#include "b200_internal.h"
#include "b200_tma.cuh"
#include "b200_dia.cuh"

constexpr int LAT_MAX_NS = 6;                          // deepest slice ring
constexpr int LAT_MAX_NV = 4;                          // deepest value ring
constexpr int LAT_RB = 4;                              // consecutive rows (along i) of one task

struct LatRun { int dk, rowoff, sp, w; };              // slice (0: k-1, 1: k, 2: k+1), row offset inside a slice, value slot, width
struct LatParams {
	int s1, my;                                        // line length, lines per plane
	int TI, TJ, NTI, NTJ;                              // tile, tiles per plane
	int pitch;                                         // rows per line of a slice: TI + 2, or TI + 3 to make it odd
	int p_begin, p_end, KL, nseg;                      // local planes [p_begin, p_end) in nseg segments of KL planes
	int xshift;                                        // plane coordinate of local plane 0 in the x tensor map
	int ng, ndp, zero_run, zero_pos;                   // runs, value slots per row, run holding offset 0 and its position
	int vpitch;                                        // doubles per row of a value tile in shared memory (>= ndp)
	int NS, NV;                                        // ring depths
	int slice_bytes, val_bytes;                        // one slice / one value buffer (bytes a copy delivers)
	int slice_stride, val_stride;                      // ... and their 128-byte aligned strides in the rings
	LatRun run[32];
	double coef[40];                                   // CONST: the stencil's coefficients by value slot (one row of the image)
};

// CONST: the operator is a constant stencil (every row carries the same coefficients, entries exist exactly where
// the neighbour is inside the lattice): the coefficients come from the kernel parameters, no value tile is loaded, and
// rows outside the lattice contribute a_d * 0 because the copy engine zero-fills them -- +-0 added to an accumulator
// that starts at +0.0 changes nothing, so the result is still the reference's, bit for bit, for every finite x.
template <int KP, int NT, bool DOT, bool CONST>
__global__ void __launch_bounds__(NT + 32, 1)
spmm_lat_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmv,
                const __grid_constant__ LatParams P, double *y, int ldy, const int *__restrict__ gate, double *dot_part)
{
	if (gate != nullptr && *gate == 0) return;
	constexpr int K = 2 * KP;
	constexpr int RB = LAT_RB;
	constexpr int NG = NT / KP;                        // row groups
	extern __shared__ __align__(128) unsigned char smem_raw[];
	__shared__ unsigned long long full[LAT_MAX_NS], empty[LAT_MAX_NS], vfull[LAT_MAX_NV], vempty[LAT_MAX_NV];
	const int NS = P.NS, NV = P.NV;
	if (threadIdx.x == 0) {
		for (int s = 0; s < NS; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, NT / 32); }
		for (int s = 0; s < NV; ++s) { mbar_init(vfull + s, 1); mbar_init(vempty + s, NT / 32); }
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
	}
	__syncthreads();
	unsigned char *vbuf = smem_raw + (size_t)NS * P.slice_stride;
	const int tiles = P.NTJ * P.NTI, nitems = tiles * P.nseg;

	if (threadIdx.x >= NT) {
		// ------------------------------------------------------------------ producer warp
		if (threadIdx.x == NT) {
			unsigned long long pol;
			asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
			int slot = 0, vslot = 0; unsigned phase = 0, vphase = 0;
			for (int it = blockIdx.x; it < nitems; it += gridDim.x) {
				const int seg = it / tiles, rem = it - seg * tiles, tj = rem / P.NTI, ti = rem - tj * P.NTI;
				const int k0 = P.p_begin + seg * P.KL;
				const int len = min(P.KL, P.p_end - k0);
				const int I0 = ti * P.TI, J0 = tj * P.TJ;
				for (int t = 0; t < len + 2; ++t) {
					mbar_spin(empty + slot, phase ^ 1u);
					mbar_expect_tx(full + slot, (unsigned)P.slice_bytes);
					tma_load_4d(smem_raw + (size_t)slot * P.slice_stride, &tmx, 0, I0 - 1, J0 - 1, k0 - 1 + t + P.xshift, full + slot);
					if (++slot == NS) { slot = 0; phase ^= 1u; }
					if (!CONST && t >= 2) {
						// the values of output plane k0 + t - 2, needed together with the slice just requested
						mbar_spin(vempty + vslot, vphase ^ 1u);
						mbar_expect_tx(vfull + vslot, (unsigned)P.val_bytes);
						tma_load_4d_hint(vbuf + (size_t)vslot * P.val_stride, &tmv, 0, I0, J0, k0 + t - 2, vfull + vslot, pol);
						if (++vslot == NV) { vslot = 0; vphase ^= 1u; }
					}
				}
			}
		}
		return;
	}
	// ---------------------------------------------------------------------- consumer warps
	const int lane = threadIdx.x & 31;
	const int group = threadIdx.x / KP, gl = threadIdx.x - group * KP;
	const bool live = group < NG;                      // the NT % KP leftover threads only keep the barriers company
	const int c = 2 * gl;
	const int CH = P.TI / RB, ntasks = P.TJ * CH;      // tasks of one plane step: (line, chunk of RB rows)
	const int pitch = P.pitch;                         // rows per line of a slice
	const int ch_first = (live ? group : 0) / P.TJ;
	double dot[2] = {0.0, 0.0};
	int slot = 0, vslot = 0; unsigned phase = 0, vphase = 0;
	int ring0 = 0, ring1 = 0, ring2 = 0;               // slots of the three most recent slices: planes k-1, k, k+1
	for (int it = blockIdx.x; it < nitems; it += gridDim.x) {
		const int seg = it / tiles, rem = it - seg * tiles, tj = rem / P.NTI, ti = rem - tj * P.NTI;
		const int k0 = P.p_begin + seg * P.KL;
		const int len = min(P.KL, P.p_end - k0);
		const int I0 = ti * P.TI, J0 = tj * P.TJ;
		for (int t = 0; t < len + 2; ++t) {
			mbar_spin(full + slot, phase);
			ring0 = ring1; ring1 = ring2; ring2 = slot;
			if (++slot == NS) { slot = 0; phase ^= 1u; }
			if (t < 2) continue;
			if (!CONST) mbar_spin(vfull + vslot, vphase);
			const double *vals = reinterpret_cast<const double *>(vbuf + (size_t)vslot * P.val_stride);
			const long long prow = (long long)(k0 + t - 2) * P.s1 * P.my;     // first row of the output plane
			if (live) {
				for (int task = group; task < ntasks; task += NG) {
					// neighbouring row groups take neighbouring LINES: their x rows are `pitch` rows apart, and with an
					// odd pitch the 16-byte pieces two groups read in one quarter-warp never meet in a bank
					// (the group's first task -- usually its only one per plane step -- was decoded once, up front)
					const int ch = (task == group) ? ch_first : task / P.TJ;
					const int jj = task - ch * P.TJ, ii0 = ch * RB;
					double acc[RB][2];
					double2 pst[RB][1];
#pragma unroll
					for (int i = 0; i < RB; ++i) { acc[i][0] = 0.0; acc[i][1] = 0.0; pst[i][0] = make_double2(0.0, 0.0); }
					const double *vrow = vals + (jj * P.TI + ii0) * P.vpitch;
					const int rbase = jj * pitch + ii0;
					for (int g = 0; g < P.ng; ++g) {
						const LatRun r = P.run[g];
						const int sl = r.dk == 0 ? ring0 : (r.dk == 1 ? ring1 : ring2);
						const double *tile = reinterpret_cast<const double *>(smem_raw + (size_t)sl * P.slice_stride) +
						                     (rbase + r.rowoff) * K + c;
						// the run that holds offset 0 also keeps the block's own x rows for the fused dot; every other run goes
						// through the instantiation WITHOUT that code (if-converted selects would otherwise issue in all of them:
						// ncu showed as many IMAD.MOV as DADD per task)
						if (DOT && g == P.zero_run) {
							const int zrow = P.zero_pos;
							if (CONST) {
								const double a0 = P.coef[r.sp], a1 = P.coef[r.sp + 1], a2 = P.coef[r.sp + 2];
								if (r.w == 2)      dia_run_const<RB, 2, K, KP, true>(acc, tile, a0, a1, a2, pst, zrow);
								else if (r.w == 3) dia_run_const<RB, 3, K, KP, true>(acc, tile, a0, a1, a2, pst, zrow);
								else               dia_run_const<RB, 1, K, KP, true>(acc, tile, a0, a1, a2, pst, zrow);
							}
							else if (r.w == 2) dia_run_ct<RB, 2, K, KP, 1, true>(acc, tile, vrow + r.sp, P.vpitch, pst, zrow);
							else if (r.w == 3) dia_run_ct<RB, 3, K, KP, 1, true>(acc, tile, vrow + r.sp, P.vpitch, pst, zrow);
							else               dia_run_ct<RB, 1, K, KP, 1, true>(acc, tile, vrow + r.sp, P.vpitch, pst, zrow);
						} else if (CONST) {
							const double a0 = P.coef[r.sp], a1 = P.coef[r.sp + 1], a2 = P.coef[r.sp + 2];
							if (r.w == 2)      dia_run_const<RB, 2, K, KP, false>(acc, tile, a0, a1, a2, pst, -1);
							else if (r.w == 3) dia_run_const<RB, 3, K, KP, false>(acc, tile, a0, a1, a2, pst, -1);
							else               dia_run_const<RB, 1, K, KP, false>(acc, tile, a0, a1, a2, pst, -1);
						}
						else if (r.w == 2) dia_run_ct<RB, 2, K, KP, 1, false>(acc, tile, vrow + r.sp, P.vpitch, pst, -1);
						else if (r.w == 3) dia_run_ct<RB, 3, K, KP, 1, false>(acc, tile, vrow + r.sp, P.vpitch, pst, -1);
						else               dia_run_ct<RB, 1, K, KP, 1, false>(acc, tile, vrow + r.sp, P.vpitch, pst, -1);
					}
					const int j = J0 + jj;
					if (j < P.my) {
						double *yr = y + (size_t)(prow + (long long)j * P.s1 + I0 + ii0) * ldy + c;
#pragma unroll
						for (int i = 0; i < RB; ++i) {
							if (I0 + ii0 + i < P.s1) {
								// streaming store: y is not read again by this kernel and must not push x rows out of L2
								__stcs(reinterpret_cast<double2 *>(yr + (size_t)i * ldy), make_double2(acc[i][0], acc[i][1]));
								if (DOT) {
									dot[0] = fma(pst[i][0].x, acc[i][0], dot[0]);
									dot[1] = fma(pst[i][0].y, acc[i][1], dot[1]);
								}
							}
						}
					}
				}
			}
			// the loads from the slice and the values must have been performed before they are handed back
			// (an mbarrier arrive does not wait for loads in flight; see lincomb_tma_body in b200_dense.cu)
			asm volatile("fence.acq_rel.cta;" ::: "memory");
			__syncwarp();
			if (lane == 0) {
				if (!CONST) mbar_arrive(vempty + vslot);
				mbar_arrive(empty + ring0);                    // plane k - 1 of this step is not needed again
				if (t == len + 1) { mbar_arrive(empty + ring1); mbar_arrive(empty + ring2); }      // end of the segment
			}
			if (++vslot == NV) { vslot = 0; vphase ^= 1u; }
		}
	}
	if (DOT) {
		// per-CTA column sums in a fixed order: groups 0 .. NG-1 (the slices are dead: reuse slice 0)
		asm volatile("bar.sync 1, %0;" ::"n"(NT));
		double *red = reinterpret_cast<double *>(smem_raw);
		if (live) { red[group * K + c] = dot[0]; red[group * K + c + 1] = dot[1]; }
		asm volatile("bar.sync 1, %0;" ::"n"(NT));
		for (int cc = threadIdx.x; cc < K; cc += NT) {
			double s = 0.0;
			for (int gq = 0; gq < NG; ++gq) s += red[gq * K + cc];
			dot_part[(size_t)blockIdx.x * K + cc] = s;
		}
	}
}

// ---- lattice recognition ---------------------------------------------------------------------------
// Candidate strides come from the diagonal offsets; a candidate is accepted when every offset decomposes
// as di + dj s1 + dk s2 with |di|, |dj|, |dk| <= 1 (one (dj, dk) per run) and NO non-zero value of the image
// couples across a lattice face (checked on the device over this rank's rows).
__global__ void lat_violations_kernel(int nrows, long long row0, int s1, int my, long long nz, int ng,
                                      const int *__restrict__ off, const int *__restrict__ grp, int ndp,
                                      const double *__restrict__ val, int *count)
{
	const int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= nrows) return;
	const long long R = row0 + r, s2 = (long long)s1 * my;
	const int i = (int)(R % s1), j = (int)((R / s1) % my);
	const long long k = R / s2;
	int bad = 0;
	for (int g = 0; g < ng; ++g) {
		const int w = grp[2 * g + 1], sp = grp[2 * g];
		for (int t = 0; t < w; ++t) {
			if (val[(size_t)r * ndp + sp + t] == 0.0) continue;
			const long long d = (long long)off[g] + t;
			long long q = d + s2 / 2;                     // dk = floor((d + s2/2) / s2)
			const long long dk = q >= 0 ? q / s2 : -((-q + s2 - 1) / s2);
			const long long rem = d - dk * s2;
			q = rem + s1 / 2;
			const long long dj = q >= 0 ? q / s1 : -((-q + s1 - 1) / s1);
			const long long di = rem - dj * s1;
			if (i + di < 0 || i + di >= s1 || j + dj < 0 || j + dj >= my || k + dk < 0 || k + dk >= nz) ++bad;
		}
	}
	if (bad) atomicAdd(count, bad);
}

// rows whose image differs from the constant stencil `coef` (coefficient where the neighbour is inside the lattice,
// +0.0 where it is not; padding slots are zero in both)
__global__ void lat_const_kernel(int nrows, long long row0, int s1, int my, long long nz, int ng,
                                 const int *__restrict__ off, const int *__restrict__ grp, int ndp,
                                 const double *__restrict__ val, const double *__restrict__ coef, int *count)
{
	const int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= nrows) return;
	const long long R = row0 + r, s2 = (long long)s1 * my;
	const int i = (int)(R % s1), j = (int)((R / s1) % my);
	const long long k = R / s2;
	int bad = 0;
	for (int g = 0; g < ng; ++g) {
		const int w = grp[2 * g + 1], sp = grp[2 * g];
		for (int t = 0; t < w; ++t) {
			const long long d = (long long)off[g] + t;
			long long q = d + s2 / 2;
			const long long dk = q >= 0 ? q / s2 : -((-q + s2 - 1) / s2);
			const long long rem = d - dk * s2;
			q = rem + s1 / 2;
			const long long dj = q >= 0 ? q / s1 : -((-q + s1 - 1) / s1);
			const long long di = rem - dj * s1;
			const bool inside = i + di >= 0 && i + di < s1 && j + dj >= 0 && j + dj < my && k + dk >= 0 && k + dk < nz;
			const double want = inside ? coef[sp + t] : 0.0;
			if (!(val[(size_t)r * ndp + sp + t] == want)) ++bad;
		}
	}
	if (bad) atomicAdd(count, bad);
}

// Every run of consecutive offsets must lie on one (dj, dk) line of the lattice: first offset = di0 + dj s1 + dk s2
// with -1 <= di0 and di0 + w - 1 <= 1, one run per line.  runs[g].rowoff comes back as ((1 + dj) << 8) | (1 + di0);
// the launch turns it into a row offset once the tile width is known.
static bool lat_decompose(const b200_mat *A, long long s1, long long s2, LatRun *runs, int *zero_run, int *zero_pos)
{
	bool seen[3][3] = {{false, false, false}, {false, false, false}, {false, false, false}};
	if (zero_run) *zero_run = -1;
	for (int g = 0; g < A->dia_ng; ++g) {
		const long long d0 = A->dia_off_h[g];
		const int w = A->dia_grp_h[2 * g + 1];
		bool ok = false;
		for (int di0 = -1; di0 <= 1 && !ok && di0 + w - 1 <= 1; ++di0)
			for (int dk = -1; dk <= 1 && !ok; ++dk)
				for (int dj = -1; dj <= 1 && !ok; ++dj) {
					if (d0 - di0 != dj * s1 + dk * s2) continue;
					if (seen[dk + 1][dj + 1]) return false;
					seen[dk + 1][dj + 1] = true;
					if (runs) { runs[g].dk = dk + 1; runs[g].rowoff = ((1 + dj) << 8) | (1 + di0); runs[g].sp = A->dia_grp_h[2 * g]; runs[g].w = w; }
					if (zero_run && dk == 0 && dj == 0 && di0 <= 0 && di0 + w > 0) { *zero_run = g; *zero_pos = -di0; }
					ok = true;
				}
		if (!ok) return false;
	}
	return true;
}

// called once per matrix, after its diagonal image exists (b200_mat.cu); sets A->lat_s1 / lat_s2 (0: not a lattice)
int b200k_lat_detect(b200_mat *A)
{
	A->lat_s1 = 0; A->lat_s2 = 0; A->lat_const = 0;
	if (A->dia_nd <= 0 || A->nrows <= 0 || b200_opt(B200_OPT_NO_LAT)) return 0;
	const long long n = A->nrows_global;
	// the central run must hold offset 0; s1 comes from the first run above it, s2 from the runs beyond
	const int zc = dia_zero_run(A);
	if (zc < 0 || zc + 1 >= A->dia_ng) return 0;
	const long long a = A->dia_off_h[zc + 1];
	long long best1 = 0, best2 = 0;
	for (long long s1 = a; s1 <= a + 1 && !best1; ++s1) {
		if (s1 < 4) continue;
		for (int g = zc + 2; g < A->dia_ng && !best1; ++g) {
			// a run with dk = +1: its first offset is s2 + dj s1 + di0
			for (int dj = -1; dj <= 1 && !best1; ++dj)
				for (int di0 = -1; di0 <= 1 && !best1; ++di0) {
					const long long s2 = A->dia_off_h[g] - dj * s1 - di0;
					if (s2 < 2 * s1 || s2 % s1 || n % s2 || n / s2 < 3) continue;
					if (!lat_decompose(A, s1, s2, nullptr, nullptr, nullptr)) continue;
					int *cnt = (int *)b200_scratch(3, 64);
					if (!cnt) return 1;
					B200_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int), g_b200.stream));
					lat_violations_kernel<<<b200_ceil_div(A->nrows, 256), 256, 0, g_b200.stream>>>(
						A->nrows, A->row0, (int)s1, (int)(s2 / s1), n / s2, A->dia_ng, A->dia_off, A->dia_grp, A->dia_ndp, A->dia_val, cnt);
					B200_KERNEL_CHECK();
					int bad = 1;
					if (b200k_d2h(&bad, cnt, sizeof(int))) return 1;
					if (bad == 0) { best1 = s1; best2 = s2; }
				}
		}
	}
	if (!best1) return 0;
	// several ranks: slabs must be whole planes, and every rank must see the same lattice
	if (A->row0 % best2 || A->nrows % best2) return 0;
	A->lat_s1 = (int)best1; A->lat_s2 = (int)best2;
	// ---- constant stencil?  take the coefficients of one interior row and compare every row of the slab with
	// (coefficient where the neighbour is inside the lattice, 0 where it is not)
	A->lat_const = 0;
	const int s1 = A->lat_s1, my = A->lat_s2 / A->lat_s1, np = A->nrows / A->lat_s2;
	const long long nz = n / best2, gk0 = A->row0 / best2;
	int kk = -1;
	for (int q = 0; q < np && kk < 0; ++q) if (gk0 + q >= 1 && gk0 + q <= nz - 2) kk = q;
	if (kk >= 0 && s1 >= 3 && my >= 3 && A->dia_ndp <= 40) {
		const size_t rstar = (size_t)kk * best2 + (size_t)(my / 2) * s1 + s1 / 2;
		double *coef_dev = (double *)b200_scratch(3, sizeof(double) * 40 + 64);
		if (!coef_dev) return 1;
		int *cnt = (int *)(coef_dev + 40);
		B200_CUDA(cudaMemcpyAsync(coef_dev, A->dia_val + rstar * A->dia_ndp, sizeof(double) * A->dia_ndp, cudaMemcpyDeviceToDevice, g_b200.stream));
		B200_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int), g_b200.stream));
		lat_const_kernel<<<b200_ceil_div(A->nrows, 256), 256, 0, g_b200.stream>>>(
			A->nrows, A->row0, s1, my, nz, A->dia_ng, A->dia_off, A->dia_grp, A->dia_ndp, A->dia_val, coef_dev, cnt);
		B200_KERNEL_CHECK();
		int bad = 1;
		if (b200k_d2h(&bad, cnt, sizeof(int))) return 1;
		if (bad == 0) {
			if (b200k_d2h(A->lat_coef, coef_dev, sizeof(double) * A->dia_ndp)) return 1;
			A->lat_const = 1;
		}
	}
	return 0;
}

// Rows of a slice line.  Row groups that share a quarter-warp read 16-byte pieces of x rows `pitch` rows apart
// (neighbouring groups work on neighbouring lines): when a row is not a whole number of 128-byte bank rounds, an
// odd pitch keeps those pieces in different banks (k = 40: rows of 320 bytes, 23 rows apart = 64 mod 128; with the
// even pitch 22 every group boundary inside a quarter-warp is a two-way conflict, +24 % wavefronts on the x reads).
static int lat_pitch(int TI, int K)
{
	int pitch = TI + 2;
	if ((K * 8) % 128 != 0 && pitch % 2 == 0) ++pitch;
	return pitch;
}

// Doubles per row of a value tile in shared memory.  The lanes of a row group read the same matrix value (a
// broadcast), but a warp holds lanes of two or three groups, whose rows are a multiple of RB = 4 rows apart: with
// 128-byte rows (16 slots) all of them sit in the same banks and every value load is a 2-3 way conflict (ncu:
// 8 conflict wavefronts per matrix row, +25 % on the whole kernel).  Rows of 8 q bytes with q = 2 (mod 4) put
// rows 4 apart 64 bytes apart; the tensor-map box is simply wider than the image and the padding arrives as zeros.
static int lat_vpitch(int ndp)
{
	return ndp % 4 == 0 ? ndp + 2 : ndp;
}

// returns 0 launched, 1 error, 2 not applicable; mode 0: all planes, 1: interior planes (no halo plane needed),
// 2: the boundary planes; *nparts (DOT): per-CTA partial rows written to dot_part
template <int KP, int NT, bool DOT, bool CONST>
static int launch_spmm_lat(const b200_mat *M, const double *x, int ldx, double *y, int ldy, const int *gate,
                           double *dot_part, int dot_cap, int *nparts, int mode)
{
	constexpr int K = 2 * KP;
	constexpr int NG = NT / KP;
	if (DOT) *nparts = 0;
	const int s1 = M->lat_s1, s2 = M->lat_s2, my = s2 / s1, np = M->nrows / s2;
	LatParams P;
	memset(&P, 0, sizeof(P));
	P.s1 = s1; P.my = my; P.ng = M->dia_ng; P.ndp = M->dia_ndp;
	if (!lat_decompose(M, s1, s2, P.run, &P.zero_run, &P.zero_pos)) return 2;
	if (DOT && P.zero_run < 0) return 2;
	// ---- tile: TI x TJ rows of a plane, ring depth; estimated shared-memory cycles per matrix row decide
	const size_t smem_cap = 227 * 1024 - 1024;
	int sum_reads = 0, n3 = 0;
	for (int g = 0; g < P.ng; ++g) { sum_reads += LAT_RB + P.run[g].w - 1; n3 += P.run[g].w == 3; }
	double best = 1e300; int bTI = 0, bTJ = 0, bNS = 0;
	for (int TI = 8; TI <= 64; TI += LAT_RB) {
		for (int TJ = 1; TJ <= 16; ++TJ) {
			// TMA destinations are 128-byte aligned
			const int pitch = lat_pitch(TI, K);
			const size_t slice = ((size_t)pitch * (TJ + 2) * K * 8 + 127) & ~(size_t)127;
			const size_t vb = CONST ? 0 : (((size_t)TI * TJ * lat_vpitch(P.ndp) * 8 + 127) & ~(size_t)127);
			for (int NS = 4; NS <= LAT_MAX_NS; ++NS) {
				const int NV = NS - 2;
				if (NS * slice + NV * vb > smem_cap) continue;
				const int nti = (s1 + TI - 1) / TI, ntj = (my + TJ - 1) / TJ;
				const int tasks = TJ * (TI / LAT_RB), rounds = (tasks + NG - 1) / NG;
				const double cover = (double)nti * TI * ntj * TJ / ((double)s1 * my);      // rows computed per row wanted
				const double busy = (double)rounds * NG / tasks;                           // 1 / (share of groups with a task)
				// shared-memory wavefronts (128 bytes) per matrix row: sliding x reads, broadcast value reads, TMA writes
				const double reads = cover * busy * (sum_reads / (double)LAT_RB) * K * 8 / 128.0;
				// (a broadcast LDS.128 costs a wavefront per quarter-warp: 4 per warp instruction, like distinct data)
				const double vals = CONST ? 0.0 : cover * busy * (4.0 * P.ng + 2.0 * n3) * KP / 32.0;
				const double writes = (double)nti * ntj * pitch * (TJ + 2) / ((double)s1 * my) * K * 8 / 128.0 +
				                      (CONST ? 0.0 : cover * P.ndp * 8 / 128.0);
				// a ring of 4 leaves the copy engine one plane step of lead; 5 and more hide its latency fully
				const double est = (reads + vals + writes) * (NS >= 5 ? 1.0 : 1.06);
				if (est < best) { best = est; bTI = TI; bTJ = TJ; bNS = NS; }
			}
		}
	}
	if (!bTI) return 2;
	P.TI = bTI; P.TJ = bTJ; P.NS = bNS; P.NV = CONST ? 0 : bNS - 2;
	if (CONST) for (int i = 0; i < 40; ++i) P.coef[i] = i < M->dia_ndp ? M->lat_coef[i] : 0.0;
	P.NTI = (s1 + P.TI - 1) / P.TI; P.NTJ = (my + P.TJ - 1) / P.TJ;
	P.pitch = lat_pitch(P.TI, K);
	P.slice_bytes = P.pitch * (P.TJ + 2) * K * 8;           // bytes one copy delivers; the ring strides are rounded up
	P.vpitch = lat_vpitch(P.ndp);
	P.val_bytes = CONST ? 0 : P.TI * P.TJ * P.vpitch * 8;
	P.slice_stride = (P.slice_bytes + 127) & ~127;
	P.val_stride = (P.val_bytes + 127) & ~127;
	for (int g = 0; g < P.ng; ++g) {
		const int dj1 = P.run[g].rowoff >> 8, di1 = P.run[g].rowoff & 0xff;             // 1 + dj, 1 + di0
		P.run[g].rowoff = dj1 * P.pitch + di1;
	}
	const size_t smem = (size_t)P.NS * P.slice_stride + (size_t)P.NV * P.val_stride;
	// ---- tensor maps: x as (K, s1, my, planes) with a halo plane in front / behind where a slab neighbour exists
	tmap_encode_fn enc = tmap_encoder();
	if (!enc) return 2;
	const int hb = M->halo_below, ha = M->nhalo - hb;
	const bool below = hb >= s2, above = ha >= s2;
	if ((hb && !below) || (ha && !above)) return 2;      // a partial halo plane: not this kernel
	const double *base = x - (below ? (size_t)s2 * ldx : 0);
	P.xshift = below ? 1 : 0;
	CUtensorMap tmx, tmv;
	{
		const cuuint64_t gdim[4] = {(cuuint64_t)K, (cuuint64_t)s1, (cuuint64_t)my, (cuuint64_t)(np + (below ? 1 : 0) + (above ? 1 : 0))};
		const cuuint64_t gstr[3] = {(cuuint64_t)ldx * 8, (cuuint64_t)ldx * 8 * s1, (cuuint64_t)ldx * 8 * s2};
		const cuuint32_t box[4] = {(cuuint32_t)K, (cuuint32_t)P.pitch, (cuuint32_t)(P.TJ + 2), 1};
		const cuuint32_t estr[4] = {1, 1, 1, 1};
		if (enc(&tmx, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 4, const_cast<double *>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
		        CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
			return 2;
	}
	if (CONST) tmv = tmx;                                // never used
	else {
		const cuuint64_t gdim[4] = {(cuuint64_t)P.ndp, (cuuint64_t)s1, (cuuint64_t)my, (cuuint64_t)np};
		const cuuint64_t gstr[3] = {(cuuint64_t)P.ndp * 8, (cuuint64_t)P.ndp * 8 * s1, (cuuint64_t)P.ndp * 8 * s2};
		// the box is wider than the image (vpitch >= ndp): the copy engine zero-fills the padding slots
		const cuuint32_t box[4] = {(cuuint32_t)P.vpitch, (cuuint32_t)P.TI, (cuuint32_t)P.TJ, 1};
		const cuuint32_t estr[4] = {1, 1, 1, 1};
		if (enc(&tmv, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 4, M->dia_val, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
		        CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
			return 2;
	}
	static bool attr_set = false;
	if (!attr_set) {
		B200_CUDA(cudaFuncSetAttribute(spmm_lat_kernel<KP, NT, DOT, CONST>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 1024));
		attr_set = true;
	}
	// ---- plane ranges: all, interior (planes whose k - 1 and k + 1 are local) or the two boundary planes
	int ranges[2][2], nr = 1;
	ranges[0][0] = 0; ranges[0][1] = np;
	if (mode == 1) { ranges[0][0] = below ? 1 : 0; ranges[0][1] = above ? np - 1 : np; }
	else if (mode == 2) {
		nr = 0;
		if (below) { ranges[nr][0] = 0; ranges[nr][1] = 1; ++nr; }
		if (above && !(below && np == 1)) { ranges[nr][0] = np - 1; ranges[nr][1] = np; ++nr; }
	}
	const int tiles = P.NTI * P.NTJ, sms = g_b200.num_sms;
	int used = 0;
	for (int q = 0; q < nr; ++q) {
		const int pl = ranges[q][1] - ranges[q][0];
		if (pl <= 0) continue;
		// segments along k: enough items to balance the SMs, each paying two extra slices
		int bnseg = 1; double bcost = 1e300;
		for (int nseg = 1; nseg <= pl; ++nseg) {
			const int KL = (pl + nseg - 1) / nseg;
			const long long items = (long long)tiles * ((pl + KL - 1) / KL);
			const double cost = (double)((items + sms - 1) / sms) * (KL + 0.7);
			if (cost < bcost - 1e-9) { bcost = cost; bnseg = nseg; }
		}
		P.p_begin = ranges[q][0]; P.p_end = ranges[q][1];
		P.KL = (pl + bnseg - 1) / bnseg; P.nseg = (pl + P.KL - 1) / P.KL;
		const long long items = (long long)tiles * P.nseg;
		const int grid = (int)(items < sms ? items : sms);
		double *dp = nullptr;
		if (DOT) {
			if (used + grid > dot_cap) return used ? 1 : 2;
			dp = dot_part + (size_t)used * K;
			used += grid;
		}
		spmm_lat_kernel<KP, NT, DOT, CONST><<<grid, NT + 32, smem, g_b200.stream>>>(tmx, tmv, P, y, ldy, gate, dp);
		B200_KERNEL_CHECK();
	}
	if (DOT) *nparts = used;
	return 0;
}

template <int KP>
static int launch_spmm_lat_kp(const b200_mat *M, const double *x, int ldx, double *y, int ldy, const int *gate,
                              double *dot_part, int dot_cap, int *nparts, int mode)
{
	const bool cst = M->lat_const && M->dia_ndp <= 40 && !b200_opt(B200_OPT_LAT_NO_CONST);
	if (dot_part && cst) return launch_spmm_lat<KP, 480, true, true>(M, x, ldx, y, ldy, gate, dot_part, dot_cap, nparts, mode);
	if (dot_part) return launch_spmm_lat<KP, 480, true, false>(M, x, ldx, y, ldy, gate, dot_part, dot_cap, nparts, mode);
	if (cst) return launch_spmm_lat<KP, 480, false, true>(M, x, ldx, y, ldy, gate, nullptr, 0, nullptr, mode);
	return launch_spmm_lat<KP, 480, false, false>(M, x, ldx, y, ldy, gate, nullptr, 0, nullptr, mode);
}

int b200k_spmm_lat(const b200_mat *M, const double *x, int ldx, double *y, int ldy, int k, const int *gate,
                   double *dot_part, int dot_cap, int *nparts, int mode)
{
	if (M->lat_s1 <= 0) return 2;
	switch (k) {
#define LT(KP_) case 2 * KP_: return launch_spmm_lat_kp<KP_>(M, x, ldx, y, ldy, gate, dot_part, dot_cap, nparts, mode);
	DIA_WS_WIDTHS(LT)
#undef LT
	default: return 2;
	}
}
