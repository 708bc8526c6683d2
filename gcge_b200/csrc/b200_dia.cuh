// Device pieces shared by the diagonal-image SpMM kernels (b200_spmm.cu: 1-D row blocks; b200_spmm_lat.cu:
// lattice tiles marching through the planes).
#pragma once
#include "b200_internal.h"
#include "b200_tma.cuh"

constexpr int DIA_WMAX = 3;                            // widest run of consecutive offsets

// The block widths k = 2 KP with a compile-time kernel, X(KP) for each: they select the warp-specialised 1-D kernel
// (b200_spmm.cu), the lattice kernel and the multi-rank overlap path; other widths take the generic kernels.
#define DIA_WS_WIDTHS(X) X(4) X(5) X(6) X(8) X(10) X(12) X(15) X(16) X(20) X(24) X(25) X(28) X(30) X(32)

// the run of M's diagonal image that holds offset 0 (the main diagonal); -1: none
static inline int dia_zero_run(const b200_mat *M)
{
	for (int g = 0; g < M->dia_ng; ++g)
		if (M->dia_off_h[g] <= 0 && M->dia_off_h[g] + M->dia_grp_h[2 * g + 1] > 0) return g;
	return -1;
}

// One run of width W on the RB rows of a row group: x rows t = 0 .. RB + W - 2 of the run's box are read once
// (128-bit) and x row t feeds matrix rows t - j, j < W.  The run's values of a matrix row sit 16-byte aligned
// in the image (runs are padded to an even number of slots): one 128-bit broadcast load (+ 64 bits for W == 3).
// Separate multiply and add, offsets ascending: the operation order of the reference's scatter loop
// (app/app_ccs.c:116-131), bit for bit.
// zrow >= 0 (fused dot only): this run contains offset 0 at position zrow, i.e. x row i + zrow of the box IS
// row i of the block itself -- keep it in pst for the p^T w epilogue instead of reading p again from memory
template <int RB, int W, int K, int KP, int CP, bool DOT>
__device__ __forceinline__ void dia_run_ct(double (&acc)[RB][2 * CP], const double *tile, const double *vrow, int ndp,
                                           double2 (&pst)[RB][CP], int zrow)
{
	double2 xv[RB + W - 1][CP];
#pragma unroll
	for (int t = 0; t < RB + W - 1; ++t)
#pragma unroll
		for (int j = 0; j < CP; ++j) xv[t][j] = *reinterpret_cast<const double2 *>(tile + t * K + 2 * KP * j);
	if (DOT && zrow >= 0) {
#pragma unroll
		for (int i = 0; i < RB; ++i)
#pragma unroll
			for (int j = 0; j < CP; ++j)
				pst[i][j] = (W >= 3 && zrow == 2) ? xv[i + (W >= 3 ? 2 : 0)][j]
				          : ((W >= 2 && zrow == 1) ? xv[i + (W >= 2 ? 1 : 0)][j] : xv[i][j]);
	}
#pragma unroll
	for (int i = 0; i < RB; ++i) {
		const double2 a01 = *reinterpret_cast<const double2 *>(vrow);
		const double a2 = (W >= 3) ? vrow[2] : 0.0;
#pragma unroll
		for (int j = 0; j < CP; ++j) {
			acc[i][2 * j]     = __dadd_rn(acc[i][2 * j],     __dmul_rn(a01.x, xv[i][j].x));
			acc[i][2 * j + 1] = __dadd_rn(acc[i][2 * j + 1], __dmul_rn(a01.x, xv[i][j].y));
			if (W >= 2) {
				acc[i][2 * j]     = __dadd_rn(acc[i][2 * j],     __dmul_rn(a01.y, xv[i + (W >= 2 ? 1 : 0)][j].x));
				acc[i][2 * j + 1] = __dadd_rn(acc[i][2 * j + 1], __dmul_rn(a01.y, xv[i + (W >= 2 ? 1 : 0)][j].y));
			}
			if (W >= 3) {
				acc[i][2 * j]     = __dadd_rn(acc[i][2 * j],     __dmul_rn(a2, xv[i + (W >= 3 ? 2 : 0)][j].x));
				acc[i][2 * j + 1] = __dadd_rn(acc[i][2 * j + 1], __dmul_rn(a2, xv[i + (W >= 3 ? 2 : 0)][j].y));
			}
		}
		vrow += ndp;
	}
}


// The same with ROW-INVARIANT coefficients (a constant stencil): the run's values a0, a1, a2 come from the caller's
// registers / the constant bank instead of a shared-memory image -- no value traffic at all.
template <int RB, int W, int K, int KP, bool DOT>
__device__ __forceinline__ void dia_run_const(double (&acc)[RB][2], const double *tile, double a0, double a1, double a2,
                                              double2 (&pst)[RB][1], int zrow)
{
	double2 xv[RB + W - 1];
#pragma unroll
	for (int t = 0; t < RB + W - 1; ++t) xv[t] = *reinterpret_cast<const double2 *>(tile + t * K);
	if (DOT && zrow >= 0) {
#pragma unroll
		for (int i = 0; i < RB; ++i)
			pst[i][0] = (W >= 3 && zrow == 2) ? xv[i + (W >= 3 ? 2 : 0)] : ((W >= 2 && zrow == 1) ? xv[i + (W >= 2 ? 1 : 0)] : xv[i]);
	}
#pragma unroll
	for (int i = 0; i < RB; ++i) {
		acc[i][0] = __dadd_rn(acc[i][0], __dmul_rn(a0, xv[i].x));
		acc[i][1] = __dadd_rn(acc[i][1], __dmul_rn(a0, xv[i].y));
		if (W >= 2) {
			acc[i][0] = __dadd_rn(acc[i][0], __dmul_rn(a1, xv[i + (W >= 2 ? 1 : 0)].x));
			acc[i][1] = __dadd_rn(acc[i][1], __dmul_rn(a1, xv[i + (W >= 2 ? 1 : 0)].y));
		}
		if (W >= 3) {
			acc[i][0] = __dadd_rn(acc[i][0], __dmul_rn(a2, xv[i + (W >= 3 ? 2 : 0)].x));
			acc[i][1] = __dadd_rn(acc[i][1], __dmul_rn(a2, xv[i + (W >= 3 ? 2 : 0)].y));
		}
	}
}

// 1-D bulk copy whose lines are the first to leave L2: the matrix values are read once per SpMM,
// the x rows pulled by the neighbouring TMA boxes up to 2 m^2 rows later must stay
__device__ __forceinline__ void bulk_load_1d_evict_first(void *dst, const void *src, unsigned bytes, unsigned long long *bar)
{
	unsigned long long pol;
	asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
	             ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol) : "memory");
}

