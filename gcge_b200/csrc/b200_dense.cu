// K2/K3: the two dense contractions of the GCG hot path, on FP64 tensor-core tiles.
//
//   gram    C(p x q)  = X(n x p)^T Y(n x q)            replaces DenseMatQtAP 'N'/'S'/'D',
//                                                       reference app/app_lapack.c:24-183
//   lincomb Y(n x q)  = X(n x p) C(p x q) + Y diag(b)   replaces MultiVecLinearComb,
//                                                       reference app/app_lapack.c:463-534
//
// sm_100a has no tcgen05 kind for f64; the FP64 tensor path is the warp-level
// mma.sync.aligned.m8n8k4.f64 (SASS DMMA.8x8x4), which is what both kernels issue.
// Fragment layout (PTX ISA, m8n8k4 .f64): lane = 4*g + t
//   A (8x4, row):  a  = A[g][t]        B (4x8, col):  b = B[t][g]
//   C/D (8x8):     c0 = C[g][2t], c1 = C[g][2t+1]
//
// Multi-vector blocks are row-major (n x ld), so for gram both operands are read exactly
// as stored ([row][col] == [k][m] and [k][n]); for lincomb X is the row-major A operand.
// Shared-memory row strides are == 4 (mod 16) doubles, which makes every fragment load a
// two-wavefront (conflict-free) 64-bit access.
#include "b200_internal.h"
#include "b200_tma.cuh"
#include "b200_stream.cuh"
#include <cmath>

__device__ __forceinline__ void dmma_8x8x4(double &c0, double &c1, double a, double b)
{
	asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
	             : "+d"(c0), "+d"(c1)
	             : "d"(a), "d"(b));
}

// ------------------------------------------------------------------ cp.async helpers
// 8-byte copies work for any column offset; the 16-byte form needs 16-byte aligned global
// addresses (even column offset and even leading dimension).  src_size 0 zero-fills.
__device__ __forceinline__ void cp_async8(double *smem_dst, const double *gsrc, bool valid)
{
	const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
	const int sz = valid ? 8 : 0;
	asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(d), "l"(gsrc), "r"(sz));
}
__device__ __forceinline__ void cp_async16(double *smem_dst, const double *gsrc, bool valid)
{
	const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
	const int sz = valid ? 16 : 0;
	asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

// =========================================================================== gram
constexpr int GR_BP = 64;     // tile of X columns (rows of C)
constexpr int GR_BQ = 64;     // tile of Y columns (cols of C)
constexpr int GR_BK = 32;     // multi-vector rows per stage
constexpr int GR_S  = 68;     // smem row stride (doubles), == 4 mod 16
constexpr int GR_STAGES = 3;
constexpr int GR_STAGE_DBL = 2 * GR_BK * GR_S;          // Xs + Ys of one stage

// Each CTA: rows [chunk*rows_per_chunk, ...) x one (p-tile, q-tile); blockIdx.x = p-tile
// (fastest, so the CTAs that share a chunk's Y rows run together and meet in L2),
// blockIdx.y = chunk, blockIdx.z = q-tile.  8 warps = 4 p-slices (16 columns of X each) x 2
// halves of the staged rows.  Global -> shared through a 3-stage cp.async ring, so the
// tensor pipe works on stage i while stages i+1, i+2 are in flight.  Partials go to
// part[chunk][q][p]; a second kernel sums the chunks in a fixed order (deterministic).
// NQ8 = 8-column groups of Y this CTA's tile really has (1..8), a compile-time constant: a DMMA
// that is merely predicated off still occupies the tensor pipe (measured: with a run-time
// `if (j < nq8)` the pipe was 80 % busy at 17 TFLOP/s for q = 40, i.e. doing 64-column work),
// so the narrow tiles get their own instantiation instead of a predicate.
template <bool AL16, int NQ8>
__device__ __forceinline__ void
gram_partial_body(long long n, int p, int q, const double *x, int ldx, const double *y, int ldy,
                  long long rows_per_chunk, double *part)
{
	extern __shared__ __align__(16) double gsm[];
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int g = lane >> 2, t = lane & 3;
	const int pw = warp & 3, kh = warp >> 2;
	const int p0 = blockIdx.x * GR_BP, q0 = blockIdx.z * GR_BQ;
	const int pt = min(GR_BP, p - p0), qt = min(GR_BQ, q - q0);
	const bool p_live = pw * 16 < pt;                    // this warp's 16 X columns exist (warp-uniform)
	const long long r_begin = (long long)blockIdx.y * rows_per_chunk;
	long long r_end = r_begin + rows_per_chunk; if (r_end > n) r_end = n;
	const int ntiles = (int)((r_end - r_begin + GR_BK - 1) / GR_BK);

	auto load_stage = [&](int stage, int tile) {
		double *Xs = gsm + (size_t)stage * GR_STAGE_DBL, *Ys = Xs + GR_BK * GR_S;
		const long long r0 = r_begin + (long long)tile * GR_BK;
		if (AL16) {
			for (int i = tid; i < GR_BK * (GR_BP / 2); i += 256) {
				const int rr = i / (GR_BP / 2), cc = (i - rr * (GR_BP / 2)) * 2;
				const long long r = r0 + rr;
				const bool ok = (r < r_end) && (cc < pt);          // pt is even on this path
				cp_async16(Xs + rr * GR_S + cc, ok ? x + (size_t)r * ldx + p0 + cc : x, ok);
			}
			for (int i = tid; i < GR_BK * (NQ8 * 4); i += 256) {
				const int rr = i / (NQ8 * 4), cc = (i - rr * (NQ8 * 4)) * 2;
				const long long r = r0 + rr;
				const bool ok = (r < r_end) && (cc < qt);
				cp_async16(Ys + rr * GR_S + cc, ok ? y + (size_t)r * ldy + q0 + cc : y, ok);
			}
		} else {
			for (int i = tid; i < GR_BK * GR_BP; i += 256) {
				const int rr = i / GR_BP, cc = i - rr * GR_BP;
				const long long r = r0 + rr;
				const bool ok = (r < r_end) && (cc < pt);
				cp_async8(Xs + rr * GR_S + cc, ok ? x + (size_t)r * ldx + p0 + cc : x, ok);
			}
			for (int i = tid; i < GR_BK * (NQ8 * 8); i += 256) {
				const int rr = i / (NQ8 * 8), cc = i - rr * (NQ8 * 8);
				const long long r = r0 + rr;
				const bool ok = (r < r_end) && (cc < qt);
				cp_async8(Ys + rr * GR_S + cc, ok ? y + (size_t)r * ldy + q0 + cc : y, ok);
			}
		}
	};

	double acc[2][NQ8][2];
#pragma unroll
	for (int i = 0; i < 2; ++i)
#pragma unroll
		for (int j = 0; j < NQ8; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

#pragma unroll
	for (int s = 0; s < GR_STAGES - 1; ++s) {
		if (s < ntiles) load_stage(s, s);
		cp_async_commit();
	}
	for (int tile = 0; tile < ntiles; ++tile) {
		cp_async_wait<GR_STAGES - 2>();
		__syncthreads();
		{   // refill the stage that was consumed in the previous iteration
			const int nt = tile + GR_STAGES - 1;
			if (nt < ntiles) load_stage(nt % GR_STAGES, nt);
			cp_async_commit();
		}
		const double *Xs = gsm + (size_t)(tile % GR_STAGES) * GR_STAGE_DBL, *Ys = Xs + GR_BK * GR_S;
		if (p_live) {
#pragma unroll
			for (int ks = 0; ks < GR_BK / 2; ks += 4) {
				const int kr = kh * (GR_BK / 2) + ks + t;
				const double a0 = Xs[kr * GR_S + pw * 16 + g];
				const double a1 = Xs[kr * GR_S + pw * 16 + 8 + g];
#pragma unroll
				for (int j = 0; j < NQ8; ++j) {
					const double b = Ys[kr * GR_S + j * 8 + g];
					dmma_8x8x4(acc[0][j][0], acc[0][j][1], a0, b);
					dmma_8x8x4(acc[1][j][0], acc[1][j][1], a1, b);
				}
			}
		}
	}
	cp_async_wait<0>();
	__syncthreads();
	// combine the two row halves through shared memory: a 64 x 68 tile in stage 0
	double *red = gsm;
	if (kh == 1) {
#pragma unroll
		for (int i = 0; i < 2; ++i)
#pragma unroll
			for (int j = 0; j < NQ8; ++j) {
				const int cr = pw * 16 + i * 8 + g;        // row of the C tile (0..63)
				red[cr * GR_S + j * 8 + 2 * t]     = acc[i][j][0];
				red[cr * GR_S + j * 8 + 2 * t + 1] = acc[i][j][1];
			}
	}
	__syncthreads();
	if (kh == 0) {
		double *out = part + (size_t)blockIdx.y * p * q;
#pragma unroll
		for (int i = 0; i < 2; ++i)
#pragma unroll
			for (int j = 0; j < NQ8; ++j) {
				const int cr = pw * 16 + i * 8 + g;
#pragma unroll
				for (int h = 0; h < 2; ++h) {
					const int cc = j * 8 + 2 * t + h;
					if (cr < pt && cc < qt)
						out[(size_t)(q0 + cc) * p + (p0 + cr)] = acc[i][j][h] + red[cr * GR_S + cc];
				}
			}
	}
}

template <bool AL16>
__global__ void __launch_bounds__(256, 2)
gram_partial_kernel(long long n, int p, int q, const double *x, int ldx, const double *y, int ldy,
                    long long rows_per_chunk, double *part)
{
	const int qt = min(GR_BQ, q - (int)blockIdx.z * GR_BQ);
	switch ((qt + 7) >> 3) {                             // uniform over the CTA
	case 1: gram_partial_body<AL16, 1>(n, p, q, x, ldx, y, ldy, rows_per_chunk, part); break;
	case 2: gram_partial_body<AL16, 2>(n, p, q, x, ldx, y, ldy, rows_per_chunk, part); break;
	case 3: gram_partial_body<AL16, 3>(n, p, q, x, ldx, y, ldy, rows_per_chunk, part); break;
	case 4: gram_partial_body<AL16, 4>(n, p, q, x, ldx, y, ldy, rows_per_chunk, part); break;
	case 5: gram_partial_body<AL16, 5>(n, p, q, x, ldx, y, ldy, rows_per_chunk, part); break;
	case 6: gram_partial_body<AL16, 6>(n, p, q, x, ldx, y, ldy, rows_per_chunk, part); break;
	case 7: gram_partial_body<AL16, 7>(n, p, q, x, ldx, y, ldy, rows_per_chunk, part); break;
	default: gram_partial_body<AL16, 8>(n, p, q, x, ldx, y, ldy, rows_per_chunk, part); break;
	}
}

// ------------------------------------------------------------------ gram, TMA-fed
// Same CTA tile (64 X columns x up to 64 Y columns over a chunk of rows), warp roles (4 column slices x 2 row
// halves) and DMMA fragments as gram_partial_body, but the ring is fed by a producer thread with tensor-map
// copies, like lincomb_tma_body: per stage of G2_BK rows, the X tile arrives as 4 boxes and the Y tile as
// ceil(qt / 16) boxes of 16 columns (128 bytes per row) with the 128-byte swizzle -- 7 copies per stage at
// q = 40 where the cp.async version spends 85 % of its instructions on copy addresses, predicates and stage
// barriers (ncu profiles/ncu_r1f_*: tensor pipe 65 % busy), and where a first bulk-copy version needed one copy
// per tile ROW (64 per stage) and was producer-bound.  Both operands are read in the 4-rows-by-8-columns
// fragment pattern; in a swizzled box the 16-byte chunk index of a row is XOR-ed with row % 8, so rows with
// row % 8 < 4 keep a slice's 8 columns in one 64-byte half of the bank round and the others in the other
// half: a k-step therefore takes the rows {0, 4, 1, 5} (then {2, 6, 3, 7}) of an 8-row group -- two rows per
// half, two wavefronts per fragment load, the minimum.  Any permutation of the rows of a stage is as good as
// any other for a sum over rows, as long as the X and Y fragments use the same one.
// Needs 16-byte aligned operands (even column offsets and leading dimensions).
constexpr int G2_BK = 32;                              // multi-vector rows per stage (== GR_BK: chunks are multiples of it)
constexpr int G2_BOX = G2_BK * 128;                    // bytes of one 16-column box
constexpr int G2_MAX_NS = 4;

template <int NQ8>
__device__ __forceinline__ void
gram_tma2_body(const CUtensorMap *tmx, const CUtensorMap *tmy, long long n, int p, int q, long long rows_per_chunk,
               int NS, double *part)
{
	extern __shared__ __align__(1024) unsigned char g2sm[];
	__shared__ unsigned long long full[G2_MAX_NS], empty[G2_MAX_NS];
	constexpr int NQB = (NQ8 + 1) / 2;                 // Y boxes
	constexpr int STAGE = (4 + NQB) * G2_BOX;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int p0 = blockIdx.x * GR_BP, q0 = blockIdx.z * GR_BQ;
	const int pt = min(GR_BP, p - p0), qt = min(GR_BQ, q - q0);
	const long long r_begin = (long long)blockIdx.y * rows_per_chunk;
	long long r_end = r_begin + rows_per_chunk; if (r_end > n) r_end = n;
	const int ntiles = (int)((r_end - r_begin + G2_BK - 1) / G2_BK);
	if (tid == 0) {
		for (int s = 0; s < NS; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 8); }
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
	}
	__syncthreads();

	if (warp == 8) {
		// ------------------------------------------------------------------ producer
		if (lane == 0) {
			int slot = 0; unsigned phase = 0;
			for (int tile = 0; tile < ntiles; ++tile) {
				const int r0 = (int)(r_begin + (long long)tile * G2_BK);
				unsigned char *st = g2sm + (size_t)slot * STAGE;
				mbar_spin(empty + slot, phase ^ 1u);
				mbar_expect_tx(full + slot, (unsigned)STAGE);
				// boxes beyond the last column / row of an operand arrive as zeros
#pragma unroll
				for (int b = 0; b < 4; ++b) tma_load_2d(st + b * G2_BOX, tmx, p0 + 16 * b, r0, full + slot);
#pragma unroll
				for (int b = 0; b < NQB; ++b) tma_load_2d(st + (4 + b) * G2_BOX, tmy, q0 + 16 * b, r0, full + slot);
				if (++slot == NS) { slot = 0; phase ^= 1u; }
			}
		}
		return;
	}
	// ---------------------------------------------------------------------- consumer warps
	const int g = lane >> 2, t = lane & 3;
	const int pw = warp & 3, kh = warp >> 2;
	const bool p_live = pw * 16 < pt;
	double acc[2][NQ8][2];
#pragma unroll
	for (int i = 0; i < 2; ++i)
#pragma unroll
		for (int j = 0; j < NQ8; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
	// row of the stage this lane reads in k-step s: kh*16 + 8*(s >> 1) + 2*(s & 1) + {0, 4, 1, 5}[t]
	const int rperm = (t & 1) * 4 + (t >> 1);
	int slot = 0; unsigned phase = 0;
	for (int tile = 0; tile < ntiles; ++tile) {
		mbar_spin(full + slot, phase);
		const double *st = reinterpret_cast<const double *>(g2sm + (size_t)slot * STAGE);
		const double *Xb = st + pw * (G2_BOX / 8);
		if (p_live) {
#pragma unroll
			for (int s = 0; s < 4; ++s) {
				const int r = kh * 16 + 8 * (s >> 1) + 2 * (s & 1) + rperm;
				const int sw = (2 * (s & 1) + rperm) & 7;                       // r % 8
				const int lo = r * 16 + ((((g >> 1)) ^ sw) << 1) + (g & 1);      // column g of a box
				const int hi = r * 16 + (((4 + (g >> 1)) ^ sw) << 1) + (g & 1);  // column 8 + g
				const double a0 = Xb[lo], a1 = Xb[hi];
#pragma unroll
				for (int j = 0; j < NQ8; ++j) {
					const double b = st[(4 + (j >> 1)) * (G2_BOX / 8) + ((j & 1) ? hi : lo)];
					dmma_8x8x4(acc[0][j][0], acc[0][j][1], a0, b);
					dmma_8x8x4(acc[1][j][0], acc[1][j][1], a1, b);
				}
			}
		}
		// the fragment loads of this stage must have been performed before the slot is handed back (see lincomb_tma_body)
		asm volatile("fence.acq_rel.cta;" ::: "memory");
		__syncwarp();
		if (lane == 0) mbar_arrive(empty + slot);
		if (++slot == NS) { slot = 0; phase ^= 1u; }
	}
	// combine the two row halves through shared memory (the ring is dead: every stage was consumed); consumer-only
	// barrier, the producer warp is gone
	asm volatile("bar.sync 1, 256;" ::: "memory");
	double *red = reinterpret_cast<double *>(g2sm);
	if (kh == 1) {
#pragma unroll
		for (int i = 0; i < 2; ++i)
#pragma unroll
			for (int j = 0; j < NQ8; ++j) {
				const int cr = pw * 16 + i * 8 + g;
				red[cr * GR_S + j * 8 + 2 * t]     = acc[i][j][0];
				red[cr * GR_S + j * 8 + 2 * t + 1] = acc[i][j][1];
			}
	}
	asm volatile("bar.sync 1, 256;" ::: "memory");
	if (kh == 0) {
		double *out = part + (size_t)blockIdx.y * p * q;
#pragma unroll
		for (int i = 0; i < 2; ++i)
#pragma unroll
			for (int j = 0; j < NQ8; ++j) {
				const int cr = pw * 16 + i * 8 + g;
#pragma unroll
				for (int h = 0; h < 2; ++h) {
					const int cc = j * 8 + 2 * t + h;
					if (cr < pt && cc < qt)
						out[(size_t)(q0 + cc) * p + (p0 + cr)] = acc[i][j][h] + red[cr * GR_S + cc];
				}
			}
	}
}

// lower != 0 ('S' with x == y on one rank): tiles strictly above the diagonal are skipped, the reduction mirrors
__global__ void __launch_bounds__(288, 2)
gram_tma2_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmy, long long n, int p, int q,
                 long long rows_per_chunk, int NS, int lower, double *part)
{
	if (lower && blockIdx.z > blockIdx.x) return;
	const int qt = min(GR_BQ, q - (int)blockIdx.z * GR_BQ);
	switch ((qt + 7) >> 3) {                             // uniform over the CTA
	case 1: gram_tma2_body<1>(&tmx, &tmy, n, p, q, rows_per_chunk, NS, part); break;
	case 2: gram_tma2_body<2>(&tmx, &tmy, n, p, q, rows_per_chunk, NS, part); break;
	case 3: gram_tma2_body<3>(&tmx, &tmy, n, p, q, rows_per_chunk, NS, part); break;
	case 4: gram_tma2_body<4>(&tmx, &tmy, n, p, q, rows_per_chunk, NS, part); break;
	case 5: gram_tma2_body<5>(&tmx, &tmy, n, p, q, rows_per_chunk, NS, part); break;
	case 6: gram_tma2_body<6>(&tmx, &tmy, n, p, q, rows_per_chunk, NS, part); break;
	case 7: gram_tma2_body<7>(&tmx, &tmy, n, p, q, rows_per_chunk, NS, part); break;
	default: gram_tma2_body<8>(&tmx, &tmy, n, p, q, rows_per_chunk, NS, part); break;
	}
}

// 0 launched, 1 error, 2 not applicable
static int gram_tma2_launch(long long n, int p, int q, const double *x, int ldx, const double *y, int ldy,
                            long long rows_per_chunk, dim3 grid, int lower, double *part)
{
	if (n < G2_BK || n > 0x7fffffffLL || ((uintptr_t)x % 16) || ((uintptr_t)y % 16) || (ldx & 1) || (ldy & 1)) return 2;
	tmap_encode_fn enc = tmap_encoder();
	if (!enc) return 2;
	CUtensorMap tmx, tmy;
	const cuuint32_t box[2] = {16, (cuuint32_t)G2_BK};
	const cuuint32_t estr[2] = {1, 1};
	{
		const cuuint64_t gdim[2] = {(cuuint64_t)p, (cuuint64_t)n};
		const cuuint64_t gstr[1] = {(cuuint64_t)ldx * 8};
		if (enc(&tmx, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(x), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
		        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
			return 2;
	}
	{
		const cuuint64_t gdim[2] = {(cuuint64_t)q, (cuuint64_t)n};
		const cuuint64_t gstr[1] = {(cuuint64_t)ldy * 8};
		if (enc(&tmy, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(y), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
		        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
			return 2;
	}
	// ring depth: four stages while two CTAs still share an SM (<= 48 Y columns per tile), else three
	const int nqb = ((q < GR_BQ ? q : GR_BQ) + 15) / 16;
	const int NS = nqb <= 3 ? 4 : 3;
	size_t smem = (size_t)NS * (4 + nqb) * G2_BOX;
	const size_t red_bytes = sizeof(double) * GR_BP * GR_S;
	if (smem < red_bytes) smem = red_bytes;
	static bool attr_set = false;
	if (!attr_set) {
		B200_CUDA(cudaFuncSetAttribute(gram_tma2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * 8 * G2_BOX));
		attr_set = true;
	}
	gram_tma2_kernel<<<grid, 288, smem, g_b200.stream>>>(tmx, tmy, n, p, q, rows_per_chunk, NS, lower, part);
	B200_KERNEL_CHECK();
	return 0;
}

// C[i + j*ldc] = sum_chunks part[chunk][i + j*p]; mode 'S' mirrors the lower triangle.
__global__ void gram_reduce_kernel(int p, int q, int chunks, const double *__restrict__ part, double alpha,
                                   double *__restrict__ c, int c_rs, int c_cs, int symmetric)
{
	const int idx = blockIdx.x * blockDim.x + threadIdx.x;
	if (idx >= p * q) return;
	const int i = idx % p, j = idx / p;
	if (symmetric && i < j) return;
	double s = 0.0;
	for (int ch = 0; ch < chunks; ++ch) s += part[(size_t)ch * p * q + idx];
	s *= alpha;
	c[(size_t)i * c_rs + (size_t)j * c_cs] = s;
	if (symmetric && i > j) c[(size_t)j * c_rs + (size_t)i * c_cs] = s;
}

// 'D': column dot products, c[col * stride] = alpha * x[:, col] . y[:, col], on the geometry of the streaming kernels
// (b200_stream.cuh): a thread owns one 16-byte column pair and every rp-th row of its CTA's chunk with ST_UNROLL rows
// of both streams in flight, so every warp request is a run of whole row segments; per-CTA partials, and the last
// CTA to arrive adds them in a fixed order (deterministic, identical on every rank).  The first version (blockDim =
// (32, 8), 8-byte loads, column passes of 32) left 24 of 32 lanes idle on the second pass at k = 40 and ran at
// 0.50-0.60 of HBM (profiles/config5_kernel_sweep_r2_n8M.log).
template <int VEC>
__global__ void __launch_bounds__(ST_THREADS)
dots_stream_kernel(long long n, int k, StreamGeom g, const double *__restrict__ x, int ldx, const double *__restrict__ y, int ldy,
                   double alpha, double *c, int stride, double *part, unsigned *ticket)
{
	const StreamThread t = stream_thread<VEC>(g);
	const long long r_begin = (long long)blockIdx.x * g.rows_per_chunk;
	long long r_end = r_begin + g.rows_per_chunk; if (r_end > n) r_end = n;
	double acc[1][VEC];
#pragma unroll
	for (int i = 0; i < VEC; ++i) acc[0][i] = 0.0;
	if (t.active) {
		for (long long row0 = r_begin + t.rl; row0 < r_end; row0 += (long long)ST_UNROLL * g.rp) {
			StV<VEC> xv[ST_UNROLL], yv[ST_UNROLL];
#pragma unroll
			for (int u = 0; u < ST_UNROLL; ++u) {
				const long long row = row0 + (long long)u * g.rp;
				if (row < r_end) { xv[u] = st_ld<VEC>(x + (size_t)row * ldx + t.c); yv[u] = st_ld<VEC>(y + (size_t)row * ldy + t.c); }
			}
#pragma unroll
			for (int u = 0; u < ST_UNROLL; ++u) {
				const long long row = row0 + (long long)u * g.rp;
				if (row < r_end) {
#pragma unroll
					for (int i = 0; i < VEC; ++i) acc[0][i] = fma(xv[u].v[i], yv[u].v[i], acc[0][i]);
				}
			}
		}
	}
	if (!stream_reduce_and_elect<VEC, 1>(acc, k, g, t, part, ticket)) return;
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	for (int col = warp; col < k; col += ST_THREADS / 32) {
		const double s = stream_total<1>(part, gridDim.x, k, 0, col);
		if (lane == 0) c[(size_t)col * stride] = alpha * s;
	}
}

__global__ void fill2d_kernel(int p, int q, double v, double *c, int c_rs, int c_cs)
{
	const int idx = blockIdx.x * blockDim.x + threadIdx.x;
	if (idx >= p * q) return;
	c[(size_t)(idx % p) * c_rs + (size_t)(idx / p) * c_cs] = v;
}

// scatter a contiguous column-major p x q block (already summed over ranks) into the caller's
// strided destination; mode 'S' mirrors the lower triangle, 'D' writes p values with stride c_rs
__global__ void gram_scatter_kernel(int p, int q, const double *__restrict__ tmp, double *__restrict__ c, int c_rs,
                                    int c_cs, int symmetric)
{
	const int idx = blockIdx.x * blockDim.x + threadIdx.x;
	if (idx >= p * q) return;
	const int i = idx % p, j = idx / p;
	if (symmetric && i < j) return;
	const double s = tmp[idx];
	c[(size_t)i * c_rs + (size_t)j * c_cs] = s;
	if (symmetric && i > j) c[(size_t)j * c_rs + (size_t)i * c_cs] = s;
}

int b200k_multi(void) { return g_b200.nranks > 1 ? g_b200.nranks : 1; }

// 'D': c_dev[i*c_rs] = alpha * x_i . y_i  (c_cs ignored)
int b200k_gram(char mode, long long n, int p, int q, double alpha, const double *x, int ldx,
               const double *y, int ldy, double *c_dev, int c_rs, int c_cs, int dist)
{
	if (p <= 0 || q <= 0) return 0;
	cudaStream_t st = g_b200.stream;
	B200Prof prof(mode == 'D' ? B200_PROF_DOTS : (n <= 1024 && !dist ? B200_PROF_SMALL : B200_PROF_GRAM),
	              mode == 'D' ? 16.0 * n * p : 8.0 * n * ((double)p + q) + 8.0 * p * q,
	              mode == 'D' ? 2.0 * n * p : 2.0 * n * p * q);
	// Several ranks: every rank reduces its slab into a contiguous block, one NCCL allreduce sums
	// the blocks (reference: MPI_Allreduce after the local inner product, src/ops_multi_vec.c:214),
	// then the block is scattered into the caller's layout.  All ranks get identical bits.
	const bool multi = dist && b200_multi();
	double *dst = c_dev; int d_rs = c_rs, d_cs = c_cs;
	const int cnt = (mode == 'D') ? p : p * q;
	if (multi) {
		dst = (double *)b200_scratch(8, sizeof(double) * (size_t)cnt + 256);
		if (!dst) return 1;
		d_rs = 1; d_cs = p;
	}
	if (mode == 'D') {
		const int k = p;
		if (n <= 0) {
			fill2d_kernel<<<b200_ceil_div(k, 128), 128, 0, st>>>(k, 1, 0.0, dst, d_rs, 0);
			B200_KERNEL_CHECK();
		} else {
			// at most DOTS_COLS columns per launch (the geometry wants a column group per thread of one CTA row pass)
			constexpr int DOTS_COLS = 128;
			for (int c0 = 0; c0 < k; c0 += DOTS_COLS) {
				const int kc = (k - c0 < DOTS_COLS) ? k - c0 : DOTS_COLS;
				const double *xc = x + c0, *yc = y + c0;
				const StreamGeom g = stream_geometry(n, kc, stream_aligned16(xc, ldx) && stream_aligned16(yc, ldy));
				char *base = (char *)b200_scratch(0, sizeof(double) * (size_t)(g.chunks + 1) * kc + 64);
				if (!base) return 1;
				double *part = (double *)base;
				unsigned *ticket = (unsigned *)(part + (size_t)(g.chunks + 1) * kc);
				B200_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned), st));
				ST_DISPATCH_VEC(g, (dots_stream_kernel<VEC><<<g.chunks, ST_THREADS, 0, st>>>(n, kc, g, xc, ldx, yc, ldy, alpha,
				                                                                          dst + (size_t)c0 * d_rs, d_rs, part, ticket)));
				B200_KERNEL_CHECK();
			}
		}
		if (multi) {
			if (b200k_allreduce_sum(dst, (size_t)k)) return 1;
			gram_scatter_kernel<<<b200_ceil_div(k, 128), 128, 0, st>>>(k, 1, dst, c_dev, c_rs, 0, 0);
			B200_KERNEL_CHECK();
		}
		return 0;
	}
	if (n <= 0) {
		fill2d_kernel<<<b200_ceil_div((long long)p * q, 256), 256, 0, st>>>(p, q, 0.0, dst, d_rs, d_cs);
		B200_KERNEL_CHECK();
	} else {
		const int ptiles = b200_ceil_div(p, GR_BP), qtiles = b200_ceil_div(q, GR_BQ);
		long long chunks = (long long)(g_b200.num_sms * 4) / ((long long)ptiles * qtiles);
		if (chunks < 1) chunks = 1;
		long long rows_per_chunk = (n + chunks - 1) / chunks;
		rows_per_chunk = ((rows_per_chunk + GR_BK - 1) / GR_BK) * GR_BK;
		if (rows_per_chunk < 4 * GR_BK) rows_per_chunk = 4 * GR_BK;
		chunks = (n + rows_per_chunk - 1) / rows_per_chunk;
		double *part = (double *)b200_scratch(0, sizeof(double) * (size_t)chunks * p * q);
		if (!part) return 1;
		dim3 grid(ptiles, (unsigned)chunks, qtiles);
		const size_t smem = sizeof(double) * (size_t)GR_STAGES * GR_STAGE_DBL;
		static bool attr_set = false;
		if (!attr_set) {
			B200_CUDA(cudaFuncSetAttribute(gram_partial_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
			B200_CUDA(cudaFuncSetAttribute(gram_partial_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
			attr_set = true;
		}
		// 16-byte copies need even column offsets (pointer alignment), even leading dimensions and
		// even tile widths; anything else takes the 8-byte path
		const bool al16 = (((uintptr_t)x | (uintptr_t)y) % 16 == 0) && (ldx % 2 == 0) && (ldy % 2 == 0) &&
		                  (p % 2 == 0) && (q % 2 == 0);
		// 'S' with one operand on one rank: only the tiles on and below the diagonal are computed
		const int lower = (!multi && mode == 'S' && x == y && ldx == ldy && p == q) ? 1 : 0;
		int rc_tma = 2;
		if (al16) {
			rc_tma = gram_tma2_launch(n, p, q, x, ldx, y, ldy, rows_per_chunk, grid, lower, part);
			if (rc_tma == 1) return 1;
		}
		if (rc_tma == 2) {
			if (al16) gram_partial_kernel<true><<<grid, 256, smem, st>>>(n, p, q, x, ldx, y, ldy, rows_per_chunk, part);
			else      gram_partial_kernel<false><<<grid, 256, smem, st>>>(n, p, q, x, ldx, y, ldy, rows_per_chunk, part);
			B200_KERNEL_CHECK();
		}
		gram_reduce_kernel<<<b200_ceil_div((long long)p * q, 256), 256, 0, st>>>(p, q, (int)chunks, part, alpha, dst,
		                                                                        d_rs, d_cs, (!multi && mode == 'S') ? 1 : 0);
		B200_KERNEL_CHECK();
	}
	if (multi) {
		if (b200k_allreduce_sum(dst, (size_t)p * q)) return 1;
		gram_scatter_kernel<<<b200_ceil_div((long long)p * q, 256), 256, 0, st>>>(p, q, dst, c_dev, c_rs, c_cs,
		                                                                         mode == 'S' ? 1 : 0);
		B200_KERNEL_CHECK();
	}
	return 0;
}

// ======================================================================== lincomb
constexpr int LC_BM = 128;    // multi-vector rows per CTA
constexpr int LC_BN = 64;     // output columns per CTA
constexpr int LC_BK = 16;     // slice of the contraction (columns of X / rows of C)
constexpr int LC_SX = 20;     // Xs row stride, == 4 mod 16
constexpr int LC_SC = 68;     // Cs row stride, == 4 mod 16
constexpr int LC_STAGES = 3;
constexpr int LC_STAGE_DBL = LC_BM * LC_SX + LC_BK * LC_SC;

// C: element (k,j) at c[k*c_rs + j*c_cs].  blockIdx.x = column tile (fastest: the CTAs that
// re-read one X row tile run together), blockIdx.y = row tile.  8 warps, warp w owns rows
// [16w,16w+16) x 64 columns; 3-stage cp.async ring over the contraction dimension.
template <bool HAS_BETA, bool AL16, int NQ8>
__device__ __forceinline__ void
lincomb_body(long long n, int p, int q, const double *x, int ldx, const double *__restrict__ c, int c_rs,
             int c_cs, const double *__restrict__ beta, int incb, double *y, int ldy)
{
	extern __shared__ __align__(16) double lsm[];
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int g = lane >> 2, t = lane & 3;
	const long long r0 = (long long)blockIdx.y * LC_BM;
	const int n0 = blockIdx.x * LC_BN;
	const int nt = min(LC_BN, q - n0);
	const int ktiles = (p + LC_BK - 1) / LC_BK;

	auto load_stage = [&](int stage, int kt) {
		double *Xs = lsm + (size_t)stage * LC_STAGE_DBL, *Cs = Xs + LC_BM * LC_SX;
		const int k0 = kt * LC_BK;
		if (AL16) {
			for (int i = tid; i < LC_BM * (LC_BK / 2); i += 256) {
				const int rr = i / (LC_BK / 2), kk = (i - rr * (LC_BK / 2)) * 2;
				const long long r = r0 + rr;
				const bool ok = (r < n) && (k0 + kk < p);          // p is even on this path
				cp_async16(Xs + rr * LC_SX + kk, ok ? x + (size_t)r * ldx + k0 + kk : x, ok);
			}
		} else {
			for (int i = tid; i < LC_BM * LC_BK; i += 256) {
				const int rr = i / LC_BK, kk = i - rr * LC_BK;
				const long long r = r0 + rr;
				const bool ok = (r < n) && (k0 + kk < p);
				cp_async8(Xs + rr * LC_SX + kk, ok ? x + (size_t)r * ldx + k0 + kk : x, ok);
			}
		}
		if (c_rs == 1) {             // column-major C: walk down columns
			for (int i = tid; i < LC_BK * (NQ8 * 8); i += 256) {
				const int cc = i / LC_BK, kk = i - cc * LC_BK;
				const bool ok = (k0 + kk < p) && (cc < nt);
				cp_async8(Cs + kk * LC_SC + cc, ok ? c + (size_t)(n0 + cc) * c_cs + k0 + kk : c, ok);
			}
		} else {                     // row-major (or general strides): walk along rows
			for (int i = tid; i < LC_BK * (NQ8 * 8); i += 256) {
				const int kk = i / (NQ8 * 8), cc = i - kk * (NQ8 * 8);
				const bool ok = (k0 + kk < p) && (cc < nt);
				cp_async8(Cs + kk * LC_SC + cc, ok ? c + (size_t)(k0 + kk) * c_rs + (size_t)(n0 + cc) * c_cs : c, ok);
			}
		}
	};

	double acc[2][NQ8][2];
#pragma unroll
	for (int i = 0; i < 2; ++i)
#pragma unroll
		for (int j = 0; j < NQ8; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

#pragma unroll
	for (int s = 0; s < LC_STAGES - 1; ++s) {
		if (s < ktiles) load_stage(s, s);
		cp_async_commit();
	}
	for (int kt = 0; kt < ktiles; ++kt) {
		cp_async_wait<LC_STAGES - 2>();
		__syncthreads();
		{
			const int nk = kt + LC_STAGES - 1;
			if (nk < ktiles) load_stage(nk % LC_STAGES, nk);
			cp_async_commit();
		}
		const double *Xs = lsm + (size_t)(kt % LC_STAGES) * LC_STAGE_DBL, *Cs = Xs + LC_BM * LC_SX;
#pragma unroll
		for (int ks = 0; ks < LC_BK; ks += 4) {
			const double a0 = Xs[(warp * 16 + g) * LC_SX + ks + t];
			const double a1 = Xs[(warp * 16 + 8 + g) * LC_SX + ks + t];
#pragma unroll
			for (int j = 0; j < NQ8; ++j) {
				const double b = Cs[(ks + t) * LC_SC + j * 8 + g];
				dmma_8x8x4(acc[0][j][0], acc[0][j][1], a0, b);
				dmma_8x8x4(acc[1][j][0], acc[1][j][1], a1, b);
			}
		}
	}
	cp_async_wait<0>();
#pragma unroll
	for (int i = 0; i < 2; ++i) {
		const long long r = r0 + warp * 16 + i * 8 + g;
		if (r >= n) continue;
#pragma unroll
		for (int j = 0; j < NQ8; ++j)
#pragma unroll
			for (int h = 0; h < 2; ++h) {
				const int cc = j * 8 + 2 * t + h;
				if (cc < nt) {
					double v = acc[i][j][h];
					double *yp = y + (size_t)r * ldy + n0 + cc;
					if (HAS_BETA) {
						const double b = beta[(size_t)incb * (n0 + cc)];
						if (b != 0.0) v += b * (*yp);      // beta == 0 overwrites (no NaN carry-over)
					}
					*yp = v;
				}
			}
	}
}

// the column tile's width in 8-column groups is a compile-time constant of the body: see
// gram_partial_body (predicated-off DMMAs still occupy the tensor pipe)
template <bool HAS_BETA, bool AL16>
__global__ void __launch_bounds__(256, 2)
lincomb_kernel(long long n, int p, int q, const double *x, int ldx, const double *__restrict__ c, int c_rs,
               int c_cs, const double *__restrict__ beta, int incb, double *y, int ldy)
{
	const int nt = min(LC_BN, q - (int)blockIdx.x * LC_BN);
	switch ((nt + 7) >> 3) {                             // uniform over the CTA
	case 1: lincomb_body<HAS_BETA, AL16, 1>(n, p, q, x, ldx, c, c_rs, c_cs, beta, incb, y, ldy); break;
	case 2: lincomb_body<HAS_BETA, AL16, 2>(n, p, q, x, ldx, c, c_rs, c_cs, beta, incb, y, ldy); break;
	case 3: lincomb_body<HAS_BETA, AL16, 3>(n, p, q, x, ldx, c, c_rs, c_cs, beta, incb, y, ldy); break;
	case 4: lincomb_body<HAS_BETA, AL16, 4>(n, p, q, x, ldx, c, c_rs, c_cs, beta, incb, y, ldy); break;
	case 5: lincomb_body<HAS_BETA, AL16, 5>(n, p, q, x, ldx, c, c_rs, c_cs, beta, incb, y, ldy); break;
	case 6: lincomb_body<HAS_BETA, AL16, 6>(n, p, q, x, ldx, c, c_rs, c_cs, beta, incb, y, ldy); break;
	case 7: lincomb_body<HAS_BETA, AL16, 7>(n, p, q, x, ldx, c, c_rs, c_cs, beta, incb, y, ldy); break;
	default: lincomb_body<HAS_BETA, AL16, 8>(n, p, q, x, ldx, c, c_rs, c_cs, beta, incb, y, ldy); break;
	}
}

// ------------------------------------------------------------------ lincomb, TMA-fed
// The cp.async version above spends 85 % of its instructions outside the DMMAs (address arithmetic of
// the copies, predicates, stage barriers: ncu profiles/ncu_r1f_*: 5.06 G warp instructions for 0.75 G
// DMMAs, tensor pipe 77 % busy).  Here a producer warp feeds the ring: the X tile (128 rows x 16
// columns = 128 bytes per row) by ONE tensor-map copy per stage with the 128-byte swizzle (the 16-byte
// chunk index of a row is XOR-ed with row % 8, which makes the A-fragment loads -- 8 consecutive rows
// x 4 consecutive columns -- two-wavefront, i.e. conflict-free), the C tile by one 1-D bulk copy per
// row into rows padded to 68 doubles (the B-fragment pattern, 4 rows x 8 consecutive columns, needs
// the padding; no swizzle mode gives it).  The 8 consumer warps do nothing but fragment loads and
// DMMAs and hand a stage back with one mbarrier arrive per warp.
// Needs 16-byte aligned operands: x (even column offset and leading dimension), row-major C with even
// row stride, even column offset and even q; everything else takes the kernel above.
constexpr int LT_NS = 4;                                     // ring depth
constexpr int LT_X_BYTES = LC_BM * LC_BK * 8;                // 16 KB, dense (swizzled) rows of 128 bytes
constexpr int LT_C_BYTES = LC_BK * LC_SC * 8;                // 16 rows padded to 68 doubles
constexpr int LT_STAGE_BYTES = LT_X_BYTES + LT_C_BYTES;

template <bool HAS_BETA, int NQ8>
__device__ __forceinline__ void
lincomb_tma_body(const CUtensorMap *tmx, long long n, int p, int q, const double *__restrict__ c, int c_rs,
                 const double *__restrict__ beta, int incb, double *y, int ldy)
{
	extern __shared__ __align__(1024) unsigned char tsm[];
	__shared__ unsigned long long full[LT_NS], empty[LT_NS];
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const long long r0 = (long long)blockIdx.y * LC_BM;
	const int n0 = blockIdx.x * LC_BN;
	const int nt = min(LC_BN, q - n0);
	const int ktiles = (p + LC_BK - 1) / LC_BK;
	unsigned char *xs_base = tsm, *cs_base = tsm + LT_NS * LT_X_BYTES;
	// the C rows of the last k tile beyond p are never copied: make sure no NaN bit pattern sits there
	// (they meet zero X columns, but 0 * NaN would poison the accumulators)
	for (int i = tid; i < LT_NS * LC_BK * LC_SC; i += blockDim.x) reinterpret_cast<double *>(cs_base)[i] = 0.0;
	if (tid == 0) {
		for (int s = 0; s < LT_NS; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 8); }
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // the zero fill before the async-proxy writes
	__syncthreads();

	if (warp == 8) {
		// ------------------------------------------------------------------ producer warp
		int slot = 0; unsigned phase = 0;
		const int cbytes = nt * 8;                     // nt is even: a multiple of 16 bytes
		for (int kt = 0; kt < ktiles; ++kt) {
			const int k0 = kt * LC_BK;
			const int krows = min(LC_BK, p - k0);
			if (lane == 0) {
				mbar_spin(empty + slot, phase ^ 1u);
				mbar_expect_tx(full + slot, (unsigned)(LT_X_BYTES + krows * cbytes));
				tma_load_2d(xs_base + (size_t)slot * LT_X_BYTES, tmx, k0, (int)r0, full + slot);
			}
			__syncwarp();
			if (lane < krows)
				bulk_load_1d(cs_base + (size_t)slot * LT_C_BYTES + (size_t)lane * LC_SC * 8,
				             c + (size_t)(k0 + lane) * c_rs + n0, (unsigned)cbytes, full + slot);
			if (++slot == LT_NS) { slot = 0; phase ^= 1u; }
		}
		return;
	}
	// ---------------------------------------------------------------------- consumer warps
	const int g = lane >> 2, t = lane & 3;
	double acc[2][NQ8][2];
#pragma unroll
	for (int i = 0; i < 2; ++i)
#pragma unroll
		for (int j = 0; j < NQ8; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
	// A fragments: element (row, k) of the swizzled X tile sits at row*16 + (((k >> 1) ^ (row & 7)) << 1) + (k & 1)
	// doubles; rows warp*16 + g and + 8 (both = g mod 8), k = ks + t
	int aoff[LC_BK / 4];
#pragma unroll
	for (int s4 = 0; s4 < LC_BK / 4; ++s4) aoff[s4] = (warp * 16 + g) * 16 + ((((4 * s4 + t) >> 1) ^ g) << 1) + (t & 1);
	int slot = 0; unsigned phase = 0;
	for (int kt = 0; kt < ktiles; ++kt) {
		mbar_spin(full + slot, phase);
		const double *Xs = reinterpret_cast<const double *>(xs_base + (size_t)slot * LT_X_BYTES);
		const double *Cs = reinterpret_cast<const double *>(cs_base + (size_t)slot * LT_C_BYTES);
#pragma unroll
		for (int s4 = 0; s4 < LC_BK / 4; ++s4) {
			const double a0 = Xs[aoff[s4]];
			const double a1 = Xs[aoff[s4] + 8 * 16];
#pragma unroll
			for (int j = 0; j < NQ8; ++j) {
				const double b = Cs[(4 * s4 + t) * LC_SC + j * 8 + g];
				dmma_8x8x4(acc[0][j][0], acc[0][j][1], a0, b);
				dmma_8x8x4(acc[1][j][0], acc[1][j][1], a1, b);
			}
		}
		// Every fragment load of this stage must have been PERFORMED before the slot is handed back.  The
		// mbarrier arrive alone does not wait for shared-memory loads still in flight, and ptxas schedules
		// it above the last DMMAs (the only instructions that wait for those loads): without this fence
		// the refill of the slot overtook the last A-fragment loads of a stage about once per 10^9
		// loads -- whole output rows wrong, only when the consumers were starved (narrow last column
		// tile, misaligned x) -- found with scripts/lincomb_race.py.
		asm volatile("fence.acq_rel.cta;" ::: "memory");
		__syncwarp();
		if (lane == 0) mbar_arrive(empty + slot);
		if (++slot == LT_NS) { slot = 0; phase ^= 1u; }
	}
#pragma unroll
	for (int i = 0; i < 2; ++i) {
		const long long r = r0 + warp * 16 + i * 8 + g;
		if (r >= n) continue;
#pragma unroll
		for (int j = 0; j < NQ8; ++j)
#pragma unroll
			for (int h = 0; h < 2; ++h) {
				const int cc = j * 8 + 2 * t + h;
				if (cc < nt) {
					double v = acc[i][j][h];
					double *yp = y + (size_t)r * ldy + n0 + cc;
					if (HAS_BETA) {
						const double b = beta[(size_t)incb * (n0 + cc)];
						if (b != 0.0) v += b * (*yp);      // beta == 0 overwrites (no NaN carry-over)
					}
					*yp = v;
				}
			}
	}
}

template <bool HAS_BETA>
__global__ void __launch_bounds__(288, 2)
lincomb_tma_kernel(const __grid_constant__ CUtensorMap tmx, long long n, int p, int q, const double *__restrict__ c, int c_rs,
                   const double *__restrict__ beta, int incb, double *y, int ldy)
{
	const int nt = min(LC_BN, q - (int)blockIdx.x * LC_BN);
	switch ((nt + 7) >> 3) {                             // uniform over the CTA
	case 1: lincomb_tma_body<HAS_BETA, 1>(&tmx, n, p, q, c, c_rs, beta, incb, y, ldy); break;
	case 2: lincomb_tma_body<HAS_BETA, 2>(&tmx, n, p, q, c, c_rs, beta, incb, y, ldy); break;
	case 3: lincomb_tma_body<HAS_BETA, 3>(&tmx, n, p, q, c, c_rs, beta, incb, y, ldy); break;
	case 4: lincomb_tma_body<HAS_BETA, 4>(&tmx, n, p, q, c, c_rs, beta, incb, y, ldy); break;
	case 5: lincomb_tma_body<HAS_BETA, 5>(&tmx, n, p, q, c, c_rs, beta, incb, y, ldy); break;
	case 6: lincomb_tma_body<HAS_BETA, 6>(&tmx, n, p, q, c, c_rs, beta, incb, y, ldy); break;
	case 7: lincomb_tma_body<HAS_BETA, 7>(&tmx, n, p, q, c, c_rs, beta, incb, y, ldy); break;
	default: lincomb_tma_body<HAS_BETA, 8>(&tmx, n, p, q, c, c_rs, beta, incb, y, ldy); break;
	}
}

// 0 launched, 1 error, 2 not applicable
static int lincomb_tma_launch(long long n, int p, int q, const double *x, int ldx, const double *c_dev, int c_rs, int c_cs,
                              const double *beta_dev, int incb, double *y, int ldy)
{
	if (n < LC_BM || c_cs != 1 || (c_rs & 1) || (q & 1) || ((uintptr_t)c_dev % 16) || ((uintptr_t)x % 16) || (ldx & 1) ||
	    n > 0x7fffffffLL)
		return 2;
	tmap_encode_fn enc = tmap_encoder();
	if (!enc) return 2;
	CUtensorMap tm;
	const cuuint64_t gdim[2] = {(cuuint64_t)p, (cuuint64_t)n};
	const cuuint64_t gstr[1] = {(cuuint64_t)ldx * 8};
	const cuuint32_t box[2] = {(cuuint32_t)LC_BK, (cuuint32_t)LC_BM};
	const cuuint32_t estr[2] = {1, 1};
	if (enc(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(x), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
	        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
		return 2;
	const size_t smem = (size_t)LT_NS * LT_STAGE_BYTES;
	static bool attr_set = false;
	if (!attr_set) {
		B200_CUDA(cudaFuncSetAttribute(lincomb_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		B200_CUDA(cudaFuncSetAttribute(lincomb_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		attr_set = true;
	}
	dim3 grid(b200_ceil_div(q, LC_BN), (unsigned)((n + LC_BM - 1) / LC_BM));
	if (beta_dev) lincomb_tma_kernel<true><<<grid, 288, smem, g_b200.stream>>>(tm, n, p, q, c_dev, c_rs, beta_dev, incb, y, ldy);
	else          lincomb_tma_kernel<false><<<grid, 288, smem, g_b200.stream>>>(tm, n, p, q, c_dev, c_rs, nullptr, 0, y, ldy);
	B200_KERNEL_CHECK();
	return 0;
}

// scaling only: y[:,c] *= beta[incb*c]  (beta == nullptr => y = 0)
__global__ void colscale_kernel(long long n, int q, int rows_per_cta, const double *__restrict__ beta, int incb,
                                double *y, int ldy)
{
	const long long r0 = (long long)blockIdx.x * rows_per_cta;
	long long nr = n - r0; if (nr > rows_per_cta) nr = rows_per_cta;
	const int total = (int)nr * q;
	for (int i = threadIdx.x; i < total; i += blockDim.x) {
		const int r = i / q, cidx = i - r * q;
		double *yp = y + (size_t)(r0 + r) * ldy + cidx;
		const double b = beta ? beta[(size_t)incb * cidx] : 0.0;
		*yp = (b == 0.0) ? 0.0 : b * (*yp);
	}
}

static int lincomb_rows(long long n, int p, int q, const double *x, int ldx, const double *c_dev, int c_rs, int c_cs,
                        const double *beta_dev, int incb, double *y, int ldy);

// Row tiles are gridDim.y of the kernels (at most 65535): blocks with more rows go in several launches.
int b200k_lincomb(long long n, int p, int q, const double *x, int ldx, const double *c_dev, int c_rs, int c_cs,
                  const double *beta_dev, int incb, double *y, int ldy)
{
	const long long max_rows = 65535LL * LC_BM;
	if (n <= max_rows) return lincomb_rows(n, p, q, x, ldx, c_dev, c_rs, c_cs, beta_dev, incb, y, ldy);
	for (long long r0 = 0; r0 < n; r0 += max_rows) {
		const long long nr = (n - r0 < max_rows) ? n - r0 : max_rows;
		if (lincomb_rows(nr, p, q, x ? x + (size_t)r0 * ldx : nullptr, ldx, c_dev, c_rs, c_cs, beta_dev, incb,
		                 y + (size_t)r0 * ldy, ldy))
			return 1;
	}
	return 0;
}

static int lincomb_rows(long long n, int p, int q, const double *x, int ldx, const double *c_dev, int c_rs, int c_cs,
                        const double *beta_dev, int incb, double *y, int ldy)
{
	if (n <= 0 || q <= 0) return 0;
	cudaStream_t st = g_b200.stream;
	const bool scale_only = (x == nullptr || c_dev == nullptr || p <= 0);
	B200Prof prof(scale_only ? B200_PROF_AXPBY : (n <= 1024 ? B200_PROF_SMALL : B200_PROF_LINCOMB),
	              scale_only ? 16.0 * n * q : 8.0 * n * ((double)p + q + (beta_dev ? q : 0)) + 8.0 * p * q,
	              scale_only ? 1.0 * n * q : 2.0 * n * p * q);
	if (scale_only) {
		// reference app/app_lapack.c:476-505: without x/coef only the dscal part runs, and
		// with beta == NULL nothing runs at all
		if (beta_dev == nullptr) return 0;
		int rows = 4096 / q; if (rows < 1) rows = 1;
		colscale_kernel<<<(unsigned)((n + rows - 1) / rows), 256, 0, st>>>(n, q, rows, beta_dev, incb, y, ldy);
		B200_KERNEL_CHECK();
		return 0;
	}
	{
		const int rc = lincomb_tma_launch(n, p, q, x, ldx, c_dev, c_rs, c_cs, beta_dev, incb, y, ldy);
		if (rc != 2) return rc;
	}
	dim3 grid(b200_ceil_div(q, LC_BN), (unsigned)((n + LC_BM - 1) / LC_BM));
	const size_t smem = sizeof(double) * (size_t)LC_STAGES * LC_STAGE_DBL;
	static bool attr_set = false;
	if (!attr_set) {
		B200_CUDA(cudaFuncSetAttribute(lincomb_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		B200_CUDA(cudaFuncSetAttribute(lincomb_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		B200_CUDA(cudaFuncSetAttribute(lincomb_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		B200_CUDA(cudaFuncSetAttribute(lincomb_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		attr_set = true;
	}
	const bool al16 = ((uintptr_t)x % 16 == 0) && (ldx % 2 == 0) && (p % 2 == 0);
	if (beta_dev) {
		if (al16) lincomb_kernel<true, true><<<grid, 256, smem, st>>>(n, p, q, x, ldx, c_dev, c_rs, c_cs, beta_dev, incb, y, ldy);
		else      lincomb_kernel<true, false><<<grid, 256, smem, st>>>(n, p, q, x, ldx, c_dev, c_rs, c_cs, beta_dev, incb, y, ldy);
	} else {
		if (al16) lincomb_kernel<false, true><<<grid, 256, smem, st>>>(n, p, q, x, ldx, c_dev, c_rs, c_cs, nullptr, 0, y, ldy);
		else      lincomb_kernel<false, false><<<grid, 256, smem, st>>>(n, p, q, x, ldx, c_dev, c_rs, c_cs, nullptr, 0, y, ldy);
	}
	B200_KERNEL_CHECK();
	return 0;
}

// y[:,j] *= s[j]  (or /= s[j])
__global__ void colscale_vec_kernel(long long n, int q, int rows_per_cta, const double *__restrict__ sv, int invert,
                                    double *y, int ldy)
{
	const long long r0 = (long long)blockIdx.x * rows_per_cta;
	long long nr = n - r0; if (nr > rows_per_cta) nr = rows_per_cta;
	const int total = (int)nr * q;
	for (int i = threadIdx.x; i < total; i += blockDim.x) {
		const int r = i / q, cidx = i - r * q;
		double *yp = y + (size_t)(r0 + r) * ldy + cidx;
		const double f = invert ? 1.0 / sv[cidx] : sv[cidx];
		*yp = f * (*yp);
	}
}

int b200k_colscale(long long n, int q, const double *s_dev, int invert, double *y, int ldy)
{
	if (n <= 0 || q <= 0) return 0;
	B200Prof prof(B200_PROF_AXPBY, 16.0 * n * q, 1.0 * n * q);
	int rows = 4096 / q; if (rows < 1) rows = 1;
	colscale_vec_kernel<<<(unsigned)((n + rows - 1) / rows), 256, 0, g_b200.stream>>>(n, q, rows, s_dev, invert, y, ldy);
	B200_KERNEL_CHECK();
	return 0;
}
