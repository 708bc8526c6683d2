// K1: CSR SpMM  y[:, 0:k] = A x[:, 0:k]  on row-major multi-vector blocks.
//
// Replaces the reference's column-parallel CCS scatter loop (app/app_ccs.c:116-131), which
// streams the whole matrix once PER COLUMN.  Here the matrix is read once for all k columns:
// a group of G lanes owns one row, lane l accumulates columns l, l+G, ... so every gathered
// x row is one contiguous k*8-byte segment (row-major store) and the matrix entry is a
// broadcast load inside the group.  HBM-bound: algorithmic bytes per launch are
//   nnz*(8+4) + (n+1)*4 + 8*n*k (x, read once) + 8*n*k (y, written once)       (SURVEY §8d)
//
// Arithmetic: separate multiply and add (no FMA contraction), entries of a row visited in
// ascending column order -- the same operation sequence as the reference's serial scatter,
// so the result is bit-identical to the reference on every input.
#include "b200_internal.h"
#include "b200_tma.cuh"
#include "b200_dia.cuh"

// Matrix entries are fetched cooperatively: the G lanes of a row group load G consecutive
// (value, column) pairs with one coalesced request each and hand them round with shuffles,
// instead of every lane issuing the same broadcast load per entry -- the L1 wavefront count
// per entry drops from 2 + ceil(8k/128) to ceil(8k/128) (+2/G), and L1TEX issue, not HBM, is
// what bounds this kernel (profiles/).  Control flow is kept warp-uniform (loop bounds are
// warp maxima) so the shuffles are always fully converged.
template <int G, int CPL>
__global__ void __launch_bounds__(256)
spmm_csr_kernel(int nrows, const int *__restrict__ rp, const int *__restrict__ ci,
                const double *__restrict__ va, const double *x, int ldx, double *y, int ldy, int k,
                const int *__restrict__ gate)
{
	if (gate != nullptr && *gate == 0) return;
	const int gl = threadIdx.x % G;                          // lane inside the row group
	const int groups_per_cta = 256 / G;
	const long long row = (long long)blockIdx.x * groups_per_cta + threadIdx.x / G;
	const bool live = row < nrows;
	const int e0 = live ? __ldg(rp + row) : 0, e1 = live ? __ldg(rp + row + 1) : 0;
	for (int cbase = 0; cbase < k; cbase += G * CPL) {
		double acc[CPL];
		bool on[CPL];
#pragma unroll
		for (int i = 0; i < CPL; ++i) { acc[i] = 0.0; on[i] = live && (cbase + gl + i * G) < k; }
		if (G >= 8) {
			const int nchunk = (e1 - e0 + G - 1) / G;
			const int nchunk_max = __reduce_max_sync(0xffffffffu, nchunk);
			for (int ch = 0; ch < nchunk_max; ++ch) {
				const int eb = e0 + ch * G;
				int cnt = e1 - eb; cnt = cnt < 0 ? 0 : (cnt > G ? G : cnt);
				const int cnt_max = __reduce_max_sync(0xffffffffu, cnt);
				double a_l = 0.0; int c_l = 0;
				if (gl < cnt) { a_l = __ldg(va + eb + gl); c_l = __ldg(ci + eb + gl); }
#pragma unroll 4
				for (int j = 0; j < cnt_max; ++j) {
					const double a = __shfl_sync(0xffffffffu, a_l, j, G);
					const int col = __shfl_sync(0xffffffffu, c_l, j, G);
					if (j < cnt) {
						const double *xr = x + (size_t)col * ldx + cbase + gl;
#pragma unroll
						for (int i = 0; i < CPL; ++i)
							if (on[i]) acc[i] = __dadd_rn(acc[i], __dmul_rn(a, xr[i * G]));
					}
				}
			}
		} else {
			for (int e = e0; e < e1; ++e) {
				const double a = __ldg(va + e);
				const double *xr = x + (size_t)__ldg(ci + e) * ldx + cbase + gl;
#pragma unroll
				for (int i = 0; i < CPL; ++i)
					if (on[i]) acc[i] = __dadd_rn(acc[i], __dmul_rn(a, xr[i * G]));
			}
		}
		if (live) {
			double *yr = y + (size_t)row * ldy + cbase + gl;
#pragma unroll
			for (int i = 0; i < CPL; ++i)
				if (on[i]) yr[i * G] = acc[i];
		}
	}
}

// Wide variant (k > 4).  G lanes (8, 16 or 32) own one row; lane l accumulates the column
// pairs (2l, 2l+1) + 2G*pass, so every matrix entry costs one 128-bit gather per pass and the
// gathered x row is one contiguous segment.  The scalar kernel above spends ~27 warp
// instructions per matrix entry (64-bit shuffles, selects) and is issue-bound (profiles/);
// here the row group stages its entries -- one coalesced load of G (value, column) pairs --
// into shared memory as 16-byte records and the inner loop per entry is
//     LDS.128 (broadcast)  IMAD.WIDE  LDG.128  2 x DMUL  2 x DADD        (per pass)
// with U independent gathers in flight.  With G = 32 the loop bounds are warp-uniform and
// nothing is predicated; narrower groups run to the warp's longest row with the accumulation
// predicated off past a row's end (padding records point at row 0 and are never added).
// VEC = false (odd offsets / leading dimensions, odd k) splits the gather into two 64-bit loads.
template <int G, int NPASS, bool VEC, int U>
__global__ void __launch_bounds__(256)
spmm_csr_wide_kernel(int nrows, const int *__restrict__ rp, const int *__restrict__ ci,
                     const double *__restrict__ va, const double *x, int ldx, double *y, int ldy, int k,
                     const int *__restrict__ gate)
{
	if (gate != nullptr && *gate == 0) return;
	constexpr int RPW = 32 / G;                       // rows per warp
	__shared__ double2 ent_s[8][RPW][G];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int gl = lane % G, rg = lane / G;
	const long long row = ((long long)blockIdx.x * 8 + warp) * RPW + rg;
	const bool live = row < nrows;
	const int e0 = live ? __ldg(rp + row) : 0, e1 = live ? __ldg(rp + row + 1) : 0;
	double2 *ent = ent_s[warp][rg];
	// column pair of this lane in each pass; lanes past the end redo the last pair (no store)
	int c[NPASS]; bool st[NPASS];
	double acc[NPASS][2];
#pragma unroll
	for (int p = 0; p < NPASS; ++p) {
		c[p] = 2 * gl + 2 * G * p;
		st[p] = live && (c[p] < k);
		if (c[p] > k - 2) c[p] = k - 2 < 0 ? 0 : k - 2;
		acc[p][0] = 0.0; acc[p][1] = 0.0;
	}
	const bool odd_tail = (k & 1);                    // VEC == false only: last pair has one column
	// gather address = x + column*ldx*8 bytes: one IMAD.WIDE per entry (32-bit column, 32-bit
	// byte stride, 64-bit base) -- ldx*8 fits an int for any leading dimension below 2^28
	const int ldx8 = ldx * 8;
	const char *xbase = reinterpret_cast<const char *>(x);
	const int nchunk = (e1 - e0 + G - 1) / G;
	const int nchunk_max = (G == 32) ? nchunk : __reduce_max_sync(0xffffffffu, nchunk);
	for (int ch = 0; ch < nchunk_max; ++ch) {
		const int eb = e0 + ch * G;
		int cnt = e1 - eb; cnt = cnt < 0 ? 0 : (cnt > G ? G : cnt);
		const int cnt_max = (G == 32) ? cnt : __reduce_max_sync(0xffffffffu, cnt);
		{
			double a_l = 0.0; int c_l = 0;
			if (gl < cnt) { a_l = __ldg(va + eb + gl); c_l = __ldg(ci + eb + gl); }
			if (gl < cnt_max) ent[gl] = make_double2(a_l, __longlong_as_double((long long)c_l));
		}
		__syncwarp();
		if (cnt_max > 0) {
			// Software pipeline over batches of U entries: the gathers of batch b+1 are issued
			// before the arithmetic of batch b, across the loop back-edge, so ptxas cannot sink
			// them next to their uses (it does inside one basic block, leaving one gather in
			// flight per warp).  Slots past the end re-read the last entry and are not added.
			double a[U]; double2 v[NPASS][U];
			auto fetch = [&](int jb, double (&aa)[U], double2 (&vv)[NPASS][U]) {
#pragma unroll
				for (int u = 0; u < U; ++u) {
					int j = jb + u; j = j < cnt_max ? j : cnt_max - 1;
					const double2 e = ent[j];
					aa[u] = e.x;
					const double *xr = reinterpret_cast<const double *>(xbase + (long long)__double2loint(e.y) * (long long)ldx8);
#pragma unroll
					for (int p = 0; p < NPASS; ++p) {
						// x columns are never written by this launch (ranges are disjoint): non-coherent loads
						if (VEC) vv[p][u] = __ldg(reinterpret_cast<const double2 *>(xr + c[p]));
						else {
							vv[p][u].x = __ldg(xr + c[p]);
							vv[p][u].y = __ldg(xr + c[p] + ((odd_tail && c[p] == k - 1) ? 0 : 1));
						}
					}
				}
			};
			fetch(0, a, v);
			for (int j0 = 0; j0 < cnt_max; j0 += U) {
				double a2[U]; double2 v2[NPASS][U];
				if (j0 + U < cnt_max) fetch(j0 + U, a2, v2);
#pragma unroll
				for (int u = 0; u < U; ++u) {
					if (j0 + u < cnt) {
#pragma unroll
						for (int p = 0; p < NPASS; ++p) {
							acc[p][0] = __dadd_rn(acc[p][0], __dmul_rn(a[u], v[p][u].x));
							acc[p][1] = __dadd_rn(acc[p][1], __dmul_rn(a[u], v[p][u].y));
						}
					}
				}
#pragma unroll
				for (int u = 0; u < U; ++u) {
					a[u] = a2[u];
#pragma unroll
					for (int p = 0; p < NPASS; ++p) v[p][u] = v2[p][u];
				}
			}
		}
		__syncwarp();
	}
#pragma unroll
	for (int p = 0; p < NPASS; ++p) {
		if (!st[p]) continue;
		double *yr = y + (size_t)row * ldy + c[p];
		if (VEC) *reinterpret_cast<double2 *>(yr) = make_double2(acc[p][0], acc[p][1]);
		else { yr[0] = acc[p][0]; if (c[p] + 1 < k) yr[1] = acc[p][1]; }
	}
}

// Block variant: the main kernel for k <= 64 on matrices with short rows (FEM / stencil).
// The wide kernel above makes every warp walk a chain of dependent global loads -- row
// pointer -> entries -> gathers -- and at ~1 us per hop the SM spends most of a row's life
// waiting (measured: time proportional to the number of warps, not to bytes; profiles/).
// Here a CTA owns a contiguous block of R = 8*RPW*rw rows: all 256 threads first pull the
// block's row pointers and then its (value, column) entries -- two fully coalesced sweeps,
// paid once per block instead of once per row -- into shared memory as 16-byte records; then
// each row group walks its rw rows entirely out of shared memory, with the whole row's gathers
// (up to U) in flight at once.  Rows handled at the same time by the 8 warps are adjacent, so
// gathered x rows shared between neighbouring matrix rows meet in L1.
constexpr int SPMM_CAP = 2048;          // entries staged per CTA (32 KB of records)

template <int G, bool VEC, int U>
__global__ void __launch_bounds__(256)
spmm_csr_block_kernel(int nrows, const int *__restrict__ rp, const int *__restrict__ ci,
                      const double *__restrict__ va, const double *x, int ldx, double *y, int ldy, int k,
                      const int *__restrict__ gate, int rw)
{
	if (gate != nullptr && *gate == 0) return;
	constexpr int RPW = 32 / G;
	extern __shared__ __align__(16) unsigned char smem_raw[];
	double2 *ent = reinterpret_cast<double2 *>(smem_raw);            // [SPMM_CAP]
	int *rp_s = reinterpret_cast<int *>(ent + SPMM_CAP);              // [R + 1]
	const int R = 8 * RPW * rw;
	const long long r0 = (long long)blockIdx.x * R;
	for (int i = threadIdx.x; i <= R; i += 256) {
		const long long r = r0 + i;
		rp_s[i] = __ldg(rp + (r < nrows ? r : nrows));
	}
	__syncthreads();
	const int eb = rp_s[0], ne = rp_s[R] - eb;
	for (int i = threadIdx.x; i < ne; i += 256)
		ent[i] = make_double2(__ldg(va + eb + i), __longlong_as_double((long long)__ldg(ci + eb + i)));
	__syncthreads();

	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int gl = lane % G, rg = lane / G;
	int c = 2 * gl;
	const bool in_cols = c < k;
	if (c > k - 2) c = k - 2 < 0 ? 0 : k - 2;
	const bool odd_tail = (k & 1);
	const int ldx8 = ldx * 8;
	const char *xbase = reinterpret_cast<const char *>(x + c);
	const int second = (!VEC && odd_tail && c == k - 1) ? 0 : 1;
	for (int j = 0; j < rw; ++j) {
		const int lr = j * (8 * RPW) + warp * RPW + rg;
		const long long row = r0 + lr;
		const int e0 = rp_s[lr] - eb, e1 = rp_s[lr + 1] - eb;
		const int cnt = e1 - e0;
		const int cnt_max = (G == 32) ? cnt : __reduce_max_sync(0xffffffffu, cnt);
		double acc0 = 0.0, acc1 = 0.0;
		for (int j0 = 0; j0 < cnt_max; j0 += U) {
			double2 v[U];
#pragma unroll
			for (int u = 0; u < U; ++u) {
				int e = j0 + u; e = e < cnt ? e : (cnt > 0 ? cnt - 1 : 0);
				const int col = (cnt > 0) ? __double2loint(ent[e0 + e].y) : 0;
				const double *xr = reinterpret_cast<const double *>(xbase + (long long)col * (long long)ldx8);
				if (VEC) v[u] = __ldg(reinterpret_cast<const double2 *>(xr));
				else { v[u].x = __ldg(xr); v[u].y = __ldg(xr + second); }
			}
#pragma unroll
			for (int u = 0; u < U; ++u) {
				if (j0 + u < cnt) {
					const double a = ent[e0 + j0 + u].x;
					acc0 = __dadd_rn(acc0, __dmul_rn(a, v[u].x));
					acc1 = __dadd_rn(acc1, __dmul_rn(a, v[u].y));
				}
			}
		}
		if (in_cols && row < nrows) {
			double *yr = y + (size_t)row * ldy + c;
			if (VEC) *reinterpret_cast<double2 *>(yr) = make_double2(acc0, acc1);
			else { yr[0] = acc0; if (c + 1 < k) yr[1] = acc1; }
		}
	}
}

// 16-byte accesses to x and y: both 16-byte aligned, even leading dimensions, an even number of columns
static inline bool spmm_aligned16(const double *x, int ldx, const double *y, int ldy, int k)
{
	return (((uintptr_t)x | (uintptr_t)y) % 16 == 0) && (ldx % 2 == 0) && (ldy % 2 == 0) && (k % 2 == 0);
}

template <int G, int U>
static int launch_spmm_block(int nrows, const int *rp, const int *ci, const double *va,
                             const double *x, int ldx, double *y, int ldy, int k, const int *gate, int rw)
{
	const int R = 8 * (32 / G) * rw;
	const unsigned grid = (unsigned)(((long long)nrows + R - 1) / R);
	const size_t smem = sizeof(double2) * SPMM_CAP + sizeof(int) * ((size_t)R + 1);
	if (spmm_aligned16(x, ldx, y, ldy, k)) spmm_csr_block_kernel<G, true, U><<<grid, 256, smem, g_b200.stream>>>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate, rw);
	else     spmm_csr_block_kernel<G, false, U><<<grid, 256, smem, g_b200.stream>>>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate, rw);
	B200_KERNEL_CHECK();
	return 0;
}

// Gathers in flight per row group: measured on B200 (P1-FEM n = 1 M, profiles/): a one-row warp
// (G = 32) is fastest with U = 4 (0.475 ms at k = 40 vs 0.557 / 0.576 ms with 8 / 16), the
// narrower groups with U = 8 (0.168 ms at k = 16 vs 0.186 / 0.227 ms with 4 / 16).
template <int G>
static int launch_spmm_block_u(int nrows, const int *rp, const int *ci, const double *va,
                               const double *x, int ldx, double *y, int ldy, int k, const int *gate, int rw)
{
	if (G == 32) return launch_spmm_block<G, 4>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate, rw);
	return launch_spmm_block<G, 8>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate, rw);
}

template <int G, int NPASS>
static int launch_spmm_wide(int nrows, const int *rp, const int *ci, const double *va,
                            const double *x, int ldx, double *y, int ldy, int k, const int *gate)
{
	const int rows_per_cta = 8 * (32 / G);
	const unsigned grid = (unsigned)(((long long)nrows + rows_per_cta - 1) / rows_per_cta);
	if (spmm_aligned16(x, ldx, y, ldy, k)) spmm_csr_wide_kernel<G, NPASS, true, 4><<<grid, 256, 0, g_b200.stream>>>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate);
	else     spmm_csr_wide_kernel<G, NPASS, false, 4><<<grid, 256, 0, g_b200.stream>>>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate);
	B200_KERNEL_CHECK();
	return 0;
}

template <int G, int CPL>
static int launch_spmm(int nrows, const int *rp, const int *ci, const double *va,
                       const double *x, int ldx, double *y, int ldy, int k, const int *gate)
{
	const int groups_per_cta = 256 / G;
	const unsigned grid = (unsigned)(((long long)nrows + groups_per_cta - 1) / groups_per_cta);
	spmm_csr_kernel<G, CPL><<<grid, 256, 0, g_b200.stream>>>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate);
	B200_KERNEL_CHECK();
	return 0;
}

// ============================================================================= diagonal SpMM
// For matrices with a diagonal image (b200_mat.cu: dia_build) -- stencils and FEM operators on
// lattices.  The CSR kernels above are bound by the L1 path: every (row, entry) pair is a
// 3-line gather and L1 retires about one line per two cycles (profiles/ncu_r1c_spmm: l1tex 85 %,
// DRAM 22 %).  Here the x rows a block of matrix rows needs never go through L1 at all:
//
//   * Offsets come in runs of consecutive values ({-1,0,1}, {m, m+1}, ...).  For a CTA that owns
//     the rows [R, R + ROWS) and a run starting at offset d, the x rows needed are the CONTIGUOUS
//     range [R + d, R + d + ROWS + 2): one 2-D box of the row-major multi-vector.  One elected
//     thread issues one TMA tile copy (cp.async.bulk.tensor.2d) per run -- all runs up front,
//     ~75 KB in flight per CTA, no registers, no LSU wavefronts -- each signalling its own
//     mbarrier.  Rows outside the matrix (Dirichlet rows at the ends; halo limits) are
//     zero-filled by the TMA unit and never used (presence mask).
//   * A row group of G lanes (lane = one column pair) owns RB consecutive matrix rows with their
//     2 RB accumulators in registers, and slides along the box: x row t of a run feeds matrix
//     rows t - j, j < run width, so each x row is read from shared memory once per run instead
//     of once per matrix row that touches it.
//   * The diagonal values of the CTA's rows are one contiguous range of the image: a coalesced
//     sweep into shared memory, then broadcast reads.
//
// Arithmetic is unchanged: per matrix row the runs, and the offsets inside a run, are visited in
// ascending order = ascending column order, separate multiply and add, entries absent from the
// CCS input are skipped by the presence mask (not multiplied by a stored zero) -- bit-identical
// to the reference's scatter loop (app/app_ccs.c:116-131).

// One run of width W on the RB rows of a row group: x rows t = 0 .. RB + W - 2 of the run's box are
// read once (128-bit) and x row t feeds matrix rows t - j, j < W.  The run's values of a matrix
// row sit 16-byte aligned in the image (runs are padded to an even number of slots), so they
// come as one 128-bit broadcast load (+ one 64-bit load for W == 3).
template <int RB, int W>
__device__ __forceinline__ void dia_run(double (&acc)[RB][2], const double *tile, int k, const double *vrow, int ndp)
{
	double2 xv[RB + W - 1];
#pragma unroll
	for (int t = 0; t < RB + W - 1; ++t) xv[t] = *reinterpret_cast<const double2 *>(tile + (size_t)t * k);
#pragma unroll
	for (int i = 0; i < RB; ++i) {
		const double2 a01 = *reinterpret_cast<const double2 *>(vrow + i * ndp);
		acc[i][0] = __dadd_rn(acc[i][0], __dmul_rn(a01.x, xv[i].x));
		acc[i][1] = __dadd_rn(acc[i][1], __dmul_rn(a01.x, xv[i].y));
		if (W >= 2) {
			acc[i][0] = __dadd_rn(acc[i][0], __dmul_rn(a01.y, xv[i + (W >= 2 ? 1 : 0)].x));
			acc[i][1] = __dadd_rn(acc[i][1], __dmul_rn(a01.y, xv[i + (W >= 2 ? 1 : 0)].y));
		}
		if (W >= 3) {
			const double a2 = vrow[i * ndp + 2];
			acc[i][0] = __dadd_rn(acc[i][0], __dmul_rn(a2, xv[i + (W >= 3 ? 2 : 0)].x));
			acc[i][1] = __dadd_rn(acc[i][1], __dmul_rn(a2, xv[i + (W >= 3 ? 2 : 0)].y));
		}
	}
}

// tmx: 2-D tensor map of the x block: dim0 = the k columns, dim1 = the hb + nloc + ha rows of the
// window (halo rows in front of and behind the local rows), box = (k, ROWS + 2).
// Persistent CTAs walk the flattened sequence of (row block, run) items through a ring of NS
// shared-memory tiles: while the warps consume the x box of one run, the TMA unit fills the
// tiles of the next NS-1 items (one mbarrier per tile).  The diagonal values of a row block come
// by one 1-D bulk copy into a double buffer.  Accumulators stay in registers across the runs of
// a block.  Entries absent from the CCS input are stored as +0.0 in the image: 0.0 * x adds a
// signed zero, which never changes an accumulator (it starts at +0.0 and can never become
// -0.0), so the result is bit-identical to the reference for every finite x.
template <int G, int RB, int NS>
__global__ void __launch_bounds__(256)
spmm_dia_tma_kernel(const __grid_constant__ CUtensorMap tmx, int nrows, int nblocks, int nd, const int *__restrict__ off,
                    const double *__restrict__ val, int ng, const int *__restrict__ grp, int hb, int tile_bytes,
                    double *y, int ldy, int k, const int *__restrict__ gate)
{
	if (gate != nullptr && *gate == 0) return;
	constexpr int CPW = 32 / G;                      // row chunks per warp
	constexpr int ROWS = 8 * CPW * RB;               // rows per block
	extern __shared__ __align__(128) unsigned char smem_raw[];
	// [NS x-tiles of tile_bytes][2 value buffers of ROWS x nd doubles]
	__shared__ unsigned long long bars[NS], vbars[2];
	__shared__ int grp_s[64];
	__shared__ int d0_s[32];
	if (threadIdx.x < 2 * ng) grp_s[threadIdx.x] = __ldg(grp + threadIdx.x);
	if (threadIdx.x < ng) d0_s[threadIdx.x] = __ldg(off + threadIdx.x);      // first offset of each run
	if (threadIdx.x == 0) {
		for (int s = 0; s < NS; ++s) mbar_init(bars + s, 1);
		mbar_init(vbars, 1); mbar_init(vbars + 1, 1);
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
	}
	__syncthreads();
	const unsigned x_bytes = (unsigned)((ROWS + DIA_WMAX - 1) * k * 8);
	const unsigned val_bytes = (unsigned)(ROWS * nd * 8);
	unsigned char *vbuf = smem_raw + (size_t)NS * tile_bytes;
	const int my_blocks = (nblocks - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
	const int items = my_blocks * ng;
	auto issue_x = [&](int item) {                   // one thread
		const int blk = blockIdx.x + (item / ng) * gridDim.x, g = item % ng, slot = item % NS;
		mbar_expect_tx(bars + slot, x_bytes);
		tma_load_2d(smem_raw + (size_t)slot * tile_bytes, &tmx, 0, blk * ROWS + d0_s[g] + hb, bars + slot);
	};
	auto issue_val = [&](int lb) {                    // one thread; lb = local block counter
		const int blk = blockIdx.x + lb * gridDim.x;
		mbar_expect_tx(vbars + (lb & 1), val_bytes);
		// the image is padded to whole blocks (b200_mat.cu): full-size copies are always in bounds
		bulk_load_1d(vbuf + (size_t)(lb & 1) * val_bytes, val + (size_t)blk * ROWS * nd, val_bytes, vbars + (lb & 1));
	};
	if (threadIdx.x == 0) {
		if (my_blocks > 0) issue_val(0);
		for (int i = 0; i < NS - 1 && i < items; ++i) issue_x(i);
	}
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int gl = lane % G, chunk = warp * CPW + lane / G;
	int c = 2 * gl;
	const bool in_cols = c < k;
	if (c > k - 2) c = k - 2;
	const int lr0 = chunk * RB;                      // first row of this group inside the block
	double acc[RB][2];
	int item = 0;
	for (int lb = 0; lb < my_blocks; ++lb) {
		if (threadIdx.x == 0 && lb + 1 < my_blocks) issue_val(lb + 1);   // its buffer was released with block lb-1
		mbar_wait(vbars + (lb & 1), (unsigned)((lb >> 1) & 1));
		const double *vrow = reinterpret_cast<const double *>(vbuf + (size_t)(lb & 1) * val_bytes) + (size_t)lr0 * nd;
#pragma unroll
		for (int i = 0; i < RB; ++i) { acc[i][0] = 0.0; acc[i][1] = 0.0; }
		for (int g = 0; g < ng; ++g, ++item) {
			// refill the tile released by the barrier at the end of the previous item
			if (threadIdx.x == 0 && item + NS - 1 < items) issue_x(item + NS - 1);
			const int slot = item % NS;
			mbar_wait(bars + slot, (unsigned)((item / NS) & 1));
			const int sp = grp_s[2 * g], w = grp_s[2 * g + 1];     // padded first slot, width
			const double *tile = reinterpret_cast<const double *>(smem_raw + (size_t)slot * tile_bytes) + (size_t)lr0 * k + c;
			if (w == 2)      dia_run<RB, 2>(acc, tile, k, vrow + sp, nd);
			else if (w == 3) dia_run<RB, 3>(acc, tile, k, vrow + sp, nd);
			else             dia_run<RB, 1>(acc, tile, k, vrow + sp, nd);
			__syncthreads();                         // every warp is done with this tile
		}
		if (in_cols) {
			const long long r0 = ((long long)blockIdx.x + (long long)lb * gridDim.x) * ROWS + lr0;
#pragma unroll
			for (int i = 0; i < RB; ++i)
				if (r0 + i < nrows)
					*reinterpret_cast<double2 *>(y + (size_t)(r0 + i) * ldy + c) = make_double2(acc[i][0], acc[i][1]);
		}
	}
}

// 2-D tensor map of the x window of the 1-D diagonal kernels: dim0 = the k columns, dim1 = the hb + nloc + ha rows
// (halo rows in front of and behind the local rows), box = (k, box_rows).  false: not available
static bool dia_x_tmap(CUtensorMap *tm, const b200_mat *M, const double *x, int ldx, int k, int box_rows)
{
	tmap_encode_fn enc = tmap_encoder();
	if (!enc) return false;
	const double *base = x - (size_t)M->halo_below * ldx;   // first row of the window
	const cuuint64_t gdim[2] = {(cuuint64_t)k, (cuuint64_t)(M->nrows + M->nhalo)};
	const cuuint64_t gstr[1] = {(cuuint64_t)ldx * 8};
	const cuuint32_t box[2] = {(cuuint32_t)k, (cuuint32_t)box_rows};
	const cuuint32_t estr[2] = {1, 1};
	return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(base), gdim, gstr, box, estr,
	           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
	           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// returns 0 launched, 1 error, 2 not applicable (caller falls back to the CSR kernels)
template <int G, int RB, int NS>
static int launch_spmm_dia(const b200_mat *M, const double *x, int ldx, double *y, int ldy, int k, const int *gate)
{
	constexpr int ROWS = 8 * (32 / G) * RB;
	static_assert(ROWS <= B200_DIA_PAD && B200_DIA_PAD % ROWS == 0, "diagonal image padding does not fit the row block");
	const int ng = M->dia_ng, nd = M->dia_ndp;               // slots per row incl. the run padding
	const int tile_bytes = (((ROWS + DIA_WMAX - 1) * k * 8) + 127) & ~127;
	const size_t smem = (size_t)NS * tile_bytes + 2 * (size_t)ROWS * nd * 8;
	if (smem > 200 * 1024) return 2;
	CUtensorMap tm;
	if (!dia_x_tmap(&tm, M, x, ldx, k, ROWS + DIA_WMAX - 1)) return 2;
	const int hb = M->halo_below;
	static bool attr_set = false;
	if (!attr_set) {
		B200_CUDA(cudaFuncSetAttribute(spmm_dia_tma_kernel<G, RB, NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
		attr_set = true;
	}
	const int nblocks = (int)(((long long)M->nrows + ROWS - 1) / ROWS);
	int per_sm = (int)((224 * 1024) / (smem + 2048)); if (per_sm < 1) per_sm = 1; if (per_sm > 3) per_sm = 3;
	int grid = g_b200.num_sms * per_sm; if (grid > nblocks) grid = nblocks;
	spmm_dia_tma_kernel<G, RB, NS><<<grid, 256, smem, g_b200.stream>>>(tm, M->nrows, nblocks, nd, M->dia_off, M->dia_val, ng,
		M->dia_grp, hb, tile_bytes, y, ldy, k, gate);
	B200_KERNEL_CHECK();
	return 0;
}


// ============================================================ diagonal SpMM, warp-specialised
// Second generation of the kernel above for the common even block widths (k known at compile
// time).  What the first one left on the table (profiles/ncu_r1d_spmm: 248 warp instructions per
// matrix row of which 60 are FP64, FP64 pipe 43 % busy, stalls on the CTA barrier after every
// run) and what this one does about it:
//
//   * lane map: a row group is KP consecutive THREADS (not a power-of-two slice of a warp), so at
//     k = 40 no lane idles -- the FP64 pipe, which the separate multiply and add of the
//     bit-exact accumulation load twice as hard as an FMA would, sees > 90 % useful lanes
//     instead of 62 %;
//   * every shared-memory offset (tile pitch k*8, row t of the box) is an immediate;
//   * a dedicated producer warp issues the TMA box copies; consumer warps hand a tile back
//     with one mbarrier arrive per warp (full/empty barrier pair per ring slot) -- no
//     __syncthreads anywhere in the main loop;
//   * CP column pairs per lane (template; shipped with CP = 1): the kernel runs at 88 % of the
//     shared-memory pipe (profiles/ncu_r1e_spmm) -- per matrix row 2880 B of x-row reads, 2333 B
//     of TMA writes and 2560 B of broadcast matrix values.  Two pairs per lane halve the value
//     traffic but measured slower (0.226 vs 0.204 ms at k = 40): fewer, fatter warps hide the
//     shared-memory latency worse than the saved wavefronts gain;
//   * DOT: the CG step needs diag(p^T A p) right after w = A p (reference
//     src/ops_lin_sol.c:300-325).  The accumulators hold the finished w rows, the p rows were
//     just pulled through L2 by the TMA unit, so the dot is a few FMAs in the epilogue and the
//     separate 16nk-byte streaming pass over p and w disappears.  Per-CTA partial sums go to
//     dot_part[cta][k]; the caller adds them in a fixed order (deterministic).
constexpr int DIA2_MAX_NS = 8;                         // deepest tile ring

// The CTAs walk the row blocks blk(idx) = blk_base + idx + (idx >= blk_split ? blk_skip : 0), idx <
// nblocks: all blocks, only the interior ones (whose x rows are all local) or only the boundary ones
// (the two ends of the slab) -- several ranks multiply the interior while the halo rows travel.
// k = 2 KP CP columns; NT consumer threads (NT / 32 warps) + one producer warp; a row group is KP
// consecutive threads and owns RB consecutive rows; lane gl of a group owns the column pairs
// gl, gl + KP, ... (so every 128-bit request of a warp covers one contiguous piece of an x row).
template <int KP, int CP, int RB, int NT, bool DOT, int MINB>
__global__ void __launch_bounds__(NT + 32, MINB)
spmm_dia_ws_kernel(const __grid_constant__ CUtensorMap tmx, int nrows, int nblocks, int nd, const int *__restrict__ off,
                   const double *__restrict__ val, int ng, const int *__restrict__ grp, int hb, int tile_bytes, int NS,
                   const double *x, int ldx, double *y, int ldy, const int *__restrict__ gate, double *dot_part,
                   int blk_base, int blk_split, int blk_skip)
{
	if (gate != nullptr && *gate == 0) return;
	constexpr int K = 2 * KP * CP;
	constexpr int NG = NT / KP;                        // row groups per CTA
	constexpr int ROWS = NG * RB;
	extern __shared__ __align__(128) unsigned char smem_raw[];
	// [NS x-tiles of tile_bytes][2 value buffers of ROWS x nd doubles]
	__shared__ unsigned long long full[DIA2_MAX_NS], empty[DIA2_MAX_NS], vfull[2], vempty[2];
	__shared__ int grp_s[64];
	__shared__ int d0_s[32];
	if (threadIdx.x < 2 * ng) grp_s[threadIdx.x] = __ldg(grp + threadIdx.x);
	if (threadIdx.x < ng) d0_s[threadIdx.x] = __ldg(off + threadIdx.x);      // first offset of each run
	if (threadIdx.x == 0) {
		for (int s = 0; s < NS; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, NT / 32); }
		for (int s = 0; s < 2; ++s) { mbar_init(vfull + s, 1); mbar_init(vempty + s, NT / 32); }
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
	}
	__syncthreads();
	const unsigned x_bytes = (unsigned)((ROWS + DIA_WMAX - 1) * K * 8);
	const unsigned val_bytes = (unsigned)(ROWS * nd * 8);
	unsigned char *vbuf = smem_raw + (size_t)NS * tile_bytes;
	const int my_blocks = (nblocks - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

	if (threadIdx.x >= NT) {
		// ------------------------------------------------------------------ producer warp
		if (threadIdx.x == NT) {
			int slot = 0; unsigned phase = 0;
			for (int lb = 0; lb < my_blocks; ++lb) {
				const int idx = blockIdx.x + lb * gridDim.x;
				const int blk = blk_base + idx + (idx >= blk_split ? blk_skip : 0);
				mbar_spin(vempty + (lb & 1), (unsigned)(((lb >> 1) & 1) ^ 1));
				mbar_expect_tx(vfull + (lb & 1), val_bytes);
				// the image is padded behind its last row (b200_mat.cu): full-size copies stay in bounds
				bulk_load_1d_evict_first(vbuf + (size_t)(lb & 1) * val_bytes, val + (size_t)blk * ROWS * nd, val_bytes, vfull + (lb & 1));
				for (int g = 0; g < ng; ++g) {
					mbar_spin(empty + slot, phase ^ 1u);
					mbar_expect_tx(full + slot, x_bytes);
					tma_load_2d(smem_raw + (size_t)slot * tile_bytes, &tmx, 0, blk * ROWS + d0_s[g] + hb, full + slot);
					if (++slot == NS) { slot = 0; phase ^= 1u; }
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
	const int lr0 = (live ? group : 0) * RB;           // first row of this group inside the block
	double acc[RB][2 * CP];
	double dot[2 * CP];
	double2 pst[RB][CP];                               // DOT: the block's own x rows, kept from the run that holds offset 0
#pragma unroll
	for (int j = 0; j < 2 * CP; ++j) dot[j] = 0.0;
#pragma unroll
	for (int i = 0; i < RB; ++i)
#pragma unroll
		for (int j = 0; j < CP; ++j) pst[i][j] = make_double2(0.0, 0.0);
	int slot = 0; unsigned phase = 0;
	for (int lb = 0; lb < my_blocks; ++lb) {
		mbar_spin(vfull + (lb & 1), (unsigned)((lb >> 1) & 1));
		const double *vrow = reinterpret_cast<const double *>(vbuf + (size_t)(lb & 1) * val_bytes) + (size_t)lr0 * nd;
#pragma unroll
		for (int i = 0; i < RB; ++i)
#pragma unroll
			for (int j = 0; j < 2 * CP; ++j) acc[i][j] = 0.0;
		for (int g = 0; g < ng; ++g) {
			mbar_spin(full + slot, phase);
			const int sp = grp_s[2 * g], w = grp_s[2 * g + 1];     // padded first slot, width
			const double *tile = reinterpret_cast<const double *>(smem_raw + (size_t)slot * tile_bytes) + lr0 * K + c;
			if (live) {
				// position of offset 0 inside this run (-1: not in it)
				const int zrow = (DOT && d0_s[g] <= 0 && d0_s[g] + w > 0) ? -d0_s[g] : -1;
				if (w == 2)      dia_run_ct<RB, 2, K, KP, CP, DOT>(acc, tile, vrow + sp, nd, pst, zrow);
				else if (w == 3) dia_run_ct<RB, 3, K, KP, CP, DOT>(acc, tile, vrow + sp, nd, pst, zrow);
				else             dia_run_ct<RB, 1, K, KP, CP, DOT>(acc, tile, vrow + sp, nd, pst, zrow);
			}
			// the loads from the tile must have been performed before it is handed back (the arrive does not
			// wait for loads in flight and ptxas may schedule it above the arithmetic that does; see
			// lincomb_tma_body in b200_dense.cu, where exactly that corrupted results)
			asm volatile("fence.acq_rel.cta;" ::: "memory");
			__syncwarp();
			if (lane == 0) mbar_arrive(empty + slot);          // this warp is done with the tile
			if (++slot == NS) { slot = 0; phase ^= 1u; }
		}
		__syncwarp();
		if (lane == 0) mbar_arrive(vempty + (lb & 1));         // ... and with the block's values
		if (live) {
			const int idx = blockIdx.x + lb * gridDim.x;
			const long long r0 = (long long)(blk_base + idx + (idx >= blk_split ? blk_skip : 0)) * ROWS + lr0;
#pragma unroll
			for (int i = 0; i < RB; ++i) {
				if (r0 + i < nrows) {
#pragma unroll
					for (int j = 0; j < CP; ++j) {
						// streaming store: y is not read again by this kernel and must not push x rows out of L2
						__stcs(reinterpret_cast<double2 *>(y + (size_t)(r0 + i) * ldy + c + 2 * KP * j),
						       make_double2(acc[i][2 * j], acc[i][2 * j + 1]));
						if (DOT) {
							const double2 pv = pst[i][j];
							dot[2 * j] = fma(pv.x, acc[i][2 * j], dot[2 * j]);
							dot[2 * j + 1] = fma(pv.y, acc[i][2 * j + 1], dot[2 * j + 1]);
						}
					}
				}
			}
		}
	}
	if (DOT) {
		// per-CTA column sums in a fixed order: groups 0 .. NG-1 (the tiles are dead: reuse tile 0)
		asm volatile("bar.sync 1, %0;" ::"n"(NT));
		double *red = reinterpret_cast<double *>(smem_raw);
		if (live) {
#pragma unroll
			for (int j = 0; j < CP; ++j) {
				red[group * K + c + 2 * KP * j] = dot[2 * j];
				red[group * K + c + 2 * KP * j + 1] = dot[2 * j + 1];
			}
		}
		asm volatile("bar.sync 1, %0;" ::"n"(NT));
		for (int cc = threadIdx.x; cc < K; cc += NT) {
			double s = 0.0;
			for (int gq = 0; gq < NG; ++gq) s += red[gq * K + cc];
			dot_part[(size_t)blockIdx.x * K + cc] = s;
		}
	}
}

// returns 0 launched, 1 error, 2 not applicable; *nparts = number of per-CTA dot partials written
// mode 0: every row block; 1: interior blocks (no halo row needed); 2: the boundary blocks
// MINB: CTAs per SM the kernel is compiled for (register cap) and its tile ring is sized for
template <int KP, int CP, int RB, int NT, bool DOT, int MINB>
static int launch_spmm_dia_ws(const b200_mat *M, const double *x, int ldx, double *y, int ldy, const int *gate,
                              double *dot_part, int dot_cap, int *nparts, int mode)
{
	constexpr int K = 2 * KP * CP;
	constexpr int ROWS = (NT / KP) * RB;
	static_assert(ROWS + DIA_WMAX - 1 <= 256, "TMA box too tall");
	static_assert(ROWS <= B200_DIA_PAD, "diagonal image padding does not cover the row block");
	const int ng = M->dia_ng, nd = M->dia_ndp;
	const int tile_bytes = (((ROWS + DIA_WMAX - 1) * K * 8) + 127) & ~127;
	const size_t val_smem = 2 * (size_t)ROWS * nd * 8;
	// ring depth: the deepest that still lets MINB CTAs share an SM (measured at k = 40: three
	// CTAs with 3 tiles each 0.201 ms, two with 6 tiles 0.205 ms, one with 8 tiles 0.29 ms, four with
	// 2 tiles 0.32 ms)
	const size_t budget = (size_t)(224 * 1024) / MINB - 2048;
	int NS = budget > val_smem ? (int)((budget - val_smem) / tile_bytes) : 0;
	if (NS > DIA2_MAX_NS) NS = DIA2_MAX_NS;
	if (NS < 2) NS = 2;
	const size_t smem = (size_t)NS * tile_bytes + val_smem;
	if (smem > 200 * 1024) return 2;
	CUtensorMap tm;
	if (!dia_x_tmap(&tm, M, x, ldx, K, ROWS + DIA_WMAX - 1)) return 2;
	const int hb = M->halo_below;
	static bool attr_set = false;
	if (!attr_set) {
		B200_CUDA(cudaFuncSetAttribute(spmm_dia_ws_kernel<KP, CP, RB, NT, DOT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
		attr_set = true;
	}
	const int nblocks_all = (int)(((long long)M->nrows + ROWS - 1) / ROWS);
	int nblocks = nblocks_all, blk_base = 0, split = 0x7fffffff, skip = 0;
	if (mode != 0) {
		// block b can touch halo rows iff b*ROWS < reach_below or (b+1)*ROWS + reach_above > nrows, where the
		// reach is that of the DIAGONAL IMAGE (farthest offsets), not of the halo plan: the plan's extents
		// come from the entries the first / last slab rows really have, and a row further inside may still
		// own the farthest diagonal (masked or irregular stencils, slabs not aligned to lattice planes)
		int reach_below = 0, reach_above = 0;
		for (int g = 0; g < ng; ++g) {
			const int lo = M->dia_off_h[g], hi = M->dia_off_h[g] + M->dia_grp_h[2 * g + 1] - 1;
			if (-lo > reach_below) reach_below = -lo;
			if (hi > reach_above) reach_above = hi;
		}
		if (hb > reach_below) reach_below = hb;
		if (M->nhalo - hb > reach_above) reach_above = M->nhalo - hb;
		int b_lo = (reach_below + ROWS - 1) / ROWS, b_hi = (M->nrows - reach_above) / ROWS;
		if (b_hi < 0) b_hi = 0;
		if (b_lo > nblocks_all) b_lo = nblocks_all;
		if (b_hi < b_lo) b_hi = b_lo;
		if (mode == 1) { blk_base = b_lo; nblocks = b_hi - b_lo; }
		else { split = b_lo; skip = b_hi - b_lo; nblocks = b_lo + (nblocks_all - b_hi); }
	}
	if (DOT) *nparts = 0;
	if (nblocks <= 0) return 0;
	int per_sm = (int)((224 * 1024) / (smem + 2048)); if (per_sm < 1) per_sm = 1; if (per_sm > 4) per_sm = 4;
	int grid = g_b200.num_sms * per_sm; if (grid > nblocks) grid = nblocks;
	if (DOT) {
		if (grid > dot_cap) return 2;
		*nparts = grid;
	}
	spmm_dia_ws_kernel<KP, CP, RB, NT, DOT, MINB><<<grid, NT + 32, smem, g_b200.stream>>>(tm, M->nrows, nblocks, nd, M->dia_off,
		M->dia_val, ng, M->dia_grp, hb, tile_bytes, NS, x, ldx, y, ldy, gate, dot_part, blk_base, split, skip);
	B200_KERNEL_CHECK();
	return 0;
}

// rows per group: 4 (the x rows of a run are then read 1.25 - 1.5 times), 2 where four would make
// the TMA box taller than 256 rows
template <int KP, int NT> struct Dia2Cfg {
	static constexpr int NG = NT / KP;
	static constexpr int RB = (NG * 4 + DIA_WMAX - 1 <= 256) ? 4 : 2;
};

template <int KP, int CP, int NT = 256>
static int launch_spmm_dia_ws_kp(const b200_mat *M, const double *x, int ldx, double *y, int ldy, const int *gate,
                                 double *dot_part, int dot_cap, int *nparts, int mode)
{
	constexpr int RB = Dia2Cfg<KP, NT>::RB;
	// the fused-dot variant keeps the block's own x rows in registers (96 instead of 56): two CTAs per SM with a
	// ring twice as deep.  Measured in the BlockPCG loop at n = 8 M, k = 40 (profiles/spmm_dot_variants_r2.log):
	// 2.06 ms; capped at 72 registers for three CTAs (spills) 2.32 ms; p re-read with __ldg (round 1) 2.01-2.10 ms;
	// plain kernel 1.93 ms + a separate 0.73 ms dot pass
	if (dot_part) return launch_spmm_dia_ws<KP, CP, RB, NT, true, 2>(M, x, ldx, y, ldy, gate, dot_part, dot_cap, nparts, mode);
	return launch_spmm_dia_ws<KP, CP, RB, NT, false, 3>(M, x, ldx, y, ldy, gate, nullptr, 0, nullptr, mode);
}

static bool dia_ws_has(int k)
{
	switch (k) {
#define HAS(KP_) case 2 * KP_:
	DIA_WS_WIDTHS(HAS) return true;
#undef HAS
	default: return false;
	}
}

// The block widths with a compile-time kernel (DIA_WS_WIDTHS); anything else takes the generic kernel above.
// One column pair per lane, 8 consumer warps, three CTAs per SM: measured best at every width
// (n = 1 M P1-FEM, k = 40: 0.204 ms; two pairs per lane 0.226 ms; 4-warp CTAs 0.216 - 0.249 ms;
// gpurun_out/spmm_variants3.log, summarised in profiles/).
static int spmm_dia_ws_dispatch(const b200_mat *M, const double *x, int ldx, double *y, int ldy, int k, const int *gate,
                                double *dot_part, int dot_cap, int *nparts, int mode = 0)
{
	{
		// lattice operators: plane tiles marching along k (b200_spmm_lat.cu); same bits, fewer shared-memory bytes
		const int rc = b200k_spmm_lat(M, x, ldx, y, ldy, k, gate, dot_part, dot_cap, nparts, mode);
		if (rc != 2) return rc;
	}
	switch (k) {
#define WS(KP_) case 2 * KP_: return launch_spmm_dia_ws_kp<KP_, 1>(M, x, ldx, y, ldy, gate, dot_part, dot_cap, nparts, mode);
	DIA_WS_WIDTHS(WS)
#undef WS
	default: return 2;
	}
}

// ---- diagonal image, 1 ... 4 columns ---------------------------------------------------------------------------
// The reference's OrthSelf multiplies B by ONE column at a time (src/ops_orth.c:45-118: thousands of calls per solve
// when its own code runs over the slots), and small block sizes give 2 ... 4.  The CSR kernels then stream 12 bytes per
// entry to multiply it with 8 k bytes of x; here a thread owns a row, walks its slots of the image in ascending
// column order (runs ascending, offsets inside a run ascending: the order of every other kernel in this file) and
// gathers the x rows itself -- neighbouring threads want neighbouring rows, so the gathers meet in L1.  Entries the
// CCS input does not hold are +0.0 in the image and add a signed zero; columns outside the window are skipped.
template <int K>
__global__ void __launch_bounds__(256)
spmm_dia_narrow_kernel(int nloc, int ng, const int *__restrict__ off, const int *__restrict__ grp, const double *__restrict__ val,
                       int ndp, const double *x, int ldx, int lo, int hi, double *y, int ldy, const int *__restrict__ gate)
{
	if (gate != nullptr && *gate == 0) return;
	__shared__ int off_s[32], slot_s[32], w_s[32];
	if ((int)threadIdx.x < ng) {
		off_s[threadIdx.x] = off[threadIdx.x]; slot_s[threadIdx.x] = grp[2 * threadIdx.x]; w_s[threadIdx.x] = grp[2 * threadIdx.x + 1];
	}
	__syncthreads();
	const long long row = (long long)blockIdx.x * 256 + threadIdx.x;
	if (row >= nloc) return;
	const double *v = val + (size_t)row * ndp;
	double acc[K];
#pragma unroll
	for (int c = 0; c < K; ++c) acc[c] = 0.0;
	for (int g = 0; g < ng; ++g) {
		const long long c0 = row + off_s[g];
		const double *vs = v + slot_s[g];
		for (int j = 0; j < w_s[g]; ++j) {
			const long long col = c0 + j;
			if (col < lo || col >= hi) continue;
			const double a = __ldg(vs + j);
			const double *xr = x + col * (long long)ldx;
#pragma unroll
			for (int c = 0; c < K; ++c) acc[c] = __dadd_rn(acc[c], __dmul_rn(a, xr[c]));
		}
	}
#pragma unroll
	for (int c = 0; c < K; ++c) y[(size_t)row * ldy + c] = acc[c];
}

static int launch_spmm_dia_narrow(const b200_mat *M, const double *x, int ldx, double *y, int ldy, int k, const int *gate)
{
	const int hb = M->halo_below, lo = -hb, hi = M->nrows + M->nhalo - hb;
	const unsigned grid = (unsigned)(((long long)M->nrows + 255) / 256);
#define NARROW(K_) spmm_dia_narrow_kernel<K_><<<grid, 256, 0, g_b200.stream>>>(M->nrows, M->dia_ng, M->dia_off, M->dia_grp, \
		M->dia_val, M->dia_ndp, x, ldx, lo, hi, y, ldy, gate)
	switch (k) {
	case 1: NARROW(1); break;
	case 2: NARROW(2); break;
	case 3: NARROW(3); break;
	case 4: NARROW(4); break;
	default: return 2;
	}
#undef NARROW
	B200_KERNEL_CHECK();
	return 0;
}

// diagonal image, at most 64 columns
static int spmm_dia_dispatch(const b200_mat *M, const double *x, int ldx, double *y, int ldy, int k, const int *gate)
{
	if (!spmm_aligned16(x, ldx, y, ldy, k)) return 2;
	{
		const int rc = spmm_dia_ws_dispatch(M, x, ldx, y, ldy, k, gate, nullptr, 0, nullptr);
		if (rc != 2) return rc;
	}
	// row-block heights and ring depths measured on B200 (profiles/spmm_sweep_r1_dia_tma.log)
	if (k <= 16) return launch_spmm_dia<8, 4, 4>(M, x, ldx, y, ldy, k, gate);
	if (k <= 32) return launch_spmm_dia<16, 4, 4>(M, x, ldx, y, ldy, k, gate);
	return launch_spmm_dia<32, 8, 4>(M, x, ldx, y, ldy, k, gate);
}

// sendbuf[i, 0:k] = x[rows[i], 0:k]
__global__ void halo_pack_kernel(int nsend, int k, const int *__restrict__ rows, const double *__restrict__ x, int ldx,
                                 double *__restrict__ buf)
{
	const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
	if (idx >= (long long)nsend * k) return;
	const int i = (int)(idx / k), c = (int)(idx - (long long)i * k);
	buf[idx] = x[(size_t)rows[i] * ldx + c];
}

extern "C" int b200k_spmm_check_halo(const b200_mat *M, const b200_mv *x)
{
	if (!b200_multi() || !M) return 0;
	if (x->halo_cap < M->nhalo)
		return b200_fail("SpMM across ranks: the multi-vector has room for %d halo rows but the matrix needs %d "
		                 "(create matrices before their multi-vectors)", x->halo_cap, M->nhalo);
	return 0;
}

// Halo rows of the k-column block x (rows [nrows, nrows + nhalo) of the multi-vector) from the
// slab neighbours: pack the rows each neighbour needs, one grouped ncclSend/ncclRecv over
// NVLink, unpack behind the local rows (reference analogue: the scatter of off-process
// entries in app/app_phg.c:292-357, done there per column; here once for the whole block).
static int halo_exchange(const b200_mat *M, double *x, int ldx, int k)
{
	if (M->nnbr == 0) return 0;
	const int nsend = M->send_off[M->nnbr], nrecv = M->recv_off[M->nnbr];
	double *sbuf = (double *)b200_scratch(6, sizeof(double) * (size_t)(nsend > 0 ? nsend : 1) * k);
	double *rbuf = (double *)b200_scratch(7, sizeof(double) * (size_t)(nrecv > 0 ? nrecv : 1) * k);
	if (!sbuf || !rbuf) return 1;
	if (nsend > 0) {
		const long long tot = (long long)nsend * k;
		halo_pack_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, g_b200.stream>>>(nsend, k, M->send_rows_dev, x, ldx, sbuf);
		B200_KERNEL_CHECK();
	}
	size_t so[64], sc[64], ro[64], rc[64];
	B200_CHECK(M->nnbr <= 64, "halo exchange: %d neighbours (at most 64)", M->nnbr);
	for (int i = 0; i < M->nnbr; ++i) {
		so[i] = (size_t)M->send_off[i] * k; sc[i] = (size_t)(M->send_off[i + 1] - M->send_off[i]) * k;
		ro[i] = (size_t)M->recv_off[i] * k; rc[i] = (size_t)(M->recv_off[i + 1] - M->recv_off[i]) * k;
	}
	if (b200k_neighbor_exchange(M->nnbr, M->nbr, sbuf, so, sc, rbuf, ro, rc)) return 1;
	if (nrecv > 0 && M->halo_contiguous) {
		// the receive buffer is ordered like the halo list: the rows below the slab, then above
		const int hb = M->halo_below, ha = nrecv - hb;
		if (hb > 0 && b200k_axpby(hb, k, 1.0, rbuf, k, 0.0, x - (size_t)hb * ldx, ldx)) return 1;
		if (ha > 0 && b200k_axpby(ha, k, 1.0, rbuf + (size_t)hb * k, k, 0.0, x + (size_t)M->nrows * ldx, ldx)) return 1;
		return 0;
	}
	if (nrecv > 0) return b200k_axpby(nrecv, k, 1.0, rbuf, k, 0.0, x + (size_t)M->nrows * ldx, ldx);
	return 0;
}

// local multiply with the CSR kernels (any matrix, any alignment)
static int spmm_csr_local(const b200_mat *M, int trans, const double *x, int ldx, double *y, int ldy, int k,
                          const int *gate)
{
	const int nrows = trans ? M->ncols : M->nrows;
	const int *rp = trans ? M->t_rp : M->rp, *ci = trans ? M->t_ci : M->ci;
	const double *va = trans ? M->t_va : M->va;
	if (k == 1)       return launch_spmm<1, 1>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate);
	else if (k == 2)  return launch_spmm<2, 1>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate);
	else if (k <= 4)  return launch_spmm<4, 1>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate);
	const int mrn = trans ? M->t_max_row_nnz : M->max_row_nnz;
	if (k <= 64 && mrn > 0 && (long long)mrn * 8 <= SPMM_CAP) {
		const int rpw = k <= 16 ? 4 : (k <= 32 ? 2 : 1);
		int rw = 8;                                             // rows per row group
		while (rw > 1 && (long long)8 * rpw * rw * mrn > SPMM_CAP) rw >>= 1;
		if ((long long)8 * rpw * rw * mrn <= SPMM_CAP) {
			if (k <= 16)      return launch_spmm_block_u<8>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate, rw);
			else if (k <= 32) return launch_spmm_block_u<16>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate, rw);
			return launch_spmm_block_u<32>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate, rw);
		}
	}
	if (k <= 16) return launch_spmm_wide<8, 1>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate);
	else if (k <= 32) return launch_spmm_wide<16, 1>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate);
	else if (k <= 64) return launch_spmm_wide<32, 1>(nrows, rp, ci, va, x, ldx, y, ldy, k, gate);
	// wider blocks: 128 columns per launch pass
	for (int c0 = 0; c0 < k; c0 += 128) {
		const int kc = k - c0 < 128 ? k - c0 : 128;
		int rc;
		if (kc <= 64) rc = launch_spmm_wide<32, 1>(nrows, rp, ci, va, x + c0, ldx, y + c0, ldy, kc, gate);
		else          rc = launch_spmm_wide<32, 2>(nrows, rp, ci, va, x + c0, ldx, y + c0, ldy, kc, gate);
		if (rc) return rc;
	}
	return 0;
}

// several ranks, diagonal image, a width the warp-specialised kernel has, and a halo the mailboxes take
static bool spmm_overlap_ok(const b200_mat *M, int trans, const double *x, int ldx, const double *y, int ldy, int k)
{
	if (!b200_multi() || trans || M->nnbr == 0 || M->dia_nd <= 0 || M->nrows <= 0 || !g_b200.comm_stream) return false;
	if (!spmm_aligned16(x, ldx, y, ldy, k) || !dia_ws_has(k)) return false;
	// the dot partials of the two launches must fit the caller's buffer: at most 4 CTAs per SM each
	return b200k_p2p_usable(M, k) != 0;
}

// y = A x (b200k_spmm) or, with dot_part, y = A x and the per-CTA partials of diag(x^T w) through the warp-specialised
// diagonal kernel (b200k_spmm_dot, which has checked that it applies): the halo exchange (several ranks: copy engines
// overlapped with the interior blocks, or NCCL), the profiler scope and the launches.  Returns that kernel's 2 when it
// does not take the block after all.
static int spmm_body(const b200_mat *M, int trans, const double *x, int ldx, double *y, int ldy, int k, const int *gate,
                     double *dot_part, int dot_cap, int *nparts)
{
	const int nrows = trans ? M->ncols : M->nrows;
	const double bytes = 12.0 * M->nnz + 4.0 * (nrows + 1) + 8.0 * k * ((double)M->nrows + M->ncols);
	const double flops = dot_part ? 2.0 * M->nnz * k + 2.0 * M->nrows * k : 2.0 * M->nnz * k;
	if (spmm_overlap_ok(M, trans, x, ldx, y, ldy, k)) {
		// the halo rows travel on the comm stream (copy engines) while the interior blocks multiply
		if (b200k_p2p_halo_exchange(M, const_cast<double *>(x), ldx, k)) return 1;
		B200Prof prof(B200_PROF_SPMM, bytes, flops);
		int n1 = 0, n2 = 0;
		if (spmm_dia_ws_dispatch(M, x, ldx, y, ldy, k, gate, dot_part, dot_cap, &n1, 1)) return 1;
		B200_CUDA(cudaStreamWaitEvent(g_b200.stream, g_b200.ev_halo_done, 0));
		if (spmm_dia_ws_dispatch(M, x, ldx, y, ldy, k, gate, dot_part ? dot_part + (size_t)n1 * k : nullptr, dot_cap - n1,
		                         &n2, 2))
			return 1;
		if (dot_part) *nparts = n1 + n2;
		return 0;
	}
	if (b200_multi() && halo_exchange(M, const_cast<double *>(x), ldx, k)) return 1;
	if (nrows <= 0) return 0;
	B200Prof prof(B200_PROF_SPMM, bytes, flops);
	if (dot_part) return spmm_dia_ws_dispatch(M, x, ldx, y, ldy, k, gate, dot_part, dot_cap, nparts);
	if (!trans && M->dia_nd > 0 && M->nrows > 0) {
		// diagonal image, 64 columns per pass (1 ... 4 columns: the narrow kernel); whatever it cannot take
		// (a misaligned or odd block) goes to the CSR kernels
		int c0 = 0;
		for (; c0 < k; c0 += 64) {
			const int kc = k - c0 < 64 ? k - c0 : 64;
			const int rc = (kc > 4) ? spmm_dia_dispatch(M, x + c0, ldx, y + c0, ldy, kc, gate)
			                        : launch_spmm_dia_narrow(M, x + c0, ldx, y + c0, ldy, kc, gate);
			if (rc == 1) return 1;
			if (rc == 2) break;
		}
		if (c0 >= k) return 0;
		return spmm_csr_local(M, 0, x + c0, ldx, y + c0, ldy, k - c0, gate);
	}
	return spmm_csr_local(M, trans, x, ldx, y, ldy, k, gate);
}

int b200k_spmm(const b200_mat *M, int trans, const double *x, int ldx, double *y, int ldy, int k,
               const int *gate)
{
	if (trans && !M->t_rp) {
		// row-partitioned matrix: only the forward image is kept; A^T x == A x when A is symmetric
		// (the reference assumes that for every matrix, app/app_ccs.c:140-150)
		B200_CHECK(M->symmetric, "transposed SpMM of a non-symmetric matrix is not available across ranks");
		trans = 0;
	}
	if (k <= 0) return 0;
	return spmm_body(M, trans, x, ldx, y, ldy, k, gate, nullptr, 0, nullptr);
}

// w = A x together with the per-CTA partial sums of diag(x^T w) (fused BlockPCG step).  Only the
// warp-specialised diagonal kernel can do this; returns 2 (nothing launched) when it does not
// apply, and the caller runs the plain SpMM followed by the streaming dot kernel.
int b200k_spmm_dot(const b200_mat *M, const double *x, int ldx, double *y, int ldy, int k, const int *gate,
                   double *dot_part, int dot_cap, int *nparts)
{
	*nparts = 0;
	if (!(M->dia_nd > 0 && k > 4 && k <= 64 && M->nrows > 0) || b200_opt(B200_OPT_NO_FUSED_DOT)) return 2;
	// the epilogue takes p from the run that holds offset 0 (the main diagonal): without one, no fusion
	if (dia_zero_run(M) < 0) return 2;
	if (!spmm_aligned16(x, ldx, y, ldy, k)) return 2;
	return spmm_body(M, 0, x, ldx, y, ldy, k, gate, dot_part, dot_cap, nparts);
}

extern "C" int b200_mat_dot_multivec(const b200_mat *A, int trans, const b200_mv *x, b200_mv *y,
                                     const int *start, const int *end)
{
	B200_REQUIRE_INIT();
	B200_CHECK(x && y && start && end, "b200_mat_dot_multivec: bad arguments");
	const int k = end[0] - start[0];
	B200_CHECK(k == end[1] - start[1], "b200_mat_dot_multivec: column counts differ (%d vs %d)", k,
	           end[1] - start[1]);
	if (k == 0) return 0;
	B200_CHECK(start[0] >= 0 && end[0] <= x->ncols && start[1] >= 0 && end[1] <= y->ncols,
	           "b200_mat_dot_multivec: column range out of bounds");
	if (!A) {
		// reference app/app_ccs.c:134-137: NULL matrix means copy
		B200_CHECK(x->nrows == y->nrows, "b200_mat_dot_multivec: row counts differ");
		return b200k_axpby(y->nrows, k, 1.0, x->d + start[0], x->ld, 0.0, y->d + start[1], y->ld);
	}
	const int out_rows = trans ? A->ncols : A->nrows, in_rows = trans ? A->nrows : A->ncols;
	B200_CHECK(x->nrows == in_rows && y->nrows == out_rows,
	           "b200_mat_dot_multivec: shapes do not match the matrix (%d x %d)", A->nrows, A->ncols);
	if (x == y) {
		const bool overlap = start[0] < end[1] && start[1] < end[0];
		B200_CHECK(!overlap, "b200_mat_dot_multivec: x and y column ranges overlap on one multi-vector");
	}
	if (b200k_spmm_check_halo(A, x)) return 1;
	return b200k_spmm(A, trans, x->d + start[0], x->ld, y->d + start[1], y->ld, k, nullptr);
}
