// Internal declarations shared by the CUDA translation units of libgcge_b200.so.
// Public surface: include/gcge_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <cstdarg>
#include "gcge_b200.h"

#include "../host/b200_dev.h"

struct b200_ctx {
	int initialised;
	int device;
	int num_sms;
	cudaStream_t stream;
	// growable device scratch: [0] reduction partials, [1] coefficient staging,
	// [2] host<->device column-major staging, [3] small results
	// [4] BlockPCG state, [5] Jacobi work, [6] halo send buffer, [7] halo receive buffer,
	// [8] contiguous Gram block for the allreduce, [9] the GCG driver's small device arrays,
	// [10] BlockPCG's Jacobi preconditioner D^-1 and its diagonal check
	void *scratch[11];
	size_t scratch_bytes[11];
	// pinned host staging for small results / coefficients
	void *pinned[2];
	size_t pinned_bytes[2];
	long long launches;
	char err[512];
	// multi-GPU layout (b200_comm.cu): rank of this process, number of ranks (0/1 = single GPU)
	int rank, nranks;
	// halo exchange off the critical path: a second stream driven by copy engines and stream memory
	// operations only (b200_comm.cu), and the two events that tie it to the library stream;
	// comm_stream == nullptr: exchanges run on the library stream through NCCL
	cudaStream_t comm_stream;
	cudaEvent_t ev_x_ready, ev_halo_done;
	// halo rows a multi-vector with n global rows must be able to hold behind its local rows:
	// the largest halo of any matrix with that many columns created so far
	long long halo_n[8];
	int halo_cap[8];
	// != 0: narrow axpby calls are waiting to be launched as one kernel (b200_mv.cu, b200k_pending_flush)
	int pending;
};

int b200k_allreduce_sum(double *buf_dev, size_t count);
int b200k_neighbor_exchange(int nnbr, const int *nbr, const double *send_dev, const size_t *send_off,
                            const size_t *send_cnt, double *recv_dev, const size_t *recv_off, const size_t *recv_cnt);
// Small allreduce INSIDE a kernel (b200_comm.cu sets it up, b200_stream.cuh has the device side): every
// rank's inbox and flags are IPC-mapped on every other rank.  nranks == 0: not available (use NCCL).
constexpr int B200_AR_MAX_RANKS = 8;
constexpr int B200_AR_MAX_COUNT = 256;
struct B200ArCtx {
	int nranks, rank;
	double *inbox[B200_AR_MAX_RANKS];      // rank q's inbox: [2 parities][nranks][B200_AR_MAX_COUNT]; [rank] is the local one
	unsigned *flags[B200_AR_MAX_RANKS];    // rank q's flags: [2 parities][nranks]
	unsigned *seq;                         // local: number of in-kernel allreduces done
	int *status;                           // local: != 0 after a time-out
};
B200ArCtx b200k_ar_ctx();
// halo exchange by copy engines on the comm stream (b200_comm.cu)
int b200k_p2p_register(int rows, int *all_ranks_ok);
int b200k_p2p_usable(const b200_mat *M, int k);
int b200k_p2p_halo_exchange(const b200_mat *M, double *x, int ldx, int k);

// lattice SpMM (b200_spmm_lat.cu): recognition at matrix creation; multiply: 0 launched, 1 error, 2 not applicable
int b200k_lat_detect(b200_mat *A);
int b200k_spmm_lat(const b200_mat *M, const double *x, int ldx, double *y, int ldy, int k, const int *gate,
                   double *dot_part, int dot_cap, int *nparts, int mode);

// ---- run-time switches (b200_runtime.cu): one table, filled ONCE from the environment (B200_<NAME>) at b200_init,
// changeable through b200_option_set / the OPS adaptor's -b200_<name> command-line options; kernels read the cached ints
enum { B200_OPT_NO_DIA = 0, B200_OPT_NO_LAT, B200_OPT_SPMM_OLD_DIA, B200_OPT_NO_FUSED_DOT, B200_OPT_NO_TMA_DENSE,
       B200_OPT_HOST_BUILD, B200_OPT_NO_OVERLAP, B200_OPT_NO_P2P, B200_OPT_NO_KERNEL_ALLREDUCE, B200_OPT_SYEV_PROF,
       B200_OPT_BPCG_TRACE, B200_OPT_SPMM_CTAS, B200_OPT_SPMM_NS, B200_OPT_LAT_TI, B200_OPT_LAT_TJ, B200_OPT_LAT_NS,
       B200_OPT_LAT_EVEN_PITCH, B200_OPT_LAT_NO_VPAD, B200_OPT_LAT_VERBOSE, B200_OPT_LAT_NO_CONST, B200_OPT_ORTH_TRACE, B200_OPT_NO_AXPBY_BATCH, B200_OPT_BPCG_CTAS, B200_OPT_COUNT };
extern int g_b200_opt[B200_OPT_COUNT];
static inline int b200_opt(int id) { return g_b200_opt[id]; }
static_assert(B200_OPT_BPCG_TRACE == B200K_OPT_BPCG_TRACE && B200_OPT_ORTH_TRACE == B200K_OPT_ORTH_TRACE, "b200_dev.h option id out of step");

extern b200_ctx g_b200;
static inline bool b200_multi() { return g_b200.nranks > 1; }

#define B200_CUDA(call)                                                            \
	do {                                                                           \
		cudaError_t e_ = (call);                                                   \
		if (e_ != cudaSuccess)                                                     \
			return b200_fail("%s:%d %s: %s", __FILE__, __LINE__, #call,           \
			                 cudaGetErrorString(e_));                              \
	} while (0)

// every entry point that touches device data starts here: the library is up, and deferred work (the batch of narrow
// axpby calls, b200_mv.cu) has been launched
#define B200_REQUIRE_INIT()                                                        \
	do {                                                                           \
		if (!g_b200.initialised) {                                                 \
			int rc_ = b200_init(-1);                                               \
			if (rc_) return rc_;                                                   \
		}                                                                          \
		if (g_b200.pending) {                                                      \
			int rc_ = b200k_pending_flush();                                       \
			if (rc_) return rc_;                                                   \
		}                                                                          \
	} while (0)

#define B200_CHECK(cond, ...)                                                      \
	do {                                                                           \
		if (!(cond)) return b200_fail(__VA_ARGS__);                                \
	} while (0)

#define B200_LAUNCHED() (++g_b200.launches)
#define B200_KERNEL_CHECK()                                                        \
	do {                                                                           \
		B200_LAUNCHED();                                                           \
		cudaError_t e_ = cudaGetLastError();                                       \
		if (e_ != cudaSuccess)                                                     \
			return b200_fail("%s:%d kernel launch: %s", __FILE__, __LINE__,        \
			                 cudaGetErrorString(e_));                              \
	} while (0)

// rows the diagonal image of a matrix is padded to a multiple of (largest SpMM row block)
constexpr int B200_DIA_PAD = 256;

static inline int b200_ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }


// ---- per-kernel-class device timing (b200_prof_*, include/gcge_b200.h) ---------------------
// A scope object brackets the launches of one b200k_* call with two CUDA events on the library
// stream and books the call's ALGORITHMIC bytes / flops (SURVEY.md §8d) to its class.  Free
// when profiling is off.  Scopes do not nest: an inner scope is a no-op.
enum { B200_PROF_SPMM = 0, B200_PROF_GRAM, B200_PROF_LINCOMB, B200_PROF_AXPBY, B200_PROF_DOTS,
       B200_PROF_BPCG, B200_PROF_PANEL, B200_PROF_SYEV, B200_PROF_SMALL, B200_PROF_NCLS };
struct B200Prof {
	int slot;
	B200Prof(int cls, double bytes, double flops);
	~B200Prof();
};
