// Runtime: device selection, library stream, growable scratch, error reporting.
#include "b200_internal.h"
#include <chrono>

b200_ctx g_b200 = {};

extern "C" int b200_fail(const char *fmt, ...)
{
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_b200.err, sizeof(g_b200.err), fmt, ap);
	va_end(ap);
	return 1;
}

extern "C" const char *b200_last_error(void) { return g_b200.err; }

extern "C" int b200_device_count(void)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
	return n;
}

static void options_from_environment(void);

extern "C" int b200_init(int device)
{
	if (g_b200.initialised && (device < 0 || device == g_b200.device)) return 0;
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess || n == 0)
		return b200_fail("b200_init: no CUDA device (%s); this library has no CPU fallback",
		                 e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
	if (device < 0) {
		const char *lr = getenv("LOCAL_RANK");
		device = lr ? atoi(lr) % n : 0;
	}
	B200_CHECK(device < n, "b200_init: device %d out of range (%d visible)", device, n);
	B200_CUDA(cudaSetDevice(device));
	cudaDeviceProp prop;
	B200_CUDA(cudaGetDeviceProperties(&prop, device));
	B200_CHECK(prop.major >= 10, "b200_init: device %d is sm_%d%d; this library is built for sm_100a only",
	           device, prop.major, prop.minor);
	options_from_environment();
	if (g_b200.initialised) b200_finalize();
	g_b200.device = device;
	g_b200.num_sms = prop.multiProcessorCount;
	B200_CUDA(cudaStreamCreateWithFlags(&g_b200.stream, cudaStreamNonBlocking));
	g_b200.launches = 0;
	g_b200.initialised = 1;
	return 0;
}

// ---- run-time switches -------------------------------------------------------------------------------------
int g_b200_opt[B200_OPT_COUNT];
static const char *const g_opt_names[B200_OPT_COUNT] = {
#define OPT_NAME(id, name) #name,
	B200_OPTIONS(OPT_NAME)
#undef OPT_NAME
};

// B200_<NAME> in the environment: a number is taken as is, anything else (incl. an empty value) means 1
static void options_from_environment(void)
{
	static bool done = false;
	if (done) return;
	done = true;
	for (int i = 0; i < B200_OPT_COUNT; ++i) {
		char env[64] = "B200_";
		size_t n = strlen(env);
		for (const char *c = g_opt_names[i]; *c && n + 1 < sizeof(env); ++c) env[n++] = (char)((*c >= 'a' && *c <= 'z') ? *c - 32 : *c);
		env[n] = 0;
		const char *v = getenv(env);
		if (!v) continue;
		char *end = nullptr;
		const long x = strtol(v, &end, 10);
		g_b200_opt[i] = (end != v && *end == 0) ? (int)x : 1;
	}
}

extern "C" int b200_option_count(void) { return B200_OPT_COUNT; }
extern "C" const char *b200_option_name(int i) { return (i >= 0 && i < B200_OPT_COUNT) ? g_opt_names[i] : nullptr; }

extern "C" int b200_option_set(const char *name, int value)
{
	options_from_environment();
	for (int i = 0; i < B200_OPT_COUNT; ++i)
		if (name && 0 == strcmp(name, g_opt_names[i])) { g_b200_opt[i] = value; return 0; }
	return b200_fail("b200_option_set: unknown option '%s'", name ? name : "(null)");
}

extern "C" int b200_option_get(const char *name, int *value)
{
	options_from_environment();
	for (int i = 0; i < B200_OPT_COUNT; ++i)
		if (name && 0 == strcmp(name, g_opt_names[i])) { if (value) *value = g_b200_opt[i]; return 0; }
	return b200_fail("b200_option_get: unknown option '%s'", name ? name : "(null)");
}

extern "C" int b200k_opt(int id) { options_from_environment(); return (id >= 0 && id < B200_OPT_COUNT) ? g_b200_opt[id] : 0; }

extern "C" void b200_finalize(void)
{
	if (!g_b200.initialised) return;
	if (g_b200.pending) b200k_pending_flush();
	cudaStreamSynchronize(g_b200.stream);
	b200_gcg_free_cache();
	for (int i = 0; i < 11; ++i) {
		if (g_b200.scratch[i]) cudaFree(g_b200.scratch[i]);
		g_b200.scratch[i] = nullptr; g_b200.scratch_bytes[i] = 0;
	}
	for (int i = 0; i < 2; ++i) {
		if (g_b200.pinned[i]) cudaFreeHost(g_b200.pinned[i]);
		g_b200.pinned[i] = nullptr; g_b200.pinned_bytes[i] = 0;
	}
	cudaStreamDestroy(g_b200.stream);
	g_b200.initialised = 0;
}

extern "C" void *b200_scratch(int slot, size_t bytes)
{
	if (bytes <= g_b200.scratch_bytes[slot]) return g_b200.scratch[slot];
	// growing a slot: every kernel that used the old buffer must be done first
	cudaStreamSynchronize(g_b200.stream);
	if (g_b200.scratch[slot]) cudaFree(g_b200.scratch[slot]);
	g_b200.scratch[slot] = nullptr; g_b200.scratch_bytes[slot] = 0;
	size_t want = bytes + bytes / 4 + 4096;
	cudaError_t e = cudaMalloc(&g_b200.scratch[slot], want);
	if (e != cudaSuccess) {
		b200_fail("scratch[%d]: cudaMalloc(%zu) failed: %s", slot, want, cudaGetErrorString(e));
		return nullptr;
	}
	g_b200.scratch_bytes[slot] = want;
	return g_b200.scratch[slot];
}

extern "C" void *b200_pinned(int slot, size_t bytes)
{
	if (bytes <= g_b200.pinned_bytes[slot]) return g_b200.pinned[slot];
	cudaStreamSynchronize(g_b200.stream);
	if (g_b200.pinned[slot]) cudaFreeHost(g_b200.pinned[slot]);
	g_b200.pinned[slot] = nullptr; g_b200.pinned_bytes[slot] = 0;
	size_t want = bytes + bytes / 4 + 4096;
	cudaError_t e = cudaMallocHost(&g_b200.pinned[slot], want);
	if (e != cudaSuccess) {
		b200_fail("pinned[%d]: cudaMallocHost(%zu) failed: %s", slot, want, cudaGetErrorString(e));
		return nullptr;
	}
	g_b200.pinned_bytes[slot] = want;
	return g_b200.pinned[slot];
}

extern "C" int b200_sync(void)
{
	B200_REQUIRE_INIT();
	B200_CUDA(cudaStreamSynchronize(g_b200.stream));
	return 0;
}

extern "C" double b200_wtime(void)
{
	if (g_b200.initialised && g_b200.pending) b200k_pending_flush();
	if (g_b200.initialised) cudaStreamSynchronize(g_b200.stream);
	using clk = std::chrono::steady_clock;
	return std::chrono::duration<double>(clk::now().time_since_epoch()).count();
}

extern "C" long long b200_kernel_launches(void) { return g_b200.launches; }

extern "C" int b200k_num_sms(void) { return g_b200.num_sms; }

extern "C" int b200k_d2h(void *host, const void *dev, size_t bytes)
{
	if (bytes == 0) return 0;
	void *pin = b200_pinned(0, bytes);
	if (!pin) return 1;
	B200_CUDA(cudaMemcpyAsync(pin, dev, bytes, cudaMemcpyDeviceToHost, g_b200.stream));
	B200_CUDA(cudaStreamSynchronize(g_b200.stream));
	memcpy(host, pin, bytes);
	return 0;
}

extern "C" int b200k_h2d(void *dev, const void *host, size_t bytes)
{
	if (bytes == 0) return 0;
	B200_CUDA(cudaStreamSynchronize(g_b200.stream));   // pinned staging may still be in flight
	void *pin = b200_pinned(0, bytes);
	if (!pin) return 1;
	memcpy(pin, host, bytes);
	B200_CUDA(cudaMemcpyAsync(dev, pin, bytes, cudaMemcpyHostToDevice, g_b200.stream));
	return 0;
}

extern "C" int b200k_memset(void *dev, int value, size_t bytes)
{
	if (bytes == 0) return 0;
	B200_CUDA(cudaMemsetAsync(dev, value, bytes, g_b200.stream));
	return 0;
}

extern "C" int b200k_malloc(void **dev, size_t bytes)
{
	B200_REQUIRE_INIT();
	cudaError_t e = cudaMalloc(dev, bytes ? bytes : 8);
	if (e != cudaSuccess) return b200_fail("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
	B200_CUDA(cudaMemsetAsync(*dev, 0, bytes ? bytes : 8, g_b200.stream));
	return 0;
}

extern "C" int b200k_free(void *dev)
{
	if (!dev) return 0;
	if (g_b200.initialised) cudaStreamSynchronize(g_b200.stream);
	cudaFree(dev);
	return 0;
}

static cudaEvent_t g_ev[2];
static bool g_ev_ok = false;

extern "C" int b200_timer_start(void)
{
	B200_REQUIRE_INIT();
	if (!g_ev_ok) {
		B200_CUDA(cudaEventCreate(&g_ev[0]));
		B200_CUDA(cudaEventCreate(&g_ev[1]));
		g_ev_ok = true;
	}
	B200_CUDA(cudaEventRecord(g_ev[0], g_b200.stream));
	return 0;
}

extern "C" int b200_timer_stop(double *ms)
{
	B200_CHECK(g_ev_ok && ms, "b200_timer_stop: timer not started");
	if (g_b200.pending && b200k_pending_flush()) return 1;
	B200_CUDA(cudaEventRecord(g_ev[1], g_b200.stream));
	B200_CUDA(cudaEventSynchronize(g_ev[1]));
	float f = 0.f;
	B200_CUDA(cudaEventElapsedTime(&f, g_ev[0], g_ev[1]));
	*ms = f;
	return 0;
}

extern "C" int b200_flush_l2(void)
{
	B200_REQUIRE_INIT();
	const size_t bytes = (size_t)256 << 20;      // 2 x the 126 MB L2
	static void *buf = nullptr;
	if (!buf) B200_CUDA(cudaMalloc(&buf, bytes));
	B200_CUDA(cudaMemsetAsync(buf, 1, bytes, g_b200.stream));
	return 0;
}

// ------------------------------------------------------------------ per-class profiling
#include <vector>
namespace {
struct ProfRec { int cls; cudaEvent_t a, b; };
struct ProfState {
	bool on = false, open = false;
	std::vector<ProfRec> pend;          // recorded, not yet resolved
	std::vector<cudaEvent_t> pool;      // free events
	double ms[B200_PROF_NCLS] = {}, bytes[B200_PROF_NCLS] = {}, flops[B200_PROF_NCLS] = {};
	double gap_ms[B200_PROF_NCLS] = {};  // stream time between the previous scope's end and this scope's start
	long long calls[B200_PROF_NCLS] = {};
} g_prof;
const char *g_prof_names[B200_PROF_NCLS] = {"spmm", "gram", "lincomb", "axpby", "dots", "bpcg_fused",
                                            "orth_panel", "syev_jacobi", "small_dense"};
cudaEvent_t prof_event()
{
	if (!g_prof.pool.empty()) { cudaEvent_t e = g_prof.pool.back(); g_prof.pool.pop_back(); return e; }
	cudaEvent_t e = nullptr;
	cudaEventCreate(&e);
	return e;
}
void prof_resolve()
{
	if (g_prof.pend.empty()) return;
	cudaEventSynchronize(g_prof.pend.back().b);
	for (size_t i = 0; i < g_prof.pend.size(); ++i) {
		const ProfRec &r = g_prof.pend[i];
		float f = 0.f;
		if (cudaEventElapsedTime(&f, r.a, r.b) == cudaSuccess) g_prof.ms[r.cls] += f;
		// what ran (or idled) on the stream between two scopes: unclassified kernels, copies, NCCL, host latency
		if (i > 0 && cudaEventElapsedTime(&f, g_prof.pend[i - 1].b, r.a) == cudaSuccess) g_prof.gap_ms[r.cls] += f;
	}
	for (const ProfRec &r : g_prof.pend) {
		g_prof.pool.push_back(r.a); g_prof.pool.push_back(r.b);
	}
	g_prof.pend.clear();
}
}  // namespace

B200Prof::B200Prof(int cls, double bytes, double flops) : slot(-1)
{
	if (!g_prof.on || g_prof.open) return;
	ProfRec r; r.cls = cls; r.a = prof_event(); r.b = prof_event();
	if (!r.a || !r.b) return;
	cudaEventRecord(r.a, g_b200.stream);
	g_prof.pend.push_back(r);
	g_prof.open = true;
	g_prof.calls[cls] += 1; g_prof.bytes[cls] += bytes; g_prof.flops[cls] += flops;
	slot = (int)g_prof.pend.size() - 1;
}

B200Prof::~B200Prof()
{
	if (slot < 0) return;
	cudaEventRecord(g_prof.pend[slot].b, g_b200.stream);
	g_prof.open = false;
	if (g_prof.pend.size() >= 4096) prof_resolve();
}

extern "C" int b200_prof_enable(int on)
{
	B200_REQUIRE_INIT();
	prof_resolve();
	if (on) {
		for (int i = 0; i < B200_PROF_NCLS; ++i) { g_prof.ms[i] = g_prof.bytes[i] = g_prof.flops[i] = g_prof.gap_ms[i] = 0.0; g_prof.calls[i] = 0; }
	}
	g_prof.on = on != 0;
	return 0;
}

extern "C" int b200_prof_classes(void) { return B200_PROF_NCLS; }

extern "C" int b200_prof_get(int cls, const char **name, double *ms, long long *calls, double *bytes, double *flops)
{
	B200_CHECK(cls >= 0 && cls < B200_PROF_NCLS, "b200_prof_get: class %d out of range", cls);
	prof_resolve();
	if (name) *name = g_prof_names[cls];
	if (ms) *ms = g_prof.ms[cls];
	if (calls) *calls = g_prof.calls[cls];
	if (bytes) *bytes = g_prof.bytes[cls];
	if (flops) *flops = g_prof.flops[cls];
	return 0;
}

// stream time that elapsed between the end of the previous profiled call and the start of the
// calls of class `cls`: kernels outside the classes, copies, collectives, and idle stream time
extern "C" int b200_prof_get_gap(int cls, double *ms)
{
	B200_CHECK(cls >= 0 && cls < B200_PROF_NCLS && ms, "b200_prof_get_gap: bad arguments");
	prof_resolve();
	*ms = g_prof.gap_ms[cls];
	return 0;
}

extern "C" int b200_host_register(void *host, unsigned long long bytes)
{
	B200_REQUIRE_INIT();
	B200_CHECK(host && bytes, "b200_host_register: bad arguments");
	B200_CUDA(cudaHostRegister(host, (size_t)bytes, cudaHostRegisterDefault));
	return 0;
}

extern "C" int b200_host_unregister(void *host)
{
	B200_CHECK(host, "b200_host_unregister: bad arguments");
	B200_CUDA(cudaHostUnregister(host));
	return 0;
}
