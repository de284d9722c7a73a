// C ABI of libmegalania_cuda.so (see include/megalania_cuda.h).  Host-side glue only: device
// memory, launches, format conversion.  No CPU implementation of the hot path lives here.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <new>
#include <vector>
#include <unistd.h>

#include "../../include/megalania_cuda.h"
#include "mg_kernels.cuh"

using namespace mg;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...)
{
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_err, sizeof(g_err), fmt, ap);
	va_end(ap);
	return code;
}

#define CU(call)                                                                                   \
	do {                                                                                           \
		cudaError_t e_ = (call);                                                                   \
		if (e_ != cudaSuccess)                                                                     \
			return fail(e_ == cudaErrorMemoryAllocation ? MG_ENOMEM : MG_ECUDA, "%s: %s", #call,   \
			            cudaGetErrorString(e_));                                                   \
	} while (0)

extern "C" MG_API const char* mg_last_error(void) { return g_err; }
// ---- device memory pool -----------------------------------------------------------------------------------
// A one-shot call (mg_ctx_create + mg_anneal_oneshot) allocates and frees ~90 GB of chain state; cudaMalloc and
// cudaFree of that size cost 0.15 s per call, more than a tenth of a one-second annealing step.  Blocks released
// by the library are kept per device and handed back to the next request of the same size; everything cached is
// returned to the driver when an allocation fails, and by mg_pool_trim().
#include <map>
#include <mutex>
#include <unordered_map>
namespace {
struct DevicePool {
	std::mutex lock;
	std::unordered_map<void*, std::pair<int, size_t>> live;       // pointer -> (device, bytes)
	std::multimap<std::pair<int, size_t>, void*> cached;          // (device, bytes) -> pointer
};
DevicePool& pool()
{
	static DevicePool* p = new DevicePool;  // leaked on purpose: contexts may be destroyed from static destructors
	return *p;
}
void pool_release_device(int device)
{
	DevicePool& P = pool();
	for (auto it = P.cached.begin(); it != P.cached.end();) {
		if (device < 0 || it->first.first == device) {
			cudaFree(it->second);
			it = P.cached.erase(it);
		} else {
			++it;
		}
	}
}
}  // namespace

static cudaError_t pool_malloc_raw(void** out, size_t bytes)
{
	if (bytes == 0) bytes = 16;
	int device = 0;
	cudaError_t e = cudaGetDevice(&device);
	if (e != cudaSuccess) return e;
	DevicePool& P = pool();
	std::lock_guard<std::mutex> g(P.lock);
	auto hit = P.cached.find({device, bytes});
	if (hit != P.cached.end()) {
		*out = hit->second;
		P.cached.erase(hit);
	} else {
		e = cudaMalloc(out, bytes);
		if (e == cudaErrorMemoryAllocation) {
			cudaGetLastError();
			pool_release_device(device);
			e = cudaMalloc(out, bytes);
		}
		if (e != cudaSuccess) return e;
	}
	P.live[*out] = {device, bytes};
	return cudaSuccess;
}
template <class T> static cudaError_t pool_malloc(T** out, size_t bytes) { return pool_malloc_raw(reinterpret_cast<void**>(out), bytes); }

static void pool_free(void* p)
{
	if (!p) return;
	DevicePool& P = pool();
	std::lock_guard<std::mutex> g(P.lock);
	auto it = P.live.find(p);
	if (it == P.live.end()) {
		cudaFree(p);
		return;
	}
	P.cached.insert({it->second, p});
	P.live.erase(it);
}

extern "C" MG_API void mg_pool_trim(void)
{
	DevicePool& P = pool();
	std::lock_guard<std::mutex> g(P.lock);
	int device = 0;
	cudaGetDevice(&device);
	for (auto it = P.cached.begin(); it != P.cached.end();) {
		cudaSetDevice(it->first.first);
		cudaFree(it->second);  // not pool_free(): the lock is held, and a cached block is not live
		it = P.cached.erase(it);
	}
	cudaSetDevice(device);
}

extern "C" MG_API uint32_t mg_version(void) { return (0u << 16) | 4u; }

struct mg_comm_state;

struct mg_ctx {
	mg_comm_state* comm = nullptr;  // NCCL communicator + exchange buffers (mg_comm_init), see mg_comm.inc
	int device = 0;
	uint32_t n = 0;
	cudaStream_t stream = nullptr;
	uint8_t* d_data = nullptr;      // n + 32 bytes, zero padded
	uint32_t* d_occ_start = nullptr;  // 65537
	uint32_t* d_occ = nullptr;        // n
	uint32_t* d_trans = nullptr;
	uint32_t* d_recip = nullptr;
	uint4* d_litq = nullptr;          // literal queues, one per whole 32-byte window (litq_build_kernel)
	Tables tables{};
	int sm_count = 0;
	double index_ms = 0;
	std::vector<mg_anneal*> annealers;  // live chain populations on this context (destroyed with it)
	double last_topk_ms = 0;          // mg_find_topk: device time and candidates of the last call
	unsigned long long last_topk_candidates = 0;
	FindLimits limits{0, 0};          // mg_ctx_set_finder_limits (0, 0 = the reference's unbounded enumeration)
	double last_encode_ms = 0;        // mg_encode_slab*: device time and events of the last call
	unsigned long long last_encode_events = 0;
	double last_decode_ms = 0;        // mg_decode_stream: device time and events of the last call
	unsigned long long last_decode_events = 0;
	double last_optimal_ms = 0;       // mg_anneal_optimal_init: device time and nodes of the last call
	unsigned long long last_optimal_nodes = 0;
	double last_xz_plan_ms = 0;       // mg_encode_slab_xz: device time of the plan walk and of the chunk kernel,
	double last_xz_code_ms = 0;       // chunks and events of the last call
	uint32_t last_xz_chunks = 0;
	unsigned long long last_xz_events = 0;
};

struct DevBuf {
	void* p = nullptr;
	~DevBuf() { if (p) pool_free(p); }
	template <class T> T* as() { return static_cast<T*>(p); }
};

static int dev_alloc(DevBuf& b, size_t bytes)
{
	CU(pool_malloc(&b.p, bytes ? bytes : 16));
	return 0;
}

static int grid_for(size_t items, int threads, int cap)
{
	size_t g = (items + threads - 1) / threads;
	if (g > (size_t)cap) g = cap;
	return g ? (int)g : 1;
}

// Function attributes belong to a device's context: every context creation sets them for its own device (a host
// with one thread per GPU creates eight).
static int set_smem_attrs()
{
	CU(cudaFuncSetAttribute(score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CtaShared)));
	CU(cudaFuncSetAttribute(topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CtaShared)));
	CU(cudaFuncSetAttribute(anneal_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CtaShared)));
	CU(cudaFuncSetAttribute(greedy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CtaShared)));
	CU(cudaFuncSetAttribute(encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(EncodeShared)));
	CU(cudaFuncSetAttribute(encode_chunks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CHUNK_SMEM));
	// the model lives in shared memory: ask for the largest carve-out so that occupancy is set by registers
	CU(cudaFuncSetAttribute(score_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
	CU(cudaFuncSetAttribute(topk_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
	CU(cudaFuncSetAttribute(anneal_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
	CU(cudaFuncSetAttribute(greedy_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
	return 0;
}

// K1: bigram index on the device
static int build_index(mg_ctx* ctx)
{
	const uint32_t n = ctx->n;
	CU(pool_malloc(&ctx->d_occ_start, sizeof(uint32_t) * (INDEX_KEYS + 1)));
	CU(pool_malloc(&ctx->d_occ, sizeof(uint32_t) * (size_t)(n ? n : 1)));
	if (n < 2) {
		CU(cudaMemsetAsync(ctx->d_occ_start, 0, sizeof(uint32_t) * (INDEX_KEYS + 1), ctx->stream));
		return 0;
	}
	const uint32_t total = n - 1;
	// one histogram row per warp; bound the rows to 64 MiB
	uint32_t nwarps = 256;
	uint32_t per_warp = (total + nwarps - 1) / nwarps;
	per_warp = (per_warp + 31) & ~31u;
	if (per_warp < 32) per_warp = 32;
	nwarps = (total + per_warp - 1) / per_warp;
	DevBuf rows, totals;
	if (int rc = dev_alloc(rows, sizeof(uint32_t) * (size_t)nwarps * INDEX_KEYS)) return rc;
	if (int rc = dev_alloc(totals, sizeof(uint32_t) * INDEX_KEYS)) return rc;
	cudaEvent_t e0, e1;
	CU(cudaEventCreate(&e0));
	CU(cudaEventCreate(&e1));
	CU(cudaEventRecord(e0, ctx->stream));
	CU(cudaMemsetAsync(rows.p, 0, sizeof(uint32_t) * (size_t)nwarps * INDEX_KEYS, ctx->stream));
	const int threads = 128;
	const int blocks = (int)((nwarps * 32 + threads - 1) / threads);
	index_count_kernel<<<blocks, threads, 0, ctx->stream>>>(ctx->d_data, n, rows.as<uint32_t>(), per_warp);
	index_prefix_kernel<<<INDEX_KEYS / 256, 256, 0, ctx->stream>>>(rows.as<uint32_t>(), nwarps, totals.as<uint32_t>());
	index_scan_kernel<<<1, 1024, 0, ctx->stream>>>(totals.as<uint32_t>(), ctx->d_occ_start);
	index_scatter_kernel<<<blocks, threads, 0, ctx->stream>>>(ctx->d_data, n, rows.as<uint32_t>(), per_warp,
	                                                          ctx->d_occ_start, ctx->d_occ);
	CU(cudaEventRecord(e1, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	CU(cudaGetLastError());
	float ms = 0;
	cudaEventElapsedTime(&ms, e0, e1);
	ctx->index_ms = ms;
	cudaEventDestroy(e0);
	cudaEventDestroy(e1);
	return 0;
}

extern "C" MG_API int mg_ctx_create(const uint8_t* data, size_t n, LZMAProperties props, int device, mg_ctx** out)
{
	if (!data || !out || n == 0) return fail(MG_EINVAL, "mg_ctx_create: data, out and a non-zero size are required");
	if (props.lc || props.lp || props.pb) return fail(MG_EINVAL, "only lc = lp = pb = 0 is supported (as in the reference)");
	if (n >= 0x7fffff00ull) return fail(MG_EINVAL, "inputs of 2 GiB and more are not supported");
	int count = 0;
	cudaError_t probe = cudaErrorUnknown;
	for (int attempt = 0; attempt < 5; attempt++) {
		// back-to-back processes on one GPU: the driver can answer "unavailable" for a moment while the
		// previous process is still being torn down
		probe = cudaGetDeviceCount(&count);
		if (probe == cudaSuccess && count > 0) break;
		if (probe == cudaErrorNoDevice || probe == cudaErrorInsufficientDriver) break;
		cudaGetLastError();
		usleep(200 * 1000);
	}
	if (probe != cudaSuccess || count == 0)
		return fail(MG_ECUDA, "no CUDA device available (this library has no CPU path): %s", cudaGetErrorString(probe));
	if (device < 0 || device >= count) return fail(MG_EINVAL, "device %d out of range (%d devices)", device, count);
	CU(cudaSetDevice(device));
	mg_ctx* ctx = new (std::nothrow) mg_ctx;
	if (!ctx) return fail(MG_ENOMEM, "out of host memory");
	ctx->device = device;
	ctx->n = (uint32_t)n;
	cudaDeviceProp prop;
	CU(cudaGetDeviceProperties(&prop, device));
	ctx->sm_count = prop.multiProcessorCount;
	int rc = 0;
	do {
		if ((rc = set_smem_attrs())) break;
#define CUB(call)                                                                 \
	if (cudaError_t e_ = (call); e_ != cudaSuccess) {                             \
		rc = fail(MG_ECUDA, "%s: %s", #call, cudaGetErrorString(e_));             \
		break;                                                                    \
	}
		CUB(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
		CUB(pool_malloc(&ctx->d_data, n + 32));
		CUB(cudaMemsetAsync(ctx->d_data + n, 0, 32, ctx->stream));
		CUB(cudaMemcpyAsync(ctx->d_data, data, n, cudaMemcpyHostToDevice, ctx->stream));
		// price table: reference generate_table.py:7-9, -int(log2(i/2048.)*2048); fused with the
		// probability update of src/probability_model.c:5-15 into one transition table
		std::vector<uint32_t> price(2048);
		price[0] = 0;
		for (int i = 1; i < 2048; i++) price[i] = (uint32_t)(-(long)(std::log2((double)i / 2048.0) * 2048.0));
		// sections of 2048 entries indexed by p; entry = stored probability after (p << PROB_SHIFT) | price << 16
		auto step = [&](uint32_t p, uint32_t bit, uint32_t& cost) {
			cost += bit ? price[(2048u - p) & 2047u] : price[p];
			return bit ? p - (p >> 5) : p + ((2048u - p) >> 5);
		};
		std::vector<uint32_t> trans(TRANS_WORDS, 0);
		for (uint32_t p = 1; p < 2048; p++) {
			for (uint32_t bit = 0; bit < 2; bit++) {
				uint32_t cost = 0;
				const uint32_t p1 = step(p, bit, cost);
				trans[bit * 2048 + p] = (p1 << PROB_SHIFT) | (cost << 16);
			}
			// two steps on one slot (literal queues): bits (a, b) in that order
			for (uint32_t ab = 0; ab < 4; ab++) {
				uint32_t cost = 0;
				const uint32_t p2 = step(step(p, ab >> 1, cost), ab & 1, cost);
				trans[(2 + ab) * 2048 + p] = (p2 << PROB_SHIFT) | (cost << 16);
			}
		}
		// probability 0 never occurs in a model: entry 0 of every section is a zero-price fixed point (the spare
		// slots' value, see the slot map in mg_device.cuh)
		std::vector<uint32_t> recip(RECIP_ENTRIES, 0);
		for (uint32_t i = 1; i < RECIP_ENTRIES; i++) recip[i] = 0xffffffffu / i + 1u;
		CUB(pool_malloc(&ctx->d_trans, TRANS_WORDS * sizeof(uint32_t)));
		CUB(pool_malloc(&ctx->d_recip, RECIP_ENTRIES * sizeof(uint32_t)));
		CUB(cudaMemcpyAsync(ctx->d_trans, trans.data(), TRANS_WORDS * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
		CUB(cudaMemcpyAsync(ctx->d_recip, recip.data(), RECIP_ENTRIES * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
		const uint32_t nwin = (uint32_t)(n / 32);
		if (nwin != 0 && !getenv("MEGALANIA_NO_LITQ")) {
			CUB(pool_malloc(&ctx->d_litq, (size_t)nwin * QUEUE_BLOCKS * 32 * sizeof(uint4)));
			litq_build_kernel<<<(nwin + 7) / 8, 256, 0, ctx->stream>>>(ctx->d_data, (uint32_t)n, nwin, ctx->d_litq);
			CUB(cudaGetLastError());
		}
		CUB(cudaStreamSynchronize(ctx->stream));
		ctx->tables.trans = ctx->d_trans;
		ctx->tables.litq = ctx->d_litq;
		ctx->tables.recip = ctx->d_recip;
		rc = build_index(ctx);
#undef CUB
	} while (0);
	if (rc) {
		mg_ctx_destroy(ctx);
		return rc;
	}
	*out = ctx;
	return MG_OK;
}

extern "C" MG_API void mg_ctx_destroy(mg_ctx* ctx)
{
	if (!ctx) return;
	cudaSetDevice(ctx->device);
	mg_comm_destroy(ctx);
	// chain populations hold pointers into the context: they go first (their handles die with it)
	while (!ctx->annealers.empty()) mg_anneal_destroy(ctx->annealers.back());
	if (ctx->stream) cudaStreamSynchronize(ctx->stream);
	pool_free(ctx->d_data);
	pool_free(ctx->d_occ_start);
	pool_free(ctx->d_occ);
	pool_free(ctx->d_trans);
	pool_free(ctx->d_recip);
	pool_free(ctx->d_litq);
	if (ctx->stream) cudaStreamDestroy(ctx->stream);
	delete ctx;
}

extern "C" MG_API size_t mg_ctx_size(const mg_ctx* ctx) { return ctx ? ctx->n : 0; }
extern "C" MG_API int mg_find_topk_stats(const mg_ctx* ctx, double* kernel_ms, uint64_t* candidates)
{
	if (!ctx) return fail(MG_EINVAL, "mg_find_topk_stats: null context");
	if (kernel_ms) *kernel_ms = ctx->last_topk_ms;
	if (candidates) *candidates = ctx->last_topk_candidates;
	return MG_OK;
}
extern "C" MG_API int mg_ctx_device(const mg_ctx* ctx) { return ctx ? ctx->device : -1; }
extern "C" MG_API int mg_ctx_set_finder_limits(mg_ctx* ctx, size_t window, uint32_t max_occurrences)
{
	if (!ctx) return fail(MG_EINVAL, "mg_ctx_set_finder_limits: null context");
	ctx->limits.window = window > 0xffffffffull ? 0xffffffffu : (uint32_t)window;
	ctx->limits.max_occ = max_occurrences;
	return MG_OK;
}
extern "C" MG_API uint32_t mg_ctx_full_wave(const mg_ctx* ctx) { return ctx ? (uint32_t)ctx->sm_count * (uint32_t)WARPS_PER_CTA : 0u; }
extern "C" MG_API uint32_t mg_ctx_sm_clock_khz(const mg_ctx* ctx)
{
	int khz = 0;
	if (!ctx || cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device) != cudaSuccess || khz <= 0) return 0u;
	return (uint32_t)khz;
}
extern "C" MG_API int mg_encode_stats(const mg_ctx* ctx, double* kernel_ms, uint64_t* events)
{
	if (!ctx) return fail(MG_EINVAL, "mg_encode_stats: null context");
	if (kernel_ms) *kernel_ms = ctx->last_encode_ms;
	if (events) *events = ctx->last_encode_events;
	return MG_OK;
}

extern "C" MG_API int mg_debug_index(mg_ctx* ctx, uint32_t* occ_start, uint32_t* occ)
{
	if (!ctx || !occ_start || !occ) return fail(MG_EINVAL, "mg_debug_index: null argument");
	CU(cudaSetDevice(ctx->device));
	CU(cudaMemcpyAsync(occ_start, ctx->d_occ_start, sizeof(uint32_t) * (INDEX_KEYS + 1), cudaMemcpyDeviceToHost, ctx->stream));
	if (ctx->n > 1) CU(cudaMemcpyAsync(occ, ctx->d_occ, sizeof(uint32_t) * (size_t)(ctx->n - 1), cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	return MG_OK;
}

// Upload `count` host packets (12 B each) and pack them into dst (device, u64 each).
static int upload_packed(mg_ctx* ctx, const LZMAPacket* host, size_t count, uint64_t* dst)
{
	static_assert(sizeof(LZMAPacket) == 12, "LZMAPacket must keep the reference layout");
	const size_t chunk = (size_t)8 << 20;  // packets per staging round
	DevBuf raw;
	const size_t stage = count < chunk ? count : chunk;
	if (int rc = dev_alloc(raw, stage * 12)) return rc;
	for (size_t off = 0; off < count; off += stage) {
		const size_t c = count - off < stage ? count - off : stage;
		CU(cudaMemcpyAsync(raw.p, host + off, c * 12, cudaMemcpyHostToDevice, ctx->stream));
		pack_kernel<<<grid_for(c, 256, ctx->sm_count * 8), 256, 0, ctx->stream>>>(raw.as<uint32_t>(), dst + off, c);
		CU(cudaStreamSynchronize(ctx->stream));
	}
	CU(cudaGetLastError());
	return 0;
}

static int download_unpacked(mg_ctx* ctx, const uint64_t* src, size_t count, LZMAPacket* host)
{
	DevBuf raw;
	if (int rc = dev_alloc(raw, count * 12)) return rc;
	unpack_kernel<<<grid_for(count, 256, ctx->sm_count * 8), 256, 0, ctx->stream>>>(src, raw.as<uint32_t>(), count);
	CU(cudaGetLastError());
	// the host struct has padding bytes; give them a defined value
	CU(cudaMemcpyAsync(host, raw.p, count * 12, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	return 0;
}

static const char* walk_error(uint32_t err)
{
	if (err & ERR_BAD_PACKET) return "slab holds a packet that cannot be coded at its position";
	if (err & ERR_NOT_BOUNDARY) return "position is not a live packet boundary of the slab";
	if (err & ERR_OUTPUT_FULL) return "output buffer too small";
	return "unknown";
}

static uint32_t default_stride(uint32_t n)
{
	// ~256 checkpoints per slab, never closer than 512 bytes (a packet spans at most 273)
	uint32_t s = n / 256;
	if (s < 512) s = 512;
	return (s + 31) & ~31u;
}

// ---- cost -------------------------------------------------------------------------------------------
static int score_device(mg_ctx* ctx, const uint64_t* d_slabs, uint32_t nslabs, uint32_t stop_pos, uint64_t* d_cost,
                        uint32_t* d_count, uint32_t* d_err, Record* ck, uint32_t* ck_pos, CkMeta* ck_meta,
                        uint32_t stride, uint32_t nslots, Record* final_model)
{
	ScoreArgs a;
	a.data = ctx->d_data;
	a.n = ctx->n;
	a.slabs = d_slabs;
	a.nslabs = nslabs;
	a.stop_pos = stop_pos;
	a.out_cost = d_cost;
	a.out_count = d_count;
	a.out_err = d_err;
	a.ck = ck;
	a.ck_pos = ck_pos;
	a.ck_meta = ck_meta;
	a.stride = stride;
	a.nslots = nslots ? nslots : 1;
	a.ck_chain_stride = a.nslots - 1;
	a.final_model = final_model;
	a.tables = ctx->tables;
	const int blocks = (int)((nslabs + WARPS_PER_CTA - 1) / WARPS_PER_CTA);
	score_kernel<<<blocks, CTA_THREADS, sizeof(CtaShared), ctx->stream>>>(a);
	CU(cudaGetLastError());
	return 0;
}

extern "C" MG_API int mg_score_slabs(mg_ctx* ctx, const LZMAPacket* slabs, size_t nslabs, uint64_t* out_cost)
{
	if (!ctx || !slabs || !out_cost) return fail(MG_EINVAL, "mg_score_slabs: null argument");
	if (nslabs == 0) return MG_OK;
	CU(cudaSetDevice(ctx->device));
	const size_t n = ctx->n;
	// batches bounded to ~2 GiB of packed slabs
	size_t batch = ((size_t)2 << 30) / (n * 8);
	if (batch < 1) batch = 1;
	if (batch > nslabs) batch = nslabs;
	DevBuf packed, cost, err;
	if (int rc = dev_alloc(packed, batch * n * 8)) return rc;
	if (int rc = dev_alloc(cost, batch * 8)) return rc;
	if (int rc = dev_alloc(err, batch * 4)) return rc;
	std::vector<uint32_t> herr(batch);
	for (size_t off = 0; off < nslabs; off += batch) {
		const size_t c = nslabs - off < batch ? nslabs - off : batch;
		if (int rc = upload_packed(ctx, slabs + off * n, c * n, packed.as<uint64_t>())) return rc;
		if (int rc = score_device(ctx, packed.as<uint64_t>(), (uint32_t)c, ctx->n, cost.as<uint64_t>(), nullptr,
		                          err.as<uint32_t>(), nullptr, nullptr, nullptr, default_stride(ctx->n), 1, nullptr))
			return rc;
		CU(cudaMemcpyAsync(out_cost + off, cost.p, c * 8, cudaMemcpyDeviceToHost, ctx->stream));
		CU(cudaMemcpyAsync(herr.data(), err.p, c * 4, cudaMemcpyDeviceToHost, ctx->stream));
		CU(cudaStreamSynchronize(ctx->stream));
		for (size_t i = 0; i < c; i++)
			if (herr[i]) return fail(MG_ESLAB, "slab %zu: %s", off + i, walk_error(herr[i]));
	}
	return MG_OK;
}

// Reference-layout index of a device slot (src/lzma_state.h:15-55)
static void export_model(const Record& r, mg_model_dump* out)
{
	for (int i = 0; i < 2615; i++) out->probs[i] = 1024;
	auto put = [&](uint32_t ref_index, uint32_t slot) { out->probs[ref_index] = (uint16_t)(r.probs[slot] >> PROB_SHIFT); };
	for (uint32_t node = 0; node < 768; node++)
		if (node & 0xff) put(node, lit_slot(node));  // node 0 of each tree is never coded
	const uint32_t ref_len[2] = {768, 768 + 514};
	const uint32_t dev_len[2] = {S_LEN, S_REPLEN};
	for (int t = 0; t < 2; t++) {
		put(ref_len[t] + 0, dev_len[t] + 0);
		put(ref_len[t] + 1, dev_len[t] + 1);
		for (uint32_t i = 0; i < 8; i++) {
			put(ref_len[t] + 2 + i, dev_len[t] + LEN_LOW + i);         // low_coder[0][i]
			put(ref_len[t] + 2 + 128 + i, dev_len[t] + LEN_MID + i);   // mid_coder[0][i]
		}
		for (uint32_t i = 0; i < 256; i++) put(ref_len[t] + 2 + 256 + i, dev_len[t] + LEN_HIGH + i);
	}
	const uint32_t ref_dist = 768 + 2 * 514;
	for (uint32_t i = 0; i < 256 + 16 + 115; i++) put(ref_dist + i, S_POSSLOT + i);
	const uint32_t ref_ctx = ref_dist + 387;
	for (uint32_t s = 0; s < 12; s++) {
		put(ref_ctx + (s << 4), S_ISMATCH + s);
		put(ref_ctx + 192 + s, S_ISREP + s);
		put(ref_ctx + 204 + s, S_ISREPG0 + s);
		put(ref_ctx + 216 + s, S_ISREPG1 + s);
		put(ref_ctx + 228 + s, S_ISREPG2 + s);
		put(ref_ctx + 240 + (s << 4), S_ISREP0LONG + s);
	}
	out->ctx_state = (uint8_t)r.ctx;
	for (int i = 0; i < 4; i++) out->dists[i] = r.rep[i];
	out->position = r.pos;
	out->cost = r.cost;
}

extern "C" MG_API int mg_debug_model_after_prefix(mg_ctx* ctx, const LZMAPacket* slab, size_t stop, mg_model_dump* out)
{
	if (!ctx || !slab || !out || stop > ctx->n) return fail(MG_EINVAL, "mg_debug_model_after_prefix: bad argument");
	CU(cudaSetDevice(ctx->device));
	DevBuf packed, cost, err, model;
	if (int rc = dev_alloc(packed, (size_t)ctx->n * 8)) return rc;
	if (int rc = dev_alloc(cost, 8)) return rc;
	if (int rc = dev_alloc(err, 4)) return rc;
	if (int rc = dev_alloc(model, sizeof(Record))) return rc;
	if (int rc = upload_packed(ctx, slab, ctx->n, packed.as<uint64_t>())) return rc;
	if (int rc = score_device(ctx, packed.as<uint64_t>(), 1, (uint32_t)stop, cost.as<uint64_t>(), nullptr, err.as<uint32_t>(),
	                          nullptr, nullptr, nullptr, default_stride(ctx->n), 1, model.as<Record>()))
		return rc;
	Record r;
	uint32_t herr = 0;
	CU(cudaMemcpyAsync(&r, model.p, sizeof(Record), cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaMemcpyAsync(&herr, err.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	if (herr) return fail(MG_ESLAB, "%s", walk_error(herr));
	memset(out, 0, sizeof(*out));
	export_model(r, out);
	return MG_OK;
}

// ---- top-k ---------------------------------------------------------------------------------------------
extern "C" MG_API int mg_find_topk(mg_ctx* ctx, const LZMAPacket* slab, int state_mode, const uint64_t* positions,
                            size_t npos, int k, LZMAPacket* out_pops, uint32_t* out_prices, int32_t* out_counts)
{
	if (!ctx || !slab || !positions || !out_pops || !out_counts) return fail(MG_EINVAL, "mg_find_topk: null argument");
	if (k < 1 || k > MAX_K) return fail(MG_EINVAL, "mg_find_topk: k must be in 1..%d", MAX_K);
	if (state_mode != 0 && state_mode != 1) return fail(MG_EINVAL, "mg_find_topk: state_mode must be 0 or 1");
	if (npos == 0) return MG_OK;
	if (npos > 0xffffffffull / (size_t)k) return fail(MG_EINVAL, "mg_find_topk: too many queries");
	CU(cudaSetDevice(ctx->device));
	const uint32_t n = ctx->n;
	std::vector<uint32_t> pos32(npos);
	for (size_t i = 0; i < npos; i++) {
		if (positions[i] >= n) return fail(MG_EINVAL, "mg_find_topk: position %llu outside the input", (unsigned long long)positions[i]);
		pos32[i] = (uint32_t)positions[i];
	}
	const uint32_t stride = default_stride(n);
	const uint32_t nslots = (n + stride - 1) / stride;
	DevBuf packed, dpos, opk, oprice, ocount, oerr, cost, serr, ck, ckpos, cand;
	if (int rc = dev_alloc(packed, (size_t)n * 8)) return rc;
	if (int rc = dev_alloc(dpos, npos * 4)) return rc;
	if (int rc = dev_alloc(opk, npos * k * 8)) return rc;
	if (int rc = dev_alloc(oprice, npos * k * 4)) return rc;
	if (int rc = dev_alloc(ocount, npos * 4)) return rc;
	if (int rc = dev_alloc(oerr, npos * 4)) return rc;
	if (int rc = dev_alloc(cand, 8)) return rc;
	if (int rc = upload_packed(ctx, slab, n, packed.as<uint64_t>())) return rc;
	CU(cudaMemcpyAsync(dpos.p, pos32.data(), npos * 4, cudaMemcpyHostToDevice, ctx->stream));
	CU(cudaMemsetAsync(cand.p, 0, 8, ctx->stream));
	if (state_mode == 1) {
		if (int rc = dev_alloc(cost, 8)) return rc;
		if (int rc = dev_alloc(serr, 4)) return rc;
		if (int rc = dev_alloc(ck, sizeof(Record) * (size_t)nslots)) return rc;
		if (int rc = dev_alloc(ckpos, 4 * (size_t)nslots)) return rc;
		if (int rc = score_device(ctx, packed.as<uint64_t>(), 1, n, cost.as<uint64_t>(), nullptr, serr.as<uint32_t>(),
		                          ck.as<Record>(), ckpos.as<uint32_t>(), nullptr, stride, nslots, nullptr))
			return rc;
		uint32_t herr = 0;
		CU(cudaMemcpyAsync(&herr, serr.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
		CU(cudaStreamSynchronize(ctx->stream));
		if (herr) return fail(MG_ESLAB, "mg_find_topk: %s", walk_error(herr));
	}
	TopkArgs a;
	a.data = ctx->d_data;
	a.n = n;
	a.occ_start = ctx->d_occ_start;
	a.occ = ctx->d_occ;
	a.slab = packed.as<uint64_t>();
	a.state_mode = state_mode;
	a.positions = dpos.as<uint32_t>();
	a.npos = (uint32_t)npos;
	a.k = (uint32_t)k;
	a.ck = ck.as<Record>();
	a.ck_pos = ckpos.as<uint32_t>();
	a.nslots = nslots;
	a.stride = stride;
	a.out_pk = opk.as<uint64_t>();
	a.out_price = oprice.as<uint32_t>();
	a.out_count = ocount.as<int32_t>();
	a.out_err = oerr.as<uint32_t>();
	a.candidates = cand.as<unsigned long long>();
	a.limits = ctx->limits;
	a.tables = ctx->tables;
	size_t blocks = (npos + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
	const size_t cap = (size_t)ctx->sm_count * 4 * 8;
	if (blocks > cap) blocks = cap;
	cudaEvent_t t0, t1;
	CU(cudaEventCreate(&t0));
	CU(cudaEventCreate(&t1));
	CU(cudaEventRecord(t0, ctx->stream));
	topk_kernel<<<(int)blocks, CTA_THREADS, sizeof(CtaShared), ctx->stream>>>(a);
	CU(cudaEventRecord(t1, ctx->stream));
	CU(cudaGetLastError());
	std::vector<uint64_t> hpk(npos * k);
	std::vector<uint32_t> hprice(npos * k), herr(npos);
	CU(cudaMemcpyAsync(hpk.data(), opk.p, npos * k * 8, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaMemcpyAsync(hprice.data(), oprice.p, npos * k * 4, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaMemcpyAsync(out_counts, ocount.p, npos * 4, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaMemcpyAsync(herr.data(), oerr.p, npos * 4, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaMemcpyAsync(&ctx->last_topk_candidates, cand.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	{
		float ms = 0;
		cudaEventElapsedTime(&ms, t0, t1);
		ctx->last_topk_ms = ms;
		cudaEventDestroy(t0);
		cudaEventDestroy(t1);
	}
	for (size_t q = 0; q < npos; q++) {
		if (herr[q]) return fail(MG_ESLAB, "mg_find_topk: query %zu (position %u): %s", q, pos32[q], walk_error(herr[q]));
		for (int i = 0; i < k; i++) {
			LZMAPacket p;
			memset(&p, 0, sizeof(p));
			uint32_t price = 0;
			if (i < out_counts[q]) {
				const uint64_t v = hpk[q * k + i];
				p.type = (uint8_t)pk_type(v);
				p.dist = pk_dist(v);
				p.len = (uint16_t)pk_len(v);
				price = hprice[q * k + i];
			}
			out_pops[q * k + i] = p;
			if (out_prices) out_prices[q * k + i] = price;
		}
	}
	return MG_OK;
}

// ---- bytes ---------------------------------------------------------------------------------------------
static int encode_to_host(mg_ctx* ctx, const LZMAPacket* slab, std::vector<uint8_t>& payload)
{
	const uint32_t n = ctx->n;
	const uint32_t cap = n + n / 2 + 4096;
	DevBuf packed, out, len, err;
	if (int rc = dev_alloc(packed, (size_t)n * 8)) return rc;
	if (int rc = dev_alloc(out, cap)) return rc;
	if (int rc = dev_alloc(len, 32)) return rc;
	if (int rc = dev_alloc(err, 4)) return rc;
	if (int rc = upload_packed(ctx, slab, n, packed.as<uint64_t>())) return rc;
	EncodeArgs a;
	a.data = ctx->d_data;
	a.n = n;
	a.slab = packed.as<uint64_t>();
	a.out = out.as<uint8_t>();
	a.cap = cap;
	a.out_len = len.as<uint32_t>();
	a.out_err = err.as<uint32_t>();
	a.out_events = len.as<uint32_t>() + 1;
	const bool debug_wait = getenv("MEGALANIA_ENCODE_DEBUG") != nullptr;
	a.out_wait = debug_wait ? reinterpret_cast<unsigned long long*>(len.as<uint32_t>() + 2) : nullptr;
	a.tables = ctx->tables;
	cudaEvent_t t0, t1;
	CU(cudaEventCreate(&t0));
	CU(cudaEventCreate(&t1));
	CU(cudaEventRecord(t0, ctx->stream));
	encode_kernel<<<1, 96, sizeof(EncodeShared), ctx->stream>>>(a);
	CU(cudaEventRecord(t1, ctx->stream));
	CU(cudaGetLastError());
	uint32_t hlen2[8] = {0, 0, 0, 0, 0, 0, 0, 0}, herr = 0;
	CU(cudaMemcpyAsync(hlen2, len.p, 32, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaMemcpyAsync(&herr, err.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	{
		float ms = 0;
		cudaEventElapsedTime(&ms, t0, t1);
		ctx->last_encode_ms = ms;
		ctx->last_encode_events = hlen2[1];
		if (debug_wait) {
			unsigned long long w[3];
			memcpy(w, hlen2 + 2, sizeof(w));
			fprintf(stderr, "mg_encode_slab: %.2f ms, %u events; clocks waiting: producer %llu, range %llu, low %llu\n", ms, hlen2[1], w[0], w[1], w[2]);
		}
		cudaEventDestroy(t0);
		cudaEventDestroy(t1);
	}
	const uint32_t hlen = hlen2[0];
	if (herr) return fail(MG_ESLAB, "mg_encode_slab: %s", walk_error(herr));
	payload.resize(hlen);
	CU(cudaMemcpyAsync(payload.data(), out.p, hlen, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	return 0;
}

// src/lzma_header_encoder.c:5-21: props byte, dict size 0x400000 LE, size as 8 bytes LE
// (the reference widens htole32(size), so the high word is zero)
static void make_header(const mg_ctx* ctx, uint8_t hdr[13])
{
	hdr[0] = 0;
	// the reference always writes 4 MiB (its todo: "peg dict size to data size"), which makes any match
	// farther than 4 MiB undecodable; same bytes up to 4 MiB, the next power of two above it (SURVEY 8(f) #2)
	uint32_t dict = 0x400000;
	while (dict < ctx->n && dict < 0x80000000u) dict <<= 1;
	for (int i = 0; i < 4; i++) hdr[1 + i] = (uint8_t)(dict >> (8 * i));
	const uint64_t size = ctx->n;
	for (int i = 0; i < 8; i++) hdr[5 + i] = (uint8_t)(size >> (8 * i));
}

extern "C" MG_API int mg_encode_slab(mg_ctx* ctx, const LZMAPacket* slab, OutputInterface* out)
{
	if (!ctx || !slab || !out || !out->write) return fail(MG_EINVAL, "mg_encode_slab: null argument");
	CU(cudaSetDevice(ctx->device));
	std::vector<uint8_t> payload;
	if (int rc = encode_to_host(ctx, slab, payload)) return rc;
	uint8_t hdr[13];
	make_header(ctx, hdr);
	bool ok = out->write(out, hdr, 1) && out->write(out, hdr + 1, 4) && out->write(out, hdr + 5, 8);
	if (ok && !payload.empty()) ok = out->write(out, payload.data(), payload.size());
	if (!ok) return fail(MG_EOUTPUT, "mg_encode_slab: OutputInterface.write failed");
	return MG_OK;
}

extern "C" MG_API int mg_encode_slab_buffer(mg_ctx* ctx, const LZMAPacket* slab, uint8_t* out, size_t cap, size_t* out_len)
{
	if (!ctx || !slab || !out_len || (!out && cap)) return fail(MG_EINVAL, "mg_encode_slab_buffer: null argument");
	CU(cudaSetDevice(ctx->device));
	std::vector<uint8_t> payload;
	if (int rc = encode_to_host(ctx, slab, payload)) return rc;
	*out_len = 13 + payload.size();
	if (*out_len > cap) return fail(MG_EINVAL, "mg_encode_slab_buffer: need %zu bytes, have %zu", *out_len, cap);
	make_header(ctx, out);
	memcpy(out + 13, payload.data(), payload.size());
	return MG_OK;
}

// ---- .xz: LZMA2 chunks coded side by side ---------------------------------------------------------------------
constexpr uint32_t XZ_GRANULE = 4096;          // the plan walk's checkpoint stride: cut candidates every 4 KiB
constexpr uint32_t XZ_CHUNK_DEFAULT = 61440;   // liblzma's own target for an LZMA2 chunk's coded bytes
constexpr uint32_t XZ_CHUNK_MIN = 256;
constexpr uint32_t LZMA2_MAX_U = 1u << 21;     // an LZMA2 chunk holds at most 2 MiB of input ...
constexpr uint32_t LZMA2_MAX_C = 1u << 16;     // ... and at most 64 KiB of coded bytes

static uint32_t crc32_update(uint32_t crc, const uint8_t* p, size_t len)
{
	static uint32_t table[256];
	static bool ready = false;
	if (!ready) {
		for (uint32_t i = 0; i < 256; i++) {
			uint32_t c = i;
			for (int k = 0; k < 8; k++) c = (c >> 1) ^ (0xEDB88320u & (0u - (c & 1u)));
			table[i] = c;
		}
		ready = true;
	}
	crc = ~crc;
	for (size_t i = 0; i < len; i++) crc = table[(crc ^ p[i]) & 0xff] ^ (crc >> 8);
	return ~crc;
}

static uint64_t crc64_update(uint64_t crc, const uint8_t* p, size_t len)
{
	static uint64_t table[256];
	static bool ready = false;
	if (!ready) {
		for (uint64_t i = 0; i < 256; i++) {
			uint64_t c = i;
			for (int k = 0; k < 8; k++) c = (c >> 1) ^ (0xC96C5795D7870F42ull & (0ull - (c & 1ull)));
			table[i] = c;
		}
		ready = true;
	}
	crc = ~crc;
	for (size_t i = 0; i < len; i++) crc = table[(crc ^ p[i]) & 0xff] ^ (crc >> 8);
	return ~crc;
}

static void put_le(std::vector<uint8_t>& v, uint64_t x, int bytes)
{
	for (int i = 0; i < bytes; i++) v.push_back((uint8_t)(x >> (8 * i)));
}

static void put_varint(std::vector<uint8_t>& v, uint64_t x)
{
	while (x >= 0x80) {
		v.push_back((uint8_t)(x | 0x80));
		x >>= 7;
	}
	v.push_back((uint8_t)x);
}

static void pad4(std::vector<uint8_t>& v, size_t from)
{
	while ((v.size() - from) & 3) v.push_back(0);
}

// The smallest LZMA2 dictionary-size byte whose size, (2 | (b & 1)) << (b / 2 + 11), is at least max(n, 4 KiB).
static uint8_t lzma2_dict_byte(uint32_t n)
{
	uint8_t b = 0;
	while (b < 40 && ((uint64_t)(2u | (b & 1u)) << (b / 2 + 11)) < n) b++;
	return b;
}

// One .xz stream: one block, LZMA2 (lc = lp = pb = 0), check CRC64.  chunk c holds the input [bounds[c],
// bounds[c + 1]) range-coded in payload[c].
static std::vector<uint8_t> xz_stream(const uint8_t* input, uint32_t n, const std::vector<uint32_t>& bounds,
                                      const std::vector<std::vector<uint8_t>>& payload)
{
	std::vector<uint8_t> v;
	const uint8_t magic[6] = {0xFD, '7', 'z', 'X', 'Z', 0x00}, flags[2] = {0x00, 0x04};  // flags: check = CRC64
	v.insert(v.end(), magic, magic + 6);
	v.insert(v.end(), flags, flags + 2);
	put_le(v, crc32_update(0, flags, 2), 4);
	// block header: size, flags (one filter, no size fields), LZMA2 with its dictionary byte, padding, CRC32
	const size_t block = v.size();
	v.push_back(0);
	v.push_back(0x00);
	v.push_back(0x21);
	v.push_back(0x01);
	v.push_back(lzma2_dict_byte(n));
	pad4(v, block);
	v[block] = (uint8_t)((v.size() + 4 - block) / 4 - 1);
	put_le(v, crc32_update(0, v.data() + block, v.size() - block), 4);
	// LZMA2 chunks: the first resets the dictionary and state and sets the properties (byte 0: lc = lp = pb = 0), the
	// rest keep everything and restart only the range coder
	for (size_t c = 0; c + 1 < bounds.size(); c++) {
		const uint32_t u = bounds[c + 1] - bounds[c] - 1, z = (uint32_t)payload[c].size() - 1;
		v.push_back((uint8_t)((c == 0 ? 0xE0u : 0x80u) | (u >> 16)));
		v.push_back((uint8_t)(u >> 8));
		v.push_back((uint8_t)u);
		v.push_back((uint8_t)(z >> 8));
		v.push_back((uint8_t)z);
		if (c == 0) v.push_back(0x00);
		v.insert(v.end(), payload[c].begin(), payload[c].end());
	}
	v.push_back(0x00);  // end of the LZMA2 data
	const uint64_t unpadded = v.size() - block + 8;
	pad4(v, block);
	put_le(v, crc64_update(0, input, n), 8);
	// index: one record (unpadded block size, input size), padding, CRC32
	const size_t index = v.size();
	v.push_back(0x00);
	put_varint(v, 1);
	put_varint(v, unpadded);
	put_varint(v, n);
	pad4(v, index);
	put_le(v, crc32_update(0, v.data() + index, v.size() - index), 4);
	const uint32_t backward = (uint32_t)((v.size() - index) / 4 - 1);
	// stream footer: CRC32 of (backward size, flags), backward size, flags, "YZ"
	uint8_t tail[6];
	for (int i = 0; i < 4; i++) tail[i] = (uint8_t)(backward >> (8 * i));
	tail[4] = flags[0];
	tail[5] = flags[1];
	put_le(v, crc32_update(0, tail, 6), 4);
	v.insert(v.end(), tail, tail + 6);
	v.push_back('Y');
	v.push_back('Z');
	return v;
}

extern "C" MG_API int mg_encode_slab_xz(mg_ctx* ctx, const LZMAPacket* slab, uint32_t chunk_bytes, OutputInterface* out)
{
	if (!ctx || !slab || !out || !out->write) return fail(MG_EINVAL, "mg_encode_slab_xz: null argument");
	if (chunk_bytes == 0) chunk_bytes = XZ_CHUNK_DEFAULT;
	if (chunk_bytes < XZ_CHUNK_MIN || chunk_bytes > XZ_CHUNK_DEFAULT)
		return fail(MG_EINVAL, "mg_encode_slab_xz: chunk_bytes %u is outside %u..%u", chunk_bytes, XZ_CHUNK_MIN, XZ_CHUNK_DEFAULT);
	CU(cudaSetDevice(ctx->device));
	const uint32_t n = ctx->n;
	// plan walk: one score_kernel pass with a checkpoint at the first packet boundary at or after each multiple of
	// the granule (a packet is at most 273 bytes, so none is skipped; one that falls on n is not written)
	const uint32_t nrec = (n - 1) / XZ_GRANULE;
	DevBuf packed, ck, meta, cost, err;
	if (int rc = dev_alloc(packed, (size_t)n * 8)) return rc;
	if (int rc = dev_alloc(ck, (size_t)(nrec ? nrec : 1) * sizeof(Record))) return rc;
	if (int rc = dev_alloc(meta, (size_t)(nrec ? nrec : 1) * sizeof(CkMeta))) return rc;
	if (int rc = dev_alloc(cost, 8)) return rc;
	if (int rc = dev_alloc(err, 4)) return rc;
	if (int rc = upload_packed(ctx, slab, n, packed.as<uint64_t>())) return rc;
	CU(cudaMemsetAsync(meta.p, 0xff, (size_t)(nrec ? nrec : 1) * sizeof(CkMeta), ctx->stream));
	cudaEvent_t ev[4];
	for (auto& e : ev) CU(cudaEventCreate(&e));
	struct Events {
		cudaEvent_t* e;
		~Events() { for (int i = 0; i < 4; i++) cudaEventDestroy(e[i]); }
	} events_guard{ev};
	CU(cudaEventRecord(ev[0], ctx->stream));
	if (int rc = score_device(ctx, packed.as<uint64_t>(), 1, n, cost.as<uint64_t>(), nullptr, err.as<uint32_t>(),
	                          nrec ? ck.as<Record>() : nullptr, nullptr, meta.as<CkMeta>(), XZ_GRANULE, nrec + 1, nullptr))
		return rc;
	CU(cudaEventRecord(ev[1], ctx->stream));
	std::vector<CkMeta> hmeta(nrec);
	uint64_t total = 0;
	uint32_t herr = 0;
	if (nrec) CU(cudaMemcpyAsync(hmeta.data(), meta.p, nrec * sizeof(CkMeta), cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaMemcpyAsync(&total, cost.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaMemcpyAsync(&herr, err.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	if (herr) return fail(MG_ESLAB, "mg_encode_slab_xz: %s", walk_error(herr));
	float plan_ms = 0;
	cudaEventElapsedTime(&plan_ms, ev[0], ev[1]);

	// cut candidates: the checkpoints and n, with the cost of everything before them
	struct Cut {
		uint32_t pos, rec;
		uint64_t cost;
	};
	std::vector<Cut> cuts;
	cuts.push_back({0, NO_RECORD, 0});
	uint64_t acc = 0;
	for (uint32_t i = 0; i < nrec && hmeta[i].pos != 0xffffffffu; i++) {
		acc += hmeta[i].dcost;
		cuts.push_back({hmeta[i].pos, i, acc});
	}
	cuts.push_back({n, NO_RECORD, total});
	// chunk plan: from s, the farthest candidate e with cost(s, e) <= chunk_bytes * 8 bits and e - s <= 2 MiB, or the
	// nearest one when none qualifies (costs only grow with e, so the qualifying candidates are the first ones)
	const uint64_t budget = (uint64_t)chunk_bytes * 8 * 2048;
	std::vector<uint32_t> bounds, start_rec;
	for (size_t s = 0; s + 1 < cuts.size();) {
		size_t e = s + 1;
		while (e + 1 < cuts.size() && cuts[e + 1].cost - cuts[s].cost <= budget && cuts[e + 1].pos - cuts[s].pos <= LZMA2_MAX_U) e++;
		bounds.push_back(cuts[s].pos);
		start_rec.push_back(cuts[s].rec);
		s = e;
	}
	bounds.push_back(n);
	const uint32_t chunks = (uint32_t)start_rec.size();

	// the chunks, one CTA each; a slot of 64 KiB per chunk (the coder counts what it could not store)
	DevBuf dbounds, drec, dout, dres;
	if (int rc = dev_alloc(dbounds, bounds.size() * 4)) return rc;
	if (int rc = dev_alloc(drec, (size_t)chunks * 4)) return rc;
	if (int rc = dev_alloc(dout, (size_t)chunks * LZMA2_MAX_C)) return rc;
	if (int rc = dev_alloc(dres, (size_t)chunks * 12)) return rc;
	CU(cudaMemcpyAsync(dbounds.p, bounds.data(), bounds.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
	CU(cudaMemcpyAsync(drec.p, start_rec.data(), (size_t)chunks * 4, cudaMemcpyHostToDevice, ctx->stream));
	ChunkArgs a;
	a.enc.data = ctx->d_data;
	a.enc.n = n;
	a.enc.slab = packed.as<uint64_t>();
	a.enc.out = dout.as<uint8_t>();
	a.enc.cap = LZMA2_MAX_C;
	a.enc.out_len = dres.as<uint32_t>();
	a.enc.out_err = dres.as<uint32_t>() + chunks;
	a.enc.out_events = dres.as<uint32_t>() + 2 * (size_t)chunks;
	a.enc.out_wait = nullptr;
	a.enc.tables = ctx->tables;
	a.ck = ck.as<Record>();
	a.bounds = dbounds.as<uint32_t>();
	a.start_rec = drec.as<uint32_t>();
	CU(cudaEventRecord(ev[2], ctx->stream));
	encode_chunks_kernel<<<chunks, 96, CHUNK_SMEM, ctx->stream>>>(a);
	CU(cudaEventRecord(ev[3], ctx->stream));
	CU(cudaGetLastError());
	std::vector<uint32_t> res((size_t)chunks * 3);
	CU(cudaMemcpyAsync(res.data(), dres.p, res.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	float code_ms = 0;
	cudaEventElapsedTime(&code_ms, ev[2], ev[3]);
	unsigned long long events = 0;
	for (uint32_t c = 0; c < chunks; c++) events += res[2 * (size_t)chunks + c];
	ctx->last_xz_plan_ms = plan_ms;
	ctx->last_xz_code_ms = code_ms;
	ctx->last_xz_chunks = chunks;
	ctx->last_xz_events = events;
	for (uint32_t c = 0; c < chunks; c++) {
		const uint32_t len = res[c], e = res[(size_t)chunks + c];
		if (e & ERR_BAD_PACKET) return fail(MG_ESLAB, "mg_encode_slab_xz: chunk %u: %s", c, walk_error(e));
		if (len > LZMA2_MAX_C || e)
			return fail(MG_ESLAB, "mg_encode_slab_xz: chunk %u (bytes %u..%u) codes to %u bytes, more than the %u an LZMA2 chunk holds",
			            c, bounds[c], bounds[c + 1], len, LZMA2_MAX_C);
	}
	std::vector<std::vector<uint8_t>> payload(chunks);
	for (uint32_t c = 0; c < chunks; c++) {
		payload[c].resize(res[c]);
		CU(cudaMemcpyAsync(payload[c].data(), dout.as<uint8_t>() + (size_t)c * LZMA2_MAX_C, res[c], cudaMemcpyDeviceToHost, ctx->stream));
	}
	// the block's check is the CRC64 of the input; the context keeps it on the device only
	std::vector<uint8_t> input(n);
	CU(cudaMemcpyAsync(input.data(), ctx->d_data, n, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	const std::vector<uint8_t> stream = xz_stream(input.data(), n, bounds, payload);
	if (!out->write(out, stream.data(), stream.size())) return fail(MG_EOUTPUT, "mg_encode_slab_xz: OutputInterface.write failed");
	return MG_OK;
}

extern "C" MG_API int mg_encode_xz_stats(const mg_ctx* ctx, double* plan_ms, double* code_ms, uint32_t* chunks, uint64_t* events)
{
	if (!ctx) return fail(MG_EINVAL, "mg_encode_xz_stats: null context");
	if (plan_ms) *plan_ms = ctx->last_xz_plan_ms;
	if (code_ms) *code_ms = ctx->last_xz_code_ms;
	if (chunks) *chunks = ctx->last_xz_chunks;
	if (events) *events = ctx->last_xz_events;
	return MG_OK;
}

// ---- stream -> slab ------------------------------------------------------------------------------------
static const char* decode_error(uint32_t err)
{
	switch (err) {
	case DEC_FIRST_BYTE: return "the range coder's first byte is not 0";
	case DEC_LITERAL: return "a literal differs from the input";
	case DEC_SOURCE: return "a match or rep reaches before position 0";
	case DEC_PAST_END: return "a packet runs past the end of the input";
	case DEC_COPY: return "a match or rep copies bytes that differ from the input";
	case DEC_MARKER: return "an end marker where none may stand";
	case DEC_SHORT: return "the stream ends before the input does";
	case DEC_TRAILING: return "bytes follow the last packet";
	case DEC_CODE: return "the range decoder does not end at code 0";
	default: return "unknown";
	}
}

extern "C" MG_API int mg_decode_stream(mg_ctx* ctx, const uint8_t* stream, size_t len, LZMAPacket* out_slab)
{
	if (!ctx || !stream || !out_slab) return fail(MG_EINVAL, "mg_decode_stream: null argument");
	if (len < 13 + 5) return fail(MG_EINVAL, "mg_decode_stream: %zu bytes are shorter than any LZMA-alone stream", len);
	if (stream[0] != 0) {
		const unsigned props = stream[0];
		return fail(MG_EINVAL, "mg_decode_stream: properties byte %u (lc = %u, lp = %u, pb = %u); only lc = lp = pb = 0 is supported",
		            props, props % 9, props / 9 % 5, props / 45);
	}
	uint64_t size = 0;
	for (int i = 0; i < 8; i++) size |= (uint64_t)stream[5 + i] << (8 * i);
	const bool known = size != ~0ull;
	if (known && size != ctx->n)
		return fail(MG_EINVAL, "mg_decode_stream: the stream is of %llu bytes, the input of %u", (unsigned long long)size, ctx->n);
	CU(cudaSetDevice(ctx->device));
	const uint32_t n = ctx->n;
	const size_t payload = len - 13;
	DevBuf dstream, slab, status;
	if (int rc = dev_alloc(dstream, payload)) return rc;
	if (int rc = dev_alloc(slab, (size_t)n * 8)) return rc;
	if (int rc = dev_alloc(status, sizeof(DecodeStatus))) return rc;
	CU(cudaMemcpyAsync(dstream.p, stream + 13, payload, cudaMemcpyHostToDevice, ctx->stream));
	fill_literal_kernel<<<grid_for(n, 256, ctx->sm_count * 8), 256, 0, ctx->stream>>>(slab.as<uint64_t>(), n);
	CU(cudaGetLastError());
	DecodeArgs a;
	a.data = ctx->d_data;
	a.n = n;
	a.stream = dstream.as<uint8_t>();
	a.len = payload;
	a.known_size = known ? 1u : 0u;
	a.slab = slab.as<uint64_t>();
	a.status = status.as<DecodeStatus>();
	cudaEvent_t t0, t1;
	CU(cudaEventCreate(&t0));
	CU(cudaEventCreate(&t1));
	CU(cudaEventRecord(t0, ctx->stream));
	decode_kernel<<<1, 32, 0, ctx->stream>>>(a);
	CU(cudaEventRecord(t1, ctx->stream));
	CU(cudaGetLastError());
	DecodeStatus st;
	CU(cudaMemcpyAsync(&st, status.p, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	{
		float ms = 0;
		cudaEventElapsedTime(&ms, t0, t1);
		ctx->last_decode_ms = ms;
		ctx->last_decode_events = st.events;
		cudaEventDestroy(t0);
		cudaEventDestroy(t1);
	}
	if (st.err != DEC_OK)
		return fail(MG_ESLAB, "mg_decode_stream: position %u: %s (%llu of %zu payload bytes read)", st.pos, decode_error(st.err),
		            st.consumed, payload);
	return download_unpacked(ctx, slab.as<uint64_t>(), n, out_slab);
}

extern "C" MG_API int mg_decode_stats(const mg_ctx* ctx, double* kernel_ms, uint64_t* events)
{
	if (!ctx) return fail(MG_EINVAL, "mg_decode_stats: null context");
	if (kernel_ms) *kernel_ms = ctx->last_decode_ms;
	if (events) *events = ctx->last_decode_events;
	return MG_OK;
}

// ---- annealing ----------------------------------------------------------------------------------------
struct mg_anneal {
	uint32_t* d_regions = nullptr;  // [chains][2] byte ranges of the last region-mode run

	mg_ctx* ctx = nullptr;
	mg_anneal_params p{};
	uint32_t stride = 0, nslots = 0, nck = 0;
	uint64_t* d_slabs = nullptr;
	uint64_t* d_bests = nullptr;
	Record* d_ck = nullptr;
	CkMeta* d_ck_meta = nullptr;
	uint8_t* d_ck_live = nullptr;
	Edit* d_logs = nullptr;
	Edit* d_journal = nullptr;
	ChainState* d_state = nullptr;
	ChainStats* d_stats = nullptr;
	TraceRec* d_trace = nullptr;
	uint32_t* d_attempts = nullptr;
	float* d_temps = nullptr;
	// scratch for (re)scoring chains
	uint64_t* d_cost = nullptr;
	uint32_t* d_count = nullptr;
	uint32_t* d_err = nullptr;
	uint32_t* d_bad = nullptr;
	std::vector<uint8_t> have_slab;
	cudaEvent_t e0 = nullptr, e1 = nullptr;
};

static void normalise(const mg_ctx* ctx, mg_anneal_params& p)
{
	if (p.top_k == 0) p.top_k = 20;
	if (p.checkpoint_stride == 0) p.checkpoint_stride = default_stride(ctx->n);
	p.checkpoint_stride = (p.checkpoint_stride + 31) & ~31u;
	if (p.edit_log_capacity == 0) p.edit_log_capacity = 4096;
	if (p.edit_log_capacity < 16) p.edit_log_capacity = 16;
}

extern "C" MG_API size_t mg_anneal_chain_bytes(const mg_ctx* ctx, const mg_anneal_params* params)
{
	if (!ctx || !params) return 0;
	mg_anneal_params p = *params;
	normalise(ctx, p);
	if (p.checkpoint_stride < 512) return 0;
	const size_t n = ctx->n;
	const size_t nslots = (n + p.checkpoint_stride - 1) / p.checkpoint_stride;
	const size_t nck = nslots > 1 ? nslots - 1 : 1;
	size_t b = n * 8;
	if (p.track_best) b += n * 8 + (size_t)JOURNAL_CAP * sizeof(Edit);
	b += nck * 2 * (sizeof(Record) + sizeof(CkMeta)) + nck;
	b += (size_t)p.edit_log_capacity * sizeof(Edit);
	b += sizeof(ChainState) + sizeof(ChainStats) + 4 + 4 + 8 + 4 + 4;
	b += (size_t)p.trace_capacity * sizeof(TraceRec);
	return b;
}

extern "C" MG_API void mg_anneal_destroy(mg_anneal* an)
{
	if (!an) return;
	{
		std::vector<mg_anneal*>& live = an->ctx->annealers;
		for (size_t i = 0; i < live.size(); i++)
			if (live[i] == an) {
				live.erase(live.begin() + (long)i);
				break;
			}
	}
	cudaSetDevice(an->ctx->device);
	cudaStreamSynchronize(an->ctx->stream);
	pool_free(an->d_regions);
	pool_free(an->d_slabs);
	pool_free(an->d_bests);
	pool_free(an->d_ck);
	pool_free(an->d_ck_meta);
	pool_free(an->d_ck_live);
	pool_free(an->d_logs);
	pool_free(an->d_journal);
	pool_free(an->d_state);
	pool_free(an->d_stats);
	pool_free(an->d_trace);
	pool_free(an->d_attempts);
	pool_free(an->d_temps);
	pool_free(an->d_cost);
	pool_free(an->d_count);
	pool_free(an->d_err);
	pool_free(an->d_bad);
	if (an->e0) cudaEventDestroy(an->e0);
	if (an->e1) cudaEventDestroy(an->e1);
	delete an;
}

extern "C" MG_API int mg_anneal_create(mg_ctx* ctx, const mg_anneal_params* params, mg_anneal** out)
{
	if (!ctx || !params || !out) return fail(MG_EINVAL, "mg_anneal_create: null argument");
	if (params->chains == 0) return fail(MG_EINVAL, "mg_anneal_create: chains must be > 0");
	mg_anneal_params p = *params;
	normalise(ctx, p);
	if (p.top_k > (uint32_t)MAX_K) return fail(MG_EINVAL, "mg_anneal_create: top_k must be <= %d", MAX_K);
	if (p.checkpoint_stride < 512) return fail(MG_EINVAL, "mg_anneal_create: checkpoint_stride must be >= 512");
	CU(cudaSetDevice(ctx->device));
	mg_anneal* an = new (std::nothrow) mg_anneal;
	if (!an) return fail(MG_ENOMEM, "out of host memory");
	an->ctx = ctx;
	an->p = p;
	an->stride = p.checkpoint_stride;
	an->nslots = (ctx->n + an->stride - 1) / an->stride;
	an->nck = an->nslots > 1 ? an->nslots - 1 : 1;  // keep arrays non-empty
	const size_t C = p.chains, n = ctx->n, nck = an->nck;
	int rc = 0;
#define A(ptr, bytes)                                                                              \
	if (!rc) {                                                                                     \
		cudaError_t e_ = pool_malloc(&(ptr), (bytes));                                      \
		if (e_ != cudaSuccess) rc = fail(e_ == cudaErrorMemoryAllocation ? MG_ENOMEM : MG_ECUDA,  \
		                                 "cudaMalloc(%zu bytes for %s): %s", (size_t)(bytes), #ptr, cudaGetErrorString(e_)); \
	}
	A(an->d_slabs, C * n * 8);
	if (p.track_best) A(an->d_bests, C * n * 8);
	A(an->d_ck, C * 2 * nck * sizeof(Record));
	A(an->d_ck_meta, C * 2 * nck * sizeof(CkMeta));
	A(an->d_ck_live, C * nck);
	A(an->d_logs, C * (size_t)p.edit_log_capacity * sizeof(Edit));
	if (p.track_best) A(an->d_journal, C * (size_t)JOURNAL_CAP * sizeof(Edit));
	A(an->d_state, C * sizeof(ChainState));
	A(an->d_stats, C * sizeof(ChainStats));
	if (p.trace_capacity) A(an->d_trace, C * (size_t)p.trace_capacity * sizeof(TraceRec));
	A(an->d_attempts, C * 4);
	A(an->d_temps, C * 4);
	A(an->d_cost, C * 8);
	A(an->d_count, C * 4);
	A(an->d_err, C * 4);
	A(an->d_bad, 4);
#undef A
	if (!rc) {
		cudaError_t e_ = cudaEventCreate(&an->e0);
		if (e_ == cudaSuccess) e_ = cudaEventCreate(&an->e1);
		if (e_ == cudaSuccess) e_ = cudaMemsetAsync(an->d_state, 0, C * sizeof(ChainState), ctx->stream);
		if (e_ == cudaSuccess) e_ = cudaMemsetAsync(an->d_ck_live, 0, C * nck, ctx->stream);
		if (e_ != cudaSuccess) rc = fail(MG_ECUDA, "mg_anneal_create: %s", cudaGetErrorString(e_));
	}
	if (!rc) {
		// per-chain generators: splitmix64 seeded by (seed, chain), same recipe as the oracle
		std::vector<ChainState> st(C);
		for (size_t c = 0; c < C; c++) {
			uint64_t s = p.seed ^ ((uint64_t)c * 0xD1342543DE82EF95ull + 0x632BE59BD9B4E019ull);
			s += 0x9E3779B97F4A7C15ull;  // one splitmix64 step (output discarded)
			memset(&st[c], 0, sizeof(ChainState));
			st[c].rng = s;
		}
		cudaError_t e_ = cudaMemcpyAsync(an->d_state, st.data(), C * sizeof(ChainState), cudaMemcpyHostToDevice, ctx->stream);
		if (e_ == cudaSuccess) e_ = cudaStreamSynchronize(ctx->stream);
		if (e_ != cudaSuccess) rc = fail(MG_ECUDA, "mg_anneal_create: %s", cudaGetErrorString(e_));
	}
	if (rc) {
		mg_anneal_destroy(an);
		return rc;
	}
	an->have_slab.assign(C, 0);
	ctx->annealers.push_back(an);
	*out = an;
	return MG_OK;
}

// dst[c * stride_bytes + ...] = src[...] for c in [0, copies): one kernel when everything is
// 16-byte aligned, a memcpy per copy otherwise.
static int replicate(mg_ctx* ctx, const void* src, void* dst, size_t bytes, size_t stride_bytes, uint32_t copies)
{
	if (copies == 0 || bytes == 0) return 0;
	const bool aligned = (((uintptr_t)src | (uintptr_t)dst | bytes | stride_bytes) & 15) == 0;
	if (aligned) {
		const size_t words = bytes / 16;
		replicate_kernel<<<grid_for(words, 256, ctx->sm_count * 16), 256, 0, ctx->stream>>>(
		    static_cast<const uint4*>(src), static_cast<uint4*>(dst), words, stride_bytes / 16, copies);
		CU(cudaGetLastError());
		return 0;
	}
	for (uint32_t c = 0; c < copies; c++)
		CU(cudaMemcpyAsync(static_cast<char*>(dst) + (size_t)c * stride_bytes, src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
	return 0;
}

// Rescore + checkpoint chains [first, first+count) from their current device slabs.
static int refresh_chains(mg_anneal* an, uint32_t first, uint32_t count, int adopt_cost, int reset_best)
{
	mg_ctx* ctx = an->ctx;
	const size_t n = ctx->n, nck = an->nck;
	// validate every slot once (the walk may later land on any of them)
	CU(cudaMemsetAsync(an->d_bad, 0, 4, ctx->stream));
	for (uint32_t c = first; c < first + count; c++)
		validate_kernel<<<grid_for(n, 256, ctx->sm_count * 4), 256, 0, ctx->stream>>>(an->d_slabs + (size_t)c * n, ctx->n, an->d_bad);
	CU(cudaGetLastError());
	// checkpoints go to buffer 0 and become current
	for (uint32_t c = first; c < first + count; c++) {
		ScoreArgs a;
		a.data = ctx->d_data;
		a.n = ctx->n;
		a.slabs = an->d_slabs + (size_t)c * n;
		a.nslabs = 1;
		a.stop_pos = ctx->n;
		a.out_cost = an->d_cost + c;
		a.out_count = an->d_count + c;
		a.out_err = an->d_err + c;
		a.ck = an->d_ck + (size_t)c * 2 * nck;
		a.ck_pos = nullptr;
		a.ck_meta = an->d_ck_meta + (size_t)c * 2 * nck;
		a.stride = an->stride;
		a.nslots = an->nslots;
		a.ck_chain_stride = 0;
		a.final_model = nullptr;
		a.tables = ctx->tables;
		score_kernel<<<1, CTA_THREADS, sizeof(CtaShared), ctx->stream>>>(a);
	}
	CU(cudaGetLastError());
	CU(cudaMemsetAsync(an->d_ck_live + (size_t)first * nck, 0, (size_t)count * nck, ctx->stream));
	std::vector<uint64_t> cost(count);
	std::vector<uint32_t> live(count), err(count);
	uint32_t bad = 0;
	CU(cudaMemcpyAsync(cost.data(), an->d_cost + first, count * 8, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaMemcpyAsync(live.data(), an->d_count + first, count * 4, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaMemcpyAsync(err.data(), an->d_err + first, count * 4, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaMemcpyAsync(&bad, an->d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
	std::vector<ChainState> st(count);
	CU(cudaMemcpyAsync(st.data(), an->d_state + first, count * sizeof(ChainState), cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	if (bad) return fail(MG_ESLAB, "slab holds %u undecodable slot(s)", bad);
	for (uint32_t i = 0; i < count; i++) {
		if (err[i]) return fail(MG_ESLAB, "chain %u: %s", first + i, walk_error(err[i]));
		st[i].cur_cost = adopt_cost ? cost[i] : 0;
		st[i].slab_cost = cost[i];
		st[i].live_count = live[i];
		st[i].err = 0;
		st[i].eval_index = 0;
		st[i].susp_slot = 0;  // a suspended proposal belongs to the slab that was replaced
		st[i].journal_count = 0;
		st[i].journal_overflow = reset_best ? 0 : 1;  // best slab == current slab only right after a reset
		if (reset_best) st[i].best_cost = 0;
	}
	CU(cudaMemcpyAsync(an->d_state + first, st.data(), count * sizeof(ChainState), cudaMemcpyHostToDevice, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	for (uint32_t i = 0; i < count; i++) an->have_slab[first + i] = 1;
	return 0;
}

extern "C" MG_API int mg_anneal_set_slab(mg_anneal* an, uint32_t first, uint32_t count, const LZMAPacket* slab,
                                  int adopt_cost, int reset_best)
{
	if (!an) return fail(MG_EINVAL, "mg_anneal_set_slab: null handle");
	if (count == 0 || first >= an->p.chains || count > an->p.chains - first)
		return fail(MG_EINVAL, "mg_anneal_set_slab: chain range out of bounds");
	mg_ctx* ctx = an->ctx;
	CU(cudaSetDevice(ctx->device));
	const size_t n = ctx->n;
	uint64_t* dst0 = an->d_slabs + (size_t)first * n;
	if (slab) {
		if (int rc = upload_packed(ctx, slab, n, dst0)) return rc;
	} else {
		fill_literal_kernel<<<grid_for(n, 256, ctx->sm_count * 8), 256, 0, ctx->stream>>>(dst0, n);
		CU(cudaGetLastError());
	}
	if (int rc = replicate(ctx, dst0, dst0 + n, n * 8, n * 8, count - 1)) return rc;
	if (an->d_bests && reset_best)
		if (int rc = replicate(ctx, dst0, an->d_bests + (size_t)first * n, n * 8, n * 8, count)) return rc;
	// identical slabs: score the first, replicate its checkpoints
	if (int rc = refresh_chains(an, first, 1, adopt_cost, reset_best)) return rc;
	if (count > 1) {
		const size_t nck = an->nck;
		if (int rc = replicate(ctx, an->d_ck + (size_t)first * 2 * nck, an->d_ck + (size_t)(first + 1) * 2 * nck,
		                       nck * sizeof(Record), 2 * nck * sizeof(Record), count - 1))
			return rc;
		if (int rc = replicate(ctx, an->d_ck_meta + (size_t)first * 2 * nck, an->d_ck_meta + (size_t)(first + 1) * 2 * nck,
		                       nck * sizeof(CkMeta), 2 * nck * sizeof(CkMeta), count - 1))
			return rc;
		CU(cudaMemsetAsync(an->d_ck_live + (size_t)first * nck, 0, (size_t)count * nck, ctx->stream));
		std::vector<ChainState> st(count);
		CU(cudaMemcpyAsync(st.data(), an->d_state + first, count * sizeof(ChainState), cudaMemcpyDeviceToHost, ctx->stream));
		CU(cudaStreamSynchronize(ctx->stream));
		for (uint32_t i = 1; i < count; i++) {
			st[i].cur_cost = st[0].cur_cost;
			st[i].slab_cost = st[0].slab_cost;
			st[i].live_count = st[0].live_count;
			st[i].err = 0;
			st[i].eval_index = 0;
			st[i].susp_slot = 0;  // a suspended proposal belongs to the slab that was replaced
			st[i].journal_count = 0;
			st[i].journal_overflow = reset_best ? 0 : 1;
			if (reset_best) st[i].best_cost = 0;
			an->have_slab[first + i] = 1;
		}
		CU(cudaMemcpyAsync(an->d_state + first, st.data(), count * sizeof(ChainState), cudaMemcpyHostToDevice, ctx->stream));
		CU(cudaStreamSynchronize(ctx->stream));
	}
	return MG_OK;
}

extern "C" MG_API int mg_anneal_refresh_chain(mg_anneal* an, uint32_t chain, int adopt_cost)
{
	if (!an || chain >= an->p.chains) return fail(MG_EINVAL, "mg_anneal_refresh_chain: bad argument");
	CU(cudaSetDevice(an->ctx->device));
	if (int rc = refresh_chains(an, chain, 1, adopt_cost, 0)) return rc;
	return MG_OK;
}

// The launch arguments that do not depend on the call.
static void anneal_common_args(mg_anneal* an, AnnealArgs& a)
{
	mg_ctx* ctx = an->ctx;
	const uint32_t C = an->p.chains;
	a.data = ctx->d_data;
	a.n = ctx->n;
	a.occ_start = ctx->d_occ_start;
	a.occ = ctx->d_occ;
	a.tables = ctx->tables;
	a.limits = ctx->limits;
	a.chains = C;
	a.k = an->p.top_k;
	a.stride = an->stride;
	a.nslots = an->nck + 1;
	a.log_cap = an->p.edit_log_capacity;
	a.track_best = an->p.track_best && an->d_bests;
	a.slabs = an->d_slabs;
	a.bests = an->d_bests;
	a.ck = an->d_ck;
	a.ck_meta = an->d_ck_meta;
	a.ck_live = an->d_ck_live;
	a.logs = an->d_logs;
	a.journal = an->d_journal;
	a.state = an->d_state;
	a.stats = an->d_stats;
	a.trace = an->d_trace;
	a.trace_cap = an->p.trace_capacity;
	a.attempts_out = an->d_attempts;
	a.regions = nullptr;
	a.abs_dist = nullptr;
	a.chain_first = 0;
	a.repair_only = 0;
	a.suspend = 0;
	a.cycle_budget = 0;
	a.packet_budget = 0;
	a.early_exit = 0;
	a.temps = nullptr;
	a.schedule = 0;
	a.step = 0;
	a.num_iters = ctx->n;
	a.first_eval = 0xffffffffu;
	a.evals = 0;
	a.max_attempts = 0;
	if (an->nslots <= 1) a.nslots = 1;  // a single slot has no checkpoints: the kernel's nck is 0
}

extern "C" MG_API int mg_anneal_run(mg_anneal* an, const mg_anneal_run_params* run, mg_anneal_stats* stats)
{
	if (!an || !run) return fail(MG_EINVAL, "mg_anneal_run: null argument");
	mg_ctx* ctx = an->ctx;
	for (uint8_t h : an->have_slab)
		if (!h) return fail(MG_ESTATE, "mg_anneal_run: every chain needs mg_anneal_set_slab first");
	if (run->schedule > 1) return fail(MG_EINVAL, "mg_anneal_run: unknown schedule");
	if (run->schedule == MG_SCHEDULE_TEMPERATURE && !run->temperatures)
		return fail(MG_EINVAL, "mg_anneal_run: temperatures required");
	CU(cudaSetDevice(ctx->device));
	const uint32_t C = an->p.chains;
	if (run->temperatures) CU(cudaMemcpyAsync(an->d_temps, run->temperatures, (size_t)C * 4, cudaMemcpyHostToDevice, ctx->stream));
	AnnealArgs a;
	anneal_common_args(an, a);
	a.evals = run->evals;
	a.max_attempts = run->max_attempts ? run->max_attempts : run->evals * 64u + 1024u;
	a.schedule = run->schedule;
	a.step = run->step;
	a.num_iters = run->num_iters ? run->num_iters : ctx->n;
	a.first_eval = run->first_eval;
	a.packet_budget = run->packet_budget;
	a.early_exit = run->no_early_exit ? 0u : 1u;
	a.suspend = run->suspend ? 1u : 0u;
	a.cycle_budget = run->cycle_budget;
	a.temps = run->temperatures ? an->d_temps : nullptr;
	if (run->regions) {
		for (uint32_t c = 0; c < C; c++)
			if (run->regions[2 * c] >= run->regions[2 * c + 1] || run->regions[2 * c + 1] > ctx->n)
				return fail(MG_EINVAL, "mg_anneal_run: chain %u has an empty or out-of-range region", c);
		if (!an->d_regions) CU(pool_malloc(&an->d_regions, (size_t)C * 8));
		CU(cudaMemcpyAsync(an->d_regions, run->regions, (size_t)C * 8, cudaMemcpyHostToDevice, ctx->stream));
		a.regions = an->d_regions;
	}
	// one CTA per SM while the population is at most one wave, then as many CTAs as the chains need
	int blocks = (int)((C + WARPS_PER_CTA - 1) / WARPS_PER_CTA);
	if (blocks < ctx->sm_count) blocks = (int)(C < (uint32_t)ctx->sm_count ? C : (uint32_t)ctx->sm_count);
	CU(cudaEventRecord(an->e0, ctx->stream));
	anneal_kernel<<<blocks, CTA_THREADS, sizeof(CtaShared), ctx->stream>>>(a);
	CU(cudaEventRecord(an->e1, ctx->stream));
	CU(cudaGetLastError());
	CU(cudaStreamSynchronize(ctx->stream));
	float ms = 0;
	CU(cudaEventElapsedTime(&ms, an->e0, an->e1));
	std::vector<ChainStats> cs(C);
	std::vector<ChainState> st(C);
	CU(cudaMemcpy(cs.data(), an->d_stats, (size_t)C * sizeof(ChainStats), cudaMemcpyDeviceToHost));
	CU(cudaMemcpy(st.data(), an->d_state, (size_t)C * sizeof(ChainState), cudaMemcpyDeviceToHost));
	for (uint32_t c = 0; c < C; c++)
		if (st[c].err) return fail(MG_ESLAB, "mg_anneal_run: chain %u stopped: %s", c, walk_error(st[c].err));
	if (stats) {
		memset(stats, 0, sizeof(*stats));
		for (uint32_t c = 0; c < C; c++) {
			stats->evals += cs[c].evals;
			stats->attempts += cs[c].attempts;
			stats->accepted += cs[c].accepted;
			stats->new_best += cs[c].new_best;
			stats->packets_scored += cs[c].packets;
			stats->bits_scored += cs[c].bits;
			stats->slab_bytes_read += cs[c].slab_bytes;
			stats->checkpoint_bytes += cs[c].ck_bytes;
			stats->finder_calls += cs[c].finds;
			stats->finder_candidates += cs[c].candidates;
			stats->edits += cs[c].edits;
			stats->log_overflows += cs[c].overflows;
			stats->rejoined += cs[c].rejoined;
			stats->finder_cycles += cs[c].find_cycles;
			stats->finder_chunks += cs[c].chunks;
			stats->finder_gave_up += cs[c].gave_up;
			stats->chain_cycles += cs[c].chain_cycles;
			if (cs[c].chain_cycles > stats->max_chain_cycles) stats->max_chain_cycles = cs[c].chain_cycles;
		}
		stats->kernel_ms = ms;
		stats->launches = 1;
	}
	return MG_OK;
}

extern "C" MG_API int mg_anneal_costs(mg_anneal* an, uint64_t* cur_cost, uint64_t* best_cost)
{
	if (!an) return fail(MG_EINVAL, "mg_anneal_costs: null handle");
	CU(cudaSetDevice(an->ctx->device));
	const uint32_t C = an->p.chains;
	std::vector<ChainState> st(C);
	CU(cudaStreamSynchronize(an->ctx->stream));
	CU(cudaMemcpy(st.data(), an->d_state, (size_t)C * sizeof(ChainState), cudaMemcpyDeviceToHost));
	for (uint32_t c = 0; c < C; c++) {
		if (cur_cost) cur_cost[c] = st[c].cur_cost;
		if (best_cost) best_cost[c] = st[c].best_cost;
	}
	return MG_OK;
}

extern "C" MG_API int mg_anneal_get_slab(mg_anneal* an, uint32_t chain, int which, LZMAPacket* out_slab)
{
	if (!an || !out_slab || chain >= an->p.chains) return fail(MG_EINVAL, "mg_anneal_get_slab: bad argument");
	if (which == 1 && !an->d_bests) return fail(MG_ESTATE, "mg_anneal_get_slab: chains were created without track_best");
	CU(cudaSetDevice(an->ctx->device));
	const size_t n = an->ctx->n;
	const uint64_t* src = (which == 1 ? an->d_bests : an->d_slabs) + (size_t)chain * n;
	if (int rc = download_unpacked(an->ctx, src, n, out_slab)) return rc;
	return MG_OK;
}

extern "C" MG_API int mg_anneal_get_trace(mg_anneal* an, uint32_t chain, mg_trace_rec* out, size_t cap, size_t* count)
{
	if (!an || chain >= an->p.chains || !count) return fail(MG_EINVAL, "mg_anneal_get_trace: bad argument");
	if (!an->d_trace) return fail(MG_ESTATE, "mg_anneal_get_trace: chains were created without trace_capacity");
	CU(cudaSetDevice(an->ctx->device));
	uint32_t attempts = 0;
	CU(cudaMemcpy(&attempts, an->d_attempts + chain, 4, cudaMemcpyDeviceToHost));
	*count = attempts;
	size_t c = attempts < an->p.trace_capacity ? attempts : an->p.trace_capacity;
	if (c > cap) c = cap;
	static_assert(sizeof(mg_trace_rec) == sizeof(TraceRec), "trace record layout");
	if (c && out)
		CU(cudaMemcpy(out, an->d_trace + (size_t)chain * an->p.trace_capacity, c * sizeof(TraceRec), cudaMemcpyDeviceToHost));
	return MG_OK;
}

extern "C" MG_API int mg_anneal_device_slab(mg_anneal* an, uint32_t chain, int which, void** dev_ptr, size_t* bytes)
{
	if (!an || chain >= an->p.chains || !dev_ptr || !bytes) return fail(MG_EINVAL, "mg_anneal_device_slab: bad argument");
	if (which == 1 && !an->d_bests) return fail(MG_ESTATE, "mg_anneal_device_slab: chains were created without track_best");
	*dev_ptr = (which == 1 ? an->d_bests : an->d_slabs) + (size_t)chain * an->ctx->n;
	*bytes = (size_t)an->ctx->n * 8;
	return MG_OK;
}

extern "C" MG_API int mg_anneal_export_slab(mg_anneal* an, uint32_t chain, int which, void* dev_dst)
{
	if (!an || chain >= an->p.chains || !dev_dst) return fail(MG_EINVAL, "mg_anneal_export_slab: bad argument");
	if (which == 1 && !an->d_bests) return fail(MG_ESTATE, "mg_anneal_export_slab: chains were created without track_best");
	CU(cudaSetDevice(an->ctx->device));
	const size_t n = an->ctx->n;
	const uint64_t* src = (which == 1 ? an->d_bests : an->d_slabs) + (size_t)chain * n;
	CU(cudaMemcpyAsync(dev_dst, src, n * 8, cudaMemcpyDeviceToDevice, an->ctx->stream));
	CU(cudaStreamSynchronize(an->ctx->stream));
	return MG_OK;
}

extern "C" MG_API int mg_anneal_import_slab(mg_anneal* an, uint32_t chain, const void* dev_src, int adopt_cost)
{
	if (!an || chain >= an->p.chains || !dev_src) return fail(MG_EINVAL, "mg_anneal_import_slab: bad argument");
	CU(cudaSetDevice(an->ctx->device));
	const size_t n = an->ctx->n;
	CU(cudaMemcpyAsync(an->d_slabs + (size_t)chain * n, dev_src, n * 8, cudaMemcpyDeviceToDevice, an->ctx->stream));
	if (int rc = refresh_chains(an, chain, 1, adopt_cost, 0)) return rc;
	return MG_OK;
}

// Swap two chains' slabs, checkpoints and costs (replica exchange on one device).
extern "C" MG_API int mg_anneal_swap_chains(mg_anneal* an, uint32_t x, uint32_t y)
{
	if (!an || x >= an->p.chains || y >= an->p.chains) return fail(MG_EINVAL, "mg_anneal_swap_chains: bad argument");
	if (x == y) return MG_OK;
	mg_ctx* ctx = an->ctx;
	CU(cudaSetDevice(ctx->device));
	const size_t n = ctx->n, nck = an->nck;
	DevBuf tmp;
	size_t big = n * 8;
	if (2 * nck * sizeof(Record) > big) big = 2 * nck * sizeof(Record);
	if (int rc = dev_alloc(tmp, big)) return rc;
	auto swap_region = [&](void* pa, void* pb, size_t bytes) -> cudaError_t {
		cudaError_t e = cudaMemcpyAsync(tmp.p, pa, bytes, cudaMemcpyDeviceToDevice, ctx->stream);
		if (e == cudaSuccess) e = cudaMemcpyAsync(pa, pb, bytes, cudaMemcpyDeviceToDevice, ctx->stream);
		if (e == cudaSuccess) e = cudaMemcpyAsync(pb, tmp.p, bytes, cudaMemcpyDeviceToDevice, ctx->stream);
		return e;
	};
	CU(swap_region(an->d_slabs + (size_t)x * n, an->d_slabs + (size_t)y * n, n * 8));
	CU(swap_region(an->d_ck + (size_t)x * 2 * nck, an->d_ck + (size_t)y * 2 * nck, 2 * nck * sizeof(Record)));
	CU(swap_region(an->d_ck_meta + (size_t)x * 2 * nck, an->d_ck_meta + (size_t)y * 2 * nck, 2 * nck * sizeof(CkMeta)));
	CU(swap_region(an->d_ck_live + (size_t)x * nck, an->d_ck_live + (size_t)y * nck, nck));
	ChainState sx, sy;
	CU(cudaStreamSynchronize(ctx->stream));
	CU(cudaMemcpy(&sx, an->d_state + x, sizeof(ChainState), cudaMemcpyDeviceToHost));
	CU(cudaMemcpy(&sy, an->d_state + y, sizeof(ChainState), cudaMemcpyDeviceToHost));
	// the slab, its cost and live count move; generators and best records stay with the chain id
	ChainState nx = sx, ny = sy;
	nx.cur_cost = sy.cur_cost;
	nx.slab_cost = sy.slab_cost;
	nx.live_count = sy.live_count;
	ny.cur_cost = sx.cur_cost;
	ny.slab_cost = sx.slab_cost;
	ny.live_count = sx.live_count;
	nx.journal_count = ny.journal_count = 0;
	nx.susp_slot = ny.susp_slot = 0;  // suspended proposals do not move with the slabs: dropped
	nx.journal_overflow = ny.journal_overflow = 1;  // the best slabs stayed, the current ones moved
	CU(cudaMemcpy(an->d_state + x, &nx, sizeof(ChainState), cudaMemcpyHostToDevice));
	CU(cudaMemcpy(an->d_state + y, &ny, sizeof(ChainState), cudaMemcpyHostToDevice));
	return MG_OK;
}

extern "C" MG_API int mg_anneal_merge_export(mg_anneal* an, uint32_t nregions, const uint32_t* bounds, const uint32_t* owners,
                                      void* dev_slab, void* dev_abs)
{
	if (!an || !bounds || !owners || nregions == 0 || !dev_slab || !dev_abs)
		return fail(MG_EINVAL, "mg_anneal_merge_export: bad argument");
	mg_ctx* ctx = an->ctx;
	const size_t n = ctx->n;
	if (bounds[0] != 0 || bounds[nregions] != n) return fail(MG_EINVAL, "mg_anneal_merge_export: regions must cover the input");
	for (uint32_t r = 0; r < nregions; r++) {
		if (bounds[r] >= bounds[r + 1]) return fail(MG_EINVAL, "mg_anneal_merge_export: region %u is empty", r);
		if (owners[r] != MG_NO_OWNER && owners[r] >= an->p.chains)
			return fail(MG_EINVAL, "mg_anneal_merge_export: region %u has no such owner", r);
	}
	CU(cudaSetDevice(ctx->device));
	DevBuf d_bounds, d_owners;
	if (int rc = dev_alloc(d_bounds, (size_t)(nregions + 1) * 4)) return rc;
	if (int rc = dev_alloc(d_owners, (size_t)nregions * 4)) return rc;
	CU(cudaMemcpyAsync(d_bounds.p, bounds, (size_t)(nregions + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
	CU(cudaMemcpyAsync(d_owners.p, owners, (size_t)nregions * 4, cudaMemcpyHostToDevice, ctx->stream));
	CU(cudaMemsetAsync(dev_slab, 0, n * 8, ctx->stream));
	CU(cudaMemsetAsync(dev_abs, 0, n * 4, ctx->stream));
	// pass A: what every LONG_REP of the owners' regions stands for (distance + 1)
	region_abs_reps_kernel<<<grid_for(nregions, 128, 1 << 20), 128, 0, ctx->stream>>>(
	    an->d_slabs, (uint32_t)n, d_bounds.as<uint32_t>(), d_owners.as<uint32_t>(), nregions, an->d_ck, an->d_ck_meta, an->d_ck_live,
	    (uint32_t)an->nck, an->nslots > 1 ? 1u : 0u, an->stride, static_cast<uint32_t*>(dev_abs));
	CU(cudaGetLastError());
	merge_regions_kernel<<<grid_for(nregions, 1, ctx->sm_count * 8), 256, 0, ctx->stream>>>(
	    an->d_slabs, (uint32_t)n, d_bounds.as<uint32_t>(), d_owners.as<uint32_t>(), nregions, static_cast<uint64_t*>(dev_slab));
	CU(cudaGetLastError());
	CU(cudaStreamSynchronize(ctx->stream));
	return MG_OK;
}

extern "C" MG_API int mg_anneal_merge_import(mg_anneal* an, const void* dev_slab, const void* dev_abs, uint32_t dst_chain,
                                      uint64_t* cost_out)
{
	if (!an || !dev_slab || !dev_abs || dst_chain >= an->p.chains) return fail(MG_EINVAL, "mg_anneal_merge_import: bad argument");
	mg_ctx* ctx = an->ctx;
	const size_t n = ctx->n;
	CU(cudaSetDevice(ctx->device));
	CU(cudaMemsetAsync(an->d_bad, 0, 4, ctx->stream));
	validate_kernel<<<grid_for(n, 256, ctx->sm_count * 4), 256, 0, ctx->stream>>>(static_cast<const uint64_t*>(dev_slab), ctx->n, an->d_bad);
	CU(cudaGetLastError());
	uint32_t bad = 0;
	CU(cudaMemcpyAsync(&bad, an->d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaMemcpyAsync(an->d_slabs + (size_t)dst_chain * n, dev_slab, n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
	// the destination's bookkeeping no longer describes its slab: the forced pass below rebuilds it
	ChainState st;
	CU(cudaStreamSynchronize(ctx->stream));
	if (bad) return fail(MG_ESLAB, "mg_anneal_merge_import: merged slab holds %u undecodable slot(s)", bad);
	CU(cudaMemcpy(&st, an->d_state + dst_chain, sizeof(ChainState), cudaMemcpyDeviceToHost));
	st.susp_slot = 0;
	st.journal_count = 0;
	st.journal_overflow = 1;
	st.err = 0;
	CU(cudaMemcpy(an->d_state + dst_chain, &st, sizeof(ChainState), cudaMemcpyHostToDevice));
	// one forced pass over the merged slab: repair what the seams broke (SHORT_REP / LONG_REP packets
	// whose rep distances changed; src/packet_slab_neighbour.c:82-117), price it, rewrite the checkpoints
	AnnealArgs a;
	anneal_common_args(an, a);
	a.chains = 1;
	a.chain_first = dst_chain;
	a.repair_only = 1;
	a.abs_dist = static_cast<const uint32_t*>(dev_abs);
	a.evals = 1;
	a.max_attempts = 1;
	anneal_kernel<<<1, CTA_THREADS, sizeof(CtaShared), ctx->stream>>>(a);
	CU(cudaGetLastError());
	CU(cudaStreamSynchronize(ctx->stream));
	CU(cudaMemcpy(&st, an->d_state + dst_chain, sizeof(ChainState), cudaMemcpyDeviceToHost));
	if (st.err) return fail(MG_ESLAB, "mg_anneal_merge_import: merged slab: %s", walk_error(st.err));
	an->have_slab[dst_chain] = 1;
	if (cost_out) *cost_out = st.slab_cost;
	return MG_OK;
}

extern "C" MG_API int mg_anneal_merge_regions(mg_anneal* an, uint32_t nregions, const uint32_t* bounds, const uint32_t* owners,
                                       uint32_t dst_chain, uint64_t* cost_out)
{
	if (!an || !bounds || !owners || nregions == 0 || dst_chain >= an->p.chains)
		return fail(MG_EINVAL, "mg_anneal_merge_regions: bad argument");
	for (uint32_t r = 0; r < nregions; r++)
		if (owners[r] == MG_NO_OWNER) return fail(MG_EINVAL, "mg_anneal_merge_regions: region %u has no owner", r);
	CU(cudaSetDevice(an->ctx->device));
	DevBuf slab, abs;
	if (int rc = dev_alloc(slab, (size_t)an->ctx->n * 8)) return rc;
	if (int rc = dev_alloc(abs, (size_t)an->ctx->n * 4)) return rc;
	if (int rc = mg_anneal_merge_export(an, nregions, bounds, owners, slab.p, abs.p)) return rc;
	return mg_anneal_merge_import(an, slab.p, abs.p, dst_chain, cost_out);
}

extern "C" MG_API int mg_anneal_greedy_init(mg_anneal* an, uint32_t nregions, uint32_t dst_chain, uint64_t* cost_out)
{
	if (!an || dst_chain >= an->p.chains) return fail(MG_EINVAL, "mg_anneal_greedy_init: bad argument");
	mg_ctx* ctx = an->ctx;
	const uint32_t n = ctx->n;
	if (nregions == 0) nregions = 1;
	if (nregions > n / 64 + 1) nregions = n / 64 + 1;  // a region is at least 64 bytes
	CU(cudaSetDevice(ctx->device));
	std::vector<uint32_t> bounds(nregions + 1);
	for (uint32_t r = 0; r <= nregions; r++) bounds[r] = (uint32_t)((uint64_t)n * r / nregions);
	DevBuf slab, abs, dbounds, derr;
	if (int rc = dev_alloc(slab, (size_t)n * 8)) return rc;
	if (int rc = dev_alloc(abs, (size_t)n * 4)) return rc;
	if (int rc = dev_alloc(dbounds, sizeof(uint32_t) * (nregions + 1))) return rc;
	if (int rc = dev_alloc(derr, 4)) return rc;
	CU(cudaMemcpyAsync(dbounds.p, bounds.data(), sizeof(uint32_t) * (nregions + 1), cudaMemcpyHostToDevice, ctx->stream));
	CU(cudaMemsetAsync(abs.p, 0, (size_t)n * 4, ctx->stream));
	CU(cudaMemsetAsync(derr.p, 0, 4, ctx->stream));
	fill_literal_kernel<<<grid_for(n, 256, ctx->sm_count * 8), 256, 0, ctx->stream>>>(slab.as<uint64_t>(), n);
	CU(cudaGetLastError());
	GreedyArgs g;
	g.data = ctx->d_data;
	g.n = n;
	g.occ_start = ctx->d_occ_start;
	g.occ = ctx->d_occ;
	g.tables = ctx->tables;
	g.limits = ctx->limits;
	g.k = an->p.top_k;
	g.bounds = dbounds.as<uint32_t>();
	g.nregions = nregions;
	g.slab = slab.as<uint64_t>();
	g.abs_dist = abs.as<uint32_t>();
	g.err = derr.as<uint32_t>();
	int blocks = (int)((nregions + WARPS_PER_CTA - 1) / WARPS_PER_CTA);
	if (blocks > ctx->sm_count) blocks = ctx->sm_count;
	greedy_kernel<<<blocks, CTA_THREADS, sizeof(CtaShared), ctx->stream>>>(g);
	CU(cudaGetLastError());
	uint32_t herr = 0;
	CU(cudaMemcpyAsync(&herr, derr.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	if (herr) return fail(MG_ESLAB, "mg_anneal_greedy_init: %s", walk_error(herr));
	return mg_anneal_merge_import(an, slab.p, abs.p, dst_chain, cost_out);
}

extern "C" MG_API int mg_anneal_optimal_init(mg_anneal* an, uint32_t nregions, uint32_t max_occ, uint32_t dst_chain,
                                             uint64_t* cost_out)
{
	if (!an || dst_chain >= an->p.chains) return fail(MG_EINVAL, "mg_anneal_optimal_init: bad argument");
	mg_ctx* ctx = an->ctx;
	const uint32_t n = ctx->n;
	if (nregions == 0) nregions = 1;
	if (nregions > n / 64 + 1) nregions = n / 64 + 1;  // a region is at least 64 bytes
	if (max_occ == 0) max_occ = 64;
	CU(cudaSetDevice(ctx->device));
	std::vector<uint32_t> bounds(nregions + 1);
	for (uint32_t r = 0; r <= nregions; r++) bounds[r] = (uint32_t)((uint64_t)n * r / nregions);
	// the parse's warps each keep one block of nodes (L2-resident scratch); regions are dealt over them
	uint32_t blocks = (uint32_t)ctx->sm_count * 8;
	if (blocks > nregions) blocks = nregions;
	DevBuf slab, abs, dbounds, lists, counts, nodes, dnodes;
	if (int rc = dev_alloc(slab, (size_t)n * 8)) return rc;
	if (int rc = dev_alloc(abs, (size_t)n * 4)) return rc;
	if (int rc = dev_alloc(dbounds, sizeof(uint32_t) * (nregions + 1))) return rc;
	if (int rc = dev_alloc(lists, (size_t)n * OPT_LIST * sizeof(uint2))) return rc;
	if (int rc = dev_alloc(counts, n)) return rc;
	if (int rc = dev_alloc(nodes, (size_t)blocks * (OPT_BLOCK + 1) * 2 * sizeof(uint4))) return rc;
	if (int rc = dev_alloc(dnodes, sizeof(unsigned long long))) return rc;
	CU(cudaMemcpyAsync(dbounds.p, bounds.data(), sizeof(uint32_t) * (nregions + 1), cudaMemcpyHostToDevice, ctx->stream));
	CU(cudaMemsetAsync(abs.p, 0, (size_t)n * 4, ctx->stream));
	CU(cudaMemsetAsync(dnodes.p, 0, sizeof(unsigned long long), ctx->stream));
	fill_literal_kernel<<<grid_for(n, 256, ctx->sm_count * 8), 256, 0, ctx->stream>>>(slab.as<uint64_t>(), n);
	CU(cudaGetLastError());
	MatchListArgs ml;
	ml.data = ctx->d_data;
	ml.n = n;
	ml.occ_start = ctx->d_occ_start;
	ml.occ = ctx->d_occ;
	ml.max_occ = max_occ;
	ml.lists = lists.as<uint2>();
	ml.counts = counts.as<uint8_t>();
	OptimalArgs o;
	o.data = ctx->d_data;
	o.n = n;
	o.trans = ctx->d_trans;
	o.lists = lists.as<uint2>();
	o.counts = counts.as<uint8_t>();
	o.bounds = dbounds.as<uint32_t>();
	o.nregions = nregions;
	o.nodes = nodes.as<uint4>();
	o.slab = slab.as<uint64_t>();
	o.abs_dist = abs.as<uint32_t>();
	o.nodes_relaxed = dnodes.as<unsigned long long>();
	cudaEvent_t t0, t1;
	CU(cudaEventCreate(&t0));
	CU(cudaEventCreate(&t1));
	CU(cudaEventRecord(t0, ctx->stream));
	matchlist_kernel<<<grid_for((size_t)n * 32, 256, ctx->sm_count * 64), 256, 0, ctx->stream>>>(ml);
	optimal_kernel<<<blocks, 32, 0, ctx->stream>>>(o);
	CU(cudaEventRecord(t1, ctx->stream));
	CU(cudaGetLastError());
	unsigned long long relaxed = 0;
	CU(cudaMemcpyAsync(&relaxed, dnodes.p, sizeof(relaxed), cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	{
		float ms = 0;
		cudaEventElapsedTime(&ms, t0, t1);
		ctx->last_optimal_ms = ms;
		ctx->last_optimal_nodes = relaxed;
		cudaEventDestroy(t0);
		cudaEventDestroy(t1);
	}
	return mg_anneal_merge_import(an, slab.p, abs.p, dst_chain, cost_out);
}

extern "C" MG_API int mg_optimal_stats(const mg_ctx* ctx, double* kernel_ms, uint64_t* nodes)
{
	if (!ctx) return fail(MG_EINVAL, "mg_optimal_stats: null context");
	if (kernel_ms) *kernel_ms = ctx->last_optimal_ms;
	if (nodes) *nodes = ctx->last_optimal_nodes;
	return MG_OK;
}

extern "C" MG_API int mg_anneal_broadcast_chain(mg_anneal* an, uint32_t src_chain)
{
	if (!an || src_chain >= an->p.chains) return fail(MG_EINVAL, "mg_anneal_broadcast_chain: bad argument");
	mg_ctx* ctx = an->ctx;
	CU(cudaSetDevice(ctx->device));
	const size_t n = ctx->n, nck = an->nck;
	const uint32_t C = an->p.chains;
	if (C == 1) return MG_OK;
	if (src_chain != 0) {
		CU(cudaMemcpyAsync(an->d_slabs, an->d_slabs + (size_t)src_chain * n, n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
		if (nck) {
			CU(cudaMemcpyAsync(an->d_ck, an->d_ck + (size_t)src_chain * 2 * nck, 2 * nck * sizeof(Record), cudaMemcpyDeviceToDevice, ctx->stream));
			CU(cudaMemcpyAsync(an->d_ck_meta, an->d_ck_meta + (size_t)src_chain * 2 * nck, 2 * nck * sizeof(CkMeta), cudaMemcpyDeviceToDevice, ctx->stream));
			CU(cudaMemcpyAsync(an->d_ck_live, an->d_ck_live + (size_t)src_chain * nck, nck, cudaMemcpyDeviceToDevice, ctx->stream));
		}
	}
	if (int rc = replicate(ctx, an->d_slabs, an->d_slabs + n, n * 8, n * 8, C - 1)) return rc;
	if (nck) {
		if (int rc = replicate(ctx, an->d_ck, an->d_ck + 2 * nck, 2 * nck * sizeof(Record), 2 * nck * sizeof(Record), C - 1)) return rc;
		if (int rc = replicate(ctx, an->d_ck_meta, an->d_ck_meta + 2 * nck, 2 * nck * sizeof(CkMeta), 2 * nck * sizeof(CkMeta), C - 1)) return rc;
		if (int rc = replicate(ctx, an->d_ck_live, an->d_ck_live + nck, nck, nck, C - 1)) return rc;
	}
	std::vector<ChainState> st(C);
	CU(cudaStreamSynchronize(ctx->stream));
	CU(cudaMemcpy(st.data(), an->d_state, (size_t)C * sizeof(ChainState), cudaMemcpyDeviceToHost));
	const ChainState src = st[src_chain];
	for (uint32_t c = 0; c < C; c++) {
		st[c].cur_cost = src.slab_cost;
		st[c].slab_cost = src.slab_cost;
		st[c].live_count = src.live_count;
		st[c].susp_slot = 0;
		st[c].err = 0;
		st[c].journal_count = 0;
		st[c].journal_overflow = 1;  // the best slabs stay where they are, the current ones moved
		an->have_slab[c] = 1;
	}
	CU(cudaMemcpy(an->d_state, st.data(), (size_t)C * sizeof(ChainState), cudaMemcpyHostToDevice));
	return MG_OK;
}

extern "C" MG_API int mg_anneal_oneshot(mg_ctx* ctx, const mg_anneal_params* params, const mg_anneal_run_params* run,
                                 const LZMAPacket* init, LZMAPacket* best_slab_out, uint64_t* best_cost,
                                 mg_anneal_stats* stats)
{
	if (!ctx || !params || !run || !best_slab_out) return fail(MG_EINVAL, "mg_anneal_oneshot: null argument");
	mg_anneal_params p = *params;
	p.track_best = 1;
	mg_anneal* an = nullptr;
	int rc = mg_anneal_create(ctx, &p, &an);
	if (rc) return rc;
	rc = mg_anneal_set_slab(an, 0, p.chains, init, init ? 1 : 0, 1);
	if (!rc) rc = mg_anneal_run(an, run, stats);
	if (!rc) {
		std::vector<uint64_t> best(p.chains);
		rc = mg_anneal_costs(an, nullptr, best.data());
		if (!rc) {
			uint32_t arg = 0;
			for (uint32_t c = 1; c < p.chains; c++)
				if (best[c] != 0 && (best[arg] == 0 || best[c] < best[arg])) arg = c;
			if (best[arg] == 0) {
				rc = fail(MG_ESTATE, "mg_anneal_oneshot: no chain completed an evaluation");
			} else {
				if (best_cost) *best_cost = best[arg];
				rc = mg_anneal_get_slab(an, arg, 1, best_slab_out);
			}
		}
	}
	mg_anneal_destroy(an);
	return rc;
}

#include "mg_comm.inc"
