// mgb_engine.cu -- host side of libmgb200.so: model construction, batch dispatcher and the C ABI (include/mgb200.h).
//
// Compiled by nvcc for sm_100a into the product library.  With -DMGB_HOSTSIM the same file is compiled by g++ into
// tests/hostsim/libmgb_hostsim.so, where "device memory" is host memory and a "launch" is a loop over reads with a
// single lane: that build exists only so that the CPU-only unit tests can exercise the control flow of the kernels.
// It is never loaded by the product path; the product library refuses to work without a CUDA device.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <vector>
#include <algorithm>
#include <string>
#include <chrono>
#include <thread>
#include <mutex>
#include <condition_variable>
#include <functional>
#include <unordered_map>
#include "mgb_hostpool.h"

#include "../../include/mgb200.h"
#include "mgb_galign.cuh"
#include "mgb_gaf.cuh"

#ifndef MGB_HOSTSIM
#include <cuda_runtime.h>
#include "mgb_index.cuh"
#endif

using namespace mgb;

// ---------------------------------------------------------------------------------------------------------------
// errors, parameters
// ---------------------------------------------------------------------------------------------------------------

static std::string g_last_error;
static void set_error(const std::string &s) { g_last_error = s; fprintf(stderr, "[E::mgb200] %s\n", s.c_str()); }

static int64_t p_arena_mb = 6;        // per worker, first pass
static int64_t p_arena_big_mb = 1024; // per worker, retry pass
static int64_t p_workers_per_sm = 32;
static int64_t p_device = 0;
static int64_t p_host_threads = 0; // 0: min(16, hardware threads)
static int64_t p_slots = 3;            // mg_map_batch calls that may run at once on one index (each on its own slot: stream, buffers, arenas)
static int64_t p_slot_workers = 0;
static int64_t p_tier_learn = 1;       // 0: every gap tries every tier (no routing)
static int64_t p_index_dev = 1;        // 0: the minimizer table is grouped and laid out on the host (std::sort) instead of on the device
static int64_t p_gpu_lock = 1;         // 0: the kernels of concurrent calls may interleave on the device
static int64_t p_pack2 = 1;            // 0: reads are uploaded as ASCII (1 byte per base) instead of 2 bits per base
static int64_t p_lab_cache = 1;        // 0: graph chaining searches its walks per read instead of keeping per-source labels in HBM (mgb_gclabel.cuh)

// ---- the kernel stages, one row each ----
// A stage's number is its key in mgb_set_param ("sw<N>", "mb<N>"), its slot in mgb_stats_t::t_kernel_ms (stages below 10) and what
// the profiles call it.  Columns: kernel, stage, number; the kernel's __launch_bounds__ (threads per block, blocks per SM); the
// launch shape (warps per block, blocks per SM wanted) until "sw<N>" / "mb<N>" lower it; shared memory per warp; how an item is
// entered; items taken per ticket.  Entry: ENTER_WARP, all lanes of the warp run the item; ENTER_LANE0, lane 0 alone with the whole
// arena of its warp; ENTER_THREAD, every thread runs its own item in 1/32 of the warp's arena (the hardware interleaves the 32
// diverged lanes, so their memory latencies overlap).  k_wfa_mid is the one kernel launched in smaller blocks than it is compiled for.
#ifndef MGB_BIG_MINB
#define MGB_BIG_MINB 4 // blocks of k_wfa_big per SM (its register budget follows: 80 at 6, 96 at 5, 128 at 4)
#endif
#ifndef MGB_GWFA_MINB
#define MGB_GWFA_MINB 4
#endif
#define MGB_STAGES(X) \
	X(k_seed,          ST_SEED,          0, (128, 8),             4, 8,             SKETCH_SMEM_BYTES,       ENTER_WARP,   1) /* K1-K3: sketch, index lookup, seed sort */ \
	X(k_chain,         ST_CHAIN,         1, (224, 2),             7, 2,             CHAIN_SMEM_BYTES,        ENTER_WARP,   1) /* K4/K5: linear chaining on chip (seeds bulk-loaded into shared memory; 2 x 7 slices of 16 KB per SM) */ \
	X(k_gchain,        ST_GCHAIN,        2, (128, 8),             4, 8,             0,                       ENTER_WARP,   1) /* K6: graph chaining DP + k-shortest walks, overlap resolution, bridging plan */ \
	X(k_index_sketch,  ST_INDEX_SKETCH,  3, (128, 8),             4, 8,             0,                       ENTER_LANE0,  1) /* index build: sketch of graph segments */ \
	X(k_wfa_small,     ST_WFA1,          4, (128, 5),             4, 5,             WfTier1::STRIDE,         ENTER_WARP,   4) /* K8a tier 1: small gaps, wavefronts + traceback bytes in shared memory */ \
	X(k_finish,        ST_FINISH,        5, (128, 8),             4, 8,             0,                       ENTER_WARP,   1) /* K8b: CIGAR stitching, ds strings, result blobs */ \
	X(k_wfa_mid,       ST_WFA2,          6, (128, 5),             2, 7,             WfTier2::STRIDE,         ENTER_WARP,   4) /* K8a tier 2: mid-size gaps, wavefronts in shared memory */ \
	X(k_wfa_big,       ST_WFA3,          7, (128, MGB_BIG_MINB),  4, MGB_BIG_MINB,  0,                       ENTER_WARP,   1) /* K8a tier 3: anything else, wavefronts in the worker arena */ \
	X(k_gwfa,          ST_GWFA,          8, (128, MGB_GWFA_MINB), 4, MGB_GWFA_MINB, GWFA_SMEM_ARENA,         ENTER_WARP,   1) /* K7a: bridging alignments (graph wavefront), one warp per bridge */ \
	X(k_gchain_gen,    ST_GCHAIN_GEN,    9, (128, 4),             4, 4,             0,                       ENTER_WARP,   1) /* K7b: graph-chain materialisation, post filters, mapq, alignment plan */ \
	X(k_gc_labels,     ST_LABELS,       17, (128, 8),             4, 8,             0,                       ENTER_THREAD, 1) /* reachability labels of new source vertices (mgb_gclabel.cuh) */ \
	X(k_gc_labels_big, ST_LABELS_BIG,   18, (128, 8),             4, 8,             0,                       ENTER_LANE0,  1) /* the few sources whose search outgrew a thread's share of the arena */ \
	X(k_chain_rescue,  ST_CHAIN_RESCUE, 19, (192, 2),             6, 2,             CHAIN_RESCUE_SMEM_BYTES, ENTER_WARP,   1) /* K5: long-join rescue (RMQ chaining) of the reads k_chain listed (2 x 6 slices of 18 KB) */ \
	X(k_gaf_size,      ST_GAF_SIZE,     10, (128, 8),             4, 8,             0,                       ENTER_WARP,   1) /* mgb_map_batch_gaf: bytes and dv:f fix-ups of a read's GAF text (mgb_gaf.cuh) */ \
	X(k_gaf_write,     ST_GAF_WRITE,    11, (128, 8),             4, 8,             0,                       ENTER_WARP,   1) /* mgb_map_batch_gaf: the text itself, at the read's place after the scan */
enum StageEntry { ENTER_WARP, ENTER_LANE0, ENTER_THREAD };
enum Stage {
#define MGB_STAGE_ENUM(kern, st, num, ...) st = num,
	MGB_STAGES(MGB_STAGE_ENUM)
#undef MGB_STAGE_ENUM
};
struct StageShapes { int warps[20], minb[20]; }; // indexed by stage number
static StageShapes default_shapes()
{
	StageShapes s = {};
#define MGB_STAGE_SHAPE(kern, st, num, bounds, w, b, ...) s.warps[num] = (w), s.minb[num] = (b);
	MGB_STAGES(MGB_STAGE_SHAPE)
#undef MGB_STAGE_SHAPE
	return s;
}
static StageShapes g_shape = default_shapes(); // the launch shape in use

extern "C" const char *mgb_last_error(void) { return g_last_error.c_str(); }
extern "C" const char *mgb_version(void) { return "mgb200-r1"; }
extern "C" int mgb_set_param(const char *key, int64_t value)
{
	if (!strcmp(key, "arena_mb")) p_arena_mb = value;
	else if (!strcmp(key, "arena_big_mb")) p_arena_big_mb = value;
	else if (!strcmp(key, "workers_per_sm")) p_workers_per_sm = value;
	else if (!strcmp(key, "device")) p_device = value;
	else if (!strcmp(key, "host_threads")) p_host_threads = value;
	else if (!strcmp(key, "slots")) p_slots = value;
	else if (!strcmp(key, "slot_workers")) p_slot_workers = value;
	else if (!strcmp(key, "lab_cache")) p_lab_cache = value;
	else if (!strcmp(key, "pack2")) p_pack2 = value;
	else if (!strcmp(key, "gpu_lock")) p_gpu_lock = value;
	else if (!strcmp(key, "index_dev")) p_index_dev = value;
	else if (!strcmp(key, "tier_learn")) p_tier_learn = value;
	else if (!strncmp(key, "sw", 2) && key[2] >= '0' && key[2] <= '9' && !key[3] && value >= 1 && value <= 4) g_shape.warps[key[2] - '0'] = (int)value;
	else if (!strncmp(key, "mb", 2) && key[2] >= '0' && key[2] <= '9' && !key[3] && value >= 1 && value <= 32) g_shape.minb[key[2] - '0'] = (int)value;
	else return -1;
	return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// device memory shim
// ---------------------------------------------------------------------------------------------------------------

static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
// kernels launched by the calling thread (every launcher counts its own): mgb_stats_t::n_launches is the difference over a batch
static thread_local int64_t t_launches = 0;

#ifdef MGB_HOSTSIM
typedef void *DevStream;
typedef double DevEvent; // the host clock when it was recorded
struct MgbError { int code; };
static bool dev_ok(int dev = -1) { (void)dev; return true; }
static void set_device(int dev) { (void)dev; }
static void set_stream(DevStream s) { (void)s; }
static void *dmalloc(size_t n) { void *p = malloc(n? n : 16); return p; }
static void dfree(void *p) { free(p); }
static void h2d(void *d, const void *h, size_t n) { if (n) memcpy(d, h, n); }
static void d2h(void *h, const void *d, size_t n) { if (n) memcpy(h, d, n); }
static void dzero(void *d, size_t n) { if (n) memset(d, 0, n); }
static void d2d(void *d, const void *s, size_t n) { if (n) memcpy(d, s, n); }
static void dfill(void *d, int v, size_t n) { if (n) memset(d, v, n); }
static void dsync() {}
static void h2d_async(void *d, const void *h, size_t n) { if (n) memcpy(d, h, n); }
static void d2h_async(void *h, const void *d, size_t n) { if (n) memcpy(h, d, n); }
static void ev_record(DevEvent &e) { e = now_ms(); }
static void ev_wait(DevEvent e) { (void)e; }
static double ev_elapsed_ms(DevEvent a, DevEvent b) { return b - a; }
static int dev_sm_count() { return 2; }
static size_t dev_free_mem() { return (size_t)8 << 30; }
struct EvTimer { double t0 = 0, t1 = 0; void start() { t0 = now_ms(); } void stop() { t1 = now_ms(); } double ms() { return t1 - t0; } void clear() { t0 = t1 = 0; } };
#else
// A failed CUDA call (out of memory, a fault in a kernel) unwinds to the C entry point, which returns NULL / a negative code with
// the reason in mgb_last_error(); the library never ends the host process on its own.
struct MgbError { int code; };
#define CUDA_OK(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) { set_error(std::string(#call) + ": " + cudaGetErrorString(_e)); throw MgbError{MGB_E_INTERNAL}; } } while (0)
typedef cudaStream_t DevStream;
typedef cudaEvent_t DevEvent;
// every host thread that drives a slot of the batch pipeline works on its own stream
static thread_local cudaStream_t t_stream = 0;
static bool dev_ok(int dev = -1)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return false;
	if (cudaSetDevice(dev >= 0? dev : (int)p_device) != cudaSuccess) return false;
	return true;
}
static void set_device(int dev) { cudaSetDevice(dev); }
static void set_stream(DevStream s) { t_stream = s; }
static void *dmalloc(size_t n) { void *p = 0; CUDA_OK(cudaMalloc(&p, n? n : 16)); return p; }
static void dfree(void *p) { if (p) cudaFree(p); }
static void dsync() { CUDA_OK(cudaStreamSynchronize(t_stream)); }
static void h2d(void *d, const void *h, size_t n) { if (n) { CUDA_OK(cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, t_stream)); dsync(); } }
static void d2h(void *h, const void *d, size_t n) { if (n) { CUDA_OK(cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, t_stream)); dsync(); } }
static void dzero(void *d, size_t n) { if (n) CUDA_OK(cudaMemsetAsync(d, 0, n, t_stream)); }
static void d2d(void *d, const void *s, size_t n) { if (n) CUDA_OK(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToDevice, t_stream)); }
static void dfill(void *d, int v, size_t n) { if (n) CUDA_OK(cudaMemsetAsync(d, v, n, t_stream)); }
static void h2d_async(void *d, const void *h, size_t n) { if (n) CUDA_OK(cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, t_stream)); }
static void d2h_async(void *h, const void *d, size_t n) { if (n) CUDA_OK(cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, t_stream)); }
static void ev_record(DevEvent e) { CUDA_OK(cudaEventRecord(e, t_stream)); }
static void ev_wait(DevEvent e) { CUDA_OK(cudaEventSynchronize(e)); }
static double ev_elapsed_ms(DevEvent a, DevEvent b) { float t = 0; return cudaEventElapsedTime(&t, a, b) == cudaSuccess? t : 0; }
struct EvTimer {
	cudaEvent_t a, b; bool used;
	EvTimer() : used(false) { cudaEventCreate(&a); cudaEventCreate(&b); }
	~EvTimer() { cudaEventDestroy(a); cudaEventDestroy(b); }
	void start() { cudaEventRecord(a, t_stream); used = true; }
	void stop() { cudaEventRecord(b, t_stream); }
	double ms() { if (!used) return 0; float t = 0; cudaEventSynchronize(b); cudaEventElapsedTime(&t, a, b); return t; }
	void clear() { used = false; }
};
static int dev_sm_count() { static int v = 0; if (v == 0) { int d = 0; CUDA_OK(cudaGetDevice(&d)); CUDA_OK(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, d)); } return v; } // (the devices of one box are alike)
static size_t dev_free_mem() { size_t f = 0, t = 0; CUDA_OK(cudaMemGetInfo(&f, &t)); return f; }
#endif

// the timers of a batch's first pass
struct SlotTimers {
	EvTimer h2d, seed, chain, align, wfa, fin, d2h, lab, gaf_size, gaf_write, k[10]; // k: per kernel slot of mgb_stats_t::t_kernel_ms
	void reset() { EvTimer *all[] = {&h2d, &seed, &chain, &align, &wfa, &fin, &d2h, &lab, &gaf_size, &gaf_write}; for (EvTimer *t : all) t->clear(); for (int i = 0; i < 10; ++i) k[i].clear(); }
};
// a timer around a scope; none: the scope is not timed
struct Span {
	EvTimer *t;
	explicit Span(EvTimer *t_) : t(t_) { if (t) t->start(); }
	~Span() { if (t) t->stop(); }
};

template<typename T> static T *dalloc_copy(const std::vector<T> &v)
{
	T *d = (T*)dmalloc(v.size() * sizeof(T));
	h2d(d, v.data(), v.size() * sizeof(T));
	return d;
}

// grow-only buffers kept across batches: device memory, or page-locked host memory for fast H2D/D2H
struct GrowBuf {
	void *p; size_t cap; bool host;
	GrowBuf(bool host_ = false) : p(0), cap(0), host(host_) {}
	GrowBuf(const GrowBuf &) = delete;
	~GrowBuf() { release(); }
	void release()
	{
		if (p == 0) return;
#ifdef MGB_HOSTSIM
		free(p);
#else
		if (host) cudaFreeHost(p); else cudaFree(p);
#endif
		p = 0, cap = 0;
	}
	void *ensure(size_t n)
	{
		if (n <= cap && p) return p;
		release();
		size_t c = n + n / 4 + 4096;
#ifdef MGB_HOSTSIM
		p = malloc(c);
#else
		if (host) CUDA_OK(cudaHostAlloc(&p, c, cudaHostAllocDefault)); else CUDA_OK(cudaMalloc(&p, c));
#endif
		cap = c;
		return p;
	}
};

static int n_host_threads() // "host_threads"; 0: min(16, hardware threads)
{
	const int nt = (int)p_host_threads;
	if (nt > 0) return nt;
	return std::min(16, std::max(1, (int)std::thread::hardware_concurrency()));
}

namespace {
static mgb::HostPool g_host_pool; // packing, result assembly, index build (one caller at a time)
template<typename F> void parallel_for(int64_t n, F fn)
{
	const int nt = n_host_threads();
	if (n < 64 || nt == 1) { for (int64_t i = 0; i < n; ++i) fn(i); return; }
	const std::function<void(int64_t)> f = fn;
	g_host_pool.run(n, nt, f);
}
}

// ---------------------------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------------------------

struct LaunchArgs {
	PipeCtx c;
	ReadOut *routs;
	const int32_t *rid_list; // NULL: reads 0..n-1
	int32_t n_work;
	const unsigned int *n_work_dev; // non-NULL: the number of items is read on the device (known only after the kernel in front)
	char *arena_base;
	uint64_t arena_bytes;
	uint64_t *arena_peak;    // per worker
	int64_t job_start;       // first job of this launch (stage 4)
	// segment sketch (index build)
	Pool *pool_mz; u128 *mz;
	const GafCtx *gaf;       // k_gaf_size / k_gaf_write (device memory)
};

// the columns of the stage table that the device code reads
template<int STAGE> struct StageRow;
#define MGB_STAGE_ROW(kern, st, num, bounds, warps, blocks, smem, entry, grab) \
	template<> struct StageRow<st> { static constexpr int SMEM = smem, GRAB = grab; static constexpr StageEntry ENTRY = entry; };
MGB_STAGES(MGB_STAGE_ROW)
#undef MGB_STAGE_ROW

template<int STAGE>
MG_HD inline int run_stage(const LaunchArgs &L, int item, Arena &A, int lane, int32_t *smem)
{
	switch (STAGE) {
	case ST_SEED: return stage_seed(L.c, item, A, lane, smem);
	case ST_CHAIN: return stage_chain<0>(L.c, item, A, lane, smem);
	case ST_CHAIN_RESCUE: return stage_chain<1>(L.c, L.c.rescue_list[item], A, lane, smem); // the reads k_chain listed
	case ST_GCHAIN: return stage_gchain(L.c, L.routs, item, A, lane);
	case ST_LABELS: return label_job(A, L.c.g, L.c.lab, item, 0);
	case ST_LABELS_BIG: return label_job(A, L.c.g, L.c.lab, item, 1);
	case ST_FINISH: return stage_finish(L.c, L.routs, item, A, lane);
	case ST_GWFA: return gwfa_job_run(A, L.c, L.job_start + item, lane, smem);
	case ST_GCHAIN_GEN: return stage_gchain_gen(L.c, L.routs, item, A, lane);
	case ST_WFA1: return wfa_job_run(A, L.c, L.job_start + item, lane, smem, 1);
	case ST_WFA2: return wfa_job_run(A, L.c, L.c.jobq[0][item], lane, smem, 2);
	case ST_WFA3: return wfa_job_run(A, L.c, L.c.jobq[1][item], lane, smem, 3);
	case ST_GAF_SIZE: return stage_gaf_size(*L.gaf, L.c, L.routs, item, lane);
	case ST_GAF_WRITE: return stage_gaf_write(*L.gaf, L.c, L.routs, item, lane);
	case ST_INDEX_SKETCH: { // sketch one graph segment for the index (reference: index.c:200-205)
		AVec<u128> mv;
		avec_init(mv);
		int32_t len = L.c.g.seg_len[item];
		if (len <= 0) return 0;
		MGB_TRY(sketch_seq(A, g_vseq(L.c.g, (uint32_t)item << 1), len, L.c.ix.w, L.c.ix.k, (uint32_t)item, mv));
		int64_t off = pool_alloc(L.pool_mz, (uint64_t)mv.n * sizeof(u128));
		if (off < 0) return MGB_E_POOL;
		u128 *dst = L.mz + off / (int64_t)sizeof(u128);
		for (int64_t i = 0; i < mv.n; ++i) dst[i] = mv.a[i];
		return 0;
	}
	}
	return MGB_E_INTERNAL;
}

// record a failure: per read for the mapping stages, a single status word for the index build
template<int STAGE>
MG_HD inline void stage_fail(const LaunchArgs &L, int item, int rc)
{
	int rid = item; // the read the item belongs to
	switch (STAGE) {
	case ST_LABELS: case ST_LABELS_BIG: return; // a source that could not be finished is searched again by the read that needs it
	case ST_INDEX_SKETCH:
#if MGB_ON_DEVICE
		atomicMin((int*)L.routs, rc);
#else
		if (rc < *(int*)L.routs) *(int*)L.routs = rc;
#endif
		return;
	case ST_CHAIN_RESCUE: rid = L.c.rescue_list[item]; break;
	case ST_GWFA: rid = L.c.gjobs[L.job_start + item].rid; break;
	case ST_WFA1: rid = L.c.jobs[L.job_start + item].rid; break;
	case ST_WFA2: rid = L.c.jobs[L.c.jobq[0][item]].rid; break;
	case ST_WFA3: rid = L.c.jobs[L.c.jobq[1][item]].rid; break;
	default: break;
	}
	L.c.meta[rid].status = rc; // benign race between jobs of one read: any negative code triggers the redo
	L.routs[rid].status = rc;
}

#ifndef MGB_HOSTSIM
// One warp per work item; items are pulled from a global counter so that long items do not stall a wave.
// Every mapping stage is warp-uniform (all lanes enter the stage function, see mgb_common.cuh).
template<int STAGE>
__device__ __forceinline__ void stage_loop(const LaunchArgs &L)
{
	const int lane = threadIdx.x & 31;
	const int worker = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
	Arena A;
	arena_init(A, L.arena_base + (uint64_t)worker * L.arena_bytes, L.arena_bytes);
	extern __shared__ int4 dyn_smem[];
	const int smem_stride = StageRow<STAGE>::SMEM;
	int32_t *smem = smem_stride? (int32_t*)((char*)dyn_smem + (size_t)(threadIdx.x >> 5) * smem_stride) : 0;
	if (STAGE == ST_CHAIN || STAGE == ST_CHAIN_RESCUE) chain_smem_init(smem, lane);
	if ((STAGE == ST_WFA1 || STAGE == ST_WFA2) && lane == 0) { unsigned long long *ck = wfa_cig_chunk(smem, STAGE == ST_WFA1? 1 : 2); ck[0] = ck[1] = 0; } // no slice of the CIGAR pool yet
	prof_block_begin();
	const int n_work = L.n_work_dev? (int)*L.n_work_dev : L.n_work;
	const int grab = StageRow<STAGE>::GRAB; // the short jobs of the on-chip WFA tiers are taken four at a time: one contended ticket per four jobs
	int next_item = 0, have = 0;
	for (;;) {
		if (have == 0) {
			if (lane == 0) next_item = (int)atomicAdd(L.c.next_read, (unsigned int)grab);
			next_item = __shfl_sync(0xffffffffu, next_item, 0);
			have = grab;
		}
		int item = next_item++;
		--have;
		if (item >= n_work) break;
		if (L.rid_list) item = L.rid_list[item];
		if (StageRow<STAGE>::ENTRY == ENTER_WARP) {
			A.top = 0;
			int rc = run_stage<STAGE>(L, item, A, lane, smem);
			if (rc < 0 && lane == 0) stage_fail<STAGE>(L, item, rc);
		} else if (lane == 0) {
			A.top = 0;
			int rc = run_stage<STAGE>(L, item, A, 0, 0);
			if (rc < 0) stage_fail<STAGE>(L, item, rc);
		}
		__syncwarp();
	}
	if (lane == 0 && L.arena_peak) L.arena_peak[worker] = A.peak > L.arena_peak[worker]? A.peak : L.arena_peak[worker];
	prof_block_end(L.c.prof);
}

// Thread-per-item variant (ENTER_THREAD) for the stages whose control flow is sequential: every THREAD pulls its own item
// and owns 1/32 of the warp's arena.  The 32 lanes of a warp diverge completely, but the hardware interleaves the diverged
// lanes, so 32x more items are in flight per warp and their memory latencies overlap.
template<int STAGE>
__device__ __forceinline__ void stage_loop_thread(const LaunchArgs &L)
{
	const int lane = threadIdx.x & 31;
	const int worker = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
	const uint64_t sub = (L.arena_bytes / 32) & ~(uint64_t)15;
	Arena A;
	arena_init(A, L.arena_base + (uint64_t)worker * L.arena_bytes + (uint64_t)lane * sub, sub);
	prof_block_begin();
	const int n_work = L.n_work_dev? (int)*L.n_work_dev : L.n_work;
	for (;;) {
		int item = (int)atomicAdd(L.c.next_read, 1u);
		if (item >= n_work) break;
		if (L.rid_list) item = L.rid_list[item];
		A.top = 0;
		int rc = run_stage<STAGE>(L, item, A, -1, 0);
		if (rc < 0) stage_fail<STAGE>(L, item, rc);
	}
	if (L.arena_peak) atomicMax((unsigned long long*)&L.arena_peak[worker], (unsigned long long)A.peak);
	prof_block_end(L.c.prof);
}

// One named kernel per stage (so that profiles read well), each running the one loop its entry needs.  The choice is a plain if
// on a constant, not if constexpr: with the unused loop left out of the source, nvcc stops inlining chain_rmq_fill_seq into
// k_chain_rescue, which then needs more registers and stack.
typedef void (*StageFn)(LaunchArgs);
template<int STAGE> static StageFn stage_kernel();
#define MGB_STAGE_KERNEL(kern, st, num, bounds, ...) \
	__global__ void __launch_bounds__ bounds kern(LaunchArgs L) \
	{ if (StageRow<st>::ENTRY == ENTER_THREAD) stage_loop_thread<st>(L); else stage_loop<st>(L); } \
	template<> StageFn stage_kernel<st>() { return kern; }
MGB_STAGES(MGB_STAGE_KERNEL)
#undef MGB_STAGE_KERNEL
#endif

// Longest-first order of a job list (a tail of a few long jobs otherwise decides the kernel time).  Jobs are binned by
// size, four bins per octave, largest first; the order inside a bin does not matter (results do not depend on it).
MG_HD inline int order_bin(uint32_t key)
{
	uint32_t x = key + 1, lz = 0;
	while ((x >> lz) > 1) ++lz; // floor(log2(x))
	int b = (int)(lz * 4 + (lz >= 2? ((x >> (lz - 2)) & 3) : 0));
	return 63 - (b > 63? 63 : b);
}
// ORDER_BRIDGES: bridging jobs [job_start, job_start+n), key = query length; ORDER_GAPS: alignment jobs listed in q[0..n), key = tl + ql;
// ORDER_READS: reads 0..n-1, key = number of linear chains
enum { NO_ORDER = -1, ORDER_BRIDGES, ORDER_GAPS, ORDER_READS };
MG_HD inline uint32_t order_key(const LaunchArgs &L, int kind, const int32_t *q, int i)
{
	if (kind == ORDER_BRIDGES) return (uint32_t)L.c.gjobs[L.job_start + i].ql;
	if (kind == ORDER_READS) return (uint32_t)L.c.meta[i].n_lc; // reads by their number of linear chains (graph chaining is roughly quadratic in it)
	const WfaJob &J = L.c.jobs[q[i]];
	return (uint32_t)(J.tl + J.ql);
}
#ifndef MGB_HOSTSIM
__global__ void __launch_bounds__(1024) k_job_order(LaunchArgs L, int kind, const int32_t *q, int n, const unsigned int *n_dev, int32_t *order)
{
	if (n_dev) n = (int)*n_dev;
	__shared__ unsigned int cnt[64];
	const int tid = threadIdx.x;
	if (tid < 64) cnt[tid] = 0;
	__syncthreads();
	for (int i = tid; i < n; i += 1024) atomicAdd(&cnt[order_bin(order_key(L, kind, q, i))], 1u);
	__syncthreads();
	if (tid == 0) { unsigned int acc = 0; for (int b = 0; b < 64; ++b) { unsigned int c = cnt[b]; cnt[b] = acc; acc += c; } }
	__syncthreads();
	for (int i = tid; i < n; i += 1024) order[atomicAdd(&cnt[order_bin(order_key(L, kind, q, i))], 1u)] = i;
}
#endif
static void make_job_order(const LaunchArgs &L, int kind, const int32_t *q, int n, int32_t *order, const unsigned int *n_dev)
{
	++t_launches;
#ifndef MGB_HOSTSIM
	k_job_order<<<1, 1024, 0, t_stream>>>(L, kind, q, n, n_dev, order);
	CUDA_OK(cudaGetLastError());
#else
	if (n_dev) n = (int)*n_dev;
	unsigned int cnt[65] = {0};
	for (int i = 0; i < n; ++i) ++cnt[order_bin(order_key(L, kind, q, i)) + 1];
	for (int b = 0; b < 64; ++b) cnt[b + 1] += cnt[b];
	for (int i = 0; i < n; ++i) order[cnt[order_bin(order_key(L, kind, q, i))]++] = i;
#endif
}

// ---- result blobs in read order ----
// The kernels allocate a read's two result blobs from the output pool in completion order.  Before the copy to the host they are
// closed up in read order, so that the copy can go in a few pieces and the host threads can build the mg_gchains_t of one piece
// while the next one is still on the wire.
struct PackArgs { ReadOut *routs; const ReadMeta *meta; int n; const char *pool; char *packed; uint64_t *off; };
MG_HD inline uint64_t pack_size(const PackArgs &P, int r)
{
	const ReadOut &ro = P.routs[r];
	if (P.meta[r].status != 0 || ro.status != 0 || ro.n_gc <= 0) return 0;
	return (((uint64_t)ro.blob_size + 15) & ~(uint64_t)15) + (((uint64_t)ro.blob2_size + 15) & ~(uint64_t)15);
}
MG_HD inline void pack_read(const PackArgs &P, int r, int lane, int nl)
{
	ReadOut &ro = P.routs[r];
	const uint64_t sz = P.off[r + 1] - P.off[r];
	if (sz == 0) return;
	const uint64_t n1 = ((uint64_t)ro.blob_size + 15) & ~(uint64_t)15, n2 = sz - n1;
	const uint64_t *s1 = (const uint64_t*)(P.pool + ro.blob_off), *s2 = (const uint64_t*)(P.pool + ro.blob2_off);
	uint64_t *d1 = (uint64_t*)(P.packed + P.off[r]), *d2 = d1 + n1 / 8;
	for (uint64_t i = lane; i < n1 / 8; i += nl) d1[i] = s1[i];
	for (uint64_t i = lane; i < n2 / 8; i += nl) d2[i] = s2[i];
#if MGB_ON_DEVICE
	__syncwarp();
#endif
	const int64_t delta = (int64_t)(P.off[r] + n1) - ro.blob2_off;
	GChain *gc = (GChain*)d1;
	for (int i = lane; i < ro.n_gc; i += nl)
		if (gc[i].has_cigar) gc[i].cigar_off += delta, gc[i].ds_off += delta, gc[i].dsoff_off += delta;
	if (lane == 0) ro.blob_off = (int64_t)P.off[r], ro.blob2_off = (int64_t)(P.off[r] + n1);
}
#ifndef MGB_HOSTSIM
__global__ void __launch_bounds__(1024) k_out_scan(PackArgs P)
{
	__shared__ uint64_t part[1024];
	const int tid = threadIdx.x, per = (P.n + 1023) / 1024;
	const int r0 = tid * per < P.n? tid * per : P.n, r1 = r0 + per < P.n? r0 + per : P.n;
	uint64_t sum = 0;
	for (int r = r0; r < r1; ++r) sum += pack_size(P, r);
	part[tid] = sum;
	__syncthreads();
	if (tid == 0) { uint64_t acc = 0; for (int i = 0; i < 1024; ++i) { uint64_t c = part[i]; part[i] = acc; acc += c; } P.off[P.n] = acc; }
	__syncthreads();
	uint64_t acc = part[tid];
	for (int r = r0; r < r1; ++r) { P.off[r] = acc; acc += pack_size(P, r); }
}
__global__ void __launch_bounds__(256) k_out_pack(PackArgs P)
{
	const int lane = threadIdx.x & 31, warp = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), n_warp = (int)((gridDim.x * blockDim.x) >> 5);
	for (int r = warp; r < P.n; r += n_warp) pack_read(P, r, lane, 32);
}
#endif
static void pack_results(const PackArgs &P)
{
	t_launches += 2;
#ifndef MGB_HOSTSIM
	k_out_scan<<<1, 1024, 0, t_stream>>>(P);
	k_out_pack<<<dev_sm_count() * 8, 256, 0, t_stream>>>(P);
	CUDA_OK(cudaGetLastError());
#else
	uint64_t acc = 0;
	for (int r = 0; r < P.n; ++r) { P.off[r] = acc; acc += pack_size(P, r); }
	P.off[P.n] = acc;
	for (int r = 0; r < P.n; ++r) pack_read(P, r, 0, 1);
#endif
}

// ---- GAF text: exclusive scan of the per-read sizes and fix-up counts, in place ([n] receives the totals), shaped like k_out_scan ----
#ifndef MGB_HOSTSIM
__global__ void __launch_bounds__(1024) k_gaf_scan(uint64_t *a, uint64_t *b, int n)
{
	__shared__ uint64_t pa[1024], pb[1024];
	const int tid = threadIdx.x, per = (n + 1023) / 1024;
	const int r0 = tid * per < n? tid * per : n, r1 = r0 + per < n? r0 + per : n;
	uint64_t sa = 0, sb = 0;
	for (int r = r0; r < r1; ++r) sa += a[r], sb += b[r];
	pa[tid] = sa, pb[tid] = sb;
	__syncthreads();
	if (tid == 0) {
		uint64_t xa = 0, xb = 0;
		for (int i = 0; i < 1024; ++i) { const uint64_t ca = pa[i], cb = pb[i]; pa[i] = xa, pb[i] = xb; xa += ca, xb += cb; }
		a[n] = xa, b[n] = xb;
	}
	__syncthreads();
	uint64_t xa = pa[tid], xb = pb[tid];
	for (int r = r0; r < r1; ++r) { const uint64_t ca = a[r], cb = b[r]; a[r] = xa, b[r] = xb; xa += ca, xb += cb; }
}
#endif
static void gaf_scan(uint64_t *a, uint64_t *b, int n)
{
	++t_launches;
#ifndef MGB_HOSTSIM
	k_gaf_scan<<<1, 1024, 0, t_stream>>>(a, b, n);
	CUDA_OK(cudaGetLastError());
#else
	uint64_t xa = 0, xb = 0;
	for (int r = 0; r < n; ++r) { const uint64_t ca = a[r], cb = b[r]; a[r] = xa, b[r] = xb; xa += ca, xb += cb; }
	a[n] = xa, b[n] = xb;
#endif
}

// ---- reads cross PCIe 2 bits per base ----
// Host: A/C/G/T -> 0..3 (the order of seq_nt4_table, sketch.c:9-26), 32 bases per 64-bit word, base i in bits 2*(i%32).  Returns false
// when the read holds any other byte (N, lower case, IUPAC): such a read travels as ASCII, because the alignment compares raw bytes.
static bool pack_read_scalar(const char *s, int len, uint64_t *out)
{
	static uint8_t tab[256];
	static bool init = false;
	if (!init) { for (int i = 0; i < 256; ++i) tab[i] = 4; tab['A'] = 0, tab['C'] = 1, tab['G'] = 2, tab['T'] = 3; init = true; }
	unsigned bad = 0;
	for (int w = 0; w * 32 < len; ++w) {
		uint64_t x = 0;
		const int n = len - w * 32 < 32? len - w * 32 : 32;
		for (int j = 0; j < n; ++j) { const unsigned c = tab[(uint8_t)s[w * 32 + j]]; bad |= c; x |= (uint64_t)(c & 3) << (2 * j); }
		out[w] = x;
	}
	return (bad & 4) == 0;
}
#if defined(__x86_64__) && !defined(MGB_NO_SIMD_PACK)
#include <immintrin.h>
// 16 bases per step: code = (b >> 1 & 3) with G and T swapped back, checked by mapping the codes to letters again
__attribute__((target("ssse3,sse4.1,bmi2"))) static bool pack_read_simd(const char *s, int len, uint64_t *out)
{
	const __m128i letters = _mm_setr_epi8('A', 'C', 'G', 'T', 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0), three = _mm_set1_epi8(3), one = _mm_set1_epi8(1);
	int i = 0;
	unsigned ok = 0xffffu;
	for (; i + 32 <= len; i += 32) {
		uint64_t word = 0;
		for (int h = 0; h < 2; ++h) {
			const __m128i x = _mm_loadu_si128((const __m128i*)(s + i + 16 * h));
			__m128i c = _mm_and_si128(_mm_srli_epi16(x, 1), three);              // A0 C1 T2 G3
			c = _mm_xor_si128(c, _mm_and_si128(_mm_srli_epi16(c, 1), one));       // A0 C1 G2 T3
			ok &= (unsigned)_mm_movemask_epi8(_mm_cmpeq_epi8(_mm_shuffle_epi8(letters, c), x));
			const uint64_t lo = _pext_u64((uint64_t)_mm_cvtsi128_si64(c), 0x0303030303030303ULL), hi = _pext_u64((uint64_t)_mm_extract_epi64(c, 1), 0x0303030303030303ULL);
			word |= (lo | hi << 16) << (32 * h);
		}
		out[i >> 5] = word;
	}
	bool good = ok == 0xffffu;
	if (i < len) good &= pack_read_scalar(s + i, len - i, out + (i >> 5));
	return good;
}
static bool pack_read(const char *s, int len, uint64_t *out)
{
	static const bool simd = __builtin_cpu_supports("ssse3") && __builtin_cpu_supports("bmi2") && __builtin_cpu_supports("sse4.1");
	return simd? pack_read_simd(s, len, out) : pack_read_scalar(s, len, out);
}
#else
static bool pack_read(const char *s, int len, uint64_t *out) { return pack_read_scalar(s, len, out); }
#endif

// Device: the ASCII copy of the packed reads (alignment, ds strings and the sequential sketch read bytes): one 64-bit word = 32 bases =
// two 16-byte stores per lane, a warp per read.
struct UnpackArgs { const uint64_t *pk, *pk_off, *seq_off; const int32_t *seq_len; char *seq; int n_reads; };
MG_HD inline void unpack_word(const UnpackArgs &U, int r, int64_t wd)
{
	const int32_t len = U.seq_len[r];
	const uint64_t x = U.pk[U.pk_off[r] + (uint64_t)wd];
	uint32_t q[8];
	for (int j = 0; j < 8; ++j) { // four bases -> four letters: 'A' + {0, 2, 6, 19}
		uint32_t o = 0;
		for (int b = 0; b < 4; ++b) { const uint32_t c = (uint32_t)(x >> (2 * (4 * j + b))) & 3u; o |= (0x41u + ((0x13060200u >> (8 * c)) & 0xffu)) << (8 * b); }
		q[j] = o;
	}
	uint32_t *dst = (uint32_t*)(U.seq + U.seq_off[r] + (uint64_t)wd * 32);
	for (int h = 0; h < 2; ++h) // a half that starts at or behind the end of the read is not the read's to write
		if (wd * 32 + 16 * h < (int64_t)len) {
#if MGB_ON_DEVICE
			*(uint4*)(dst + 4 * h) = make_uint4(q[4 * h], q[4 * h + 1], q[4 * h + 2], q[4 * h + 3]);
#else
			for (int j = 0; j < 4; ++j) dst[4 * h + j] = q[4 * h + j];
#endif
		}
}
#ifndef MGB_HOSTSIM
__global__ void __launch_bounds__(256) k_unpack(UnpackArgs U)
{
	const int lane = threadIdx.x & 31, warp = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), n_warp = (int)((gridDim.x * blockDim.x) >> 5);
	for (int r = warp; r < U.n_reads; r += n_warp) {
		if (U.pk_off[r] == ~0ULL) continue; // uploaded as ASCII
		const int64_t nw = ((int64_t)U.seq_len[r] + 31) >> 5;
		for (int64_t wd = lane; wd < nw; wd += 32) unpack_word(U, r, wd);
	}
}
#endif
static void unpack_reads(const UnpackArgs &U)
{
	++t_launches;
#ifndef MGB_HOSTSIM
	k_unpack<<<dev_sm_count() * 8, 256, 0, t_stream>>>(U);
	CUDA_OK(cudaGetLastError());
#else
	for (int r = 0; r < U.n_reads; ++r) if (U.pk_off[r] != ~0ULL) for (int64_t wd = 0; wd * 32 < U.seq_len[r]; ++wd) unpack_word(U, r, wd);
#endif
}

// ---- the few words the host needs between two kernels (pool fill levels, queue lengths) ----
// They do not travel by cudaMemcpy: a copy of 16 bytes queues behind whatever another call in flight has put on the copy engines
// (a few hundred MB of results, tens of ms).  A one-warp kernel writes them into page-locked host memory the device can address.
struct Mail { Pool pools[16]; unsigned int jobq_n[2], lab_n[2]; unsigned long long prof[32]; unsigned int tier_hist[128]; unsigned long long arena_peak; };
struct MailSrc { const Pool *pools; const unsigned int *jobq_n, *lab_n; const unsigned long long *prof; const unsigned int *tier_hist; const uint64_t *peak; int n_workers; };
#ifndef MGB_HOSTSIM
__global__ void k_mail(MailSrc m, Mail *out)
{
	const int t = threadIdx.x;
	if (t < 16) out->pools[t] = m.pools[t];
	if (t < 2) out->jobq_n[t] = m.jobq_n[t], out->lab_n[t] = m.lab_n? m.lab_n[t] : 0;
	out->prof[t] = m.prof[t];
	for (int i = t; i < 128; i += 32) out->tier_hist[i] = m.tier_hist[i];
	unsigned long long pk = 0;
	for (int i = t; i < m.n_workers; i += 32) pk = m.peak[i] > pk? m.peak[i] : pk;
	for (int o = 16; o > 0; o >>= 1) { const unsigned long long y = __shfl_xor_sync(0xffffffffu, pk, o); pk = y > pk? y : pk; }
	if (t == 0) out->arena_peak = pk;
	__threadfence_system();
}
#endif
// how many bridging jobs / gap jobs the kernels in front have appended to their pools since `done`: the job kernels read it on the device
MG_HD inline void job_counts(const Pool *pools, int i_gjobs, int i_jobs, unsigned int gjobs_done, unsigned int jobs_done, unsigned int *cnt)
{
	const Pool &pg = pools[i_gjobs], &pj = pools[i_jobs];
	cnt[0] = (unsigned int)((pg.used < pg.cap? pg.used : pg.cap) / sizeof(GwfaJob)) - gjobs_done;
	cnt[1] = (unsigned int)((pj.used < pj.cap? pj.used : pj.cap) / sizeof(WfaJob)) - jobs_done;
}
#ifndef MGB_HOSTSIM
__global__ void k_job_counts(const Pool *pools, int i_gjobs, int i_jobs, unsigned int gjobs_done, unsigned int jobs_done, unsigned int *cnt) { job_counts(pools, i_gjobs, i_jobs, gjobs_done, jobs_done, cnt); }
#endif
static void count_jobs(const Pool *pools, int i_gjobs, int i_jobs, unsigned int gjobs_done, unsigned int jobs_done, unsigned int *cnt)
{
	++t_launches;
#ifndef MGB_HOSTSIM
	k_job_counts<<<1, 1, 0, t_stream>>>(pools, i_gjobs, i_jobs, gjobs_done, jobs_done, cnt);
	CUDA_OK(cudaGetLastError());
#else
	job_counts(pools, i_gjobs, i_jobs, gjobs_done, jobs_done, cnt);
#endif
}
static void fetch_mail(const MailSrc &m, Mail *mail)
{
	++t_launches;
#ifndef MGB_HOSTSIM
	k_mail<<<1, 32, 0, t_stream>>>(m, mail);
	CUDA_OK(cudaGetLastError());
	dsync();
#else
	memcpy(mail->pools, m.pools, sizeof(mail->pools));
	memcpy(mail->jobq_n, m.jobq_n, sizeof(mail->jobq_n));
	if (m.lab_n) memcpy(mail->lab_n, m.lab_n, sizeof(mail->lab_n)); else mail->lab_n[0] = mail->lab_n[1] = 0;
	memcpy(mail->prof, m.prof, sizeof(mail->prof));
	memcpy(mail->tier_hist, m.tier_hist, sizeof(mail->tier_hist));
	mail->arena_peak = 0;
	for (int i = 0; i < m.n_workers; ++i) if (m.peak[i] > mail->arena_peak) mail->arena_peak = m.peak[i];
#endif
}

struct Workers {
	int n_workers;
	uint64_t arena_bytes;
	char *arena;
	uint64_t *peak;
	void release() { dfree(arena), dfree(peak); memset(this, 0, sizeof(*this)); }
};

template<int STAGE>
static void launch_stage(LaunchArgs &L, const Workers &W)
{
	L.arena_base = W.arena, L.arena_bytes = W.arena_bytes, L.arena_peak = W.peak;
	dzero(L.c.next_read, sizeof(unsigned int)); // in stream order: no host round trip per launch
	++t_launches;
#ifdef MGB_HOSTSIM
	constexpr StageEntry entry = StageRow<STAGE>::ENTRY;
	Arena A;
	arena_init(A, W.arena, entry == ENTER_THREAD? (W.arena_bytes / 32) & ~(uint64_t)15 : W.arena_bytes); // one item per thread: a thread's share, as on the device
#define MGB_STAGE_SMEM(kern, st, num, bounds, warps, blocks, smem, ...) , (int)(smem)
	std::vector<int32_t> sim_smem(std::max({0 MGB_STAGES(MGB_STAGE_SMEM)}) / 4); // the largest of all stages
#undef MGB_STAGE_SMEM
	if (STAGE == ST_CHAIN || STAGE == ST_CHAIN_RESCUE) { mbar_init((uint64_t*)sim_smem.data(), 1); sim_smem[2] = 0; }
	const int n_work_sim = L.n_work_dev? (int)*L.n_work_dev : L.n_work;
	for (int it = 0; it < n_work_sim; ++it) {
		int item = L.rid_list? L.rid_list[it] : it;
		A.top = 0;
		int rc;
#if MGB_W > 1
		if (entry == ENTER_WARP) { // all lanes of the simulated warp enter, each with its own copy of the arena header (as in registers on the device)
			int rcs[MGB_W];
			uint64_t peaks[MGB_W];
			sim::tag()[0] = STAGE, sim::tag()[1] = item;
			sim::run_warp(MGB_W, [&](int lane) {
				Arena Al = A;
				rcs[lane] = run_stage<STAGE>(L, item, Al, lane, sim_smem.data());
				peaks[lane] = Al.peak;
			});
			rc = rcs[0];
			for (int l = 1; l < MGB_W; ++l) if (rcs[l] != rc) { set_error("simulated warp: lanes returned different codes from one stage"); abort(); }
			for (int l = 0; l < MGB_W; ++l) if (peaks[l] > A.peak) A.peak = peaks[l];
		} else
#endif
		rc = run_stage<STAGE>(L, item, A, 0, entry == ENTER_WARP? sim_smem.data() : 0);
		if (rc < 0 && getenv("MGB_HOSTSIM_TRACE")) fprintf(stderr, "[hostsim] stage %d item %d failed with %d\n", STAGE, item, rc);
		if (rc < 0) stage_fail<STAGE>(L, item, rc);
	}
	if (W.peak && A.peak > W.peak[0]) W.peak[0] = A.peak;
#else
	const int warps = g_shape.warps[STAGE];
	const int want = dev_sm_count() * g_shape.minb[STAGE] * warps; // resident warps this stage can keep on the chip
	const int blocks = std::max(1, std::min(W.n_workers, want) / warps);
	const size_t smem = (size_t)warps * StageRow<STAGE>::SMEM;
	const StageFn kern = stage_kernel<STAGE>();
	if (smem > 48 * 1024) CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	kern<<<blocks, warps * 32, smem, t_stream>>>(L);
	CUDA_OK(cudaGetLastError());
#endif
}

// ---------------------------------------------------------------------------------------------------------------
// model: flattened graph + minimizer index, host copy and device image
// ---------------------------------------------------------------------------------------------------------------

struct Model {
	// host copies
	std::vector<int32_t> seg_len;
	std::vector<uint64_t> vseq_off;
	std::vector<char> seq;
	std::vector<uint64_t> arc_idx;
	std::vector<DevArc> arc;
	std::vector<u128> slot;
	std::vector<uint64_t> pos;
	std::vector<uint32_t> occ;      // occurrences per distinct minimizer (for the quantiles)
	uint64_t n_slots_mask;
	int k, w;
	uint32_t *d_occ_sorted = 0; uint64_t n_keys = 0, n_pos = 0; // device-built index: ascending occurrence counts; host copies of slot/pos are made on demand
	std::mutex host_ix_mutex;
	// device image
	GraphDev g;
	IndexDev ix;
	std::vector<void*> dev_ptrs;
	// per-model scratch reused across batches
	std::vector<int32_t> seg_name_id, seg_soff; // MG_M_NO_DIAG: the name a segment goes by (id into name_ids) and its offset there
	std::unordered_map<std::string, int32_t> name_ids;
	Workers W, Wbig;
	int32_t skip1_len = INT32_MAX, skip2_len = INT32_MAX; // WFA tier routing learned from earlier batches (wfa_job_run)
	std::vector<float> logf_tab; float *d_logf; int n_logf;
	mgb_stats_t stats;
	gfa_edseq_t *es;
	// the batch pipeline: a batch is cut into sub-batches, each driven by its own host thread on its own stream ("slot"),
	// so that kernels, copies and host-side result assembly of different sub-batches overlap
	struct Slot {
		GrowBuf h_seq{true}, h_out{true}, h_small{true}, h_pk{true}, h_mail{true}, h_routs{true}, d_pk, d_seq, d_meta, d_routs, d_small, d_jobq, d_order, d_packed, d_packoff, d_segs, d_lab_new, d_pool[10];
		GrowBuf h_rname{true}, d_rname, d_gafctx, d_gafoff, d_text, d_fix; // the text route (mgb_map_batch_gaf)
		mgb::HostPool host_pool; // packing and result assembly of the batch on this slot
		Workers W;
		mgb_stats_t st;
		DevStream stream;
		DevEvent ev_first, ev_last, ev_piece[4]; // first kernel start, last kernel end; the pieces of the result copy
		SlotTimers *timers = 0;
		bool ready;
		Slot() : ready(false) { memset(&W, 0, sizeof(W)); }
		~Slot() // (on the model's device; the GrowBufs release themselves)
		{
			delete timers;
			W.release();
#ifndef MGB_HOSTSIM
			if (ready) { cudaStreamDestroy(stream); cudaEventDestroy(ev_first); cudaEventDestroy(ev_last); for (int i = 0; i < 4; ++i) cudaEventDestroy(ev_piece[i]); }
#endif
		}
	};
	enum { MAX_SLOTS = 8 };
	Slot slots[MAX_SLOTS];
	std::mutex big_mutex; // the large-arena retry pass, the label table and the learned routing are shared by the slots
	std::condition_variable slot_cv;
	std::mutex gpu_mutex;         // the kernels of one call at a time: calls in flight overlap their copies and host work with them, not with each other's kernels
	int device = 0;               // the GPU this image lives on
	std::vector<Model*> peers;    // MGB_DEVICES: the same index on further GPUs; a batch is cut into one contiguous part per device
	bool slot_busy[MAX_SLOTS] = {};
	int in_flight = 0;    // calls inside map_batch_impl
	bool lab_growing = false; // a call is waiting to replace the label pool: new calls wait
	// reachability labels of the graph (mgb_gclabel.cuh): built on demand, kept across batches, grown between them
	long long *d_lab_off = 0; Pool *d_lab_hdr = 0; char *d_lab_pool = 0;
	uint64_t lab_cap = 0; int32_t lab_max_dist_g = -1; int64_t lab_sources = 0;
	// the names the GAF kernels print (graph part of GafCtx): uploaded at the first mgb_map_batch_gaf() on this device
	GafCtx gaf_graph = {}; bool gaf_ready = false;
};

static void model_free(Model *M)
{
	for (Model *P : M->peers) model_free(P);
	M->peers.clear();
	set_device(M->device);
	for (void *p : M->dev_ptrs) dfree(p);
	M->W.release(), M->Wbig.release();
	if (M->d_logf) dfree(M->d_logf);
	dfree(M->d_lab_off), dfree(M->d_lab_hdr), dfree(M->d_lab_pool), dfree(M->d_occ_sorted);
	delete M; // (the slots release their own)
}

static unsigned char comp_tab[256];
static void init_comp_tab() // reference: gfa-base.c:509-526 gfa_comp_table
{
	static const char *from = "ABCDEFGHIJKLMNOPQRSTUVWXYZ", *to = "TVGHEFCDIJMLKNOPQYSAABWXRZ";
	for (int i = 0; i < 256; ++i) comp_tab[i] = (unsigned char)i;
	for (int i = 0; i < 26; ++i) {
		comp_tab[(unsigned char)from[i]] = (unsigned char)to[i];
		comp_tab[(unsigned char)(from[i] + 32)] = (unsigned char)(to[i] + 32);
	}
}

static void ensure_workers(Workers &W, int n_workers, uint64_t arena_bytes)
{
	if (W.arena && W.n_workers == n_workers && W.arena_bytes == arena_bytes) return;
	W.release();
	W.n_workers = n_workers, W.arena_bytes = arena_bytes;
	W.arena = (char*)dmalloc((size_t)n_workers * arena_bytes);
	W.peak = (uint64_t*)dmalloc((size_t)n_workers * sizeof(uint64_t));
	dzero(W.peak, (size_t)n_workers * sizeof(uint64_t));
}

static int default_workers()
{
#ifdef MGB_HOSTSIM
	return 1;
#else
	return dev_sm_count() * (int)p_workers_per_sm;
#endif
}

// The minimizer table built on the host: grouped by minimizer, occurrence lists ascending (reference: index.c:115-165 mg_idx_a2h)
static void index_on_host(Model *M, std::vector<u128> &mz)
{
	std::sort(mz.begin(), mz.end(), [](const u128 &a, const u128 &b) { return (a.x >> 8) != (b.x >> 8)? (a.x >> 8) < (b.x >> 8) : a.y < b.y; });
	size_t n_keys = 0;
	for (size_t i = 0; i < mz.size(); ++i) if (i == 0 || (mz[i].x >> 8) != (mz[i-1].x >> 8)) ++n_keys;
	uint64_t n_slots = 16;
	while (n_slots < n_keys * 2) n_slots <<= 1;
	M->n_slots_mask = n_slots - 1;
	M->slot.assign(n_slots, u128{~0ULL, ~0ULL});
	M->occ.reserve(n_keys);
	for (size_t i = 0; i < mz.size();) {
		size_t j = i;
		uint64_t key = mz[i].x >> 8;
		while (j < mz.size() && (mz[j].x >> 8) == key) ++j;
		uint64_t h = idx_slot_hash(key) & M->n_slots_mask;
		while (M->slot[h].x != ~0ULL) h = (h + 1) & M->n_slots_mask;
		if (j - i == 1) {
			M->slot[h].x = key << 1 | 1, M->slot[h].y = mz[i].y;
			M->occ.push_back(1);
		} else {
			M->slot[h].x = key << 1, M->slot[h].y = (uint64_t)M->pos.size() << 32 | (uint64_t)(j - i);
			for (size_t t = i; t < j; ++t) M->pos.push_back(mz[t].y);
			M->occ.push_back((uint32_t)(j - i));
		}
		i = j;
	}
	M->ix.n_slots_mask = M->n_slots_mask;
	M->ix.slot = dalloc_copy(M->slot), M->dev_ptrs.push_back((void*)M->ix.slot);
	M->ix.pos = dalloc_copy(M->pos), M->dev_ptrs.push_back((void*)M->ix.pos);
}

static Model *model_build(gfa_t *g, int k, int w)
{
	Model *M = new Model();
	M->k = k, M->w = w, M->d_logf = 0, M->n_logf = 0, M->es = 0;
	memset(&M->W, 0, sizeof(Workers)), memset(&M->Wbig, 0, sizeof(Workers));
	memset(&M->stats, 0, sizeof(M->stats));
	init_comp_tab();
	const uint32_t n_seg = g->n_seg, n_vtx = n_seg * 2;
	M->seg_len.resize(n_seg);
	M->vseq_off.resize(n_vtx);
	uint64_t tot = 0;
	for (uint32_t i = 0; i < n_seg; ++i) {
		M->seg_len[i] = g->seg[i].len;
		M->vseq_off[i << 1] = tot, tot += (uint64_t)g->seg[i].len + 8;   // 8 bytes of slack after every copy
		M->vseq_off[i << 1 | 1] = tot, tot += (uint64_t)g->seg[i].len + 8;
	}
	M->seq.assign(tot + 16, 0);
	for (uint32_t i = 0; i < n_seg; ++i) {
		const gfa_seg_t *s = &g->seg[i];
		char *f = &M->seq[M->vseq_off[i << 1]], *r = &M->seq[M->vseq_off[i << 1 | 1]];
		for (int32_t j = 0; j < s->len; ++j) f[j] = s->seq[j];
		for (int32_t j = 0; j < s->len; ++j) r[s->len - j - 1] = (char)comp_tab[(uint8_t)s->seq[j]]; // reference: gfa-ed.c:33-36
	}
	M->arc_idx.assign(g->idx, g->idx + n_vtx);
	M->arc.resize(g->n_arc);
	for (uint64_t i = 0; i < g->n_arc; ++i) { // verbatim order (SURVEY H10b)
		DevArc a;
		a.w = g->arc[i].w, a.lv = (uint32_t)g->arc[i].v_lv, a.rank = g->arc[i].rank, a.ow = g->arc[i].ow;
		M->arc[i] = a;
	}
	M->seg_name_id.resize(n_seg), M->seg_soff.resize(n_seg);
	for (uint32_t i = 0; i < n_seg; ++i) { // reference: map-algo.c:168-174
		const gfa_seg_t *s = &g->seg[i];
		const bool stable = s->snid >= 0 && g->sseq;
		const char *gname = stable? g->sseq[s->snid].name : s->name;
		auto it = M->name_ids.emplace(std::string(gname? gname : ""), (int32_t)M->name_ids.size()).first;
		M->seg_name_id[i] = it->second, M->seg_soff[i] = stable? s->soff : 0;
	}
	// upload the graph
	M->g.n_seg = (int32_t)n_seg;
	M->g.seg_name_id = dalloc_copy(M->seg_name_id), M->dev_ptrs.push_back((void*)M->g.seg_name_id);
	M->g.seg_soff = dalloc_copy(M->seg_soff), M->dev_ptrs.push_back((void*)M->g.seg_soff);
	M->g.seg_len = dalloc_copy(M->seg_len), M->dev_ptrs.push_back((void*)M->g.seg_len);
	M->g.vseq_off = dalloc_copy(M->vseq_off), M->dev_ptrs.push_back((void*)M->g.vseq_off);
	M->g.seq = dalloc_copy(M->seq), M->dev_ptrs.push_back((void*)M->g.seq);
	M->g.arc_idx = dalloc_copy(M->arc_idx), M->dev_ptrs.push_back((void*)M->g.arc_idx);
	M->g.arc = dalloc_copy(M->arc), M->dev_ptrs.push_back((void*)M->g.arc);
	M->ix.k = k, M->ix.w = w, M->ix.slot = 0, M->ix.pos = 0, M->ix.n_slots_mask = 0;

	// sketch every segment on the device (K1 reused), then build the table on the host
	std::vector<u128> mz;
	{
		uint64_t tot_len = 0;
		int32_t max_len = 1;
		for (uint32_t i = 0; i < n_seg; ++i) { tot_len += (uint64_t)g->seg[i].len; if (g->seg[i].len > max_len) max_len = g->seg[i].len; }
		uint64_t cap = (tot_len / 2 + 64 * (uint64_t)n_seg + 1024) * sizeof(u128);
		// a worker sketches one whole segment inside its arena: ~ (len/w + growth slack) records
		uint64_t need = (uint64_t)max_len * 16 + ((uint64_t)1 << 20);
		uint64_t arena_b = std::max<uint64_t>((uint64_t)p_arena_mb << 20, need);
		int nw = default_workers();
		while (nw > 1 && (uint64_t)nw * arena_b > dev_free_mem() / 2) nw /= 2;
		for (;;) {
			ensure_workers(M->W, nw, arena_b);
			Pool hp; hp.used = 0, hp.cap = cap;
			Pool *d_pool = (Pool*)dmalloc(sizeof(Pool));
			u128 *d_mz = (u128*)dmalloc(cap);
			int *d_status = (int*)dmalloc(sizeof(int));
			unsigned int *d_next = (unsigned int*)dmalloc(sizeof(unsigned int));
			int st0 = 0;
			h2d(d_pool, &hp, sizeof(Pool));
			h2d(d_status, &st0, sizeof(int));
			LaunchArgs L;
			memset(&L, 0, sizeof(L));
			L.c.g = M->g, L.c.ix = M->ix, L.c.next_read = d_next;
			L.routs = (ReadOut*)d_status, L.rid_list = 0, L.n_work = (int32_t)n_seg, L.pool_mz = d_pool, L.mz = d_mz;
			launch_stage<ST_INDEX_SKETCH>(L, M->W);
			dsync();
			d2h(&st0, d_status, sizeof(int));
			d2h(&hp, d_pool, sizeof(Pool));
			bool retry = false;
			if (st0 == MGB_E_POOL) cap *= 2, retry = true;
			else if (st0 == MGB_E_ARENA) arena_b *= 2, nw = std::max(1, nw / 2), retry = true;
			else if (st0 < 0) { set_error("segment sketch failed with code " + std::to_string(st0)); throw MgbError{st0}; }
#ifndef MGB_HOSTSIM
			if (!retry && p_index_dev) { // group, lay out and insert on the device (mgb_index.cuh)
				DevIndexOut out;
				M->W.release(); // the sketch arenas are not needed again; the sort wants the memory
				cudaError_t e = build_index_device(d_mz, hp.used / sizeof(u128), 2 * k, t_stream, &out);
				dfree(d_pool), dfree(d_mz), dfree(d_status), dfree(d_next);
				if (e != cudaSuccess) { set_error(std::string("index build on the device: ") + cudaGetErrorString(e)); throw MgbError{MGB_E_INTERNAL}; }
				M->n_slots_mask = out.n_slots - 1, M->n_keys = out.n_keys, M->n_pos = out.n_pos, M->d_occ_sorted = out.occ_sorted;
				M->ix.n_slots_mask = M->n_slots_mask, M->ix.slot = out.slot, M->ix.pos = out.pos;
				M->dev_ptrs.push_back((void*)out.slot), M->dev_ptrs.push_back((void*)out.pos);
				return M;
			}
#endif
			if (!retry) {
				mz.resize(hp.used / sizeof(u128));
				d2h(mz.data(), d_mz, hp.used);
			}
			dfree(d_pool), dfree(d_mz), dfree(d_status), dfree(d_next);
			if (!retry) break;
		}
	}
	// the sketch arenas are not needed again (every mapping slot owns its arenas)
	M->W.release();
	index_on_host(M, mz);
	return M;
}


static const Model *model_of(const mg_idx_t *gi) { return (const Model*)gi->B; }

// ---------------------------------------------------------------------------------------------------------------
// C ABI: index
// ---------------------------------------------------------------------------------------------------------------

extern "C" void mg_idx_cal_quantile(const mg_idx_t *gi, int32_t m, float f[], int32_t q[])
{
	const Model *M = model_of(gi);
#ifndef MGB_HOSTSIM
	if (M->d_occ_sorted) { // the table was built on the device: the counts are there, sorted
		const uint64_t n = M->n_keys;
		for (int32_t i = 0; i < m; ++i) {
			size_t kk = (size_t)((1.0 - (double)f[i]) * (double)n);
			if (n == 0) { q[i] = 0; continue; }
			if (kk >= n) kk = n - 1;
			uint32_t v = 0;
			cudaSetDevice(M->device);
			cudaMemcpy(&v, M->d_occ_sorted + kk, 4, cudaMemcpyDeviceToHost);
			q[i] = (int32_t)v;
		}
		return;
	}
#endif
	std::vector<uint32_t> a(M->occ);
	uint64_t n = a.size();
	for (int32_t i = 0; i < m; ++i) {
		size_t kk = (size_t)((1.0 - (double)f[i]) * (double)n);
		if (n == 0) { q[i] = 0; continue; }
		if (kk >= n) kk = n - 1;
		std::nth_element(a.begin(), a.begin() + kk, a.end());
		q[i] = (int32_t)a[kk];
	}
}

extern "C" const uint64_t *mg_idx_get(const mg_idx_t *gi, uint64_t minier, int *n)
{
	Model *M = (Model*)model_of(gi);
#ifndef MGB_HOSTSIM
	if (M->slot.empty() && M->ix.slot) { // device-built table: the host view is fetched the first time somebody asks for it
		std::lock_guard<std::mutex> lk(M->host_ix_mutex);
		if (M->slot.empty()) {
			cudaSetDevice(M->device);
			M->pos.resize(M->n_pos? M->n_pos : 1);
			cudaMemcpy(M->pos.data(), M->ix.pos, M->n_pos * 8, cudaMemcpyDeviceToHost);
			std::vector<u128> sl(M->n_slots_mask + 1);
			cudaMemcpy(sl.data(), M->ix.slot, sl.size() * sizeof(u128), cudaMemcpyDeviceToHost);
			M->slot.swap(sl);
		}
	}
#endif
	IndexDev ix;
	ix.k = M->k, ix.w = M->w, ix.n_slots_mask = M->n_slots_mask, ix.slot = M->slot.data(), ix.pos = M->pos.data();
	return idx_get(ix, minier, n);
}

extern "C" mg_idx_t *mg_index(gfa_t *g, const mg_idxopt_t *io, int n_threads, mg_mapopt_t *mo)
{
	(void)n_threads;
	// MGB_DEVICES=0-7 | 0,2,5: the index is replicated on every listed GPU and each batch is cut into one part per GPU (the reference's
	// "-t": gmap.c:163-211 hands its mini-batch to n_threads workers; here the workers are devices).  Unset: the "device" parameter.
	std::vector<int> devs;
	if (const char *e = getenv("MGB_DEVICES")) {
		for (const char *q = e; *q;) {
			char *end;
			long a = strtol(q, &end, 10), b2 = a;
			if (end == q) break;
			if (*end == '-') { q = end + 1; b2 = strtol(q, &end, 10); }
			for (long d = a; d <= b2 && devs.size() < 64; ++d) devs.push_back((int)d);
			q = *end == ','? end + 1 : end;
			if (*end && *end != ',') break;
		}
	}
	if (devs.empty()) devs.push_back((int)p_device);
	for (int d : devs) if (!dev_ok(d)) { set_error("no CUDA device " + std::to_string(d) + " available: libmgb200 has no CPU path"); return 0; }
	dev_ok(devs[0]);
	for (uint32_t i = 0; i < g->n_seg; ++i) { // reference: index.c:215-220
		gfa_seg_t *s = &g->seg[i];
		for (int32_t j = 0; j < s->len; ++j)
			if (s->seq[j] >= 'a' && s->seq[j] <= 'z') s->seq[j] -= 32;
	}
	for (uint64_t i = 0; i < g->n_arc; ++i) // reference: index.c:176-183,192-196
		if (g->arc[i].ov != 0 || g->arc[i].ow != 0) {
			fprintf(stderr, "[E::%s] minigraph doesn't work with graphs containing overlapping segments\n", __func__);
			return 0;
		}
	int k = io->k, w = io->w, b = io->bucket_bits;
	if (k * 2 < b) b = k * 2;
	if (w < 1) w = 1;
	Model *M = 0;
	try { M = model_build(g, k, w); } catch (const MgbError &) { return 0; }
	M->device = devs[0];
	if (devs.size() > 1) { // every further device builds its own copy (sketch on that device, table on the host), all at once
		M->peers.resize(devs.size() - 1, (Model*)0);
		std::vector<std::thread> th;
		for (size_t i = 1; i < devs.size(); ++i)
			th.emplace_back([&, i]() { try { if (dev_ok(devs[i])) { M->peers[i - 1] = model_build(g, k, w); M->peers[i - 1]->device = devs[i]; } } catch (const MgbError &) {} });
		for (auto &t : th) t.join();
		dev_ok(devs[0]);
		for (Model *P : M->peers) if (P == 0) { model_free(M); return 0; } // mgb_last_error() has the reason
	}
	mg_idx_t *gi = (mg_idx_t*)calloc(1, sizeof(mg_idx_t));
	gi->g = g, gi->b = b, gi->w = w, gi->k = k, gi->n_seg = (int32_t)g->n_seg;
	gi->B = (struct mg_idx_bucket_s*)M;
	// host view of both strands for callers that read gi->es (reference: gfa-ed.c:24-42)
	gi->es = (gfa_edseq_t*)malloc(sizeof(gfa_edseq_t) * 2 * (size_t)g->n_seg);
	for (uint32_t i = 0; i < g->n_seg; ++i) {
		gi->es[i << 1].seq = g->seg[i].seq, gi->es[i << 1].len = g->seg[i].len;
		gi->es[i << 1 | 1].seq = &M->seq[M->vseq_off[i << 1 | 1]], gi->es[i << 1 | 1].len = g->seg[i].len;
	}
	if (mo) { // reference: options.c:120-134 mg_opt_update
		float f[2];
		int32_t q[2];
		f[0] = 0.1f, f[1] = mo->occ_max1_frac;
		mg_idx_cal_quantile(gi, 2, f, q);
		if (q[0] > mo->lc_max_occ) mo->lc_max_occ = q[0];
		if (mo->lc_max_occ > mo->occ_max1_cap) mo->lc_max_occ = mo->occ_max1_cap;
		if (q[1] > mo->occ_max1) mo->occ_max1 = q[1];
		if (mo->occ_max1 > mo->occ_max1_cap) mo->occ_max1 = mo->occ_max1_cap;
		if (mo->bw_long < mo->bw) mo->bw_long = mo->bw;
	}
	return gi;
}

extern "C" void mg_idx_destroy(mg_idx_t *gi)
{
	if (gi == 0) return;
	if (gi->B) model_free((Model*)gi->B);
	free(gi->es);
	free(gi);
}

extern "C" void mg_idx_hfree(void *h) { (void)h; } // reference callers only pass NULL (shortk.c:191)

struct mg_tbuf_s { int dummy; };
extern "C" mg_tbuf_t *mg_tbuf_init(void) { return (mg_tbuf_t*)calloc(1, sizeof(mg_tbuf_t)); }
extern "C" void mg_tbuf_destroy(mg_tbuf_t *b) { free(b); }

extern "C" void mg_gchain_free(mg_gchains_t *gs)
{
	if (gs == 0) return;
	for (int32_t i = 0; i < gs->n_gc; ++i) {
		free(gs->gc[i].p);
		free(gs->gc[i].ds.ds);
		free(gs->gc[i].ds.off);
	}
	free(gs->gc); free(gs->a); free(gs->lc);
	free(gs);
}

extern "C" void mgb_free_batch(int n_reads, mg_gchains_t **gcs)
{
	for (int i = 0; i < n_reads; ++i) { mg_gchain_free(gcs[i]); gcs[i] = 0; }
}

// ---------------------------------------------------------------------------------------------------------------
// batch dispatcher
// ---------------------------------------------------------------------------------------------------------------

static void fill_opt(MapOptDev &o, const mg_mapopt_t *opt, int k)
{
	memset(&o, 0, sizeof(o));
	o.flag = opt->flag, o.seed = opt->seed, o.max_qlen = opt->max_qlen, o.occ_max1 = opt->occ_max1;
	o.bw = opt->bw, o.bw_long = opt->bw_long, o.rmq_size_cap = opt->rmq_size_cap, o.rmq_rescue_size = opt->rmq_rescue_size;
	o.rmq_rescue_ratio = opt->rmq_rescue_ratio;
	o.max_gap_pre = opt->max_gap_pre, o.max_gap = opt->max_gap, o.max_gap_ref = opt->max_gap_ref, o.max_frag_len = opt->max_frag_len;
	{ // reference: map-algo.c:388-390; expf() must be the host libm (SURVEY H3)
		float tmp = expf(-opt->div * k);
		o.chn_pen_gap = opt->chn_pen_gap * tmp;
		o.chn_pen_skip = opt->chn_pen_skip * tmp;
	}
	o.max_lc_skip = opt->max_lc_skip, o.max_lc_iter = opt->max_lc_iter, o.max_gc_skip = opt->max_gc_skip;
	o.min_lc_cnt = opt->min_lc_cnt, o.min_lc_score = opt->min_lc_score, o.min_gc_cnt = opt->min_gc_cnt, o.min_gc_score = opt->min_gc_score;
	o.gdp_max_ed = opt->gdp_max_ed, o.lc_max_trim = opt->lc_max_trim, o.lc_max_occ = opt->lc_max_occ;
	o.mask_level = opt->mask_level, o.sub_diff = opt->sub_diff, o.best_n = opt->best_n, o.pri_ratio = opt->pri_ratio, o.ref_bonus = opt->ref_bonus;
}

// mg_gchain_t::div (reference: gchain1.c:295) with the host's libm log (SURVEY H3): the result objects and the `dv:f` fix-ups of
// the text route both take it from here
static float gchain_div(int32_t n_mini, int32_t n_anchor, int32_t q_span)
{
	return n_mini >= n_anchor? (float)(log((double)n_mini / n_anchor) / q_span) : (float)(log((double)n_anchor / n_mini) / q_span);
}

static mg_gchains_t *build_result(const ReadOut &ro, const char *pool)
{
	const char *blob = pool + ro.blob_off;
	mg_gchains_t *gs = (mg_gchains_t*)calloc(1, sizeof(mg_gchains_t));
	gs->rep_len = ro.rep_len;
	if (ro.n_gc == 0) return gs; // reference: gchain1.c:460 returns the bare struct
	gs->n_gc = ro.n_gc, gs->n_lc = ro.n_lc, gs->n_a = ro.n_a;
	gs->gc = (mg_gchain_t*)calloc((size_t)ro.n_gc, sizeof(mg_gchain_t));
	gs->lc = (mg_llchain_t*)malloc((size_t)(ro.n_lc > 0? ro.n_lc : 1) * sizeof(mg_llchain_t));
	gs->a = (mg128_t*)malloc((size_t)(ro.n_a > 0? ro.n_a : 1) * sizeof(mg128_t));
	const GChain *d = (const GChain*)blob;
	uint64_t off_lc = align8((uint64_t)ro.n_gc * sizeof(GChain));
	uint64_t off_a = off_lc + align8((uint64_t)ro.n_lc * sizeof(LLChain));
	memcpy(gs->lc, blob + off_lc, (size_t)ro.n_lc * sizeof(mg_llchain_t));
	memcpy(gs->a, blob + off_a, (size_t)ro.n_a * sizeof(mg128_t));
	for (int32_t i = 0; i < ro.n_gc; ++i) {
		mg_gchain_t *p = &gs->gc[i];
		const GChain *s = &d[i];
		p->id = s->id, p->parent = s->parent, p->off = s->off, p->cnt = s->cnt, p->n_anchor = s->n_anchor, p->score = s->score;
		p->qs = s->qs, p->qe = s->qe, p->plen = s->plen, p->ps = s->ps, p->pe = s->pe, p->blen = s->blen, p->mlen = s->mlen;
		p->hash = s->hash, p->subsc = s->subsc, p->n_sub = s->n_sub, p->mapq = (uint32_t)s->mapq, p->flt = (uint32_t)s->flt;
		p->div = gchain_div(s->n_mini, s->n_anchor, s->q_span);
		if (s->has_cigar) {
			p->p = (mg_cigar_t*)calloc(1, (size_t)s->n_cigar * 8 + sizeof(mg_cigar_t));
			p->p->n_cigar = s->n_cigar, p->p->mlen = s->c_mlen, p->p->blen = s->c_blen, p->p->aplen = s->c_aplen, p->p->ss = s->c_ss, p->p->ee = s->c_ee;
			memcpy(p->p->cigar, pool + s->cigar_off, (size_t)s->n_cigar * 8);
			p->ds.len = s->ds_len, p->ds.n_off = s->n_dsoff;
			p->ds.ds = (char*)calloc((size_t)s->ds_len + 1, 1);
			memcpy(p->ds.ds, pool + s->ds_off, (size_t)s->ds_len);
			p->ds.off = (int32_t*)calloc((size_t)(s->n_dsoff > 0? s->n_dsoff : 1), sizeof(int32_t));
			memcpy(p->ds.off, pool + s->dsoff_off, (size_t)s->n_dsoff * sizeof(int32_t));
		}
	}
	return gs;
}

// The text route (mgb_map_batch_gaf): the graph whose names are printed, and the caller's buffer, with the rules of
// mgb_write_gaf_batch() for (*out, *out_len, *out_cap)
struct GafRoute { const gfa_t *g; char **out; size_t *len, *cap; };
// room for tot bytes and the terminator: the caller's buffer if out_cap says it is large enough, else a fresh malloc() block
static char *gaf_reserve(const GafRoute &R, size_t tot)
{
	char *o = R.cap? *R.out : 0;
	size_t cap = o? *R.cap : 0;
	if (cap < tot + 1) {
		free(o);
		cap = tot + tot / 8 + 1;
		o = (char*)malloc(cap);
		if (o == 0) { set_error("out of host memory for the GAF text"); throw MgbError{MGB_E_INTERNAL}; }
	}
	*R.out = o;
	if (R.cap) *R.cap = cap;
	o[tot] = 0;
	return o;
}

// The names the GAF kernels print, on the model's device, once (mg_index is not asked to pay for them)
static void gaf_upload_graph(Model *M, const gfa_t *g)
{
	std::lock_guard<std::mutex> lk(M->big_mutex);
	if (M->gaf_ready) return;
	std::vector<char> sn, qn;
	std::vector<uint64_t> sn_off(1, 0), qn_off(1, 0);
	std::vector<int32_t> snid(g->n_seg), soff(g->n_seg), rank(g->n_sseq), mn(g->n_sseq), mx(g->n_sseq);
	for (uint32_t i = 0; i < g->n_seg; ++i) {
		const char *nm = g->seg[i].name? g->seg[i].name : "";
		sn.insert(sn.end(), nm, nm + strlen(nm)), sn_off.push_back(sn.size());
		snid[i] = g->seg[i].snid, soff[i] = g->seg[i].soff;
	}
	for (uint32_t i = 0; i < g->n_sseq; ++i) {
		const char *nm = g->sseq[i].name? g->sseq[i].name : "";
		qn.insert(qn.end(), nm, nm + strlen(nm)), qn_off.push_back(qn.size());
		rank[i] = g->sseq[i].rank, mn[i] = g->sseq[i].min, mx[i] = g->sseq[i].max;
	}
	auto up = [&](const auto &v) { auto *d = dalloc_copy(v); M->dev_ptrs.push_back((void*)d); return d; };
	GafCtx &x = M->gaf_graph;
	x.seg_name = up(sn), x.seg_name_off = up(sn_off), x.seg_snid = up(snid), x.seg_soff = up(soff);
	x.ss_name = up(qn), x.ss_name_off = up(qn_off), x.ss_rank = up(rank), x.ss_min = up(mn), x.ss_max = up(mx);
	x.comp = up(std::vector<unsigned char>(comp_tab, comp_tab + 256));
	M->gaf_ready = true;
}

// The label table of graph chaining: allocated at the first batch, emptied when a batch asks for longer walks than it was built for.
static bool lab_prepare(Model *M, int32_t max_dist_g)
{
	std::unique_lock<std::mutex> lock(M->big_mutex);
	const size_t n_vtx = (size_t)M->g.n_seg * 2;
	if (M->lab_max_dist_g >= max_dist_g && M->d_lab_off) return true; // labels are exact for every bound up to the one they were searched with
	// (re)start the table: it must be ours alone.  No new call starts until those in flight are done; a second call that gets here
	// meanwhile searches per read this once (it is one of those the first is waiting for).
	if (M->lab_growing) return false;
	M->lab_growing = true;
	M->slot_cv.wait(lock, [&]() { return M->in_flight <= 1; });
	struct Done { Model *M; ~Done() { M->lab_growing = false; M->slot_cv.notify_all(); } } done{M};
	if (M->d_lab_off == 0) {
		M->d_lab_off = (long long*)dmalloc(n_vtx * sizeof(long long));
		M->d_lab_hdr = (Pool*)dmalloc(sizeof(Pool));
		M->lab_cap = std::min<uint64_t>(std::max<uint64_t>((uint64_t)256 << 20, (uint64_t)n_vtx * 8192), std::max<uint64_t>((uint64_t)64 << 20, dev_free_mem() / 16));
		M->d_lab_pool = (char*)dmalloc(M->lab_cap);
	}
	dfill(M->d_lab_off, 0xff, n_vtx * sizeof(long long));
	Pool hp; hp.used = 0, hp.cap = M->lab_cap;
	h2d(M->d_lab_hdr, &hp, sizeof(Pool));
	M->lab_max_dist_g = max_dist_g;
	dsync();
	return true;
}
// after a batch: a label pool that overflowed is enlarged for the batches to come (the sources that did not fit were searched per read)
static void lab_after_batch(Model *M, unsigned int n_new)
{
	std::unique_lock<std::mutex> lock(M->big_mutex);
	M->lab_sources += n_new;
	Pool hp;
	d2h(&hp, M->d_lab_hdr, sizeof(Pool));
	if (hp.used <= hp.cap || M->lab_growing) return;
	// kernels of other calls may be reading the pool: no new call starts until those in flight are done, then the pool is replaced
	M->lab_growing = true;
	M->slot_cv.wait(lock, [&]() { return M->in_flight <= 1; });
	struct Done { Model *M; ~Done() { M->lab_growing = false; M->slot_cv.notify_all(); } } done{M};
	const uint64_t want = std::max<uint64_t>((uint64_t)hp.used * 2, M->lab_cap * 2);
	if (want > dev_free_mem() / 2) return;
	char *np = (char*)dmalloc(want);
	d2d(np, M->d_lab_pool, M->lab_cap);
	dsync();
	dfree(M->d_lab_pool);
	hp.used = M->lab_cap, hp.cap = want; // everything that was written lies below the old capacity
	M->d_lab_pool = np, M->lab_cap = want;
	h2d(M->d_lab_hdr, &hp, sizeof(Pool));
}

enum { P_ANCHOR, P_MINIPOS, P_LCHAIN, P_OUT, P_PLAN, P_JOBS, P_CIG, P_GSTATE, P_GJOBS, P_WALK, N_POOLS };

// What the phases of one sub-batch share: its reads, where they and the per-read arrays live on both sides, the pool capacities
// and the launch arguments of the pass.  All buffers are the slot's and persistent: cudaMalloc/cudaFree would serialise the slots.
struct Batch {
	Model *M; Model::Slot &sl; mgb_stats_t &S; SlotTimers &TM; const MapOptDev &o;
	int n_reads; const int *qlens; const char *const *seqs; const char *const *names; mg_gchains_t **gcs; GafRoute *gaf; int host_threads; // gaf: the text route (gcs == NULL)
	const std::vector<int32_t> *seg_off, *seg_len;
	int32_t skip1_len, skip2_len; // the tier routing this batch runs with
	double t_host0;
	// host side, page-locked
	uint64_t *seq_off = 0; char *hseq = 0; size_t hseq_bytes = 0;
	ReadOut *routs = 0; ReadMeta *meta = 0; Mail *mail = 0; char *hout = 0;
	std::vector<uint64_t> pack_off;
	std::vector<uint64_t> gaf_off; size_t fix_at = 0; const uint64_t *d_rname_off = 0; const char *d_rname = 0; // text route: text and fix-up offsets ([n+1] each); where the fix-ups sit in hout; the read names
	// device side
	bool packed = false, use_lab = false, first_kernel = true;
	char *d_seq = 0; uint64_t *d_pk = 0, *d_pk_off = 0, *d_seq_off = 0; int32_t *d_seq_len = 0; uint32_t *d_name_hash = 0;
	int32_t *d_list_buf = 0, *d_self_id = 0, *d_rescue = 0, *d_seg_off = 0, *d_seg_len = 0, *d_lab_new = 0;
	unsigned int *d_next = 0, *d_jobq_n = 0, *d_rescue_n = 0, *d_cnt = 0, *d_tier_hist = 0, *d_lab_n = 0;
	unsigned long long *d_prof = 0; Pool *d_pools = 0; ReadMeta *d_meta = 0; ReadOut *d_routs = 0;
	uint64_t cap[N_POOLS] = {}; void *d_buf[N_POOLS] = {};
	int64_t max_jobs = 0, jobs_done = 0, gjobs_done = 0; int32_t *jobq_buf = 0, *order_buf = 0;
	LaunchArgs L = {};
	MailSrc msrc = {};
	int read_status(int i) const { return meta[i].status < 0? meta[i].status : routs[i].status; }
	void pfor(int64_t n, const std::function<void(int64_t)> &fn)
	{
		if (n < 256 || host_threads <= 1) { for (int64_t i = 0; i < n; ++i) fn(i); return; }
		sl.host_pool.run(n, host_threads, fn);
	}
};

// Reads go to and results come from the device in a few pieces, so that the copy of one piece overlaps the host work on the next.
template<typename F> static void for_pieces(int n_reads, const F &fn)
{
	const int n_piece = n_reads >= 2048? 4 : 1;
	for (int pc = 0; pc < n_piece; ++pc) fn(pc, (int64_t)n_reads * pc / n_piece, (int64_t)n_reads * (pc + 1) / n_piece);
}
// fill(r) writes read r into the staging copy h, at element off[r]; each piece goes up as soon as it is filled.  Returns the host
// time spent filling.
template<typename T, typename F> static double upload_pieces(Batch &B, T *d, const T *h, const uint64_t *off, uint64_t end, const F &fill)
{
	double t = 0;
	for_pieces(B.n_reads, [&](int, int64_t r0, int64_t r1) {
		const double t0 = now_ms();
		B.pfor(r1 - r0, [&](int64_t i) { fill(r0 + i); });
		t += now_ms() - t0;
		const uint64_t e0 = off[r0], e1 = r1 < B.n_reads? off[r1] : end;
		h2d_async(d + e0, h + e0, (e1 - e0) * sizeof(T));
	});
	return t;
}

// Phase 2: the per-read arrays and the counters of the sub-batch, carved from one device buffer
static void carve_small(Batch &B)
{
	const int n = B.n_reads;
	char *ds = (char*)B.sl.d_small.ensure((size_t)n * (8 + 4 + 4 + 4 + 4 + 4) + 4096 + 1024);
	B.d_seq_off = (uint64_t*)ds;
	B.d_seq_len = (int32_t*)(B.d_seq_off + n);
	B.d_name_hash = (uint32_t*)(B.d_seq_len + n);
	B.d_list_buf = (int32_t*)(B.d_name_hash + n); // n entries: read list of the retry pass
	B.d_self_id = B.d_list_buf + n; // n entries, MG_M_NO_DIAG only
	B.d_rescue = B.d_self_id + n; // n entries: reads handed from k_chain to k_chain_rescue
	char *dsm = (char*)(((uintptr_t)(B.d_rescue + n) + 255) & ~(uintptr_t)255);
	B.d_next = (unsigned int*)dsm;
	B.d_jobq_n = B.d_next + 4;
	B.d_rescue_n = B.d_next + 8;
	B.d_cnt = B.d_next + 10; // [0] bridging jobs, [1] gap jobs the next job kernel has to take
	B.d_prof = (unsigned long long*)(dsm + 64);
	B.d_pools = (Pool*)(dsm + 64 + sizeof(unsigned long long) * PROF_N);
	B.d_tier_hist = (unsigned int*)((char*)(B.d_pools + 16) + 64); // 32 x 4 counters behind the pool headers
}

// Phase 1, packed: 2 bits per base (a quarter of the bytes; k_unpack writes the ASCII copy on the device).  A read with any byte
// other than A/C/G/T goes up as ASCII; false when such reads are too many to be worth a copy each: the whole batch goes up as ASCII.
static bool upload_packed(Batch &B)
{
	mgb_stats_t &S = B.S;
	const int n = B.n_reads;
	const size_t n8 = ((size_t)n + 7) & ~(size_t)7;
	uint64_t *pk_off = (uint64_t*)B.sl.h_pk.ensure((size_t)n * 8 + 64 + (size_t)(S.n_bases / 4) + (size_t)n * 16);
	uint64_t wtot = 0;
	for (int i = 0; i < n; ++i) { pk_off[i] = wtot; wtot += (uint64_t)((B.qlens[i] > 0? B.qlens[i] : 0) + 31) / 32 + 1; }
	uint64_t *hpk = pk_off + n8;
	B.d_pk_off = (uint64_t*)B.sl.d_pk.ensure((n8 + wtot + 8) * 8);
	B.d_pk = B.d_pk_off + n8;
	std::vector<uint8_t> raw((size_t)n, 0);
	const double t_pack = upload_pieces(B, B.d_pk, hpk, pk_off, wtot, [&](int64_t r) {
		if (B.qlens[r] > 0 && !pack_read(B.seqs[r], B.qlens[r], hpk + pk_off[r])) raw[(size_t)r] = 1;
	});
	int64_t n_raw = 0;
	for (int i = 0; i < n; ++i) n_raw += raw[(size_t)i];
	if (n_raw > 64) return false;
	S.t_pack_ms = t_pack;
	S.h2d_bytes = (int64_t)(wtot * 8);
	for (int i = 0; i < n; ++i)
		if (raw[(size_t)i]) {
			memcpy(B.hseq + B.seq_off[i], B.seqs[i], (size_t)B.qlens[i]);
			h2d_async(B.d_seq + B.seq_off[i], B.hseq + B.seq_off[i], (size_t)B.qlens[i]);
			pk_off[i] = ~0ULL, S.h2d_bytes += B.qlens[i];
		}
	h2d(B.d_pk_off, pk_off, (size_t)n * 8);
	return true;
}

// Phase 1: the reads into page-locked memory and to the device, 2 bits per base unless the fragments have segments
static void upload_reads(Batch &B)
{
	mgb_stats_t &S = B.S;
	const int n = B.n_reads;
	uint64_t *seq_off = B.seq_off = (uint64_t*)B.sl.h_small.ensure((size_t)n * (8 + 4 + 4) + 256);
	int32_t *seq_len = (int32_t*)(seq_off + n);
	uint32_t *name_hash = (uint32_t*)(seq_len + n);
	uint64_t tot = 0;
	for (int i = 0; i < n; ++i) {
		seq_off[i] = tot, seq_len[i] = B.qlens[i];
		tot += (uint64_t)(B.qlens[i] > 0? B.qlens[i] : 0) + 8;
		tot = (tot + 15) & ~(uint64_t)15;
		name_hash[i] = B.names && B.names[i]? hash_str(B.names[i]) : 0;
		S.n_bases += B.qlens[i] > 0? B.qlens[i] : 0;
	}
	S.n_reads = n;
	B.hseq_bytes = tot + 16;
	B.hseq = (char*)B.sl.h_seq.ensure(B.hseq_bytes);
	B.d_seq = (char*)B.sl.d_seq.ensure(B.hseq_bytes);
	B.TM.h2d.start();
	B.packed = p_pack2 && B.seg_off == 0 && upload_packed(B);
	if (!B.packed) {
		S.t_pack_ms += upload_pieces(B, B.d_seq, B.hseq, B.seq_off, B.hseq_bytes, [&](int64_t r) {
			if (B.qlens[r] > 0) memcpy(B.hseq + B.seq_off[r], B.seqs[r], (size_t)B.qlens[r]);
		});
		dsync();
		S.h2d_bytes = (int64_t)B.hseq_bytes;
	}
	carve_small(B);
	h2d(B.d_seq_off, seq_off, (size_t)n * 16); // seq_off, seq_len and name_hash are contiguous on both sides
	S.h2d_bytes += (int64_t)n * 16;
	if (B.packed) {
		UnpackArgs U;
		U.pk = B.d_pk, U.pk_off = B.d_pk_off, U.seq_off = B.d_seq_off, U.seq_len = B.d_seq_len, U.seq = B.d_seq, U.n_reads = n;
		unpack_reads(U);
	}
	B.TM.h2d.stop();
	if (B.o.flag & F_NO_DIAG) { // which segment name, if any, is the read's own (exact string match on the host)
		std::vector<int32_t> self((size_t)n, -1);
		for (int i = 0; i < n; ++i)
			if (B.names && B.names[i]) { auto it = B.M->name_ids.find(B.names[i]); if (it != B.M->name_ids.end()) self[(size_t)i] = it->second; }
		h2d(B.d_self_id, self.data(), sizeof(int32_t) * (size_t)n);
	}
	if (B.seg_off && B.seg_len) { // multi-segment fragments only (mg_map_frag with n_segs > 1)
		B.d_seg_off = (int32_t*)B.sl.d_segs.ensure(sizeof(int32_t) * (B.seg_off->size() + B.seg_len->size()));
		B.d_seg_len = B.d_seg_off + B.seg_off->size();
		h2d(B.d_seg_off, B.seg_off->data(), sizeof(int32_t) * B.seg_off->size());
		h2d(B.d_seg_len, B.seg_len->data(), sizeof(int32_t) * B.seg_len->size());
	}
	B.d_meta = (ReadMeta*)B.sl.d_meta.ensure(sizeof(ReadMeta) * (size_t)n);
	B.d_routs = (ReadOut*)B.sl.d_routs.ensure(sizeof(ReadOut) * (size_t)n);
	dzero(B.d_meta, sizeof(ReadMeta) * (size_t)n);
	dzero(B.d_routs, sizeof(ReadOut) * (size_t)n);
	dzero(B.d_prof, sizeof(unsigned long long) * PROF_N);
	dzero(B.d_tier_hist, sizeof(unsigned int) * 128);
	if (B.gaf) { // the text route prints the read names: their offsets, then the names back to back (a NULL name travels as "*")
		uint64_t tot_n = 0;
		for (int i = 0; i < n; ++i) tot_n += B.names && B.names[i]? strlen(B.names[i]) : 1;
		const size_t hdr = ((size_t)n + 1) * 8;
		uint64_t *h = (uint64_t*)B.sl.h_rname.ensure(hdr + tot_n + 16);
		char *blob = (char*)(h + n + 1);
		h[0] = 0;
		for (int i = 0; i < n; ++i) {
			const char *nm = B.names && B.names[i]? B.names[i] : "*";
			const size_t l = strlen(nm);
			memcpy(blob + h[i], nm, l), h[i + 1] = h[i] + l;
		}
		char *d = (char*)B.sl.d_rname.ensure(hdr + tot_n + 16);
		h2d(d, h, hdr + tot_n);
		B.d_rname_off = (const uint64_t*)d, B.d_rname = d + hdr;
		S.h2d_bytes += (int64_t)(hdr + tot_n);
	}
}

// Phase 3: the first pool sizes, and what every pass of the sub-batch reports into (statuses, label sources, mailbox)
static void size_pools(Batch &B)
{
	const uint64_t nb = (uint64_t)B.S.n_bases, nr = (uint64_t)B.n_reads;
	uint64_t *cap = B.cap;
	cap[P_ANCHOR] = std::max<uint64_t>(nb / 4 * sizeof(u128), (uint64_t)1 << 22);
	cap[P_MINIPOS] = std::max<uint64_t>(nb * sizeof(int32_t) / 2, (uint64_t)1 << 20);
	cap[P_LCHAIN] = std::max<uint64_t>(nr * 64 * sizeof(LChain), (uint64_t)1 << 20);
	cap[P_OUT] = std::max<uint64_t>(nb * 4, (uint64_t)1 << 22);
	cap[P_PLAN] = std::max<uint64_t>(nb / 8 * 8, (uint64_t)1 << 20);
	cap[P_JOBS] = std::max<uint64_t>(nb / 40 * sizeof(WfaJob), (uint64_t)1 << 20);
	cap[P_CIG] = std::max<uint64_t>(nb, (uint64_t)1 << 20) + (uint64_t)B.sl.W.n_workers * CIG_CHUNK_BYTES * 4; // + the unused ends of the warps' slices (three tier kernels per pass)
	cap[P_GSTATE] = std::max<uint64_t>(nr * 2048, (uint64_t)1 << 20);
	cap[P_GJOBS] = std::max<uint64_t>(nr * 24 * sizeof(GwfaJob), (uint64_t)1 << 20);
	cap[P_WALK] = std::max<uint64_t>(nr * 256, (uint64_t)1 << 20);
	for (int i = 0; i < N_POOLS; ++i) if (B.sl.d_pool[i].cap > cap[i]) cap[i] = B.sl.d_pool[i].cap & ~(size_t)4095; // keep what earlier batches needed
	B.routs = (ReadOut*)B.sl.h_routs.ensure((sizeof(ReadOut) + sizeof(ReadMeta)) * nr + 64); // page-locked: a pageable destination makes the copy a blocking, staged one
	B.meta = (ReadMeta*)(B.routs + B.n_reads);
	B.use_lab = p_lab_cache && lab_prepare(B.M, B.o.bw_long);
	B.mail = (Mail*)B.sl.h_mail.ensure(sizeof(Mail));
	if (B.use_lab) { // this call's list of sources to search
		B.d_lab_n = (unsigned int*)B.sl.d_lab_new.ensure(((size_t)B.M->g.n_seg * 2 + 4) * sizeof(int32_t));
		B.d_lab_new = (int32_t*)(B.d_lab_n + 4);
	}
	MailSrc &m = B.msrc;
	m.pools = B.d_pools, m.jobq_n = B.d_jobq_n, m.lab_n = B.d_lab_n, m.prof = B.d_prof, m.tier_hist = B.d_tier_hist, m.peak = B.sl.W.peak, m.n_workers = B.sl.W.n_workers;
}

// Phase 4: empty pools of the current sizes and the launch arguments of a pass over them
static void fill_launch_args(Batch &B)
{
	const Model *M = B.M;
	const uint64_t *cap = B.cap;
	Pool hp[N_POOLS];
	for (int i = 0; i < N_POOLS; ++i) B.d_buf[i] = B.sl.d_pool[i].ensure(cap[i]), hp[i].used = 0, hp[i].cap = cap[i];
	h2d(B.d_pools, hp, sizeof(hp));
	dfill(B.d_buf[P_GJOBS], 0xff, cap[P_GJOBS]); // reserved-but-unused bridging job slots read as rid == -1
	dfill(B.d_buf[P_JOBS], 0xff, cap[P_JOBS]);   // the same for gap jobs: slots of an allocation that overflowed the pool are never written
	LaunchArgs &L = B.L;
	memset(&L, 0, sizeof(L));
	L.c.g = M->g, L.c.ix = M->ix, L.c.opt = B.o;
	L.c.b.n_reads = B.n_reads, L.c.b.seq = B.d_seq, L.c.b.seq_off = B.d_seq_off, L.c.b.seq_len = B.d_seq_len, L.c.b.name_hash = B.d_name_hash;
	L.c.b.seg_off = B.d_seg_off, L.c.b.seg_len = B.d_seg_len, L.c.b.self_id = (B.o.flag & F_NO_DIAG)? B.d_self_id : 0;
	L.c.b.pk = B.packed? B.d_pk : 0, L.c.b.pk_off = B.packed? B.d_pk_off : 0;
	L.c.meta = B.d_meta;
	L.c.pool_anchor = &B.d_pools[P_ANCHOR], L.c.anchor = (u128*)B.d_buf[P_ANCHOR];
	L.c.pool_minipos = &B.d_pools[P_MINIPOS], L.c.minipos = (int32_t*)B.d_buf[P_MINIPOS];
	L.c.pool_lchain = &B.d_pools[P_LCHAIN], L.c.lchain = (LChain*)B.d_buf[P_LCHAIN];
	L.c.pool_out = &B.d_pools[P_OUT], L.c.out = (char*)B.d_buf[P_OUT];
	L.c.pool_plan = &B.d_pools[P_PLAN], L.c.plan = (uint64_t*)B.d_buf[P_PLAN];
	L.c.pool_jobs = &B.d_pools[P_JOBS], L.c.jobs = (WfaJob*)B.d_buf[P_JOBS];
	L.c.pool_cig = &B.d_pools[P_CIG], L.c.cig = (uint32_t*)B.d_buf[P_CIG];
	L.c.pool_gstate = &B.d_pools[P_GSTATE], L.c.gstate = (char*)B.d_buf[P_GSTATE];
	L.c.pool_gjobs = &B.d_pools[P_GJOBS], L.c.gjobs = (GwfaJob*)B.d_buf[P_GJOBS];
	L.c.pool_walk = &B.d_pools[P_WALK], L.c.walk = (int32_t*)B.d_buf[P_WALK];
	L.c.next_read = B.d_next;
	L.c.rescue_list = B.d_rescue, L.c.rescue_n = B.d_rescue_n;
	if (B.use_lab) {
		L.c.lab.src_off = M->d_lab_off, L.c.lab.pool_hdr = M->d_lab_hdr, L.c.lab.pool = M->d_lab_pool, L.c.lab.new_src = B.d_lab_new, L.c.lab.n_new = B.d_lab_n;
		L.c.lab.max_dist_g = M->lab_max_dist_g, L.c.lab.cap_new = M->g.n_seg * 2;
		dzero(B.d_lab_n, 2 * sizeof(unsigned int));
	}
	L.c.prof = B.d_prof;
	L.c.tier_hist = B.d_tier_hist, L.c.skip1_len = B.skip1_len, L.c.skip2_len = B.skip2_len;
	L.c.jobq_n = B.d_jobq_n;
	L.routs = B.d_routs;
	B.jobs_done = B.gjobs_done = 0;
	B.max_jobs = (int64_t)(cap[P_JOBS] / sizeof(WfaJob)) + 1;
	const int64_t max_gjobs = (int64_t)(cap[P_GJOBS] / sizeof(GwfaJob)) + 1;
	B.jobq_buf = (int32_t*)B.sl.d_jobq.ensure(sizeof(int32_t) * 2 * (size_t)B.max_jobs);
	B.order_buf = (int32_t*)B.sl.d_order.ensure(sizeof(int32_t) * (size_t)std::max<int64_t>(std::max<int64_t>(B.max_jobs, max_gjobs), B.n_reads));
}

// One stage of a pass, timed by t if given.  order: its items go longest first (make_job_order of that kind, inside the timed span).
template<int STAGE> static void launch(Batch &B, const Workers &W, EvTimer *t, int order = NO_ORDER)
{
	Span span(t);
	LaunchArgs &L = B.L;
	const int32_t *list = L.rid_list;
	if (order != NO_ORDER) {
		make_job_order(L, order, order == ORDER_GAPS? L.c.jobq[1] : 0, L.n_work, B.order_buf, L.n_work_dev);
		L.rid_list = B.order_buf;
	}
	launch_stage<STAGE>(L, W);
	L.rid_list = list;
}

// Phase 5: one pass over a set of reads (d_list == 0: the whole sub-batch).  T: the timers of the first pass; the retry pass is
// not timed.  From k_gchain on every kernel reads its number of units on the device: the whole pass is queued without a host
// round trip, so nothing another thread does in the driver (large copies, blocking waits) can open gaps between its kernels.
static void run_pass(Batch &B, const int32_t *d_list, int32_t n_list, const Workers &W, SlotTimers *T)
{
	LaunchArgs &L = B.L;
	auto tm = [T](EvTimer SlotTimers::*m) { return T? &(T->*m) : (EvTimer*)0; };
	auto tk = [T](int stage) { return T? &T->k[stage] : (EvTimer*)0; }; // (one per kernel slot)
	auto counts = [&]() { count_jobs(B.d_pools, (int)P_GJOBS, (int)P_JOBS, (unsigned int)B.gjobs_done, (unsigned int)B.jobs_done, B.d_cnt); };
	L.rid_list = d_list, L.n_work = n_list;
	if (B.first_kernel) ev_record(B.sl.ev_first), B.first_kernel = false;
	{ Span s(tm(&SlotTimers::seed)); launch<ST_SEED>(B, W, tk(ST_SEED)); }
	{
		Span s(tm(&SlotTimers::chain)), k(tk(ST_CHAIN)); // t_kernel_ms[1]: both chaining kernels
		dzero(B.d_rescue_n, sizeof(unsigned int));
		launch<ST_CHAIN>(B, W, 0);
		L.n_work_dev = B.d_rescue_n, L.rid_list = 0; // the reads k_chain put on the rescue list (count known on the device only)
		launch<ST_CHAIN_RESCUE>(B, W, 0);
		L.n_work_dev = 0, L.rid_list = d_list;
	}
	{
		Span s(tm(&SlotTimers::align));
		if (B.use_lab) { // labels of the sources k_chain listed (count known on the device only)
			L.n_work_dev = B.d_lab_n, L.rid_list = 0;
			Span lab(tm(&SlotTimers::lab));
			launch<ST_LABELS>(B, W, 0);
			L.n_work_dev = B.d_lab_n + 1;
			launch<ST_LABELS_BIG>(B, W, 0);
			L.n_work_dev = 0, L.rid_list = d_list;
		}
		// whole batch: reads with many linear chains first (a few of them set the time of this kernel)
		launch<ST_GCHAIN>(B, W, tk(ST_GCHAIN), d_list == 0 && n_list >= 1024? ORDER_READS : NO_ORDER);
		counts(); // bridging jobs planned by k_gchain, then materialisation
		L.rid_list = 0, L.job_start = B.gjobs_done, L.n_work = 0, L.n_work_dev = B.d_cnt;
		launch<ST_GWFA>(B, W, tk(ST_GWFA), ORDER_BRIDGES);
		L.rid_list = d_list, L.n_work = n_list, L.n_work_dev = 0;
		launch<ST_GCHAIN_GEN>(B, W, tk(ST_GCHAIN_GEN));
	}
	{ // three tiers; a job that does not fit one tier is queued for the next
		Span s(tm(&SlotTimers::wfa));
		counts();
		L.c.jobq[0] = B.jobq_buf, L.c.jobq[1] = B.jobq_buf + B.max_jobs;
		dzero(B.d_jobq_n, 2 * sizeof(unsigned int));
		L.rid_list = 0, L.job_start = B.jobs_done, L.n_work = 0, L.n_work_dev = B.d_cnt + 1;
		launch<ST_WFA1>(B, W, tk(ST_WFA1));
		L.n_work_dev = B.d_jobq_n;
		launch<ST_WFA2>(B, W, tk(ST_WFA2));
		L.n_work_dev = B.d_jobq_n + 1;
		launch<ST_WFA3>(B, W, tk(ST_WFA3), ORDER_GAPS);
		L.rid_list = 0, L.n_work_dev = 0;
	}
	L.rid_list = d_list, L.n_work = n_list;
	{ Span s(tm(&SlotTimers::fin)); launch<ST_FINISH>(B, W, tk(ST_FINISH)); }
	ev_record(B.sl.ev_last);
	fetch_mail(B.msrc, B.mail); // (also the one wait of the pass)
	const Pool &pg = B.mail->pools[P_GJOBS], &pj = B.mail->pools[P_JOBS];
	B.gjobs_done = (int64_t)(std::min<uint64_t>(pg.used, pg.cap) / sizeof(GwfaJob));
	B.jobs_done = (int64_t)(std::min<uint64_t>(pj.used, pj.cap) / sizeof(WfaJob));
	if (T) B.S.n_jobs_mid = B.mail->jobq_n[0], B.S.n_jobs_big = B.mail->jobq_n[1];
}

// Phase 6: the reads whose worker arena overflowed run again with large arenas and few workers (shared by the slots).  Returns
// whether an output pool overflowed: then the whole sub-batch runs again with larger pools.
static bool redo_arena_overflows(Batch &B)
{
	const int n = B.n_reads;
	auto fetch_status = [&]() {
		d2h(B.routs, B.d_routs, sizeof(ReadOut) * (size_t)n);
		d2h(B.meta, B.d_meta, sizeof(ReadMeta) * (size_t)n);
	};
	fetch_status();
	std::vector<int32_t> redo;
	bool pool_full = false;
	for (int i = 0; i < n; ++i) {
		const int st = B.read_status(i);
		if (st == MGB_E_ARENA) redo.push_back(i);
		else if (st == MGB_E_POOL) pool_full = true;
	}
	if (pool_full || redo.empty()) return pool_full;
	Model *M = B.M;
	std::lock_guard<std::mutex> lock(M->big_mutex);
	const uint64_t big = (uint64_t)p_arena_big_mb << 20;
	const int nw = (int)std::min<uint64_t>(16, std::max<uint64_t>(1, dev_free_mem() / 2 / big)); // a handful of reads per batch at most come here
	if (M->Wbig.arena == 0 || M->Wbig.arena_bytes != big) ensure_workers(M->Wbig, std::max(1, nw), big);
	h2d(B.d_list_buf, redo.data(), redo.size() * sizeof(int32_t));
	{
		std::unique_lock<std::mutex> gpu(M->gpu_mutex, std::defer_lock);
		if (p_gpu_lock) gpu.lock();
		const double tw = now_ms();
		run_pass(B, B.d_list_buf, (int32_t)redo.size(), M->Wbig, 0);
		B.S.w_redo_ms += now_ms() - tw;
	}
	B.S.n_retry += (int64_t)redo.size();
	fetch_status();
	for (int i = 0; i < n; ++i) if (B.read_status(i) == MGB_E_POOL) pool_full = true;
	return pool_full;
}

// Phase 7: the result blobs into read order, then to the host in pieces (the assembly follows piece by piece)
static void download_results(Batch &B)
{
	const int n = B.n_reads;
	B.TM.d2h.start();
	const size_t pool_bytes = (size_t)std::min<uint64_t>(B.mail->pools[P_OUT].used, B.cap[P_OUT]);
	PackArgs P;
	P.routs = B.d_routs, P.meta = B.d_meta, P.n = n, P.pool = (const char*)B.d_buf[P_OUT];
	P.packed = (char*)B.sl.d_packed.ensure(pool_bytes + 64), P.off = (uint64_t*)B.sl.d_packoff.ensure(sizeof(uint64_t) * ((size_t)n + 1));
	pack_results(P);
	d2h(B.routs, B.d_routs, sizeof(ReadOut) * (size_t)n);
	B.pack_off.resize((size_t)n + 1);
	d2h(B.pack_off.data(), P.off, sizeof(uint64_t) * ((size_t)n + 1));
	const size_t out_bytes = (size_t)B.pack_off[n];
	B.hout = (char*)B.sl.h_out.ensure(out_bytes + 64);
	for_pieces(n, [&](int pc, int64_t r0, int64_t r1) {
		const uint64_t b0 = B.pack_off[r0], b1 = B.pack_off[r1];
		d2h_async(B.hout + b0, P.packed + b0, b1 - b0);
		ev_record(B.sl.ev_piece[pc]);
	});
	B.TM.d2h.stop();
	B.S.out_bytes = (int64_t)out_bytes;
}

// Phase 7, text route: the GAF text of every read, formatted on the device (mgb_gaf.cuh) from the blobs where the kernels left
// them: k_gaf_size counts each read's bytes and dv:f fix-ups, one scan turns the counts into offsets, the host reads them back
// once to size the buffers, k_gaf_write writes.  The fix-up records go to the host first, the text follows in pieces.
static void download_gaf(Batch &B)
{
	const int n = B.n_reads;
	B.TM.d2h.start();
	GafCtx x = B.M->gaf_graph;
	x.rname = B.d_rname, x.rname_off = B.d_rname_off, x.flag = B.o.flag;
	x.text_off = (uint64_t*)B.sl.d_gafoff.ensure(sizeof(uint64_t) * 2 * ((size_t)n + 1)), x.fix_off = x.text_off + n + 1;
	x.text = 0, x.fix = 0;
	GafCtx *d_x = (GafCtx*)B.sl.d_gafctx.ensure(sizeof(GafCtx));
	h2d(d_x, &x, sizeof(x));
	LaunchArgs &L = B.L;
	L.gaf = d_x, L.rid_list = 0, L.n_work = n, L.n_work_dev = 0;
	{
		Span t(&B.TM.gaf_size);
		launch<ST_GAF_SIZE>(B, B.sl.W, 0);
		gaf_scan(x.text_off, x.fix_off, n);
	}
	B.gaf_off.resize(2 * ((size_t)n + 1));
	d2h(B.gaf_off.data(), x.text_off, sizeof(uint64_t) * B.gaf_off.size());
	const uint64_t *toff = B.gaf_off.data(), text_bytes = toff[n], n_fix = toff[2 * n + 1];
	x.text = (char*)B.sl.d_text.ensure(text_bytes + 64), x.fix = (GafFix*)B.sl.d_fix.ensure(n_fix * sizeof(GafFix) + 64);
	h2d(d_x, &x, sizeof(x));
	{ Span t(&B.TM.gaf_write); launch<ST_GAF_WRITE>(B, B.sl.W, 0); }
	B.fix_at = (text_bytes + 15) & ~(uint64_t)15;
	B.hout = (char*)B.sl.h_out.ensure(B.fix_at + n_fix * sizeof(GafFix) + 64);
	d2h_async(B.hout + B.fix_at, x.fix, n_fix * sizeof(GafFix));
	for_pieces(n, [&](int pc, int64_t r0, int64_t r1) {
		d2h_async(B.hout + toff[r0], x.text + toff[r0], toff[r1] - toff[r0]);
		ev_record(B.sl.ev_piece[pc]);
	});
	B.TM.d2h.stop();
	B.S.out_bytes = (int64_t)(text_bytes + n_fix * sizeof(GafFix));
}

// Phase 8: tier routing for the next batch: the first length bucket in which the sampled gaps mostly ended beyond a tier
static void learn_tier_routing(Batch &B)
{
	const unsigned int *h = B.mail->tier_hist;
	int32_t t1 = INT32_MAX, t2 = INT32_MAX;
	for (int b = 0; b < 32 && t1 == INT32_MAX; ++b) { unsigned int in = h[b * 4 + 1], out = h[b * 4 + 2] + h[b * 4 + 3]; if (in + out >= 8 && in < out) t1 = b * 16; }
	for (int b = 0; b < 32 && t2 == INT32_MAX; ++b) { unsigned int in = h[b * 4 + 1] + h[b * 4 + 2], out = h[b * 4 + 3]; if (in + out >= 8 && in < out) t2 = b * 16; }
	unsigned int tot = 0;
	for (int i = 0; i < 128; ++i) tot += h[i];
	if (tot >= 64 && p_tier_learn) { std::lock_guard<std::mutex> lock(B.M->big_mutex); B.M->skip1_len = t1, B.M->skip2_len = t2 < t1? t1 : t2; }
	B.S.skip1_len = B.skip1_len, B.S.skip2_len = B.skip2_len;
}

// Before phase 9: a read that failed on the device fails the call
static int check_reads(Batch &B)
{
	mgb_stats_t &S = B.S;
	for (int i = 0; i < B.n_reads; ++i) {
		const int st = B.read_status(i);
		if (st < 0) {
			char buf[256];
			snprintf(buf, sizeof(buf), "read '%s' (%d bp) failed on the device with code %d%s", B.names && B.names[i]? B.names[i] : "", B.qlens[i], st,
					 st == MGB_E_ARENA? " (worker arena exhausted even in the retry pass; raise arena_big_mb)" : "");
			set_error(buf);
			return st;
		}
		const ReadMeta &m = B.meta[i];
		S.n_seeds += m.n_seed0, S.n_anchors_out += m.n_a, S.n_chains_out += m.n_u0, S.n_minimizers += m.n_mz;
	}
	return 0;
}

// Phase 9: mg_gchains_t of every read, piece by piece as the copies land
static int assemble_results(Batch &B)
{
	mgb_stats_t &S = B.S;
	const double t_asm0 = now_ms();
	S.w_download_ms = t_asm0 - B.t_host0 - S.w_upload_ms - S.w_pass_ms - S.w_redo_ms - S.w_gpu_wait_ms;
	if (const int rc = check_reads(B)) return rc;
	for_pieces(B.n_reads, [&](int pc, int64_t r0, int64_t r1) {
		ev_wait(B.sl.ev_piece[pc]);
		B.pfor(r1 - r0, [&](int64_t k) {
			const int64_t i = r0 + k;
			if (B.read_status((int)i) == 1) B.gcs[i] = 0; // empty or over-long read: reference returns before allocating (map-algo.c:359-360)
			else B.gcs[i] = build_result(B.routs[i], B.hout);
		});
	});
	S.t_asm_ms = now_ms() - t_asm0;
	S.t_d2h_ms = B.TM.d2h.ms(); // pack kernels + the pieces of the copy (they overlap the assembly above)
	S.t_host_ms = now_ms() - B.t_host0;
	return 0;
}

// Phase 9, text route: the caller's text, piece by piece as the copies land, with every record's `dv:f` put in at the byte its
// fix-up names (the fix-ups came first: the final size is known before the first byte is copied)
static int assemble_gaf(Batch &B)
{
	mgb_stats_t &S = B.S;
	const double t_asm0 = now_ms();
	S.w_download_ms = t_asm0 - B.t_host0 - S.w_upload_ms - S.w_pass_ms - S.w_redo_ms - S.w_gpu_wait_ms;
	if (const int rc = check_reads(B)) return rc;
	const int n = B.n_reads;
	const uint64_t *toff = B.gaf_off.data(), *foff = toff + n + 1;
	ev_wait(B.sl.ev_piece[0]); // (the fix-up records were queued in front of the first piece)
	const GafFix *fx = (const GafFix*)(B.hout + B.fix_at);
	enum { DV_MAX = 16 };
	std::vector<char> dv((size_t)foff[n] * DV_MAX);
	std::vector<uint8_t> dv_len((size_t)foff[n]);
	std::vector<uint64_t> at((size_t)n + 1); // where each read's text starts in the output
	B.pfor(n, [&](int64_t r) {
		uint64_t add = 0;
		for (uint64_t k = foff[r]; k < foff[r + 1]; ++k)
			add += dv_len[k] = (uint8_t)gaf_dv_text(gchain_div(fx[k].n_mini, fx[k].n_anchor, fx[k].q_span), &dv[k * DV_MAX]);
		at[(size_t)r + 1] = add;
	});
	for (int r = 0; r < n; ++r) at[(size_t)r + 1] += at[(size_t)r];
	for (int r = 0; r <= n; ++r) at[(size_t)r] += toff[r];
	char *o = gaf_reserve(*B.gaf, at[(size_t)n]);
	for_pieces(n, [&](int pc, int64_t r0, int64_t r1) {
		ev_wait(B.sl.ev_piece[pc]);
		B.pfor(r1 - r0, [&](int64_t i) {
			const int64_t r = r0 + i;
			const char *src = B.hout + toff[r];
			char *dst = o + at[(size_t)r];
			uint64_t pos = 0;
			for (uint64_t k = foff[r]; k < foff[r + 1]; ++k) {
				memcpy(dst, src + pos, fx[k].at - pos), dst += fx[k].at - pos, pos = fx[k].at;
				memcpy(dst, &dv[k * DV_MAX], dv_len[k]), dst += dv_len[k];
			}
			memcpy(dst, src + pos, toff[r + 1] - toff[r] - pos);
		});
	});
	*B.gaf->len = at[(size_t)n];
	S.t_asm_ms = now_ms() - t_asm0;
	S.t_d2h_ms = B.TM.d2h.ms();
	S.t_host_ms = now_ms() - B.t_host0;
	return 0;
}

// Map reads [0, n_reads) of one sub-batch on the calling thread's stream (slot `sl`).  The output is either the mg_gchains_t
// objects in gcs[] or, with gaf (the text route), the GAF text in the caller's buffer.
static int map_range(Model *M, Model::Slot &sl, const MapOptDev &o, int n_reads, const int *qlens, const char *const *seqs, const char *const *names,
					 mg_gchains_t **gcs, GafRoute *gaf, int host_threads, const std::vector<int32_t> *seg_off = 0, const std::vector<int32_t> *seg_len = 0)
{
	mgb_stats_t &S = sl.st;
	memset(&S, 0, sizeof(S));
	if (n_reads <= 0) return 0;
	// the event pairs live in the slot: creating and destroying three dozen events per call contends on the driver's lock with the other calls in flight
	if (sl.timers == 0) sl.timers = new SlotTimers();
	sl.timers->reset();
	const int64_t launches0 = t_launches;
	Batch B{M, sl, S, *sl.timers, o, n_reads, qlens, seqs, names, gcs, gaf, host_threads, seg_off, seg_len, M->skip1_len, M->skip2_len, now_ms()};
	upload_reads(B);
	size_pools(B);
	int rc = 0;
	for (int attempt = 0;; ++attempt) {
		fill_launch_args(B);
		{
			const double tq = now_ms();
			if (attempt == 0) S.w_upload_ms = tq - B.t_host0;
			std::unique_lock<std::mutex> gpu(M->gpu_mutex, std::defer_lock);
			if (p_gpu_lock) gpu.lock();
			const double tw = now_ms();
			S.w_gpu_wait_ms += tw - tq;
			run_pass(B, 0, n_reads, sl.W, &B.TM);
			S.w_pass_ms += now_ms() - tw;
		}
		S.n_jobs = B.jobs_done;
		const bool pool_full = redo_arena_overflows(B);
		fetch_mail(B.msrc, B.mail);
		if (B.use_lab) { S.n_lab_new = (int64_t)B.mail->lab_n[0], S.n_lab_big = (int64_t)B.mail->lab_n[1]; lab_after_batch(M, B.mail->lab_n[0]); }
		if (!pool_full) { if (gaf) download_gaf(B); else download_results(B); break; }
		// grow whatever overflowed (used counts keep growing past cap, so they tell how much was wanted)
		for (int i = 0; i < N_POOLS; ++i) if (B.mail->pools[i].used > B.cap[i]) B.cap[i] = (B.mail->pools[i].used * 3 / 2 + 4095) & ~(uint64_t)4095;
		if (attempt == 7) { set_error("output pools kept overflowing"); rc = -2; break; }
	}
	SlotTimers &TM = B.TM;
	S.t_h2d_ms = TM.h2d.ms(), S.t_seed_ms = TM.seed.ms(), S.t_chain_ms = TM.chain.ms(), S.t_align_ms = TM.align.ms();
	S.t_wfa_ms = TM.wfa.ms(), S.t_finish_ms = TM.fin.ms();
	for (int i = 0; i < 10; ++i) S.t_kernel_ms[i] = TM.k[i].ms();
	S.t_lab_ms = TM.lab.ms();
	S.t_gaf_ms = TM.gaf_size.ms() + TM.gaf_write.ms();
	S.arena_peak = B.mail->arena_peak; // (the mailbox was last filled after the last pass of the batch)
	for (int i = 0; i < 32; ++i) S.prof[i] = (uint64_t)B.mail->prof[i];
	S.n_launches = t_launches - launches0;
	learn_tier_routing(B);
	if (rc < 0) return rc;
	return gaf? assemble_gaf(B) : assemble_results(B);
}

static void slot_prepare(Model *M, Model::Slot &sl, int n_workers)
{
#ifndef MGB_HOSTSIM
	if (!sl.ready) {
		CUDA_OK(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
		CUDA_OK(cudaEventCreate(&sl.ev_first));
		CUDA_OK(cudaEventCreate(&sl.ev_last));
		for (int i = 0; i < 4; ++i) CUDA_OK(cudaEventCreateWithFlags(&sl.ev_piece[i], cudaEventDisableTiming));
	}
#endif
	sl.ready = true;
	ensure_workers(sl.W, n_workers, (uint64_t)p_arena_mb << 20);
	(void)M;
}

static thread_local mgb_stats_t t_last_stats; // of the last batch mapped by the calling thread
static thread_local bool t_has_stats = false;

// One call = one slot: its own stream, staging buffers, pools and worker arenas.  Up to "slots" calls run at once on one index
// (callers beyond that wait), so a host that maps mini-batch i+1 on a second thread overlaps its packing, copies and result
// assembly with the kernels of mini-batch i -- what the reference's kt_pipeline does with its step threads (gmap.c:176).
static int map_batch_on(Model *M, int n_reads, const int *qlens, const char *const *seqs, const char *const *names,
						mg_gchains_t **gcs, const mg_mapopt_t *opt, const std::vector<int32_t> *seg_off = 0, const std::vector<int32_t> *seg_len = 0,
						GafRoute *gaf = 0)
{
	if (gcs) for (int i = 0; i < n_reads; ++i) gcs[i] = 0;
	if (n_reads <= 0) return 0;
	double t0 = now_ms();
	int32_t max_qlen = 0;
	for (int i = 0; i < n_reads; ++i) if (qlens[i] > max_qlen) max_qlen = qlens[i];
	int k = -1;
	{ // take a slot
		std::unique_lock<std::mutex> lk(M->big_mutex);
		const int max_slots = (int)std::max<int64_t>(1, std::min<int64_t>(p_slots, Model::MAX_SLOTS));
		M->slot_cv.wait(lk, [&]() { if (M->lab_growing) return false; for (int i = 0; i < max_slots; ++i) if (!M->slot_busy[i]) return true; return false; });
		for (int i = 0; i < max_slots && k < 0; ++i) if (!M->slot_busy[i]) k = i;
		M->slot_busy[k] = true, ++M->in_flight;
	}
	Model::Slot &sl = M->slots[k];
	const double t_slot = now_ms();
	set_device(M->device);
	int rc = 0;
	try {
		slot_prepare(M, sl, p_slot_workers > 0? (int)p_slot_workers : default_workers());
		set_stream(sl.stream);
		if (gaf) gaf_upload_graph(M, gaf->g);
		MapOptDev o;
		fill_opt(o, opt, M->k);
		{ // glibc logf table for mapq (reference: gcmisc.c:216-217); grown under the lock, old copies are kept until the model dies
			std::lock_guard<std::mutex> lk(M->big_mutex);
			int need = std::max(1 << 16, max_qlen + 4096);
			if (M->n_logf < need) {
				M->logf_tab.resize(need);
				for (int i = 0; i < need; ++i) M->logf_tab[i] = logf((float)i);
				if (M->d_logf) M->dev_ptrs.push_back(M->d_logf); // a call in flight may still read it
				M->d_logf = dalloc_copy(M->logf_tab);
				M->n_logf = need;
			}
			o.logf_tab = M->d_logf, o.n_logf_tab = M->n_logf;
		}
		rc = map_range(M, sl, o, n_reads, qlens, seqs, names, gcs, gaf, n_host_threads(), seg_off, seg_len);
	} catch (const MgbError &e) {
		rc = e.code;
	}
	set_stream(0); // the slot's stream dies with the model; later calls on this thread (mg_index of another graph) use the default one
	mgb_stats_t S = sl.st;
	S.w_slot_wait_ms = t_slot - t0;
	if (rc == 0 && sl.ready) S.t_dev_span_ms = ev_elapsed_ms(sl.ev_first, sl.ev_last);
	S.n_slots = k;
	S.t_host_ms = now_ms() - t0;
	t_last_stats = S, t_has_stats = true;
	{
		std::lock_guard<std::mutex> lk(M->big_mutex);
		M->stats = S;
		M->slot_busy[k] = false, --M->in_flight;
	}
	M->slot_cv.notify_all();
	if (rc < 0) { // no partial results are left behind
		if (gcs) for (int i = 0; i < n_reads; ++i) if (gcs[i]) { mg_gchain_free(gcs[i]); gcs[i] = 0; }
		return rc;
	}
	return 0;
}

// The batch on every device of the index: contiguous parts of about equal bases, one host thread per device, results in input order.
// The text route: every part formats its own text, and the parts are joined in input order.
static int map_batch_impl(const mg_idx_t *gi, int n_reads, const int *qlens, const char *const *seqs, const char *const *names,
						  mg_gchains_t **gcs, const mg_mapopt_t *opt, const std::vector<int32_t> *seg_off = 0, const std::vector<int32_t> *seg_len = 0,
						  GafRoute *gaf = 0)
{
	Model *M = (Model*)gi->B;
	const int n_dev = 1 + (int)M->peers.size();
	if (n_dev == 1 || seg_off || n_reads < 2 * n_dev) return map_batch_on(M, n_reads, qlens, seqs, names, gcs, opt, seg_off, seg_len, gaf);
	for (Model *P : M->peers) if (P == 0) { set_error("the index is missing on one of the MGB_DEVICES"); return MGB_E_INTERNAL; }
	int64_t tot = 0;
	for (int i = 0; i < n_reads; ++i) tot += qlens[i] > 0? qlens[i] : 0;
	std::vector<int> bound((size_t)n_dev + 1, n_reads);
	bound[0] = 0;
	{
		int64_t acc = 0; int k = 1;
		for (int i = 0; i < n_reads && k < n_dev; ++i) {
			acc += qlens[i] > 0? qlens[i] : 0;
			if (acc >= tot * k / n_dev) bound[(size_t)k++] = i + 1;
		}
	}
	std::vector<int> rcs((size_t)n_dev, 0);
	std::vector<char*> txt((size_t)n_dev, (char*)0); // the text route: each part's text
	std::vector<size_t> txt_len((size_t)n_dev, 0);
	std::vector<GafRoute> part((size_t)n_dev);
	std::vector<std::thread> th;
	for (int d = 0; d < n_dev; ++d)
		th.emplace_back([&, d]() {
			const int b = bound[(size_t)d], e = bound[(size_t)d + 1];
			if (gaf) part[(size_t)d] = GafRoute{gaf->g, &txt[(size_t)d], &txt_len[(size_t)d], 0};
			if (e > b) rcs[(size_t)d] = map_batch_on(d == 0? M : M->peers[(size_t)d - 1], e - b, qlens + b, seqs + b, names? names + b : 0, gcs? gcs + b : 0, opt, 0, 0,
													 gaf? &part[(size_t)d] : 0);
		});
	for (auto &t : th) t.join();
	int rc = 0;
	for (int d = 0; d < n_dev; ++d) if (rcs[(size_t)d] < 0 && rc == 0) rc = rcs[(size_t)d];
	if (rc < 0 && gcs) for (int i = 0; i < n_reads; ++i) if (gcs[i]) { mg_gchain_free(gcs[i]); gcs[i] = 0; } // no partial results are left behind
	if (rc == 0 && gaf) {
		size_t tot = 0;
		for (size_t l : txt_len) tot += l;
		try {
			char *o = gaf_reserve(*gaf, tot);
			for (int d = 0; d < n_dev; ++d) if (txt_len[(size_t)d]) memcpy(o, txt[(size_t)d], txt_len[(size_t)d]), o += txt_len[(size_t)d];
			*gaf->len = tot;
		} catch (const MgbError &e) { rc = e.code; }
	}
	for (char *t : txt) free(t);
	set_device(M->device);
	return rc;
}

extern "C" int mg_map_batch(const mg_idx_t *gi, int n_reads, const int *qlens, const char *const *seqs, const char *const *names,
							mg_gchains_t **gcs, const mg_mapopt_t *opt)
{
	return map_batch_impl(gi, n_reads, qlens, seqs, names, gcs, opt);
}

// The GAF text of a batch, formatted on the device (include/mgb200.h)
extern "C" int mgb_map_batch_gaf(const mg_idx_t *gi, int n_reads, const int *qlens, const char *const *seqs, const char *const *names,
								 const mg_mapopt_t *opt, char **out, size_t *out_len, size_t *out_cap)
{
	*out_len = 0;
	GafRoute R{gi->g, out, out_len, out_cap};
	int rc = 0;
	if (opt->flag & (F_WRITE_LCHAIN | F_WRITE_MZ)) {
		set_error("mgb_map_batch_gaf: the -S / --write-mz records are written from mg_gchains_t only (mg_map_batch + mgb_write_gaf_batch)");
		rc = MGB_E_UNSUPPORTED;
	} else if (n_reads <= 0) {
		try { gaf_reserve(R, 0); } catch (const MgbError &e) { rc = e.code; }
	} else rc = map_batch_impl(gi, n_reads, qlens, seqs, names, 0, opt, 0, 0, &R);
	if (rc < 0) { // no text is left behind: the caller's reusable buffer is kept, empty; a buffer of the call's own is not made
		*out_len = 0;
		if (out_cap && *out && *out_cap) (*out)[0] = 0;
		else if (!out_cap) *out = 0;
	}
	return rc;
}

// Fragments of several segments (read pairs) in one go: fragment f has n_seg[f] consecutive entries of qlens/seqs/gcs starting at
// seg_off[f] = n_seg[0] + ... + n_seg[f-1]; gcs[seg_off[f]] receives the result of the concatenated fragment and the other
// entries NULL, exactly what worker_for() leaves behind without MG_M_INDEPEND_SEG (gmap.c:46-48).  names[f] is per fragment.
extern "C" int mg_map_batch_frag(const mg_idx_t *gi, int n_frag, const int *n_seg, const int *qlens, const char *const *seqs, const char *const *names,
								 mg_gchains_t **gcs, const mg_mapopt_t *opt)
{
	if (n_frag <= 0) return 0;
	bool single = true;
	int64_t n_tot = 0;
	for (int f = 0; f < n_frag; ++f) { if (n_seg[f] != 1) single = false; n_tot += n_seg[f] > 0? n_seg[f] : 0; }
	if (single) return map_batch_impl(gi, n_frag, qlens, seqs, names, gcs, opt);
	for (int64_t i = 0; i < n_tot; ++i) gcs[i] = 0;
	std::vector<std::string> cat((size_t)n_frag);
	std::vector<int> qsum((size_t)n_frag);
	std::vector<const char*> sq((size_t)n_frag);
	std::vector<int32_t> seg_off((size_t)n_frag + 1), seg_len;
	std::vector<mg_gchains_t*> res((size_t)n_frag, (mg_gchains_t*)0);
	seg_len.reserve((size_t)n_tot);
	int64_t off = 0;
	for (int f = 0; f < n_frag; ++f) {
		seg_off[(size_t)f] = (int32_t)seg_len.size();
		const int ns = n_seg[f] > 0 && n_seg[f] <= 255? n_seg[f] : 0; // more than MG_MAX_SEG segments: no result (map-algo.c:359)
		for (int j = 0; j < ns; ++j) {
			const int l = qlens[off + j] > 0? qlens[off + j] : 0;
			seg_len.push_back(l);
			if (l > 0) cat[(size_t)f].append(seqs[off + j], (size_t)l);
		}
		qsum[(size_t)f] = (int)cat[(size_t)f].size(), sq[(size_t)f] = cat[(size_t)f].data();
		off += n_seg[f] > 0? n_seg[f] : 0;
	}
	seg_off[(size_t)n_frag] = (int32_t)seg_len.size();
	int rc = map_batch_impl(gi, n_frag, qsum.data(), sq.data(), names, res.data(), opt, &seg_off, &seg_len);
	if (rc < 0) return rc;
	off = 0;
	for (int f = 0; f < n_frag; ++f) { if (n_seg[f] > 0) gcs[off] = res[(size_t)f]; off += n_seg[f] > 0? n_seg[f] : 0; }
	return 0;
}

extern "C" void mg_map_frag(const mg_idx_t *gi, int n_segs, const int *qlens, const char **seqs, mg_gchains_t **gcs, mg_tbuf_t *b, const mg_mapopt_t *opt, const char *qname)
{
	(void)b;
	for (int i = 0; i < n_segs; ++i) gcs[i] = 0;
	if (n_segs <= 0) return;
	if (n_segs != 1) { // reference: map-algo.c:356-360,366,457-464: one result for the concatenated fragment, no CIGAR
		if (n_segs > 255) return; // MG_MAX_SEG
		std::string cat;
		std::vector<int32_t> seg_off(2), seg_len((size_t)n_segs);
		for (int i = 0; i < n_segs; ++i) { seg_len[(size_t)i] = qlens[i] > 0? qlens[i] : 0; if (qlens[i] > 0) cat.append(seqs[i], (size_t)qlens[i]); }
		seg_off[0] = 0, seg_off[1] = n_segs;
		if (cat.empty()) return;
		const int qlen_sum = (int)cat.size();
		const char *sq = cat.data(), *nm1 = qname;
		if (map_batch_impl(gi, 1, &qlen_sum, &sq, &nm1, gcs, opt, &seg_off, &seg_len) < 0) abort();
		return;
	}
	const char *nm = qname;
	if (mg_map_batch(gi, 1, qlens, seqs, &nm, gcs, opt) < 0) abort(); // the reference aborts on internal errors too
}

extern "C" mg_gchains_t *mg_map(const mg_idx_t *gi, int qlen, const char *seq, mg_tbuf_t *b, const mg_mapopt_t *opt, const char *qname)
{
	mg_gchains_t *gcs;
	mg_map_frag(gi, 1, &qlen, &seq, &gcs, b, opt, qname);
	return gcs;
}

// ---------------------------------------------------------------------------------------------------------------
// test hook: one gap alignment through the tier-3 path (exact WFA capped at max_iter cells, then the chaining
// heuristic with low-memory checkpoints every `step` scores), reference: miniwfa.c:824-834 mwf_wfa_auto
// ---------------------------------------------------------------------------------------------------------------
struct TestWfaArgs { const char *ts, *qs; int32_t tl, ql, step, cap; int64_t max_iter; uint32_t *cigar; int32_t *out; char *arena; uint64_t arena_bytes; };
MG_HD inline void test_wfa_body(const TestWfaArgs &t, int lane)
{
	Arena A;
	arena_init(A, t.arena, t.arena_bytes);
	WfResult r;
	int rc = wfa_exact(A, t.tl, t.ts, t.ql, t.qs, t.max_iter, &r, lane, t.step);
	if (rc == 0 && r.n_cigar <= t.cap) for (int32_t i = lane; i < r.n_cigar; i += MGB_W) t.cigar[i] = r.cigar[i];
	if (lane == 0) t.out[0] = rc, t.out[1] = rc == 0? r.n_cigar : 0, t.out[2] = rc == 0? r.s : 0;
}
#ifndef MGB_HOSTSIM
__global__ void k_test_wfa(TestWfaArgs t) { test_wfa_body(t, threadIdx.x & 31); }
#endif
static int test_wfa_impl(const char *ts, int tl, const char *qs, int ql, int64_t max_iter, int step, uint32_t *cigar, int cap, int *score)
{
	if (!dev_ok()) { set_error("no CUDA device available: libmgb200 has no CPU path"); return -100; }
	TestWfaArgs t;
	t.tl = tl, t.ql = ql, t.step = step, t.cap = cap, t.max_iter = max_iter, t.arena_bytes = (uint64_t)1 << 30;
	char *d_ts = (char*)dmalloc((size_t)tl + 64), *d_qs = (char*)dmalloc((size_t)ql + 64);
	h2d(d_ts, ts, (size_t)tl), h2d(d_qs, qs, (size_t)ql);
	t.ts = d_ts, t.qs = d_qs;
	t.cigar = (uint32_t*)dmalloc(sizeof(uint32_t) * (size_t)cap);
	t.out = (int32_t*)dmalloc(sizeof(int32_t) * 4);
	t.arena = (char*)dmalloc(t.arena_bytes);
	int32_t out[4] = {0, 0, 0, 0};
	{
#ifdef MGB_HOSTSIM
#if MGB_W > 1
	sim::run_warp(MGB_W, [&](int lane) { test_wfa_body(t, lane); });
#else
	test_wfa_body(t, 0);
#endif
#else
	k_test_wfa<<<1, 32>>>(t);
	CUDA_OK(cudaGetLastError());
	dsync();
#endif
	d2h(out, t.out, sizeof(out));
	}
	if (out[0] == 0 && out[1] <= cap) d2h(cigar, t.cigar, sizeof(uint32_t) * (size_t)out[1]);
	*score = out[2];
	dfree(d_ts), dfree(d_qs), dfree(t.cigar), dfree(t.out), dfree(t.arena);
	return out[0] < 0? out[0] : out[1];
}

extern "C" int mgb_test_wfa(const char *ts, int tl, const char *qs, int ql, int64_t max_iter, int step, uint32_t *cigar, int cap, int *score)
{
	try { return test_wfa_impl(ts, tl, qs, ql, max_iter, step, cigar, cap, score); } catch (const MgbError &e) { return e.code; }
}

#ifdef MGB_HOSTSIM
// TEST INFRASTRUCTURE (simulator builds only): the warp-wide exact radix sort on an array of 16-byte records, in place or with the digit
// walk, with `hot_bytes` of "on-chip" scratch (0: everything in the arena).  tests/test_hostsim32_lanes.py holds it against klib's.
extern "C" int mgb_test_radix128(u128 *a, int64_t n, int walk, int hot_bytes)
{
	std::vector<char> cold((size_t)n * 64 + (1 << 20)), hot((size_t)(hot_bytes > 0? hot_bytes : 16));
	int rc_all = 0;
#if MGB_W > 1
	int rcs[MGB_W];
	sim::run_warp(MGB_W, [&](int lane) {
		Arena A, H;
		arena_init(A, cold.data(), cold.size());
		arena_init(H, hot.data(), hot_bytes > 0? (uint64_t)hot_bytes : 0);
		rcs[lane] = radix_sort_128x_w(hot_bytes > 0? H : A, a, n, lane, &A, walk != 0);
	});
	for (int l = 0; l < MGB_W; ++l) if (rcs[l] != rcs[0]) return -99; else rc_all = rcs[0];
#else
	Arena A, H;
	arena_init(A, cold.data(), cold.size());
	arena_init(H, hot.data(), hot_bytes > 0? (uint64_t)hot_bytes : 0);
	rc_all = radix_sort_128x_w(hot_bytes > 0? H : A, a, n, 0, &A, walk != 0);
#endif
	return rc_all;
}
#endif

extern "C" void mgb_get_stats(const mg_idx_t *gi, mgb_stats_t *st) { *st = t_has_stats? t_last_stats : model_of(gi)->stats; } // the calling thread's last batch
