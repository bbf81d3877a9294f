// cuba_engine.cu -- the engine behind the C ABI of include/cuba_b200.h: device memory, the host LM
// control loop (reference src/cuda_bundle_adjustment.cpp:793-857) and the kernel launches.
//
// No CPU fallback: every compute entry point needs a CUDA device and fails loudly without one.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/cuba_b200.h"
#include "cuba_kernels.cuh"
#include "cuba_pcg2.cuh"
#include "cuba_pcg3.cuh"
#include "cuba_pcg4.cuh"
#include "cuba_pcg5.cuh"
#include "cuba_pcg5t.cuh"
#include "cuba_coarse_dense.cuh"
#include "cuba_peer_reduce.cuh"
#include "cuba_jh4.cuh"
#include "cuba_schur3.cuh"
#include "cuba_structure.h"
#include "cuba_structure_gpu.cuh"

namespace cuba_b200 {

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }

#define CUDA_TRY(expr)                                                                                      \
	do {                                                                                                    \
		cudaError_t _e = (expr);                                                                            \
		if (_e != cudaSuccess) {                                                                            \
			char _b[512];                                                                                   \
			snprintf(_b, sizeof(_b), "%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
			return fail(CUBA_ERR_CUDA, _b);                                                                 \
		}                                                                                                   \
	} while (0)

// launches a 1-D kernel over n items on the engine's stream (used inside Engine<T> member functions)
#define KLAUNCH(kernel, n, ...)                                                             \
	do {                                                                                     \
		if ((n) > 0) {                                                                       \
			kernel<<<sgpu::grid_for(n), sgpu::BLK, 0, stream>>>(__VA_ARGS__);                 \
			launches++;                                                                      \
			CUDA_TRY(cudaGetLastError());                                                    \
		}                                                                                    \
	} while (0)

static thread_local long long g_h2dBytes = 0, g_d2hBytes = 0;   // host<->device traffic of this thread's engines

// Pinned staging arena for the many small host->device uploads of the PCG setup: a cudaMemcpyAsync from pageable
// memory is staged (and effectively synchronous) inside the driver, ~20 us each; from the arena it is a plain DMA.
struct PinnedArena {
	char* p = nullptr; size_t cap = 0, off = 0;
	~PinnedArena() { if (p) cudaFreeHost(p); }
	void reset() { off = 0; }
	// returns nullptr when the arena would have to grow while earlier copies may still read it: the caller falls back
	void* put(const void* src, size_t bytes)
	{
		const size_t o = (off + 255) & ~(size_t)255;
		if (o + bytes > cap) {
			if (off != 0) return nullptr;
			if (p) cudaFreeHost(p);
			cap = std::max<size_t>(2 * (o + bytes), (size_t)1 << 20);
			if (cudaMallocHost((void**)&p, cap) != cudaSuccess) { p = nullptr; cap = 0; return nullptr; }
		}
		memcpy(p + o, src, bytes);
		off = o + bytes;
		return p + o;
	}
};

template <typename U>
struct DBuf {
	U* p = nullptr; size_t n = 0, cap = 0;
	bool view = false;   // a window into another DBuf's allocation (fused collectives): never freed, never grown here
	DBuf() {}
	DBuf(const DBuf&) = delete;
	DBuf& operator=(const DBuf&) = delete;
	~DBuf() { release(); }
	void release() { if (p && !view) cudaFree(p); p = nullptr; n = 0; cap = 0; view = false; }
	void alias(U* q, size_t count) { release(); p = q; n = count; cap = count; view = true; }
	// grow-only: re-initialising an engine with a problem of the same (or smaller) size allocates nothing
	cudaError_t alloc(size_t count)
	{
		if (p && count <= cap && !view) { n = count; return cudaSuccess; }
		release();
		n = count; cap = count ? count : 1;
		return cudaMalloc((void**)&p, sizeof(U) * cap);
	}
	cudaError_t upload(const U* h, size_t count, cudaStream_t s)
	{
		cudaError_t e = alloc(count);
		if (e != cudaSuccess || !count) return e;
		g_h2dBytes += (long long)(sizeof(U) * count);
		return cudaMemcpyAsync(p, h, sizeof(U) * count, cudaMemcpyHostToDevice, s);
	}
	cudaError_t upload(const std::vector<U>& h, cudaStream_t s) { return upload(h.data(), h.size(), s); }
	cudaError_t upload(const std::vector<U>& h, cudaStream_t s, PinnedArena& arena)
	{
		const void* src = h.empty() ? nullptr : arena.put(h.data(), sizeof(U) * h.size());
		return upload(src ? (const U*)src : h.data(), h.size(), s);
	}
	operator U*() const { return p; }
};

// ---- NCCL through dlopen: single-GPU users never need the library ---------------------------------
struct Nccl {
	void* lib = nullptr;
	typedef struct { char internal[128]; } UniqueId;
	int (*GetUniqueId)(UniqueId*) = nullptr;
	int (*CommInitRank)(void**, int, UniqueId, int) = nullptr;
	int (*CommDestroy)(void*) = nullptr;
	int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
	int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
	int (*Broadcast)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
	int (*GroupStart)() = nullptr;
	int (*GroupEnd)() = nullptr;
	const char* (*GetErrorString)(int) = nullptr;
	bool load(std::string& why)
	{
		if (lib) return true;
		const char* names[] = { "libnccl.so.2", "libnccl.so" };
		for (const char* nme : names) { lib = dlopen(nme, RTLD_NOW | RTLD_GLOBAL); if (lib) break; }
		if (!lib) { why = std::string("dlopen libnccl.so.2 failed: ") + dlerror(); return false; }
		GetUniqueId = (int (*)(UniqueId*))dlsym(lib, "ncclGetUniqueId");
		CommInitRank = (int (*)(void**, int, UniqueId, int))dlsym(lib, "ncclCommInitRank");
		CommDestroy = (int (*)(void*))dlsym(lib, "ncclCommDestroy");
		AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(lib, "ncclAllReduce");
		AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(lib, "ncclAllGather");
		Broadcast = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(lib, "ncclBroadcast");
		GroupStart = (int (*)())dlsym(lib, "ncclGroupStart");
		GroupEnd = (int (*)())dlsym(lib, "ncclGroupEnd");
		GetErrorString = (const char* (*)(int))dlsym(lib, "ncclGetErrorString");
		if (!GetUniqueId || !CommInitRank || !CommDestroy || !AllReduce || !AllGather || !Broadcast || !GroupStart || !GroupEnd) { why = "libnccl lacks expected symbols"; return false; }
		return true;
	}
};
static Nccl g_nccl;
enum { NCCL_INT8 = 0, NCCL_FLOAT32 = 7, NCCL_FLOAT64 = 8, NCCL_SUM = 0, NCCL_MAX = 2 };

struct Scalars { double v[8]; unsigned long long maxdiag; PcgStatus pcg; };

// Every C ABI entry point runs on the engine's own device, whatever the calling thread's current device is
// (two engines on two GPUs in one thread; a host that calls torch.cuda.set_device between calls).
struct DevGuard {
	int prev = -1, dev;
	explicit DevGuard(int d) : dev(d) { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; if (prev != dev) cudaSetDevice(dev); }
	~DevGuard() { if (prev >= 0 && prev != dev) cudaSetDevice(prev); }
};

struct EngineBase {
	virtual ~EngineBase() {}
	cuba_config cfg{};
	int rk_type[2] = { 0, 0 };
	double rk_delta[2] = { 0, 0 };
	int rank = 0, world = 1;
	bool structureReuse = true;   // cuba_engine_set_structure_reuse
	long long structureReuses = 0;
	int devOrdinal = 0;      // CUDA device every call of this engine runs on (set once in init)
	void* comm = nullptr;
	bool haveProblem = false;
	long long launches = 0;
	double prof[CUBA_PROF_NUM] = { 0 };

	virtual int set_problem(const cuba_problem* p) = 0;
	virtual int set_state(const double* q, const double* t, const double* Xw) = 0;
	virtual int get_sizes(cuba_sizes* out) const = 0;
	virtual int reset_state() = 0;
	virtual int get_stream(void** s) = 0;
	virtual int flush_l2() = 0;
	virtual int optimize(int niter, cuba_iter_stat* stats, int* nstats) = 0;
	virtual int get_state(double* q, double* t, double* Xw) = 0;
	virtual int get_chi2(double* out) = 0;
	virtual int get_profile(double* sec) = 0;
	virtual int stage_linearize(double* chi) = 0;
	virtual int stage_max_diagonal(double* md) = 0;
	virtual int stage_solve(double lambda, int* iters, int* ok) = 0;
	virtual int stage_update(double lambda, double* chi, double* scale) = 0;
	virtual int stage_commit(int accept) = 0;
	virtual int stage_chi2(double* chi) = 0;
	virtual int dbg_hpl_structure(int32_t* colPtr, int32_t* rowInd, int32_t* e2h) = 0;
	virtual int dbg_hsc_structure(int32_t* rowPtr, int32_t* colInd) = 0;
	virtual int dbg_system(double* Hpp, double* bp, double* Hll, double* bl, double* Hpl) = 0;
	virtual int dbg_schur(double* Hsc, double* bsc, double* invHll) = 0;
	virtual int dbg_delta(double* xp, double* xl) = 0;
	virtual int bench_stage(int stage, int reps, int flush, double lambda, double* ms) = 0;
	virtual int dbg_pcg_timing(long long* out, int maxCtas) = 0;
};

template <typename T>
struct Engine : EngineBase {
	Structure S;
	cudaStream_t stream = nullptr;
	int numSMs = 0;
	int ntiles = 0, nPoseBlocks = 0, nChiBlocks = 0;
	int nChiLin = 0;
	// warp-tile J+H landmark pass (cuba_jh4.cuh); otherwise the tile kernel k_linearize_landmark
	bool jhV4 = true;
	int ntW = 0, jh4Grid = 0, jh4HasBig = 0;
	const void* jh4AttrSet = nullptr;
	int* jh4Host = nullptr;      // pinned: {number of warp tiles, any cut landmark}
	bool jh4Pending = false;
	DBuf<int> w_levels, w_start, w_pieces, w_base, w_tilePose, w_tilePieces, w_pieceCount, w_flag;
	DBuf<jh4::WTile> w_tile;
	DBuf<jh4::Rec> w_rec;
	DBuf<double> w_bigPartial;
	int cur = 0;            // current state buffer
	bool trialValid = false;
	// state
	DBuf<T> pose[2], Xw[2], cam, pose0, Xw0;
	// edge streams
	DBuf<T> e_mx, e_my, e_mz, e_om, p_mx, p_my, p_mz, p_om;
	DBuf<int> tilePtr;   // run pointers seen by the landmark tiles (see k_tile_ptr)
	DBuf<int> e_ip, e_il, e_hpl, e_user, lmPtr, tileLm, hplLm, posePtr, p_il;
	// system
	DBuf<T> Hpp, bp, Hll, bl, Hpl, invHll, fVal, bsc, xp, xl;
	DBuf<T> uVal;            // landmark-sharded runs: upper Hsc blocks | bsc, the buffer of the per-trial all-reduce
	DBuf<float> HplF;        // mixed precision (cfg.use_fp32 == 2, fp64 engine): the Hpl blocks in fp32, 20 floats per block
	bool mixed = false;
	bool upperReduce = false;   // k_schur3 writes the upper blocks into uVal; one all-reduce of uVal | bsc, then k_expand_upper
	DBuf<int> prodPtr, prodI, prodJ, prodL, blkRow, blkCol, u2f, u2fT, fRowPtr, fColInd;
	// pcg v2 (cuba_pcg2.cuh)
	DBuf<T> fHat, Linv, vR0, vR1, vS0, vS1, vW0, vW1, vP, vY;
	DBuf<int> fLocal, ctaRow, needPtr, needCol;
	DBuf<double> pcg2Partial;
	DBuf<GridBar> gridBar;
	DBuf<long long> pcgTiming;
	DBuf<unsigned long long> llFlags;   // k_pcg3: [wFlag 2*6numP*2 | pFlag 2*2G*2 | abort word]
	int pcg2Grid = 0, pcg2Cap = 0, pcg2NeedMax = 0, pcg2MaxRows = 0;
	// two-level PCG (cuba_pcg4.cuh)
	DBuf<T> cZx, cZhat;
	DBuf<float> cAcInv;
	DBuf<double> cAcP, cPart, cU, cLp, cLd, cWp;
	DBuf<int> cAggRow, cNaPtr, cNaList, cNeedAgg, cInfo, cRowOf, cCbPtr, cCbList;
	int pcg4A = 0, pcg4Gs = 1, pcg4MaxNeedAgg = 0, pcg4Cap = 0, pcg4SliceInSmem = 0, pcg4ZhInSmem = 0;
	size_t pcg4Smem = 0, pcg4InvSmem = 0;
	bool pcg4Ok = false, tlActive = false, pcg4Cluster = false;
	PinnedArena arena;
	bool coarseValid = false;       // cAcInv holds the inverse coarse matrix of an earlier solve of this problem
	int coarseAge = 0;              // two-level solves since the coarse matrix was last rebuilt
	double coarseLambda = 0, curLambda = 0;   // damping of that rebuild / of the solve being launched
	bool pcg3Ok = false;
	size_t pcg2Smem = 0;
	// reductions
	DBuf<double> chiPartial, scalePartialL, scalePartialP, chiSq;
	DBuf<Scalars> dScal;
	Scalars* hScal = nullptr;   // pinned
	DBuf<double> flushBuf;
	std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> profEvents;
	std::vector<cudaEvent_t> eventPool;

	~Engine() override
	{
		DevGuard guard(devOrdinal);
		if (stream) cudaStreamSynchronize(stream);
		p5CloseMappings(); uCloseMappings();
		for (auto& pe : profEvents) { cudaEventDestroy(pe.second.first); cudaEventDestroy(pe.second.second); }
		for (auto ev : eventPool) cudaEventDestroy(ev);
		if (hScal) cudaFreeHost(hScal);
		if (hMeta) cudaFreeHost(hMeta);
		if (jh4Host) cudaFreeHost(jh4Host);
		if (stream) cudaStreamDestroy(stream);
		if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(comm);
	}

	int init()
	{
		int ndev = 0;
		cudaError_t e = cudaGetDeviceCount(&ndev);
		if (e != cudaSuccess || ndev <= 0)
			return fail(CUBA_ERR_CUDA, std::string("no CUDA device available (") + cudaGetErrorString(e) + "); this library has no CPU fallback");
		if (cfg.device >= 0) CUDA_TRY(cudaSetDevice(cfg.device));
		int dev = 0;
		CUDA_TRY(cudaGetDevice(&dev));
		devOrdinal = dev;
		CUDA_TRY(cudaDeviceGetAttribute(&numSMs, cudaDevAttrMultiProcessorCount, dev));
		CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
		CUDA_TRY(cudaMallocHost((void**)&hScal, sizeof(Scalars)));
		memset(hScal, 0, sizeof(Scalars));
		CUDA_TRY(dScal.alloc(1));
		CUDA_TRY(cudaMemsetAsync(dScal.p, 0, sizeof(Scalars), stream));
		return CUBA_OK;
	}

	// ---- profile helpers: CUDA events on the launching stream, resolved lazily ----------------------
	cudaEvent_t newEvent()
	{
		cudaEvent_t ev;
		if (!eventPool.empty()) { ev = eventPool.back(); eventPool.pop_back(); return ev; }
		cudaEventCreate(&ev);
		return ev;
	}
	struct ProfScope {
		Engine* e; int item; cudaEvent_t a, b;
		ProfScope(Engine* e_, int item_) : e(e_), item(item_) { a = e->newEvent(); b = e->newEvent(); cudaEventRecord(a, e->stream); }
		~ProfScope() { cudaEventRecord(b, e->stream); e->profEvents.push_back({ item, { a, b } }); }
	};
	void resolveProfile()
	{
		cudaStreamSynchronize(stream);
		for (auto& pe : profEvents) {
			float ms = 0;
			if (cudaEventElapsedTime(&ms, pe.second.first, pe.second.second) == cudaSuccess) prof[pe.first] += 1e-3 * ms;
			eventPool.push_back(pe.second.first); eventPool.push_back(pe.second.second);
		}
		profEvents.clear();
	}

	RobustParams rkParams() const
	{
		RobustParams r;
		for (int i = 0; i < 2; i++) { r.type[i] = rk_type[i]; r.delta[i] = rk_delta[i]; }
		return r;
	}

	// ---- collectives (landmark-sharded runs) ----------------------------------------------------------
	int allreduce(void* buf, size_t count, bool isT)
	{
		if (world <= 1 || !comm) return CUBA_OK;      // (!comm: CUBA_DRY_SHARD diagnosis, one shard of a sharded run timed on one GPU)
		const int dt = isT ? (sizeof(T) == 8 ? NCCL_FLOAT64 : NCCL_FLOAT32) : NCCL_FLOAT64;
		const int rc = g_nccl.AllReduce(buf, buf, count, dt, NCCL_SUM, comm, stream);
		if (rc != 0) return fail(CUBA_ERR_COMM, std::string("ncclAllReduce failed: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"));
		return CUBA_OK;
	}

	// ---- problem upload -------------------------------------------------------------------------------
	// ---- problem upload ----------------------------------------------------------------------------
	// The caller's flat fp64 arrays go to the device as they are; one kernel packs them into the padded records
	// (pose [8] = q,t,pad; cam [8]; Xw [4]) of the initial state and of both working buffers.
	DBuf<double> rawQ, rawT, rawC, rawX;
	int upload_state(const double* q, const double* t, const double* c, const double* X)
	{
		const int Pall = S.Pall, Lall = S.Lall;
		CUDA_TRY(rawQ.upload(q, 4 * (size_t)Pall, stream)); CUDA_TRY(rawT.upload(t, 3 * (size_t)Pall, stream));
		CUDA_TRY(rawX.upload(X, 3 * (size_t)Lall, stream));
		if (c) CUDA_TRY(rawC.upload(c, 5 * (size_t)Pall, stream));
		CUDA_TRY(pose0.alloc(8 * (size_t)Pall)); CUDA_TRY(Xw0.alloc(4 * (size_t)Lall));
		for (int b = 0; b < 2; b++) { CUDA_TRY(pose[b].alloc(8 * (size_t)Pall)); CUDA_TRY(Xw[b].alloc(4 * (size_t)Lall)); }
		if (c) CUDA_TRY(cam.alloc(8 * (size_t)Pall));
		const int n = std::max(Pall, Lall);
		if (n > 0) {
			k_pack_state<T><<<(n + 255) / 256, 256, 0, stream>>>(rawQ.p, rawT.p, c ? rawC.p : nullptr, rawX.p, Pall, Lall,
				pose0.p, pose[0].p, pose[1].p, c ? cam.p : nullptr, Xw0.p, Xw[0].p, Xw[1].p);
			launches++;
			CUDA_TRY(cudaGetLastError());
		}
		// no synchronisation here: set_problem / set_state synchronise before they return to the caller
		return CUBA_OK;
	}

	// set_problem wall-clock marks (CUBA_SETUP_TIMING=1 prints them)
	std::vector<std::pair<const char*, std::chrono::steady_clock::time_point>> marks;
	void tmark(const char* name) { if (markOn) marks.push_back({ name, std::chrono::steady_clock::now() }); }
	bool markOn = false;
	int set_problem(const cuba_problem* p) override
	{
		markOn = getenv("CUBA_SETUP_TIMING") != nullptr; marks.clear(); tmark("start");
		if (!p) return fail(CUBA_ERR_INVALID, "set_problem: null problem");
		if (p->Pall < 0 || p->Lall < 0 || p->numP < 0 || p->numL < 0 || p->numP > p->Pall || p->numL > p->Lall || p->E2 < 0 || p->E3 < 0)
			return fail(CUBA_ERR_INVALID, "set_problem: invalid sizes");
		if ((p->Pall > 0 && (!p->q || !p->t || !p->cam)) || (p->Lall > 0 && !p->Xw) || (p->E2 > 0 && (!p->idx2 || !p->meas2 || !p->omega2)) ||
			(p->E3 > 0 && (!p->idx3 || !p->meas3 || !p->omega3)))
			return fail(CUBA_ERR_INVALID, "set_problem: null array with a non-zero count");
		const auto t0 = std::chrono::steady_clock::now();
		// Same topology as the problem this engine already holds (sizes, fixed/free split and every (iP, iL) pair identical): only the
		// numbers changed -- the estimate after a previous optimize(), new measurements -- so every index structure, tile list,
		// product list and PCG partition on the device stays valid.  Upload the values and re-run the three kernels that scatter them.
		if (structureReuse && reusable && haveProblem && cfg.reserved[1] != 1 && same_topology(p)) {
			int rc = refresh_values(p); if (rc) return rc;
			structureReuses++;
			prof[CUBA_PROF_BUILD_STRUCTURE] += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
			return CUBA_OK;
		}
		haveProblem = false;
		reusable = false;
		hostStructureValid = false;
		shardBoundValid = false;
		// J+H landmark pass: k_linearize_landmark4 in fp64; k_linearize_landmark in fp32 and, for the agreement test, with cfg.reserved[2] == 4
		jhV4 = cfg.reserved[2] == 0 && sizeof(T) == 8;
		int rc = (cfg.reserved[1] == 1) ? build_on_host(p) : build_on_gpu(p);
		if (rc) return rc;
		tmark("structure built");
		rc = upload_state(p->q, p->t, p->cam, p->Xw); if (rc) return rc;
		tmark("state uploaded");
		rc = alloc_system(); if (rc) return rc;
		CUDA_TRY(cudaStreamSynchronize(stream));
		tmark("alloc_system done");
		if (markOn) {
			for (size_t i = 1; i < marks.size(); i++)
				fprintf(stderr, "setup %-28s %8.3f ms\n", marks[i].first, 1e3 * std::chrono::duration<double>(marks[i].second - marks[i - 1].second).count());
			fprintf(stderr, "setup total %8.3f ms\n", 1e3 * std::chrono::duration<double>(marks.back().second - marks.front().second).count());
		}
		cur = 0; trialValid = false;
		tlActive = false; coarseValid = false; coarseAge = 0; p5CoarseValid = false; p5CoarseAge = 0;
		resolveProfile();   // drop the events of earlier problems
		for (int i = 0; i < CUBA_PROF_NUM; i++) prof[i] = 0;
		const auto t1 = std::chrono::steady_clock::now();
		prof[CUBA_PROF_BUILD_STRUCTURE] += std::chrono::duration<double>(t1 - t0).count();
		haveProblem = true;
		if (cfg.reserved[1] != 1 && structureReuse) {
			lastIdx2.assign(p->idx2, p->idx2 + 2 * (size_t)p->E2); lastIdx3.assign(p->idx3, p->idx3 + 2 * (size_t)p->E3);
			const int sz[6] = { p->Pall, p->numP, p->Lall, p->numL, p->E2, p->E3 };
			memcpy(lastSizes, sz, sizeof(sz));
			reusable = true;
		}
		return CUBA_OK;
	}

	bool same_topology(const cuba_problem* p) const
	{
		const int sz[6] = { p->Pall, p->numP, p->Lall, p->numL, p->E2, p->E3 };
		if (memcmp(sz, lastSizes, sizeof(sz)) != 0) return false;
		if (p->E2 > 0 && memcmp(p->idx2, lastIdx2.data(), sizeof(int32_t) * 2 * (size_t)p->E2) != 0) return false;
		if (p->E3 > 0 && memcmp(p->idx3, lastIdx3.data(), sizeof(int32_t) * 2 * (size_t)p->E3) != 0) return false;
		return true;
	}

	// set_problem on an unchanged topology: measurements, information values and the estimate go up, the edge streams are re-scattered
	int refresh_values(const cuba_problem* p)
	{
		using namespace sgpu;
		const int E2 = p->E2, E3 = p->E3, eL = S.eLocal;
		CUDA_TRY(g_meas2.upload(p->meas2, 2 * (size_t)E2, stream)); CUDA_TRY(g_meas3.upload(p->meas3, 3 * (size_t)E3, stream));
		CUDA_TRY(g_om2.upload(p->omega2, (size_t)E2, stream)); CUDA_TRY(g_om3.upload(p->omega3, (size_t)E3, stream));
		int rc = upload_state(p->q, p->t, p->cam, p->Xw); if (rc) return rc;
		KLAUNCH(k_edge_stream<T>, eL, g_keyS.p, g_valS.p, g_ff.p, g_hplG.p, savedKBeg, eL, S.hplBase, E2, g_meas2.p, g_om2.p, g_meas3.p, g_om3.p,
			e_user.p, e_ip.p, e_il.p, e_hpl.p, e_mx.p, e_my.p, e_mz.p, e_om.p);
		KLAUNCH(k_pose_stream<T>, eL, g_psrc.p, posePtr.p, S.numP, eL, e_ip.p, e_il.p, e_mx.p, e_my.p, e_mz.p, e_om.p, p_il.p, p_mx.p, p_my.p, p_mz.p, p_om.p);
		if constexpr (sizeof(T) == 8) {
			if (jhV4 && ntW > 0) {
				const int lb = S.lmBeg, N = S.lmEnd - S.lmBeg;
				KLAUNCH(jh4::k_emit, (long long)N * 32, w_start.p, w_pieces.p, w_base.p, N, lmPtr.p, lb, w_levels.p,
					e_mx.p, e_my.p, e_mz.p, e_om.p, e_ip.p, e_il.p, e_hpl.p, w_tile.p, w_rec.p, w_tilePose.p, w_tilePieces.p);
			}
		}
		CUDA_TRY(cudaStreamSynchronize(stream));      // the caller's buffers are free again
		cur = 0; trialValid = false;
		tlActive = false; coarseValid = false; coarseAge = 0; p5CoarseValid = false; p5CoarseAge = 0;
		resolveProfile();
		for (int i = 0; i < CUBA_PROF_NUM; i++) prof[i] = 0;
		return CUBA_OK;
	}

	// host structure builder (cuba_structure.cpp): reference path for the GPU builder, cfg.reserved[1] == 1
	int build_on_host(const cuba_problem* p)
	{
		const char* err = "";
		if (!build_structure(p->Pall, p->numP, p->Lall, p->numL, p->E2, p->idx2, p->E3, p->idx3, rank, world, LM_TILE, S, &err))
			return fail(CUBA_ERR_INVALID, err);
		hostStructureValid = true;
		const int eL = S.eLocal;
		std::vector<T> mx(eL), my(eL), mz(eL), om(eL);
		for (int e = 0; e < eL; e++) {
			const int u = S.order[e];
			if (u < S.E2) { mx[e] = (T)p->meas2[2 * (size_t)u]; my[e] = (T)p->meas2[2 * (size_t)u + 1]; mz[e] = T(0); om[e] = (T)p->omega2[u]; }
			else { const size_t k = (size_t)(u - S.E2); mx[e] = (T)p->meas3[3 * k]; my[e] = (T)p->meas3[3 * k + 1]; mz[e] = (T)p->meas3[3 * k + 2]; om[e] = (T)p->omega3[k]; }
		}
		CUDA_TRY(e_mx.upload(mx, stream)); CUDA_TRY(e_my.upload(my, stream)); CUDA_TRY(e_mz.upload(mz, stream)); CUDA_TRY(e_om.upload(om, stream));
		CUDA_TRY(e_ip.upload(S.e_ip, stream)); CUDA_TRY(e_il.upload(S.e_il, stream)); CUDA_TRY(e_hpl.upload(S.e_hpl, stream));
		CUDA_TRY(e_user.upload(S.order, stream));
		CUDA_TRY(lmPtr.upload(S.lmPtr, stream)); CUDA_TRY(tilePtr.upload(S.lmPtr, stream));
		CUDA_TRY(tileLm.upload(S.tileLm, stream)); CUDA_TRY(hplLm.upload(S.hplLm, stream));
		const size_t nPe = S.p_src.size();
		std::vector<T> qx(nPe), qy(nPe), qz(nPe), qo(nPe);
		for (size_t k = 0; k < nPe; k++) { const int e = S.p_src[k]; qx[k] = mx[e]; qy[k] = my[e]; qz[k] = mz[e]; qo[k] = om[e]; }
		CUDA_TRY(p_mx.upload(qx, stream)); CUDA_TRY(p_my.upload(qy, stream)); CUDA_TRY(p_mz.upload(qz, stream)); CUDA_TRY(p_om.upload(qo, stream));
		CUDA_TRY(p_il.upload(S.p_il, stream)); CUDA_TRY(posePtr.upload(S.posePtr, stream));
		CUDA_TRY(prodPtr.upload(S.prodPtr, stream)); CUDA_TRY(prodI.upload(S.prodI, stream)); CUDA_TRY(prodJ.upload(S.prodJ, stream));
		CUDA_TRY(blkRow.upload(S.blkRow, stream)); CUDA_TRY(blkCol.upload(S.blkCol, stream));
		CUDA_TRY(u2f.upload(S.u2f, stream)); CUDA_TRY(u2fT.upload(S.u2fT, stream));
		CUDA_TRY(fRowPtr.upload(S.fRowPtr, stream)); CUDA_TRY(fColInd.upload(S.fColInd, stream));
		CUDA_TRY(cudaStreamSynchronize(stream));   // host staging vectors die here
		ntiles = (int)S.tileLm.size() - 1;
		return CUBA_OK;
	}

	// ---- device structure builder (cuba_structure_gpu.cuh) ------------------------------------------------
	DBuf<int> g_idx2, g_idx3, g_val, g_valS, g_ff, g_hplG, g_lmPtrG, g_hplRowInd, g_hplLmG, g_edge2Hpl, g_hplColPtr, g_hscRowPtr;
	DBuf<int> g_pval, g_pvalS, g_pi, g_pj, g_head, g_blkId, g_cnt, g_off, g_fval, g_fvalS, g_pkeyVal, g_psrc;
	DBuf<double> g_meas2, g_meas3, g_om2, g_om3;
	DBuf<unsigned long long> g_key, g_keyS, g_pkey, g_pkeyS, g_fkey, g_fkeyS;
	DBuf<unsigned int> g_k32, g_k32S;
	DBuf<char> cubTmp;
	DBuf<sgpu::Meta> g_meta;
	sgpu::Meta* hMeta = nullptr;
	bool hostStructureValid = false;
	// structure reuse across set_problem calls (repeated local BA on an unchanged graph): the last problem's index lists
	std::vector<int32_t> lastIdx2, lastIdx3;
	int lastSizes[6] = { -1, -1, -1, -1, -1, -1 };
	int savedKBeg = 0;
	bool reusable = false;      // the device structures of the last problem are complete and were built on the device
	int shardBound[9] = { 0 };    // first landmark of every rank's shard
	bool shardBoundValid = false;

	template <typename K>
	int sortPairs(K* kin, K* kout, int* vin, int* vout, int n, int endBit)
	{
		if (n <= 0) return CUBA_OK;
		size_t bytes = 0;
		CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, bytes, kin, kout, vin, vout, n, 0, endBit, stream));
		CUDA_TRY(cubTmp.alloc(bytes));
		CUDA_TRY(cub::DeviceRadixSort::SortPairs(cubTmp.p, bytes, kin, kout, vin, vout, n, 0, endBit, stream));
		launches += 4;
		return CUBA_OK;
	}
	int exclusiveSum(const int* in, int* out, int n)
	{
		if (n <= 0) return CUBA_OK;
		size_t bytes = 0;
		CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, n, stream));
		CUDA_TRY(cubTmp.alloc(bytes));
		CUDA_TRY(cub::DeviceScan::ExclusiveSum(cubTmp.p, bytes, in, out, n, stream));
		launches += 2;
		return CUBA_OK;
	}
	int fetchMeta()
	{
		if (!hMeta) CUDA_TRY(cudaMallocHost((void**)&hMeta, sizeof(sgpu::Meta)));
		CUDA_TRY(cudaMemcpyAsync(hMeta, g_meta.p, sizeof(sgpu::Meta), cudaMemcpyDeviceToHost, stream));
		CUDA_TRY(cudaStreamSynchronize(stream));
		if (hMeta->error == 1) return fail(CUBA_ERR_INVALID, "build_structure: edge index out of range");
		if (hMeta->error == 2) return fail(CUBA_ERR_INVALID, "build_structure: edge with both ends fixed");
		if (hMeta->error == 3) return fail(CUBA_ERR_INVALID, "build_structure: free landmark without edges (the reference's initialize() drops such vertices)");
		return CUBA_OK;
	}

	int build_on_gpu(const cuba_problem* p)
	{
		using namespace sgpu;
		S = Structure();
		const int Pall = p->Pall, numP = p->numP, Lall = p->Lall, numL = p->numL, E2 = p->E2, E3 = p->E3, E = E2 + E3;
		S.Pall = Pall; S.numP = numP; S.Lall = Lall; S.numL = numL; S.E2 = E2; S.E3 = E3; S.E = E;
		// raw problem -> device (the only bulk H2D traffic of set_problem besides the state)
		CUDA_TRY(g_idx2.upload(p->idx2, 2 * (size_t)E2, stream)); CUDA_TRY(g_idx3.upload(p->idx3, 2 * (size_t)E3, stream));
		CUDA_TRY(g_meas2.upload(p->meas2, 2 * (size_t)E2, stream)); CUDA_TRY(g_meas3.upload(p->meas3, 3 * (size_t)E3, stream));
		CUDA_TRY(g_om2.upload(p->omega2, (size_t)E2, stream)); CUDA_TRY(g_om3.upload(p->omega3, (size_t)E3, stream));
		CUDA_TRY(g_meta.alloc(1));
		CUDA_TRY(cudaMemsetAsync(g_meta.p, 0, sizeof(Meta), stream));
		// 1. canonical (iL, iP, edge id) order
		CUDA_TRY(g_key.alloc(E)); CUDA_TRY(g_keyS.alloc(E)); CUDA_TRY(g_val.alloc(E)); CUDA_TRY(g_valS.alloc(E));
		KLAUNCH(k_make_keys, E, E2, g_idx2.p, E3, g_idx3.p, Pall, numP, Lall, numL, g_key.p, g_val.p, g_meta.p);
		int rc = sortPairs(g_key.p, g_keyS.p, g_val.p, g_valS.p, E, 32 + bits_for((unsigned long long)std::max(Lall, 1))); if (rc) return rc;
		CUDA_TRY(g_lmPtrG.alloc((size_t)Lall + 1));
		KLAUNCH(k_ptr_from_high, Lall + 1, g_keyS.p, E, Lall, g_lmPtrG.p);
		KLAUNCH(k_check_nonempty, numL, g_lmPtrG.p, numL, g_meta.p);
		// 2. Hpl blocks = free-free edges in canonical order
		CUDA_TRY(g_ff.alloc(E)); CUDA_TRY(g_hplG.alloc(E));
		KLAUNCH(k_flag_freefree, E, g_keyS.p, E, numP, numL, g_ff.p);
		rc = exclusiveSum(g_ff.p, g_hplG.p, E); if (rc) return rc;
		k_shard_meta<<<1, 32, 0, stream>>>(g_lmPtrG.p, Lall, E, rank, world, g_ff.p, g_hplG.p, g_meta.p);
		launches++;
		CUDA_TRY(cudaGetLastError());
		tmark("queued to sync 1");
		rc = fetchMeta(); if (rc) return rc;                                   // sync point 1
		tmark("sync 1");
		S.nhpl = hMeta->nhpl; S.lmBeg = hMeta->lmBeg; S.lmEnd = hMeta->lmEnd; S.eLocal = hMeta->kEnd - hMeta->kBeg;
		S.hplBase = hMeta->hplBase; S.nhplLocal = hMeta->hplEnd - hMeta->hplBase;
		for (int r = 0; r < 9; r++) shardBound[r] = hMeta->bounds[r];
		shardBoundValid = true;
		const int kBeg = hMeta->kBeg, kEnd = hMeta->kEnd, eL = S.eLocal, nhpl = S.nhpl;
		savedKBeg = kBeg;
		CUDA_TRY(g_hplRowInd.alloc(nhpl)); CUDA_TRY(g_hplLmG.alloc(nhpl)); CUDA_TRY(g_edge2Hpl.alloc(E)); CUDA_TRY(g_hplColPtr.alloc((size_t)numL + 1));
		KLAUNCH(k_hpl_global, E, g_keyS.p, g_valS.p, g_ff.p, g_hplG.p, E, g_hplRowInd.p, g_hplLmG.p, g_edge2Hpl.p);
		KLAUNCH(k_hpl_colptr, numL + 1, g_lmPtrG.p, g_hplG.p, E, numL, nhpl, g_hplColPtr.p);
		// 3. landmark-major stream of the shard, tiles
		CUDA_TRY(e_user.alloc(eL)); CUDA_TRY(e_ip.alloc(eL)); CUDA_TRY(e_il.alloc(eL)); CUDA_TRY(e_hpl.alloc(eL));
		CUDA_TRY(e_mx.alloc(eL)); CUDA_TRY(e_my.alloc(eL)); CUDA_TRY(e_mz.alloc(eL)); CUDA_TRY(e_om.alloc(eL));
		KLAUNCH(k_edge_stream<T>, eL, g_keyS.p, g_valS.p, g_ff.p, g_hplG.p, kBeg, eL, S.hplBase, E2, g_meas2.p, g_om2.p, g_meas3.p, g_om3.p,
			e_user.p, e_ip.p, e_il.p, e_hpl.p, e_mx.p, e_my.p, e_mz.p, e_om.p);
		CUDA_TRY(lmPtr.alloc((size_t)Lall + 1));
		KLAUNCH(k_local_lmptr, Lall + 1, g_lmPtrG.p, Lall, kBeg, kEnd, lmPtr.p);
		CUDA_TRY(hplLm.alloc(S.nhplLocal));
		if (S.nhplLocal > 0) CUDA_TRY(cudaMemcpyAsync(hplLm.p, g_hplLmG.p + S.hplBase, sizeof(int) * (size_t)S.nhplLocal, cudaMemcpyDeviceToDevice, stream));
		CUDA_TRY(tilePtr.alloc((size_t)numL + 2));
		KLAUNCH(k_tile_ptr, numL + 2, lmPtr.p, numL, eL, tilePtr.p);
		const int tb = std::min(S.lmBeg, numL), te = std::min(S.lmEnd, numL) + (S.lmEnd > numL ? 1 : 0);
		const int nt = (eL + LM_WINDOW - 1) / LM_WINDOW;
		CUDA_TRY(tileLm.alloc((size_t)nt + 1));
		KLAUNCH(k_tiles, nt + 1, tilePtr.p, tb, te, LM_WINDOW, nt, tileLm.p);
		ntiles = nt;
		// 4. pose-major stream (free poses only)
		CUDA_TRY(g_k32.alloc(eL)); CUDA_TRY(g_k32S.alloc(eL)); CUDA_TRY(g_pval.alloc(eL)); CUDA_TRY(g_psrc.alloc(eL));
		KLAUNCH(k_pose_keys, eL, e_ip.p, eL, numP, g_k32.p, g_pval.p);
		rc = sortPairs(g_k32.p, g_k32S.p, g_pval.p, g_psrc.p, eL, bits_for((unsigned long long)numP)); if (rc) return rc;
		CUDA_TRY(posePtr.alloc((size_t)numP + 1));
		KLAUNCH(k_ptr_from_u32, numP + 1, g_k32S.p, eL, numP, posePtr.p);
		CUDA_TRY(p_il.alloc(eL)); CUDA_TRY(p_mx.alloc(eL)); CUDA_TRY(p_my.alloc(eL)); CUDA_TRY(p_mz.alloc(eL)); CUDA_TRY(p_om.alloc(eL));
		KLAUNCH(k_pose_stream<T>, eL, g_psrc.p, posePtr.p, numP, eL, e_ip.p, e_il.p, e_mx.p, e_my.p, e_mz.p, e_om.p, p_il.p, p_mx.p, p_my.p, p_mz.p, p_om.p);
		// 5. block products keyed by destination block, + one dummy per diagonal
		CUDA_TRY(g_cnt.alloc((size_t)nhpl + 1)); CUDA_TRY(g_off.alloc((size_t)nhpl + 1));
		CUDA_TRY(cudaMemsetAsync(g_cnt.p, 0, sizeof(int) * ((size_t)nhpl + 1), stream));
		KLAUNCH(k_prod_count, nhpl, g_hplLmG.p, g_hplColPtr.p, nhpl, g_cnt.p);
		rc = exclusiveSum(g_cnt.p, g_off.p, nhpl + 1); if (rc) return rc;
		long long nmul = 0;
		{
			int last = 0;
			CUDA_TRY(cudaMemcpyAsync(&last, g_off.p + nhpl, sizeof(int), cudaMemcpyDeviceToHost, stream));
			tmark("queued to sync 2");
			CUDA_TRY(cudaStreamSynchronize(stream));                              // sync point 2
			tmark("sync 2");
			nmul = last;
		}
		S.nmul = nmul;
		const long long N = nmul + numP;
		if (N > 0x7fffffffLL) return fail(CUBA_ERR_INVALID, "build_structure: more than 2^31 block products");
		S.nmulLocal = N;
		CUDA_TRY(g_pkey.alloc((size_t)N)); CUDA_TRY(g_pkeyS.alloc((size_t)N)); CUDA_TRY(g_pkeyVal.alloc((size_t)N)); CUDA_TRY(g_pvalS.alloc((size_t)N));
		CUDA_TRY(g_pi.alloc((size_t)N)); CUDA_TRY(g_pj.alloc((size_t)N));
		KLAUNCH(k_prod_emit, nhpl, g_hplLmG.p, g_hplColPtr.p, g_hplRowInd.p, g_off.p, nhpl, S.lmBeg, S.lmEnd, S.hplBase, g_pkey.p, g_pkeyVal.p, g_pi.p, g_pj.p);
		KLAUNCH(k_prod_diag, numP, numP, nmul, g_pkey.p, g_pkeyVal.p, g_pi.p, g_pj.p);
		rc = sortPairs(g_pkey.p, g_pkeyS.p, g_pkeyVal.p, g_pvalS.p, (int)N, 32 + bits_for((unsigned long long)std::max(numP, 1))); if (rc) return rc;
		CUDA_TRY(g_head.alloc((size_t)N + 1)); CUDA_TRY(g_blkId.alloc((size_t)N + 1));
		KLAUNCH(k_heads, N, g_pkeyS.p, (int)N, g_head.p);
		rc = exclusiveSum(g_head.p, g_blkId.p, (int)N); if (rc) return rc;
		k_nblk<<<1, 32, 0, stream>>>(g_head.p, g_blkId.p, (int)N, g_meta.p);
		launches++;
		tmark("queued to sync 3");
		rc = fetchMeta(); if (rc) return rc;                                   // sync point 3
		tmark("sync 3");
		const int nblk = hMeta->nblk;
		S.nblk = nblk;
		CUDA_TRY(blkRow.alloc(nblk)); CUDA_TRY(blkCol.alloc(nblk)); CUDA_TRY(prodPtr.alloc((size_t)nblk + 1));
		CUDA_TRY(prodI.alloc((size_t)N)); CUDA_TRY(prodJ.alloc((size_t)N));
		KLAUNCH(k_blocks, N + 1, g_pkeyS.p, g_pvalS.p, g_head.p, g_blkId.p, g_pi.p, g_pj.p, (int)N, blkRow.p, blkCol.p, prodPtr.p, prodI.p, prodJ.p);
		CUDA_TRY(g_hscRowPtr.alloc((size_t)numP + 1));
		KLAUNCH(k_rowptr_from_rows, numP + 1, blkRow.p, nblk, numP, g_hscRowPtr.p);
		int* dLocalCount = nullptr;
		if (world > 1) {
			// the sorted list holds every rank's products (the block numbering must be global); a destination's warp would walk all of
			// them and skip the foreign ones -- the Schur kernel then does not speed up with the rank count (measured: 1.34 ms for a
			// 1/8 shard of the 10 M-edge graph against 3.7 ms for the whole).  Keep the local products and the diagonal placeholders only.
			CUDA_TRY(g_head.alloc((size_t)N + 1)); CUDA_TRY(g_blkId.alloc((size_t)N + 1));
			KLAUNCH(k_local_flag, N + 1, prodI.p, prodJ.p, (int)N, g_head.p);
			rc = exclusiveSum(g_head.p, g_blkId.p, (int)N + 1); if (rc) return rc;
			KLAUNCH(k_compact_products, N, prodI.p, prodJ.p, g_head.p, g_blkId.p, (int)N, g_pi.p, g_pj.p);
			KLAUNCH(k_remap_ptr, nblk + 1, g_blkId.p, nblk, prodPtr.p);
			CUDA_TRY(cudaMemcpyAsync(prodI.p, g_pi.p, sizeof(int) * (size_t)N, cudaMemcpyDeviceToDevice, stream));
			CUDA_TRY(cudaMemcpyAsync(prodJ.p, g_pj.p, sizeof(int) * (size_t)N, cudaMemcpyDeviceToDevice, stream));
			dLocalCount = g_blkId.p + N;
		}
		// 6. symmetric-full BSR for the PCG
		const int nfull = 2 * nblk - numP;
		S.nfull = nfull;
		CUDA_TRY(g_fkey.alloc(2 * (size_t)nblk)); CUDA_TRY(g_fkeyS.alloc(2 * (size_t)nblk)); CUDA_TRY(g_fval.alloc(2 * (size_t)nblk)); CUDA_TRY(g_fvalS.alloc(2 * (size_t)nblk));
		KLAUNCH(k_full_entries, nblk, blkRow.p, blkCol.p, nblk, numP, g_fkey.p, g_fval.p);
		rc = sortPairs(g_fkey.p, g_fkeyS.p, g_fval.p, g_fvalS.p, 2 * nblk, 32 + bits_for((unsigned long long)std::max(numP, 1))); if (rc) return rc;
		CUDA_TRY(fColInd.alloc(nfull)); CUDA_TRY(u2f.alloc(nblk)); CUDA_TRY(u2fT.alloc(nblk)); CUDA_TRY(fRowPtr.alloc((size_t)numP + 1));
		KLAUNCH(k_full_finish, nfull, g_fkeyS.p, g_fvalS.p, nfull, blkRow.p, blkCol.p, fColInd.p, u2f.p, u2fT.p);
		KLAUNCH(k_ptr_from_high, numP + 1, g_fkeyS.p, nfull, numP, fRowPtr.p);
		// the PCG partition is computed on the host from the (small) full pattern
		S.fRowPtr.resize((size_t)numP + 1); S.fColInd.resize(nfull);
		g_d2hBytes += (long long)(sizeof(int) * ((size_t)numP + 1 + nfull));
		CUDA_TRY(cudaMemcpyAsync(S.fRowPtr.data(), fRowPtr.p, sizeof(int) * ((size_t)numP + 1), cudaMemcpyDeviceToHost, stream));
		if (nfull > 0) CUDA_TRY(cudaMemcpyAsync(S.fColInd.data(), fColInd.p, sizeof(int) * (size_t)nfull, cudaMemcpyDeviceToHost, stream));
		int localCount = (int)N;
		if (dLocalCount) CUDA_TRY(cudaMemcpyAsync(&localCount, dLocalCount, sizeof(int), cudaMemcpyDeviceToHost, stream));
		tmark("queued to sync 4");
		CUDA_TRY(cudaStreamSynchronize(stream));                                  // sync point 4
		tmark("sync 4");
		S.nmulLocal = localCount;
		return CUBA_OK;
	}

	// host copies of the index structures, only for the debug getters
	int ensureHostStructure()
	{
		if (hostStructureValid) return CUBA_OK;
		auto dl = [&](std::vector<int>& dst, const int* src, size_t n) -> cudaError_t {
			dst.resize(n);
			return n ? cudaMemcpyAsync(dst.data(), src, sizeof(int) * n, cudaMemcpyDeviceToHost, stream) : cudaSuccess;
		};
		CUDA_TRY(dl(S.hplColPtr, g_hplColPtr.p, (size_t)S.numL + 1)); CUDA_TRY(dl(S.hplRowInd, g_hplRowInd.p, S.nhpl));
		CUDA_TRY(dl(S.edge2Hpl, g_edge2Hpl.p, S.E)); CUDA_TRY(dl(S.hscRowPtr, g_hscRowPtr.p, (size_t)S.numP + 1));
		CUDA_TRY(dl(S.hscColInd, blkCol.p, S.nblk)); CUDA_TRY(dl(S.u2f, u2f.p, S.nblk)); CUDA_TRY(dl(S.u2fT, u2fT.p, S.nblk));
		CUDA_TRY(cudaStreamSynchronize(stream));
		hostStructureValid = true;
		return CUBA_OK;
	}

	int alloc_system()
	{
		const int eL = S.eLocal;
		const size_t nP = S.numP, nL = S.numL;
		// Hpp | bp | (chi2 slot) and Hsc | bsc are single allocations: one collective each in landmark-sharded runs
		CUDA_TRY(Hpp.alloc(42 * nP + 2)); bp.alias(Hpp.p + 36 * nP, 6 * nP);
		CUDA_TRY(Hll.alloc(9 * nL)); CUDA_TRY(bl.alloc(3 * nL));
		mixed = cfg.use_fp32 == 2 && sizeof(T) == 8 && jhV4;
		if (mixed) { CUDA_TRY(HplF.alloc(20 * (size_t)std::max(S.nhplLocal, 1))); CUDA_TRY(Hpl.alloc(1)); }
		else CUDA_TRY(Hpl.alloc(18 * (size_t)S.nhplLocal));
		CUDA_TRY(invHll.alloc(9 * nL));
		CUDA_TRY(fVal.alloc(36 * (size_t)S.nfull + 6 * nP)); bsc.alias(fVal.p + 36 * (size_t)S.nfull, 6 * nP);
		upperReduce = world > 1 && S.numP > 0 && S.numL > 0;
		if (upperReduce) {
			uCount = 36 * (size_t)S.nblk + 6 * nP;
			const size_t need = ((uCount + 1) & ~(size_t)1) + 64;          // + the signal block of the peer all-reduce
			if (!uVal.p || need > uVal.cap) {
				if (uMappedFor) { CUDA_TRY(cudaStreamSynchronize(stream)); uCloseMappings(); }
				CUDA_TRY(uVal.alloc(std::max(need, (size_t)1 << 18)));
				CUDA_TRY(cudaMemsetAsync(uVal.p, 0, sizeof(T) * uVal.cap, stream));
				uEpoch = 0;
			}
			bsc.alias(uVal.p + 36 * (size_t)S.nblk, 6 * nP);
			// map the peers' buffers; the signal block must sit at the same offset everywhere (it does: uCount is global)
			uPeerOk = false;
			if (!getenv("CUBA_NCCL_HSC") && comm) {
				// signals of an earlier problem may sit at another offset: start from a clean block (all ranks do, in lockstep)
				CUDA_TRY(cudaMemsetAsync(uVal.p + ((uCount + 1) & ~(size_t)1), 0, sizeof(T) * 64, stream));
				uEpoch = 0;
				int rcx = allreduce(&dScal.p->v[7], 1, false); if (rcx) return rcx;          // nobody signals into a block that is being cleared
				bool ok = false;
				rcx = ipcExchange((void*)uVal.p, uPeerBase, uMappedFor, ok); if (rcx) return rcx;
				uPeerOk = ok;
				CUDA_TRY(gridBar.alloc(1));
			}
		}
		CUDA_TRY(xp.alloc(6 * nP)); CUDA_TRY(xl.alloc(3 * nL));
		// landmarks outside this rank's shard keep zero Hll/bl/xl (they are never touched locally)
		if (nL) CUDA_TRY(cudaMemsetAsync(Hll.p, 0, sizeof(T) * 9 * nL, stream));
		if (nL) CUDA_TRY(cudaMemsetAsync(bl.p, 0, sizeof(T) * 3 * nL, stream));
		if (nL) CUDA_TRY(cudaMemsetAsync(xl.p, 0, sizeof(T) * 3 * nL, stream));
		if (nP) CUDA_TRY(cudaMemsetAsync(xp.p, 0, sizeof(T) * 6 * nP, stream));
		if (nP) CUDA_TRY(cudaMemsetAsync(Hpp.p, 0, sizeof(T) * 36 * nP, stream));
		if (nP) CUDA_TRY(cudaMemsetAsync(bp.p, 0, sizeof(T) * 6 * nP, stream));
		if (S.nmulLocal > 0) {
			CUDA_TRY(prodL.alloc((size_t)S.nmulLocal));
			KLAUNCH(schur3::k_prod_landmark, S.nmulLocal, prodI.p, hplLm.p, (int)S.nmulLocal, prodL.p);
		}
		tmark("alloc queued");
		if (jhV4) { int rc = setup_jh4(); if (rc) return rc; }
		tmark("jh4 queued");
		if (S.numP > 0) { int rc = setup_pcg2(); if (rc) return rc; }        // host-heavy: overlaps the warp-tile kernels queued above
		if (S.numP > 0 && S.numL > 0) { int rc = setup_pcg5(); if (rc) return rc; }
		tmark("pcg partition (host)");
		if (jhV4) { int rc = setup_jh4_finish(); if (rc) return rc; }
		tmark("jh4 finish");
		nChiLin = jhV4 ? jh4Grid : ntiles;
		nPoseBlocks = (S.numP + RED_BLOCK - 1) / RED_BLOCK;
		nChiBlocks = std::max(1, std::min((eL + RED_BLOCK - 1) / RED_BLOCK, numSMs * 8));
		CUDA_TRY(chiPartial.alloc((size_t)std::max(std::max(ntiles, nChiBlocks), jh4Grid) + 1));
		CUDA_TRY(scalePartialL.alloc((size_t)std::max(ntiles, (S.numL + RED_BLOCK - 1) / RED_BLOCK) + 1));
		CUDA_TRY(scalePartialP.alloc((size_t)nPoseBlocks + 1));
		CUDA_TRY(chiSq.alloc((size_t)S.E));
		return CUBA_OK;
	}

	int set_state(const double* q, const double* t, const double* X) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "set_state before set_problem");
		const int rc = upload_state(q, t, nullptr, X); if (rc) return rc;
		CUDA_TRY(cudaStreamSynchronize(stream));      // the caller's buffers are free again
		trialValid = false;
		return CUBA_OK;
	}

	int reset_state() override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "reset_state before set_problem");
		for (int b = 0; b < 2; b++) {
			CUDA_TRY(cudaMemcpyAsync(pose[b].p, pose0.p, sizeof(T) * 8 * (size_t)S.Pall, cudaMemcpyDeviceToDevice, stream));
			CUDA_TRY(cudaMemcpyAsync(Xw[b].p, Xw0.p, sizeof(T) * 4 * (size_t)S.Lall, cudaMemcpyDeviceToDevice, stream));
		}
		trialValid = false;
		return CUBA_OK;
	}
	int get_stream(void** s) override { *s = (void*)stream; return CUBA_OK; }
	int flush_l2() override
	{
		const size_t flushN = (size_t)40 << 20;
		CUDA_TRY(flushBuf.alloc(flushN));
		k_fill<<<numSMs * 8, 256, 0, stream>>>(flushBuf.p, flushN, 1.0);
		launches++;
		CUDA_TRY(cudaGetLastError());
		return CUBA_OK;
	}

	int get_sizes(cuba_sizes* o) const override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "get_sizes before set_problem");
		o->Pall = S.Pall; o->numP = S.numP; o->Lall = S.Lall; o->numL = S.numL; o->E2 = S.E2; o->E3 = S.E3;
		o->nhpl = S.nhpl; o->nblk = S.nblk; o->nmul = (int32_t)S.nmul; o->nblk_full = S.nfull;
		return CUBA_OK;
	}

	// ---- launches --------------------------------------------------------------------------------------
	ChiArgs<T> chiArgs(int buf)
	{
		ChiArgs<T> a;
		a.pose = pose[buf]; a.cam = cam; a.Xw = Xw[buf];
		a.mx = e_mx; a.my = e_my; a.mz = e_mz; a.om = e_om; a.ip = e_ip; a.il = e_il;
		a.E = S.eLocal; a.rk = rkParams(); a.chiPartial = chiPartial;
		return a;
	}

	int launch_linearize_landmark()
	{
		if (ntiles <= 0) return CUBA_OK;
		LinLmArgs<T> a;
		a.pose = pose[cur]; a.cam = cam; a.Xw = Xw[cur];
		a.mx = e_mx; a.my = e_my; a.mz = e_mz; a.om = e_om; a.ip = e_ip; a.il = e_il; a.hpl = e_hpl;
		a.lmPtr = tilePtr; a.tileLm = tileLm; a.numP = S.numP; a.numL = S.numL;
		a.Hpl = Hpl; a.Hll = Hll; a.bl = bl; a.chiPartial = chiPartial; a.rk = rkParams();
		if (jhV4) {
			if constexpr (sizeof(T) == 8) {
				if (ntW <= 0) return CUBA_OK;
				jh4::Args b;
				b.pose = pose[cur]; b.cam = cam; b.Xw = Xw[cur];
				b.rec = w_rec; b.tile = w_tile; b.tilePose = w_tilePose; b.tilePieces = w_tilePieces; b.pieceCount = w_pieceCount; b.ntiles = ntW; b.numL = S.numL;
				b.Hpl = Hpl; b.HplF = mixed ? HplF.p : nullptr; b.Hll = Hll; b.bl = bl; b.bigPartial = w_bigPartial; b.chiPartial = chiPartial; b.rk = rkParams();
				const void* fn = nullptr; size_t smem = 0;
#define JH4_PICK(MB, NS, DB) { fn = (const void*)jh4::k_linearize_landmark4<MB, NS, DB>; smem = (size_t)NS * jh4::WARPS * sizeof(jh4::StageOf<MB, NS>); }
				int dbg = 0;
#ifdef CUBA_JH4_DEBUG
				dbg = getenv("CUBA_JH4_DBG") ? atoi(getenv("CUBA_JH4_DBG")) : 0;
				switch (dbg) { case 1: JH4_PICK(4, 2, 1) break; case 2: JH4_PICK(4, 2, 2) break; case 4: JH4_PICK(4, 2, 4) break; case 6: JH4_PICK(4, 2, 6) break;
					case 7: JH4_PICK(4, 2, 7) break; case 8: JH4_PICK(4, 2, 8) break; case 15: JH4_PICK(4, 2, 15) break; default: dbg = 0; }
#endif
				if (mixed) { fn = (const void*)jh4::k_linearize_landmark4<4, 2, 0, true>; smem = (size_t)2 * jh4::WARPS * sizeof(jh4::StageOf<4, 2>); }
				if (!fn) JH4_PICK(4, 2, 0)
				if (fn != jh4AttrSet) { CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); jh4AttrSet = fn; }   // once per kernel, not per launch
				void* kargs[] = { (void*)&b };
				CUDA_TRY(cudaLaunchKernel(fn, dim3(jh4Grid), dim3(jh4::WARPS * 32), kargs, smem, stream));
#ifdef CUBA_JH4_DEBUG
				if (dbg & 8) {
					const int nw = jh4Grid * jh4::WARPS;
					std::vector<double> h(11 * (size_t)nw);
					cudaMemcpyAsync(h.data(), w_bigPartial.p, sizeof(double) * h.size(), cudaMemcpyDeviceToHost, stream);
					cudaStreamSynchronize(stream);
					double acc[8] = { 0 };
					for (int w = 0; w < nw; w++) for (int i = 0; i < 8; i++) acc[i] += h[8 * (size_t)w + i];
					static int once = 0;
					if (once++ == 3) {
						const char* nm[8] = { "cpasync_wait", "mbar_wait", "lds_inputs", "math+hpl_staging", "fence+bulk_store", "wait_read+issue", "reduce+stores", "rotate(descr)" };
						double tot = 0; for (int i = 0; i < 8; i++) tot += acc[i];
						for (int i = 0; i < 8; i++) fprintf(stderr, "jh4 phase %-18s %9.0f cycles/warp  %5.1f %%\n", nm[i], acc[i] / nw, 100 * acc[i] / tot);
						fprintf(stderr, "jh4 total %9.0f cycles/warp, %d warps, %d tiles\n", tot / nw, nw, ntW);
						double s0 = 1e300, s1 = 0, l0 = 1e300, l1 = 0, e0 = 1e300, e1 = 0;
						for (int w = 0; w < nw; w++) {
							const double* g = h.data() + 8 * (size_t)nw + 3 * (size_t)w;
							s0 = std::min(s0, g[0]); s1 = std::max(s1, g[0]); l0 = std::min(l0, g[1]); l1 = std::max(l1, g[1]); e0 = std::min(e0, g[2]); e1 = std::max(e1, g[2]);
						}
						fprintf(stderr, "jh4 globaltimer (ns, rel. first start): start %.0f..%.0f  loop entry %.0f..%.0f  loop exit %.0f..%.0f\n", 0.0, s1 - s0, l0 - s0, l1 - s0, e0 - s0, e1 - s0);
					}
				}
#endif
			}
		}
		else k_linearize_landmark<T, LM_TILE, 6><<<ntiles, LM_TILE, 0, stream>>>(a);
		launches++;
		CUDA_TRY(cudaGetLastError());
		return CUBA_OK;
	}
	int launch_linearize_pose()
	{
		if (S.numP <= 0) return CUBA_OK;
		LinPoseArgs<T> a;
		a.pose = pose[cur]; a.cam = cam; a.Xw = Xw[cur];
		a.mx = p_mx; a.my = p_my; a.mz = p_mz; a.om = p_om; a.il = p_il; a.posePtr = posePtr;
		a.Hpp = Hpp; a.bp = bp; a.rk = rkParams();
		k_linearize_pose<T><<<S.numP, POSE_BLOCK, 0, stream>>>(a);
		launches++;
		CUDA_TRY(cudaGetLastError());
		return CUBA_OK;
	}
	// sums chiPartial[0..n) (+ optional two more arrays) into dScal->v[slot..slot+2]
	int launch_sum(const double* p0, int n0, const double* p1, int n1, const double* p2, int n2, int slot)
	{
		k_sum_partials<<<1, RED_BLOCK, 0, stream>>>(p0, n0, p1, n1, p2, n2, &dScal.p->v[slot]);
		launches++;
		CUDA_TRY(cudaGetLastError());
		return CUBA_OK;
	}
	int fetchScalars()
	{
		g_d2hBytes += (long long)sizeof(Scalars);
		CUDA_TRY(cudaMemcpyAsync(hScal, dScal.p, sizeof(Scalars), cudaMemcpyDeviceToHost, stream));
		CUDA_TRY(cudaStreamSynchronize(stream));
		return CUBA_OK;
	}

	int stage_linearize(double* chi) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "linearize before set_problem");
		{
			ProfScope ps(this, CUBA_PROF_BUILD_SYSTEM);
			int rc = launch_linearize_landmark(); if (rc) return rc;
			rc = launch_linearize_pose(); if (rc) return rc;
			rc = launch_sum(chiPartial, ntiles > 0 ? nChiLin : 0, nullptr, 0, nullptr, 0, 0); if (rc) return rc;
			if (world > 1) {
				// ONE collective: Hpp | bp | chi2 are contiguous (the chi2 partial rides in the slot behind bp)
				if constexpr (sizeof(T) == 8) {
					T* slot = Hpp.p + 42 * (size_t)S.numP;
					CUDA_TRY(cudaMemcpyAsync(slot, &dScal.p->v[0], sizeof(double), cudaMemcpyDeviceToDevice, stream));
					rc = allreduce(Hpp.p, 42 * (size_t)S.numP + 1, true); if (rc) return rc;
					CUDA_TRY(cudaMemcpyAsync(&dScal.p->v[0], slot, sizeof(double), cudaMemcpyDeviceToDevice, stream));
				} else {
					if (S.numP > 0) { rc = allreduce(Hpp.p, 42 * (size_t)S.numP, true); if (rc) return rc; }
					rc = allreduce(&dScal.p->v[0], 1, false); if (rc) return rc;
				}
			}
		}
		int rc = fetchScalars(); if (rc) return rc;
		if (chi) *chi = hScal->v[0];
		return CUBA_OK;
	}

	int stage_chi2(double* chi) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "chi2 before set_problem");
		int rc = launch_chi2(cur, 0); if (rc) return rc;
		rc = fetchScalars(); if (rc) return rc;
		if (chi) *chi = hScal->v[0];
		return CUBA_OK;
	}

	int launch_chi2(int buf, int slot, bool reduce = true)
	{
		ProfScope ps(this, CUBA_PROF_COMPUTE_ERROR);
		if (S.eLocal > 0) {
			k_chi2<T><<<nChiBlocks, RED_BLOCK, 0, stream>>>(chiArgs(buf));
			launches++;
			CUDA_TRY(cudaGetLastError());
		}
		int rc = launch_sum(chiPartial, S.eLocal > 0 ? nChiBlocks : 0, nullptr, 0, nullptr, 0, slot); if (rc) return rc;
		if (world > 1 && reduce) { rc = allreduce(&dScal.p->v[slot], 1, false); if (rc) return rc; }
		return CUBA_OK;
	}

	int stage_max_diagonal(double* md) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "max_diagonal before set_problem");
		CUDA_TRY(cudaMemsetAsync(&dScal.p->maxdiag, 0, sizeof(unsigned long long), stream));
		const int n = S.numP * 6 + S.numL * 3;
		if (n > 0) {
			const int grid = std::max(1, std::min((n + 255) / 256, numSMs * 4));
			k_max_diagonal<T><<<grid, 256, 0, stream>>>(Hpp, S.numP, Hll, S.numL, &dScal.p->maxdiag);
			launches++;
			CUDA_TRY(cudaGetLastError());
		}
		if (world > 1) {
			const int rcn = comm ? g_nccl.AllReduce(&dScal.p->maxdiag, &dScal.p->maxdiag, 1, NCCL_FLOAT64, NCCL_MAX, comm, stream) : 0;
			if (rcn != 0) return fail(CUBA_ERR_COMM, "ncclAllReduce(max) failed");
		}
		int rc = fetchScalars(); if (rc) return rc;
		double m;
		memcpy(&m, &hScal->maxdiag, sizeof(double));
		if (md) *md = m;
		return CUBA_OK;
	}

	int launch_schur(T lambda)
	{
		ProfScope ps(this, CUBA_PROF_SCHUR_COMPLEMENT);
		{
			// the inverses of this rank's landmarks only (nobody reads the others here)
			const int l0 = std::min(S.lmBeg, S.numL), l1 = std::min(S.lmEnd, S.numL);
			if (l1 > l0) {
				k_inv_hll<T><<<(l1 - l0 + 255) / 256, 256, 0, stream>>>(Hll.p + 9 * (size_t)l0, l1 - l0, lambda, invHll.p + 9 * (size_t)l0);
				launches++;
				CUDA_TRY(cudaGetLastError());
			}
		}
		if (S.numP > 0 && S.numL > 0) {
			schur3::Args<T> a;
			a.Hpl = Hpl; a.invHll = invHll; a.bl = bl; a.Hpp = Hpp; a.bp = bp;
			a.prodPtr = prodPtr; a.prodI = prodI; a.prodJ = prodJ; a.prodL = prodL;
			a.blkRow = blkRow; a.blkCol = blkCol; a.u2f = u2f; a.u2fT = u2fT; a.nblk = S.nblk;
			a.lambda = lambda; a.addDiag = rank == 0 ? 1 : 0; a.fVal = fVal; a.bsc = bsc; a.uVal = upperReduce ? uVal.p : nullptr;
			if (mixed) {
				if constexpr (sizeof(T) == 8) {
					schur3::Args<double, float> m;
					m.Hpl = HplF; m.invHll = invHll; m.bl = bl; m.Hpp = Hpp; m.bp = bp; m.prodPtr = prodPtr; m.prodI = prodI; m.prodJ = prodJ; m.prodL = prodL;
					m.blkRow = blkRow; m.blkCol = blkCol; m.u2f = u2f; m.u2fT = u2fT; m.nblk = S.nblk; m.lambda = lambda; m.addDiag = a.addDiag; m.fVal = fVal; m.bsc = bsc; m.uVal = a.uVal;
					schur3::k_schur3<double, float><<<(S.nblk + schur3::WARPS - 1) / schur3::WARPS, schur3::WARPS * 32, 0, stream>>>(m);
				}
			}
			else schur3::k_schur3<T><<<(S.nblk + schur3::WARPS - 1) / schur3::WARPS, schur3::WARPS * 32, 0, stream>>>(a);
			launches++;
			CUDA_TRY(cudaGetLastError());
			if (upperReduce) {
				// upper blocks | bsc: one collective of half the bytes, then both triangles are filled locally
				static const bool timing = getenv("CUBA_SCHUR_TIMING") != nullptr;      // diagnosis: split of the stage, printed by rank 0
				cudaEvent_t ev[3];
				if (timing) { for (auto& e : ev) cudaEventCreate(&e); cudaEventRecord(ev[0], stream); }
				int rc = uPeerOk ? launch_peer_allreduce() : allreduce(uVal.p, 36 * (size_t)S.nblk + 6 * (size_t)S.numP, true); if (rc) return rc;
				if (timing) cudaEventRecord(ev[1], stream);
				KLAUNCH(schur3::k_expand_upper<T>, 36LL * S.nblk, uVal.p, u2f.p, u2fT.p, blkRow.p, blkCol.p, S.nblk, fVal.p);
				if (timing) {
					cudaEventRecord(ev[2], stream); cudaEventSynchronize(ev[2]);
					float a1 = 0, a2 = 0; cudaEventElapsedTime(&a1, ev[0], ev[1]); cudaEventElapsedTime(&a2, ev[1], ev[2]);
					static int count = 0;
					if (rank == 0 && (count++ % 16) == 8) fprintf(stderr, "schur split: all-reduce (%s) %.3f ms, expand %.3f ms, %zu elements\n", uPeerOk ? "peer" : "nccl", a1, a2, uCount);
					for (auto& e : ev) cudaEventDestroy(e);
				}
			}
			else if (world > 1) {
				int rc = allreduce(fVal.p, 36 * (size_t)S.nfull + 6 * (size_t)S.numP, true); if (rc) return rc;   // Hsc | bsc: one buffer
			}
		}
		return CUBA_OK;
	}

	// warp tiles of the J+H landmark pass (cuba_jh4.cuh): greedy packing by binary lifting, padded records, pose lists
	int setup_jh4()
	{
		ntW = 0; jh4Grid = 0; jh4HasBig = 0;
		if constexpr (sizeof(T) == 8) {
			using namespace jh4;
			const int lb = S.lmBeg, N = S.lmEnd - S.lmBeg;
			if (N <= 0 || S.eLocal <= 0) return CUBA_OK;
			int K = 1;
			while ((1LL << K) <= (long long)N) K++;
			CUDA_TRY(w_levels.alloc((size_t)K * ((size_t)N + 1)));
			CUDA_TRY(w_start.alloc((size_t)N + 1)); CUDA_TRY(w_pieces.alloc((size_t)N + 1)); CUDA_TRY(w_base.alloc((size_t)N + 1));
			CUDA_TRY(w_flag.alloc(1));
			CUDA_TRY(cudaMemsetAsync(w_flag.p, 0, sizeof(int), stream));
			KLAUNCH(jh4::k_next, N + 1, lmPtr.p, lb, N, w_levels.p);
			for (int k = 1; k < K; k++)
				KLAUNCH(jh4::k_lift, N + 1, w_levels.p + (size_t)(k - 1) * ((size_t)N + 1), N, w_levels.p + (size_t)k * ((size_t)N + 1));
			KLAUNCH(jh4::k_starts, N + 1, w_levels.p, K, N, lmPtr.p, lb, w_start.p, w_pieces.p, w_flag.p);
			int rc = exclusiveSum(w_pieces.p, w_base.p, N + 1); if (rc) return rc;
			if (!jh4Host) CUDA_TRY(cudaMallocHost((void**)&jh4Host, 2 * sizeof(int)));
			CUDA_TRY(cudaMemcpyAsync(&jh4Host[0], w_base.p + N, sizeof(int), cudaMemcpyDeviceToHost, stream));
			CUDA_TRY(cudaMemcpyAsync(&jh4Host[1], w_flag.p, sizeof(int), cudaMemcpyDeviceToHost, stream));
			jh4Pending = true;
		}
		return CUBA_OK;
	}
	// second half of the warp-tile setup: the host work of setup_pcg2 runs between the two halves, overlapping the kernels above
	int setup_jh4_finish()
	{
		if (!jh4Pending) return CUBA_OK;
		jh4Pending = false;
		if constexpr (sizeof(T) == 8) {
			using namespace jh4;
			const int lb = S.lmBeg, N = S.lmEnd - S.lmBeg;
			CUDA_TRY(cudaStreamSynchronize(stream));
			const int big = jh4Host[1];
			ntW = jh4Host[0]; jh4HasBig = big;
			if (ntW <= 0) return CUBA_OK;
			CUDA_TRY(w_tile.alloc(ntW)); CUDA_TRY(w_rec.alloc(ntW)); CUDA_TRY(w_tilePose.alloc(32 * (size_t)ntW)); CUDA_TRY(w_tilePieces.alloc(ntW)); CUDA_TRY(w_pieceCount.alloc(ntW));
			CUDA_TRY(cudaMemsetAsync(w_pieceCount.p, 0, sizeof(int) * (size_t)ntW, stream));
			CUDA_TRY(w_bigPartial.alloc(std::max<size_t>(big ? 12 * (size_t)ntW : 12, 11 * (size_t)numSMs * 6 * jh4::WARPS)));
			KLAUNCH(jh4::k_emit, (long long)N * 32, w_start.p, w_pieces.p, w_base.p, N, lmPtr.p, lb, w_levels.p,
				e_mx.p, e_my.p, e_mz.p, e_om.p, e_ip.p, e_il.p, e_hpl.p, w_tile.p, w_rec.p, w_tilePose.p, w_tilePieces.p);
			jh4Grid = std::max(1, std::min((ntW + WARPS - 1) / WARPS, numSMs * 4));      // 4 CTAs per SM: the shape's __launch_bounds__
		}
		return CUBA_OK;
	}

	// Row partition, need lists and shared-memory budget of k_pcg2.
	int setup_pcg2()
	{
		const int numP = S.numP;
		int smemMax = 0;
		CUDA_TRY(cudaDeviceGetAttribute(&smemMax, cudaDevAttrMaxSharedMemoryPerBlockOptin, devOrdinal));
		const size_t budget = (size_t)smemMax > 8192 ? (size_t)smemMax - 6144 : 0;   // leave room for the static arrays (4.4 KB in k_pcg3)
		const size_t matBytes = (size_t)S.nfull * (36 * sizeof(T) + 4);
		int G = std::max((numP + 7) / 8, (int)((matBytes + budget - 1) / std::max<size_t>(budget, 1)));
		G = std::max(1, std::min(G, std::min(numSMs, numP)));
		// row partition, need lists, block-local column positions: cuba_structure.cpp (CPU-tested)
		PcgPartition& PP = hostPP;                     // kept: k_pcg5's plan starts from the same partition when its CTA count is the same
		build_pcg_partition(numP, S.nfull, S.fRowPtr, S.fColInd, G, PP);
		const std::vector<int>& rows = PP.rows; const std::vector<int>& nptr = PP.nptr; const std::vector<int>& ncol = PP.ncol; const std::vector<int>& local = PP.local;
		const int needMax = PP.needMax, blkMax = PP.blkMax, maxRows = PP.maxRows;
		// fixed shared-memory footprint of k_pcg3 (a superset of k_pcg2's): r,s per needed column, p,y per own row, index lists
		const size_t needBytes = (size_t)needMax * (12 * sizeof(T) + 8) + (size_t)maxRows * (12 * sizeof(T) + 4) + ((size_t)maxRows + 1) * 4
			+ (size_t)PCG3_CHUNK * 6 * sizeof(T);
		pcg3Ok = maxRows * 6 <= PCG3_BLOCK && 2 * G <= 2 * PCG3_BLOCK;   // k_pcg3: one (row,component) pair per thread, two partial words per thread
		size_t cap = budget > needBytes ? (budget - needBytes) / (36 * sizeof(T) + 4) : 0;
		cap = std::min<size_t>(cap, (size_t)blkMax);
		pcg2Grid = G; pcg2Cap = (int)cap; pcg2NeedMax = needMax; pcg2MaxRows = maxRows;
		pcg2Smem = (size_t)cap * 36 * sizeof(T) + needBytes + (size_t)cap * 4 + 16;
		CUDA_TRY(cudaFuncSetAttribute(k_pcg2<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pcg2Smem));
		CUDA_TRY(cudaFuncSetAttribute(k_pcg3<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pcg2Smem));
		CUDA_TRY(llFlags.alloc(2 * (2 * 6 * (size_t)numP) + 2 * (2 * PCG3_REPL * 2 * (size_t)G) + 2));
		int perSM = 0;
		CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_pcg2<T>, PCG2_BLOCK, pcg2Smem));
		if (perSM < 1) return fail(CUBA_ERR_CUDA, "k_pcg2 cannot be resident with the requested shared memory");
		arena.reset();
		CUDA_TRY(ctaRow.upload(rows, stream, arena)); CUDA_TRY(needPtr.upload(nptr, stream, arena)); CUDA_TRY(needCol.upload(ncol, stream, arena));
		CUDA_TRY(fLocal.upload(local, stream, arena));
		const size_t n6 = 6 * (size_t)numP;
		CUDA_TRY(fHat.alloc(36 * (size_t)S.nfull)); CUDA_TRY(Linv.alloc(36 * (size_t)numP));
		CUDA_TRY(vR0.alloc(n6)); CUDA_TRY(vR1.alloc(n6)); CUDA_TRY(vS0.alloc(n6)); CUDA_TRY(vS1.alloc(n6));
		CUDA_TRY(vW0.alloc(n6)); CUDA_TRY(vW1.alloc(n6)); CUDA_TRY(vP.alloc(n6)); CUDA_TRY(vY.alloc(n6));
		CUDA_TRY(pcg2Partial.alloc(4 * (size_t)G));
		CUDA_TRY(gridBar.alloc(1));
		CUDA_TRY(cudaMemsetAsync(gridBar.p, 0, sizeof(GridBar), stream));
		tmark("  pcg2 partition + uploads");
		// ---- two-level PCG of round 1 (k_pcg4): aggregates = groups of gs consecutive CTAs (at most PCG4_MAXAGG of them).
		//      Only prepared when it can be asked for: explicitly (reserved[0] == 3), by the fp32 engine, or as the fallback for systems
		//      beyond k_pcg5's 85 rows per CTA; otherwise its host lists and uploads are skipped (k_pcg5 has its own plan) ----
		pcg4Ok = false;
		if (cfg.reserved[0] == 3 || sizeof(T) != 8 || numP > 80 * numSMs * (world > 1 && numP >= 2048 ? world : 1)) {
			// up to 74 aggregates (coarse inverse in the shared memory of an 8-CTA cluster), 37 with cfg.reserved[6] == 37 (one CTA)
			const int maxAgg = (cfg.reserved[6] > 0 && cfg.reserved[6] < PCG4_MAXAGG) ? cfg.reserved[6] : PCG4_MAXAGG;
			CoarsePartition CP;
			build_coarse_partition(numP, PP, maxAgg, CP);
			const int gs = CP.gs, A = CP.A, nc = 6 * A;
			pcg4Cluster = A > PCG4_MAXAGG1;
			pcg4A = A; pcg4Gs = gs; pcg4MaxNeedAgg = CP.maxNeedAgg;
			size_t fixed4 = (size_t)needMax * (12 * sizeof(T) + 8) + (size_t)maxRows * (6 * sizeof(T) + 8) + 8 + 2 * (size_t)nc * sizeof(T)
				+ (size_t)pcg4MaxNeedAgg * (6 * sizeof(T) + 4) + 64;
			// shared-memory priorities: all of A^ first, then Z^ of the needed columns, then the CTA's slices of the inverse coarse matrix
			const size_t matAll = (size_t)blkMax * (36 * sizeof(T) + 4);
			const size_t zhBytes = (size_t)needMax * 36 * sizeof(T);
			const size_t sliceBytes = (((size_t)pcg4MaxNeedAgg * 6 * nc + 1) & ~(size_t)1) * sizeof(float);
			pcg4ZhInSmem = budget >= fixed4 + matAll + zhBytes ? 1 : 0;
			if (pcg4ZhInSmem) fixed4 += zhBytes;
			pcg4SliceInSmem = budget >= fixed4 + matAll + sliceBytes ? 1 : 0;
			if (pcg4SliceInSmem) fixed4 += sliceBytes;
			size_t cap4 = budget > fixed4 ? (budget - fixed4) / (36 * sizeof(T) + 4) : 0;
			cap4 = std::min<size_t>(cap4, (size_t)blkMax);
			pcg4Cap = (int)cap4;
			pcg4Smem = (size_t)cap4 * (36 * sizeof(T) + 4) + fixed4;
			if (getenv("CUBA_PCG_VERBOSE")) fprintf(stderr, "pcg4: G %d A %d gs %d needMax %d maxRows %d blkMax %d maxNeedAgg %d zhInSmem %d sliceInSmem %d cap %d smem %zu\n",
				G, A, gs, needMax, maxRows, blkMax, pcg4MaxNeedAgg, pcg4ZhInSmem, pcg4SliceInSmem, pcg4Cap, pcg4Smem);
			const size_t nblkPz = (size_t)A * (A + 1) / 2;
			pcg4InvSmem = pcg4Cluster ? (((nblkPz + PCG4_CL - 1) / PCG4_CL + 2 * (size_t)A) * 36 * sizeof(double) + 2 * nblkPz + 16)
			                          : ((nblkPz + 2 * (size_t)A) * 36 * sizeof(double));
			pcg4Ok = budget > fixed4 && nc + 64 <= PCG4_BLOCK && pcg4InvSmem + 1024 <= (size_t)smemMax && numP >= 2 * A;
			if (pcg4Ok) {
				CUDA_TRY(cudaFuncSetAttribute(k_pcg4<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pcg4Smem));
				if (pcg4Cluster) CUDA_TRY(cudaFuncSetAttribute(k_coarse_chol_cluster, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pcg4InvSmem));
				else CUDA_TRY(cudaFuncSetAttribute(k_coarse_invert<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pcg4InvSmem));
				int perSM4 = 0;
				CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM4, k_pcg4<T>, PCG4_BLOCK, pcg4Smem));
				if (perSM4 < 1) pcg4Ok = false;
			}
			if (pcg4Ok) {
				CUDA_TRY(cAggRow.upload(CP.aggRow, stream, arena)); CUDA_TRY(cNaPtr.upload(CP.naPtr, stream, arena)); CUDA_TRY(cNaList.upload(CP.naList, stream, arena));
				CUDA_TRY(cNeedAgg.upload(CP.needAgg, stream, arena));
				// fine blocks of every coarse block (lower triangle), ascending -> fixed-order sums in k_coarse_assemble
				build_coarse_lists(numP, S.nfull, S.fRowPtr, S.fColInd, CP);
				CUDA_TRY(cRowOf.upload(CP.rowOf, stream, arena)); CUDA_TRY(cCbPtr.upload(CP.cbPtr, stream, arena)); CUDA_TRY(cCbList.upload(CP.cbList, stream, arena));
				CUDA_TRY(cZx.alloc(36 * (size_t)numP)); CUDA_TRY(cZhat.alloc(36 * (size_t)numP)); CUDA_TRY(cU.alloc(36 * (size_t)S.nfull));
				CUDA_TRY(cAcP.alloc((size_t)A * (A + 1) / 2 * 36)); CUDA_TRY(cAcInv.alloc((size_t)nc * nc));
				CUDA_TRY(cLp.alloc((size_t)A * (A + 1) / 2 * 36)); CUDA_TRY(cWp.alloc((size_t)A * (A + 1) / 2 * 36)); CUDA_TRY(cLd.alloc((size_t)A * 36));
				CUDA_TRY(cPart.alloc(2 * (size_t)G * PCG4_PSTRIDE)); CUDA_TRY(cInfo.alloc(1));
				CUDA_TRY(cudaMemsetAsync(cPart.p, 0, sizeof(double) * cPart.n, stream));
				// (no synchronisation: the uploads above read the pinned arena, or were staged by the driver before returning)
			}
			tlActive = false; coarseValid = false; coarseAge = 0;
		}
		return CUBA_OK;
	}

	// two-level PCG: coarse basis, coarse matrix and its inverse, then the cooperative solve
	int launch_pcg4()
	{
		ProfScope ps(this, CUBA_PROF_DECOMP_NUMERICAL);
		const int numP = S.numP, A = pcg4A, nblkP = A * (A + 1) / 2;
		KLAUNCH(k_coarse_basis<T>, numP, pose[cur].p, numP, cZx.p);
		// The coarse matrix Ac = Z^T S Z and its inverse are rebuilt only now and then: ANY symmetric positive definite
		// stand-in for Ac^-1 keeps M^-1 = D^-1 + Z B Z^T a valid preconditioner, and the coarse operator of an earlier
		// damping / linearisation preconditions as well as the current one (CPU prototype: 26..201 iterations over ten LM
		// iterations with a fresh inverse, 26..193 with one that is refreshed every fifth iteration).
		// Measured limits of that freedom: a coarse inverse from an 81x larger damping costs nothing, one from a 1e5x larger damping
		// costs 8x the iterations (1 276 vs 149 on kitti00_shaped) -> it is also rebuilt when the damping moved by more than 300x.
		const int refreshEvery = cfg.reserved[4] > 0 ? cfg.reserved[4] : 8;
		const double lamRatio = (coarseValid && coarseLambda > 0 && curLambda > 0) ? std::max(curLambda / coarseLambda, coarseLambda / curLambda) : 1.0;
		if (!coarseValid || coarseAge >= refreshEvery || lamRatio > 300.0) {
			KLAUNCH(k_coarse_project<T>, 36LL * S.nfull, fVal.p, cRowOf.p, fColInd.p, S.nfull, cZx.p, cU.p);
			KLAUNCH(k_coarse_assemble, (long long)nblkP * 36, cCbPtr.p, cCbList.p, cU.p, nblkP, cAcP.p);
			if (pcg4Cluster) {
				// Cholesky in the shared memory of an 8-CTA cluster, then the triangular inverse (one CTA per block column) and W^T W on the whole chip
				k_coarse_chol_cluster<<<PCG4_CL, 1024, pcg4InvSmem, stream>>>(cAcP.p, A, cLp.p, cLd.p, cAcInv.p, cInfo.p);
				k_coarse_trinv<<<A, 256, (size_t)A * 36 * sizeof(double), stream>>>(cLp.p, cLd.p, A, cWp.p, cInfo.p);
				k_coarse_wtw<<<(nblkP * 36 + 255) / 256, 256, 0, stream>>>(cWp.p, A, cAcInv.p, cInfo.p);
				launches += 2;
			}
			else k_coarse_invert<T><<<1, 1024, pcg4InvSmem, stream>>>(cAcP.p, A, cAcInv.p, cInfo.p);
			launches++;
			CUDA_TRY(cudaGetLastError());
			coarseValid = true; coarseAge = 0; coarseLambda = curLambda;
		}
		coarseAge++;
		Pcg4Args<T> b;
		Pcg2Args<T>& a = b.base;
		a.fRowPtr = fRowPtr; a.fColInd = fColInd; a.fLocal = fLocal; a.fVal = fVal; a.fHat = fHat;
		a.ctaRow = ctaRow; a.needPtr = needPtr; a.needCol = needCol; a.b = bsc; a.numP = S.numP; a.Linv = Linv;
		a.R0 = vR0; a.R1 = vR1; a.S0 = vS0; a.S1 = vS1; a.W0 = vW0; a.W1 = vW1; a.P = vP; a.Y = vY; a.x = xp;
		a.partial = pcg2Partial; a.bar = gridBar; a.capBlocks = pcg4Cap; a.needMax = pcg2NeedMax; a.maxRows = pcg2MaxRows;
		a.maxIters = cfg.pcg_max_iters > 0 ? cfg.pcg_max_iters : std::max(200, 40 * S.numP);
		const double tol = cfg.pcg_tol > 0 ? cfg.pcg_tol : (sizeof(T) == 8 ? 1e-11 : 1e-6);
		a.tol2 = tol * tol;
		a.status = &dScal.p->pcg;
		b.Zx = cZx; b.Zhat = cZhat; b.AcInv = cAcInv; b.aggRow = cAggRow; b.naPtr = cNaPtr; b.naList = cNaList; b.needAgg = cNeedAgg;
		b.A = A; b.gs = pcg4Gs; b.maxNeedAgg = pcg4MaxNeedAgg; b.sliceInSmem = pcg4SliceInSmem; b.zhInSmem = pcg4ZhInSmem; b.cpart = cPart;
		b.timing = nullptr;
#ifdef CUBA_PCG_TIMING
		CUDA_TRY(pcgTiming.alloc(8 * (size_t)pcg2Grid));
		b.timing = pcgTiming.p;
#endif
		void* args[] = { (void*)&b };
		CUDA_TRY(cudaLaunchCooperativeKernel((void*)k_pcg4<T>, dim3(pcg2Grid), dim3(PCG4_BLOCK), args, pcg4Smem, stream));
		launches++;
		lastPcgTwoLevel = true;
		return CUBA_OK;
	}
	bool lastPcgTwoLevel = false;
	bool forceBlockJacobi = false;   // retry of a trial whose two-level solve broke down
	// policy of the default solver: block-Jacobi (k_pcg3, ~5.4 us per iteration) while it converges quickly, two-level (k_pcg4,
	// ~9 us per iteration but 2-8x fewer of them) once a block-Jacobi solve needed more than 100 iterations -- the count grows
	// as the LM damping falls.  The decision depends on iteration counts only, so runs stay bit-reproducible.
	void note_pcg_iters(int iters) { if (!lastPcgTwoLevel && iters > (cfg.reserved[5] > 0 ? cfg.reserved[5] : 100)) tlActive = true; }

	int launch_pcg2(bool flagged)
	{
		ProfScope ps(this, CUBA_PROF_DECOMP_NUMERICAL);
		Pcg2Args<T> a;
		a.fRowPtr = fRowPtr; a.fColInd = fColInd; a.fLocal = fLocal; a.fVal = fVal; a.fHat = fHat;
		a.ctaRow = ctaRow; a.needPtr = needPtr; a.needCol = needCol; a.b = bsc; a.numP = S.numP; a.Linv = Linv;
		a.R0 = vR0; a.R1 = vR1; a.S0 = vS0; a.S1 = vS1; a.W0 = vW0; a.W1 = vW1; a.P = vP; a.Y = vY; a.x = xp;
		a.partial = pcg2Partial; a.bar = gridBar; a.capBlocks = pcg2Cap; a.needMax = pcg2NeedMax; a.maxRows = pcg2MaxRows;
		a.maxIters = cfg.pcg_max_iters > 0 ? cfg.pcg_max_iters : std::max(200, 40 * S.numP);
		const double tol = cfg.pcg_tol > 0 ? cfg.pcg_tol : (sizeof(T) == 8 ? 1e-11 : 1e-6);
		a.tol2 = tol * tol;
		a.status = &dScal.p->pcg;
		if (flagged) {
			Pcg3Args<T> b;
			b.base = a;
			b.wFlag = llFlags.p;
			b.pFlag = llFlags.p + 2 * (2 * 6 * (size_t)S.numP);
			b.abortFlag = (int*)(b.pFlag + 2 * (2 * PCG3_REPL * 2 * (size_t)pcg2Grid));
			b.timing = nullptr;
#ifdef CUBA_PCG_TIMING
			CUDA_TRY(pcgTiming.alloc(8 * (size_t)pcg2Grid));
			b.timing = pcgTiming.p;
#endif
			CUDA_TRY(cudaMemsetAsync(llFlags.p, 0, sizeof(unsigned long long) * llFlags.n, stream));
			void* args3[] = { (void*)&b };
			CUDA_TRY(cudaLaunchCooperativeKernel((void*)k_pcg3<T>, dim3(pcg2Grid), dim3(PCG3_BLOCK), args3, pcg2Smem, stream));
			launches++;
			return CUBA_OK;
		}
		void* args[] = { (void*)&a };
		CUDA_TRY(cudaLaunchCooperativeKernel((void*)k_pcg2<T>, dim3(pcg2Grid), dim3(PCG2_BLOCK), args, pcg2Smem, stream));
		launches++;
		return CUBA_OK;
	}


	// ---- k_pcg5: two-level, flag-synchronised, rows distributed over the ranks (cuba_pcg5.cuh) --------------------------
	DBuf<int> p5CtaRow, p5NeedPtr, p5NeedCol, p5Local, p5AggRow, p5NaPtr, p5NaList, p5NeedAgg, p5CbPtr, p5CbList;
	DBuf<unsigned char> p5RowPeers;
	DBuf<T> p5Linv, p5R0, p5Zhat, p5RcRow, p5Rc0;
	DBuf<float> p5AcInv;
	DBuf<double> p5AcP;
	DBuf<double> cdM, cdL, cdW, cdDinv;            // dense work matrices of k_coarse_dense
	bool p5Dense = false;
	DBuf<unsigned long long> p5Boards;
	void* p5PeerBase[PCG5_MAXWORLD] = { nullptr };   // cudaIpc mappings of the peers' boards (own entry: the local allocation)
	void* p5MappedFor = nullptr;                   // local allocation the mappings were exchanged for
	size_t p5WWords = 0, p5PWords = 0, p5RWords = 0, p5CWords = 0;
	PcgPartition hostPP;                           // host copy of k_pcg3's row partition of the current system (setup_pcg2)
	Pcg5Dims p5Dims{}, p5DimsBJ{};
	size_t p5Smem = 0;
	int p5G = 0, p5W = 1, p5A = 0, p5Gs = 1;
	bool p5Ok = false, p5Dist = false, p5Big = false, p5Tuned = false;
	p5t::Pcg5Dims p5tDims{}, p5tDimsBJ{};            // the tuned one-GPU shape (cuba_pcg5t.cuh), when p5Tuned
	const void* p5Fn = nullptr;
	int p5Block = PCG5_BLOCK;
	bool p5CoarseValid = false; int p5CoarseAge = 0; double p5CoarseLambda = 0;
	size_t p5InvSmem = 0;
	long long p5TagBound = 0;                      // conservative host-side bound on the device tag base

	Pcg5Ctl* p5Ctl(void* base) const { return (Pcg5Ctl*)((unsigned long long*)base + 2 * (p5WWords + p5PWords + p5RWords + p5CWords)); }

	void p5CloseMappings()
	{
		for (int r = 0; r < PCG5_MAXWORLD; r++) {
			if (p5PeerBase[r] && r != rank) cudaIpcCloseMemHandle(p5PeerBase[r]);
			p5PeerBase[r] = nullptr;
		}
		p5MappedFor = nullptr;
	}

	// Maps one device allocation of every peer into this process (cudaIpc over NVLink peer access); the 64-byte handles travel by
	// ncclAllGather.  All ranks agree on the outcome (sum of per-rank success flags), so either everybody uses the peer path or
	// everybody keeps the NCCL one.
	int ipcExchange(void* localBase, void** peerBase, void*& mappedFor, bool& ok)
	{
		ok = false;
		if (mappedFor == localBase) { ok = true; return CUBA_OK; }
		for (int r = 0; r < PCG5_MAXWORLD; r++) { if (peerBase[r] && r != rank) cudaIpcCloseMemHandle(peerBase[r]); peerBase[r] = nullptr; }
		mappedFor = nullptr;
		cudaIpcMemHandle_t mine;
		int good = cudaIpcGetMemHandle(&mine, localBase) == cudaSuccess ? 1 : 0;
		if (!good) cudaGetLastError();
		DBuf<char> dh;
		CUDA_TRY(dh.alloc(sizeof(cudaIpcMemHandle_t) * (size_t)world));
		CUDA_TRY(cudaMemcpyAsync(dh.p + sizeof(cudaIpcMemHandle_t) * (size_t)rank, &mine, sizeof(mine), cudaMemcpyHostToDevice, stream));
		int rc = g_nccl.AllGather(dh.p + sizeof(cudaIpcMemHandle_t) * (size_t)rank, dh.p, sizeof(cudaIpcMemHandle_t), NCCL_INT8, comm, stream);
		if (rc != 0) return fail(CUBA_ERR_COMM, "ncclAllGather (memory handles) failed");
		std::vector<cudaIpcMemHandle_t> all(world);
		CUDA_TRY(cudaMemcpyAsync(all.data(), dh.p, sizeof(cudaIpcMemHandle_t) * (size_t)world, cudaMemcpyDeviceToHost, stream));
		CUDA_TRY(cudaStreamSynchronize(stream));
		for (int r = 0; r < world && good; r++) {
			if (r == rank) { peerBase[r] = localBase; continue; }
			if (cudaIpcOpenMemHandle(&peerBase[r], all[r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); peerBase[r] = nullptr; good = 0; }
		}
		// agreement
		DBuf<double> flag;
		CUDA_TRY(flag.alloc(1));
		const double mineOk = good;
		CUDA_TRY(cudaMemcpyAsync(flag.p, &mineOk, sizeof(double), cudaMemcpyHostToDevice, stream));
		rc = allreduce(flag.p, 1, false); if (rc) return rc;
		double tot = 0;
		CUDA_TRY(cudaMemcpyAsync(&tot, flag.p, sizeof(double), cudaMemcpyDeviceToHost, stream));
		CUDA_TRY(cudaStreamSynchronize(stream));
		if ((int)(tot + 0.5) != world) {
			for (int r = 0; r < PCG5_MAXWORLD; r++) { if (peerBase[r] && r != rank) cudaIpcCloseMemHandle(peerBase[r]); peerBase[r] = nullptr; }
			return CUBA_OK;
		}
		mappedFor = localBase;
		ok = true;
		return CUBA_OK;
	}
	int p5Exchange(bool& ok) { return ipcExchange((void*)p5Boards.p, p5PeerBase, p5MappedFor, ok); }

	// ---- the per-trial Hsc | bsc all-reduce over peer memory (cuba_peer_reduce.cuh) ----
	void* uPeerBase[PCG5_MAXWORLD] = { nullptr };
	void* uMappedFor = nullptr;
	bool uPeerOk = false;
	unsigned int uEpoch = 0;
	size_t uCount = 0;             // elements of the all-reduced part of uVal
	void uCloseMappings()
	{
		for (int r = 0; r < PCG5_MAXWORLD; r++) { if (uPeerBase[r] && r != rank) cudaIpcCloseMemHandle(uPeerBase[r]); uPeerBase[r] = nullptr; }
		uMappedFor = nullptr; uPeerOk = false;
	}
	int launch_peer_allreduce()
	{
		peer::Args<T> pa;
		pa.local = uVal.p; pa.n = uCount; pa.rank = rank; pa.world = world; pa.epoch = ++uEpoch; pa.bar = gridBar;
		const size_t sigOff = (uCount + 1) & ~(size_t)1;       // the signal block sits behind the data (element units)
		for (int r = 0; r < peer::MAXW; r++) { pa.peers[r] = nullptr; pa.sigPeer[r] = nullptr; }
		for (int r = 0; r < world; r++) { pa.peers[r] = (T*)uPeerBase[r]; pa.sigPeer[r] = (unsigned int*)((T*)uPeerBase[r] + sigOff); }
		pa.sigLocal = (unsigned int*)(uVal.p + sigOff);
		void* args[] = { (void*)&pa };
		CUDA_TRY(cudaLaunchCooperativeKernel((void*)peer::k_peer_allreduce<T>, dim3(numSMs), dim3(peer::BLOCK), args, 0, stream));
		launches++;
		return CUBA_OK;
	}

	// Partition of the rows over world x G virtual CTAs, aggregates aligned with the ranks, shared-memory budget, boards.
	int setup_pcg5()
	{
		p5Ok = false; p5Dist = false; p5CoarseValid = false; p5CoarseAge = 0;
		const int numP = S.numP;
		if (numP < 1) return CUBA_OK;
		const int mode = cfg.reserved[0];
		if (mode == 2 || mode == 3 || mode == 4) return CUBA_OK;          // an older kernel was asked for explicitly
		const bool wantDist = world > 1 && comm && mode != 7 && (mode == 8 || numP >= 2048);
		const int W = wantDist ? world : 1;
		int smemMax = 0;
		CUDA_TRY(cudaDeviceGetAttribute(&smemMax, cudaDevAttrMaxSharedMemoryPerBlockOptin, devOrdinal));
		const size_t budget = (size_t)smemMax > 4096 ? (size_t)smemMax - 2048 : 0;   // static arrays of k_pcg5: < 1 KB
		// rows over world x G virtual CTAs (about eight rows each, never more than 42: one thread per (row, component) pair in the
		// row sums), rank-aligned aggregates, halo masks: cuba_structure.cpp (CPU-tested through cuba_debug_pcg5_plan)
		const int maxAgg = (cfg.reserved[6] > 0 && cfg.reserved[6] < PCG5_MAXAGG) ? cfg.reserved[6] : PCG5_MAXAGG;
		Pcg5Plan plan;
		build_pcg5_plan(numP, S.nfull, S.fRowPtr, S.fColInd, W, numSMs, maxAgg, 2 * PCG5_BLOCK / 6, plan, &hostPP);
		if (!plan.ok) return CUBA_OK;
		const int G = plan.G, gs = plan.gs, A = plan.A;
		const PcgPartition& PP = plan.P; const CoarsePartition& CP = plan.C;
		const std::vector<unsigned char>& peers = plan.rowPeers;
		const int Aloc = G / gs, NR = 3 + 6 * Aloc, nc = 6 * A;
		Pcg5Dims d{};
		d.needMax = PP.needMax; d.maxRows = PP.maxRows; d.nc = nc; d.maxNeedAgg = CP.maxNeedAgg;
		d.npv = std::max(std::max(G * 9, W * NR), 6 * CP.maxNeedAgg); d.nls = NR;
		d.sliceRows = (nc + G - 1) / G;
		const size_t per = 36 * sizeof(T) + 4;
		size_t wantCache = PP.blkMax > PCG5_REGBLK ? (size_t)(PP.blkMax - PCG5_REGBLK) : 0;
		// the tuned shape (cuba_pcg5t.cuh): a solve on one GPU whose blocks fit registers + shared memory
		p5Tuned = false;
		if (W == 1 && !getenv("CUBA_PCG5_LEGACY")) {
			using TS = p5t::Pcg5Shape;
			p5t::Pcg5Dims t{};
			t.needMax = PP.needMax; t.maxRows = PP.maxRows; t.nc = nc; t.maxNeedAgg = CP.maxNeedAgg;
			t.npv = d.npv; t.nls = NR; t.sliceRows = d.sliceRows;
			t.ccCap = PP.blkMax >= TS::CHUNK ? TS::CHUNK : std::max((std::max(PP.blkMax, PP.needMax) + 31) / 32 * 32, 32);
			t.sqWords = std::max(9 * PP.maxRows * 6, 9 * (TS::BLOCK / 32));
			t.capBlocks = 0; t.zhInSmem = 0;
			const size_t base = p5t::Pcg5Layout<T>(t).total + 64;
			const size_t zhBytes = (size_t)t.needMax * 36 * sizeof(T);
			size_t used = base + wantCache * per;
			if (used + zhBytes <= budget) { t.zhInSmem = 1; used += zhBytes; }
			if (PP.maxRows * 6 <= TS::BLOCK && used <= budget) {
				t.capBlocks = (int)wantCache;
				p5tDims = t;
				p5tDimsBJ = t; p5tDimsBJ.nc = 0; p5tDimsBJ.maxNeedAgg = 0; p5tDimsBJ.zhInSmem = 0; p5tDimsBJ.sliceRows = 0; p5tDimsBJ.nls = 3; p5tDimsBJ.npv = std::max(G * 3, W * 3);
				const size_t smemT = std::max(p5t::Pcg5Layout<T>(p5tDims).total, p5t::Pcg5Layout<T>(p5tDimsBJ).total);
				const void* fn = (const void*)p5t::k_pcg5t<T>;
				int perSM = 0;
				if (smemT <= (size_t)smemMax - 1024 && cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemT) == cudaSuccess &&
					cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, fn, TS::BLOCK, smemT) == cudaSuccess && perSM >= 1) {
					p5Tuned = true; p5Big = false; p5Fn = fn; p5Block = TS::BLOCK; p5Smem = smemT;
					p5Dims = Pcg5Dims{}; p5Dims.capBlocks = t.capBlocks;
					d.capBlocks = t.capBlocks; d.zhInSmem = t.zhInSmem;
				} else cudaGetLastError();
			}
		}
		if (!p5Tuned) {
		bool big = PP.maxRows * 6 > PCG5_BLOCK;
		{
			d.capBlocks = 0; d.zhInSmem = 0;
			const size_t base = Pcg5Layout<T>(d).total + 64;
			if (base > budget) return CUBA_OK;
			const size_t zhBytes = (size_t)d.needMax * 36 * sizeof(T);
			size_t used = base + wantCache * per;
			if (used + zhBytes <= budget) { d.zhInSmem = 1; used += zhBytes; }
			const size_t fixed = used - wantCache * per;
			d.capBlocks = (int)std::min(wantCache, (budget - fixed) / per);
			// blocks would have to be streamed from the global copy every pass: the variant without register-resident blocks streams
			// with eighteen 16-byte loads in flight per thread (the register variant can afford six 8-byte loads)
			if ((size_t)d.capBlocks < wantCache) big = true;
			if (big) d.capBlocks = (int)std::min((size_t)PP.blkMax, (budget - fixed) / per);
		}
		p5Dims = d;
		p5DimsBJ = d; p5DimsBJ.nc = 0; p5DimsBJ.maxNeedAgg = 0; p5DimsBJ.zhInSmem = 0; p5DimsBJ.sliceRows = 0; p5DimsBJ.nls = 3; p5DimsBJ.npv = std::max(G * 3, W * 3);
		p5Smem = std::max(Pcg5Layout<T>(p5Dims).total, Pcg5Layout<T>(p5DimsBJ).total);
		if (p5Smem > (size_t)smemMax - 1024) return CUBA_OK;
		p5Big = big;
		p5Fn = p5Big ? (const void*)k_pcg5<T, true> : (const void*)k_pcg5<T, false>;
		p5Block = PCG5_BLOCK;
		CUDA_TRY(cudaFuncSetAttribute(p5Fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p5Smem));
		int perSM = 0;
		if (p5Big) CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_pcg5<T, true>, PCG5_BLOCK, p5Smem));
		else CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_pcg5<T, false>, PCG5_BLOCK, p5Smem));
		if (perSM < 1) return CUBA_OK;
		}
		if (getenv("CUBA_PCG_VERBOSE")) fprintf(stderr, "pcg5: world %d G %d gs %d A %d needMax %d maxRows %d blkMax %d maxNeedAgg %d zhInSmem %d sliceRows %d cap %d smem %zu\n",
			W, G, gs, A, d.needMax, d.maxRows, PP.blkMax, d.maxNeedAgg, d.zhInSmem, d.sliceRows, d.capBlocks, p5Smem);
		if (getenv("CUBA_PCG_VERBOSE")) fprintf(stderr, "pcg5: shape %s, %d threads\n", p5Big ? "big" : p5Tuned ? "tuned" : "legacy", p5Block);
		// coarse inverse: packed block triangle in the shared memory of one CTA (A <= 37), beyond that the dense tile Cholesky on the
		// whole chip (cuba_coarse_dense.cuh)
		p5Dense = A > PCG4_MAXAGG1;
		const size_t nblkPz = (size_t)A * (A + 1) / 2;
		if (!p5Dense) {
			p5InvSmem = (nblkPz + 2 * (size_t)A) * 36 * sizeof(double);
			if (p5InvSmem + 1024 > (size_t)smemMax) return CUBA_OK;
			CUDA_TRY(cudaFuncSetAttribute(k_coarse_invert<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max(p5InvSmem, (!pcg4Cluster && pcg4Ok) ? pcg4InvSmem : 0)));
		}
		CUDA_TRY(p5CtaRow.upload(PP.rows, stream, arena)); CUDA_TRY(p5NeedPtr.upload(PP.nptr, stream, arena)); CUDA_TRY(p5NeedCol.upload(PP.ncol, stream, arena));
		CUDA_TRY(p5Local.upload(PP.local, stream, arena)); CUDA_TRY(p5RowPeers.upload(peers, stream, arena));
		CUDA_TRY(p5AggRow.upload(CP.aggRow, stream, arena)); CUDA_TRY(p5NaPtr.upload(CP.naPtr, stream, arena)); CUDA_TRY(p5NaList.upload(CP.naList, stream, arena));
		CUDA_TRY(p5NeedAgg.upload(CP.needAgg, stream, arena)); CUDA_TRY(p5CbPtr.upload(CP.cbPtr, stream, arena)); CUDA_TRY(p5CbList.upload(CP.cbList, stream, arena));
		CUDA_TRY(cRowOf.upload(CP.rowOf, stream, arena));
		const size_t nP = (size_t)numP;
		CUDA_TRY(p5Linv.alloc(36 * nP)); CUDA_TRY(p5R0.alloc(6 * nP)); CUDA_TRY(p5Zhat.alloc(36 * nP)); CUDA_TRY(p5RcRow.alloc(6 * nP)); CUDA_TRY(p5Rc0.alloc(std::max(nc, 1)));
		CUDA_TRY(cZx.alloc(36 * nP)); CUDA_TRY(cU.alloc(36 * (size_t)S.nfull)); CUDA_TRY(cInfo.alloc(1));
		CUDA_TRY(fHat.alloc(36 * (size_t)S.nfull));
		CUDA_TRY(p5AcP.alloc(nblkPz * 36)); CUDA_TRY(p5AcInv.alloc((size_t)nc * nc));
		if (p5Dense) {
			const size_t ntd = ((size_t)nc + cdense::NB - 1) / cdense::NB, npd = ntd * cdense::NB;
			CUDA_TRY(cdM.alloc(npd * npd)); CUDA_TRY(cdL.alloc(npd * npd)); CUDA_TRY(cdW.alloc(npd * npd)); CUDA_TRY(cdDinv.alloc(ntd * cdense::NB * cdense::NB));
			CUDA_TRY(gridBar.alloc(1));
		}
		// boards (16-byte words): [2 solve halves][2 pass parities] of w, of the per-CTA partials and of the rank summaries, then the control block
		const size_t wW = 4 * 6 * nP, pW = 4 * (size_t)PCG5_REPL * G * 9, rW = 4 * (size_t)PCG5_REPL * W * NR, cW = 4 * (size_t)PCG5_REPL * nc;
		const size_t words2 = 2 * (wW + pW + rW + cW) + (sizeof(Pcg5Ctl) + 7) / 8 + 2;
		const bool fresh = !p5Boards.p || words2 > p5Boards.cap || wW != p5WWords || pW != p5PWords || rW != p5RWords || cW != p5CWords;
		if (fresh) {
			// the tag protocol needs boards that start out as zeros; a layout change invalidates every mapping and every tag
			if (p5MappedFor) { CUDA_TRY(cudaStreamSynchronize(stream)); p5CloseMappings(); }
			CUDA_TRY(p5Boards.alloc(std::max(words2, (size_t)(1u << 18))));
			CUDA_TRY(cudaMemsetAsync(p5Boards.p, 0, sizeof(unsigned long long) * p5Boards.cap, stream));
			p5WWords = wW; p5PWords = pW; p5RWords = rW; p5CWords = cW;
			p5TagBound = 0;
		}
		p5G = G; p5W = W; p5A = A; p5Gs = gs;
		if (W > 1) {
			bool ok = false;
			int rc = p5Exchange(ok); if (rc) return rc;
			if (!ok) {
				if (rank == 0) fprintf(stderr, "cuba_b200: cudaIpc mapping of the peers' PCG boards failed; keeping the replicated PCG\n");
				return CUBA_OK;
			}
			p5Dist = true;
		} else p5PeerBase[rank] = (void*)p5Boards.p;
		p5Ok = true;
		return CUBA_OK;
	}

	// coarse matrix Ac = Z^T S Z of the current system and its inverse (fp32), for the aggregates behind (cbPtr, cbList)
	int launch_coarse_setup(int A, size_t invSmem, const int* cbPtr, const int* cbList, double* AcP, float* AcInv, bool dense)
	{
		const int nblkP = A * (A + 1) / 2;
		KLAUNCH(k_coarse_project<T>, 36LL * S.nfull, fVal.p, cRowOf.p, fColInd.p, S.nfull, cZx.p, cU.p);
		KLAUNCH(k_coarse_assemble, (long long)nblkP * 36, cbPtr, cbList, cU.p, nblkP, AcP);
		if (dense) {
			// dense tile Cholesky + inverse on the whole chip (cuba_coarse_dense.cuh): one persistent cooperative kernel
			CUDA_TRY(cudaMemsetAsync(cdM.p, 0, sizeof(double) * cdM.n, stream));
			cdense::Args da;
			da.AcP = AcP; da.A = A; da.M = cdM; da.Lm = cdL; da.Dinv = cdDinv; da.W = cdW; da.AcInv = AcInv; da.info = cInfo; da.bar = gridBar;
			void* dargs[] = { (void*)&da };
			CUDA_TRY(cudaLaunchCooperativeKernel((void*)cdense::k_coarse_dense, dim3(numSMs), dim3(cdense::WARPS * 32), dargs, 0, stream));
			launches++;
			return CUBA_OK;
		}
		k_coarse_invert<T><<<1, 1024, invSmem, stream>>>(AcP, A, AcInv, cInfo.p);
		launches++;
		CUDA_TRY(cudaGetLastError());
		return CUBA_OK;
	}

	int launch_pcg5(bool twoLevel)
	{
		ProfScope ps(this, CUBA_PROF_DECOMP_NUMERICAL);
		const int numP = S.numP, A = twoLevel ? p5A : 0;
		const int maxIters = cfg.pcg_max_iters > 0 ? cfg.pcg_max_iters : std::max(200, 40 * numP);
		// tags are 32 bits: long before the device tag base can wrap, every rank (same arithmetic everywhere) clears its boards
		p5TagBound += (long long)maxIters + 8;
		if (p5TagBound > (1LL << 31)) {
			if (p5Dist) { int rc0 = allreduce(&dScal.p->v[7], 1, false); if (rc0) return rc0; }   // nobody still writes into a peer's boards
			CUDA_TRY(cudaMemsetAsync(p5Boards.p, 0, sizeof(unsigned long long) * p5Boards.cap, stream));
			if (p5Dist) { int rc0 = allreduce(&dScal.p->v[7], 1, false); if (rc0) return rc0; }
			p5TagBound = (long long)maxIters + 8;
		}
		if (twoLevel) KLAUNCH(k_coarse_basis<T>, numP, pose[cur].p, numP, cZx.p);
		Pcg5PrepArgs<T> pa;
		pa.fRowPtr = fRowPtr; pa.fColInd = fColInd; pa.fVal = fVal; pa.b = bsc; pa.Zx = cZx; pa.numP = numP; pa.A = A; pa.aggRow = p5AggRow;
		pa.Linv = p5Linv; pa.R0 = p5R0; pa.Zhat = p5Zhat; pa.rcRow = p5RcRow; pa.rc0 = p5Rc0; pa.ctl = p5Ctl(p5Boards.p);
		k_pcg5_prep_rows<T><<<(numP + 127) / 128, 128, 0, stream>>>(pa);
		launches++;
		if (twoLevel) {
			k_pcg5_prep_rc<T><<<(6 * A + 127) / 128, 128, 0, stream>>>(pa);
			launches++;
			// The coarse inverse is rebuilt only now and then (see launch_pcg4: any SPD stand-in keeps M^-1 a valid preconditioner).
			const int refreshEvery = cfg.reserved[4] > 0 ? cfg.reserved[4] : 8;
			const double lamRatio = (p5CoarseValid && p5CoarseLambda > 0 && curLambda > 0) ? std::max(curLambda / p5CoarseLambda, p5CoarseLambda / curLambda) : 1.0;
			if (!p5CoarseValid || p5CoarseAge >= refreshEvery || lamRatio > 300.0) {
				int rc = launch_coarse_setup(A, p5InvSmem, p5CbPtr, p5CbList, p5AcP, p5AcInv, p5Dense); if (rc) return rc;
				p5CoarseValid = true; p5CoarseAge = 0; p5CoarseLambda = curLambda;
			}
			p5CoarseAge++;
		}
		CUDA_TRY(cudaGetLastError());
		// the same arguments for both shapes (cuba_pcg5.cuh / cuba_pcg5t.cuh differ only in their Pcg5Dims)
		auto fill = [&](auto& a) {
			using CtlPtr = decltype(a.ctl);
			a.fRowPtr = fRowPtr; a.fColInd = fColInd; a.fLocal = p5Local; a.fVal = fVal; a.fHat = fHat;
			a.ctaRow = p5CtaRow; a.needPtr = p5NeedPtr; a.needCol = p5NeedCol;
			a.numP = numP; a.G = p5G; a.rank = p5Dist ? rank : 0; a.world = p5W;
			a.Linv = p5Linv; a.R0 = p5R0; a.Zhat = p5Zhat; a.rc0 = p5Rc0; a.x = xp;
			a.maxIters = maxIters;
			const double tol = cfg.pcg_tol > 0 ? cfg.pcg_tol : (sizeof(T) == 8 ? 1e-11 : 1e-6);
			a.tol2 = tol * tol;
			a.status = &dScal.p->pcg;
			a.AcInv = p5AcInv; a.naPtr = p5NaPtr; a.naList = p5NaList; a.needAgg = p5NeedAgg; a.A = A; a.gs = p5Gs;
			for (int r = 0; r < PCG5_MAXWORLD; r++) { a.peerW[r] = nullptr; a.peerR[r] = nullptr; a.peerCtl[r] = nullptr; }
			for (int r = 0; r < p5W; r++) {
				unsigned long long* base = (unsigned long long*)p5PeerBase[p5Dist ? r : rank];
				a.peerW[r] = base; a.peerR[r] = base + 2 * (p5WWords + p5PWords); a.peerCtl[r] = reinterpret_cast<CtlPtr>(p5Ctl(base));
			}
			a.wBoard = p5Boards.p; a.pBoard = p5Boards.p + 2 * p5WWords; a.rBoard = p5Boards.p + 2 * (p5WWords + p5PWords);
			a.cBoard = p5Boards.p + 2 * (p5WWords + p5PWords + p5RWords);
			a.rowPeers = p5RowPeers; a.ctl = reinterpret_cast<CtlPtr>(p5Ctl(p5Boards.p));
			a.timing = nullptr;
		};
#ifdef CUBA_PCG_TIMING
		CUDA_TRY(pcgTiming.alloc(8 * (size_t)p5G));
#endif
		if (p5Dist) CUDA_TRY(cudaMemsetAsync(xp.p, 0, sizeof(T) * 6 * (size_t)numP, stream));     // rows of the other ranks: summed in below
		Pcg5Args<T> a;
		p5t::Pcg5Args<T> at;
		void* args[1];
		if (p5Tuned) {
			fill(at);
			at.dims = twoLevel ? p5tDims : p5tDimsBJ;
			at.dims.capBlocks = p5tDims.capBlocks;
#ifdef CUBA_PCG_TIMING
			at.timing = pcgTiming.p;
#endif
			args[0] = (void*)&at;
		} else {
			fill(a);
			a.dims = twoLevel ? p5Dims : p5DimsBJ;
			a.dims.capBlocks = p5Dims.capBlocks;
#ifdef CUBA_PCG_TIMING
			a.timing = pcgTiming.p;
#endif
			args[0] = (void*)&a;
		}
		CUDA_TRY(cudaLaunchCooperativeKernel(p5Fn, dim3(p5G), dim3(p5Block), args, p5Smem, stream));
		k_pcg5_commit<<<1, 1, 0, stream>>>(p5Ctl(p5Boards.p));
		launches += 2;
		CUDA_TRY(cudaGetLastError());
		if (p5Dist) { int rc = allreduce(xp.p, 6 * (size_t)numP, true); if (rc) return rc; }
		lastPcgTwoLevel = twoLevel;
		return CUBA_OK;
	}

	int launch_pcg()
	{
		lastPcgTwoLevel = false;
		// 0 (also 7, 8): automatic = block-Jacobi while a solve converges quickly, two-level afterwards -- k_pcg5 for the two-level solves
		// (and, when the rows are distributed over the ranks, for every solve), k_pcg3 for the quick block-Jacobi ones on one GPU;
		// 5: always two-level k_pcg5; 6: always block-Jacobi k_pcg5; 3: always k_pcg4; 4: always k_pcg3; 2: k_pcg2.
		// k_pcg3 falls back to k_pcg2 beyond ~85 rows per CTA, k_pcg5 and k_pcg4 to k_pcg3 where their setup declined the system.
		const int m = cfg.reserved[0];
		const bool two = tlActive && !forceBlockJacobi;
		if (p5Ok && (m == 5 || m == 6)) return launch_pcg5(m == 5 && !forceBlockJacobi);
		if (p5Ok && (m == 0 || m == 7 || m == 8) && (p5Dist || two)) return launch_pcg5(two);
		if (pcg4Ok && (m == 0 || m == 7 || m == 8) && two) return launch_pcg4();
		if (pcg4Ok && m == 3 && !forceBlockJacobi) return launch_pcg4();
		if (m == 2) return launch_pcg2(false);   // k_pcg2: one grid barrier per iteration
		return launch_pcg2(pcg3Ok);              // k_pcg3: flag-synchronised exchange
	}

	int launch_backsub(T lambda)
	{
		ProfScope ps(this, CUBA_PROF_SCHUR_COMPLEMENT);
		if (ntiles > 0 && S.numL > 0) {
			BacksubArgs<T> a;
			a.Hpl = Hpl; a.invHll = invHll; a.bl = bl; a.xp = xp; a.ip = e_ip; a.hpl = e_hpl; a.lmPtr = tilePtr; a.tileLm = tileLm;
			a.numL = S.numL; a.lambda = lambda; a.XwCur = Xw[cur]; a.XwTrial = Xw[cur ^ 1]; a.xl = xl; a.scalePartial = scalePartialL;
			if (mixed) {
				if constexpr (sizeof(T) == 8) {
					BacksubArgs<double, float> m;
					m.Hpl = HplF; m.invHll = invHll; m.bl = bl; m.xp = xp; m.ip = e_ip; m.hpl = e_hpl; m.lmPtr = tilePtr; m.tileLm = tileLm;
					m.numL = S.numL; m.lambda = lambda; m.XwCur = Xw[cur]; m.XwTrial = Xw[cur ^ 1]; m.xl = xl; m.scalePartial = scalePartialL;
					k_backsub<double, LM_TILE, float><<<ntiles, LM_TILE, 0, stream>>>(m);
				}
			}
			else k_backsub<T, LM_TILE><<<ntiles, LM_TILE, 0, stream>>>(a);
			launches++;
			CUDA_TRY(cudaGetLastError());
		}
		return CUBA_OK;
	}

	// Schur + PCG + back-substitution.  Leaves xp/xl, the trial landmarks and the landmark scale partials.
	int stage_solve(double lambda, int* iters, int* ok) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "solve before set_problem");
		const T lam = (T)lambda;
		curLambda = lambda;
		int rc = launch_schur(lam); if (rc) return rc;
		int nScaleL = 0;
		if (S.numP > 0 && S.numL > 0) {
			rc = launch_pcg(); if (rc) return rc;
			rc = launch_backsub(lam); if (rc) return rc;
			nScaleL = ntiles;
		} else if (S.numP > 0) {
			k_solve_poses_only<T><<<(S.numP + 127) / 128, 128, 0, stream>>>(Hpp, bp, S.numP, lam, xp);
			launches++;
			CUDA_TRY(cudaGetLastError());
			hScal->pcg.iters = 0; hScal->pcg.status = 0;
		} else if (S.numL > 0) {
			nScaleL = (S.numL + RED_BLOCK - 1) / RED_BLOCK;
			k_solve_landmarks_only<T><<<nScaleL, RED_BLOCK, 0, stream>>>(invHll, bl, S.numL, lam, Xw[cur], Xw[cur ^ 1], xl, scalePartialL);
			launches++;
			CUDA_TRY(cudaGetLastError());
		}
		nScaleLandmark = nScaleL;
		solvedLambda = lambda;
		if (iters || ok) {
			rc = fetchScalars(); if (rc) return rc;
			const bool usedPcg = S.numP > 0 && S.numL > 0;
			if (usedPcg) note_pcg_iters(hScal->pcg.iters);
			if (iters) *iters = usedPcg ? hScal->pcg.iters : 0;
			if (ok) *ok = usedPcg ? (hScal->pcg.status == 0) : 1;
		}
		return CUBA_OK;
	}
	int nScaleLandmark = 0;
	double solvedLambda = 0;

	// pose update + trial chi2 + scale; results in dScal->v[1] (chi2), v[2..3] (scale parts)
	int stage_update(double lambda, double* chi, double* scale) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "update before set_problem");
		const T lam = (T)lambda;
		{
			ProfScope ps(this, CUBA_PROF_UPDATE);
			if (S.numP > 0) {
				k_update_poses<T><<<nPoseBlocks, RED_BLOCK, 0, stream>>>(xp, bp, S.numP, lam, pose[cur], pose[cur ^ 1], scalePartialP);
				launches++;
				CUDA_TRY(cudaGetLastError());
			}
		}
		int rc = launch_chi2(cur ^ 1, 1, false); if (rc) return rc;
		// scale = sum over [xp;xl] of x (lambda x + b): pose part is replicated, landmark part is sharded
		rc = launch_sum(scalePartialL, nScaleLandmark, scalePartialP, S.numP > 0 ? nPoseBlocks : 0, nullptr, 0, 2); if (rc) return rc;
		if (world > 1) { rc = allreduce(&dScal.p->v[1], 2, false); if (rc) return rc; }   // trial chi2 and the landmark part of the scale: adjacent slots
		rc = fetchScalars(); if (rc) return rc;
		trialValid = true;
		if (chi) *chi = hScal->v[1];
		if (scale) *scale = hScal->v[2] + hScal->v[3];
		return CUBA_OK;
	}

	int stage_commit(int accept) override
	{
		if (!trialValid) return fail(CUBA_ERR_STATE, "commit without a trial state");
		if (accept) cur ^= 1;
		trialValid = false;
		return CUBA_OK;
	}

	// ---- the LM loop: reference src/cuda_bundle_adjustment.cpp:793-857 ---------------------------------
	int optimize(int niter, cuba_iter_stat* stats, int* nstats) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "optimize before set_problem");
		const int maxq = 10;
		const double tau = 1e-5;
		double nu = 2, lambda = 0, F = 0;
		int n = 0;
		tlActive = false; coarseValid = false; coarseAge = 0;     // results never depend on what the engine solved before
		p5CoarseValid = false; p5CoarseAge = 0; forceBlockJacobi = false;
		bool haveF = false;
		for (int it = 0; it < niter; it++) {
			double chi0 = 0;
			int rc = stage_linearize(&chi0); if (rc) return rc;
			// after an accepted trial the reference recomputes the same residuals (cpp:808); the value is F
			if (!haveF) F = chi0;
			F = chi0; haveF = true;
			if (it == 0) {
				double md = 0;
				rc = stage_max_diagonal(&md); if (rc) return rc;
				lambda = tau * md;
			}
			int q = 0, trials = 0, pcgIters = 0, pcgFailed = 0;
			double rho = -1;
			for (; q < maxq && rho < 0; q++) {
				trials++;
				int iters = 0, ok = 1;
				double Fhat = 0, scale = 0;
				for (int attempt = 0; attempt < 2; attempt++) {
					rc = stage_solve(lambda, nullptr, nullptr); if (rc) return rc;
					rc = stage_update(lambda, &Fhat, &scale); if (rc) return rc;
					if (!(S.numP > 0 && S.numL > 0)) break;
					const PcgStatus& ps = hScal->pcg;
					iters += ps.iters;
					if (ps.status == 3) return fail(CUBA_ERR_COMM, "PCG: a CTA or a peer GPU stopped answering (flag exchange timed out)");
					// The reference's direct solve fails only when the factorisation does (cuda_linear_solver.cpp:406-410).  Here: a solve
					// that ran into the iteration cap is still used when its residual fell far enough for an LM step; a breakdown of a
					// two-level solve (the fp32 coarse inverse lost definiteness) is retried once with block-Jacobi alone.
					const double loose = sizeof(T) == 8 ? 1e-6 : 1e-3;
					ok = ps.status == 0 || (ps.status == 1 && ps.rz0 > 0 && ps.rz <= loose * loose * ps.rz0);
					if (ps.status == 2 && lastPcgTwoLevel && attempt == 0) {
						forceBlockJacobi = true; coarseValid = false; p5CoarseValid = false;
						rc = stage_commit(0); if (rc) return rc;
						continue;
					}
					break;
				}
				forceBlockJacobi = false;
				if (S.numP > 0 && S.numL > 0) note_pcg_iters(hScal->pcg.iters);
				pcgIters += iters; if (!ok) pcgFailed++;
				scale += 1e-3;
				rho = ok ? (F - Fhat) / scale : -1;
				if (!(rho == rho)) rho = -1;   // NaN trial -> reject
				if (rho > 0) {
					const double a = 2 * rho - 1;
					lambda *= std::max(1. / 3, std::min(1 - a * a * a, 2. / 3));
					nu = 2; F = Fhat;
					rc = stage_commit(1); if (rc) return rc;
					break;
				} else {
					lambda *= nu; nu *= 2;
					rc = stage_commit(0); if (rc) return rc;
				}
			}
			if (stats) {
				stats[n].iteration = it; stats[n].trials = trials; stats[n].chi2 = F; stats[n].lambda = lambda;
				stats[n].pcg_iters = pcgIters; stats[n].pcg_failed = pcgFailed;
			}
			n++;
			if (q == maxq || rho <= 0 || !std::isfinite(lambda)) break;
		}
		if (nstats) *nstats = n;
		resolveProfile();   // the stream is idle (every trial ends with a fetch): recycle the profile events instead of hoarding them
		return CUBA_OK;
	}

	int get_state(double* q, double* t, double* X) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "get_state before set_problem");
		std::vector<T> hp((size_t)S.Pall * 8), hx((size_t)S.Lall * 4);
		g_d2hBytes += (long long)(sizeof(T) * (hp.size() + hx.size()));
		CUDA_TRY(cudaMemcpyAsync(hp.data(), pose[cur].p, sizeof(T) * hp.size(), cudaMemcpyDeviceToHost, stream));
		if (world > 1 && S.numL > 0) {
			// all-gather of the sharded landmarks: every rank broadcasts its own range in place (one grouped NCCL call).
			// The trial buffer is free between LM iterations and serves as the gather target.
			T* tmp = Xw[cur ^ 1].p;
			trialValid = false;
			CUDA_TRY(cudaMemcpyAsync(tmp, Xw[cur].p, sizeof(T) * 4 * (size_t)S.Lall, cudaMemcpyDeviceToDevice, stream));
			if (shardBoundValid) {
				const int dt = sizeof(T) == 8 ? NCCL_FLOAT64 : NCCL_FLOAT32;
				g_nccl.GroupStart();
				int rcn = 0;
				for (int r = 0; r < world; r++) {
					const int b0 = std::min(shardBound[r], S.numL), b1 = std::min(shardBound[r + 1], S.numL);     // fixed landmarks never change
					if (b1 > b0) rcn |= g_nccl.Broadcast(tmp + 4 * (size_t)b0, tmp + 4 * (size_t)b0, 4 * (size_t)(b1 - b0), dt, r, comm, stream);
				}
				rcn |= g_nccl.GroupEnd();
				if (rcn != 0) return fail(CUBA_ERR_COMM, "ncclBroadcast (landmark gather) failed");
			} else {
				// host-built structure (debug path): zero the foreign entries, sum over ranks
				CUDA_TRY(cudaMemsetAsync(tmp, 0, sizeof(T) * 4 * (size_t)S.Lall, stream));
				if (S.lmEnd > S.lmBeg)
					CUDA_TRY(cudaMemcpyAsync(tmp + 4 * (size_t)S.lmBeg, Xw[cur].p + 4 * (size_t)S.lmBeg, sizeof(T) * 4 * (size_t)(S.lmEnd - S.lmBeg), cudaMemcpyDeviceToDevice, stream));
				int rc = allreduce(tmp, 4 * (size_t)S.Lall, true); if (rc) return rc;
			}
			CUDA_TRY(cudaMemcpyAsync(hx.data(), tmp, sizeof(T) * hx.size(), cudaMemcpyDeviceToHost, stream));
			CUDA_TRY(cudaStreamSynchronize(stream));
		} else {
			CUDA_TRY(cudaMemcpyAsync(hx.data(), Xw[cur].p, sizeof(T) * hx.size(), cudaMemcpyDeviceToHost, stream));
			CUDA_TRY(cudaStreamSynchronize(stream));
		}
		for (int i = 0; i < S.Pall; i++) {
			if (q) for (int k = 0; k < 4; k++) q[4 * (size_t)i + k] = (double)hp[8 * (size_t)i + k];
			if (t) for (int k = 0; k < 3; k++) t[3 * (size_t)i + k] = (double)hp[8 * (size_t)i + 4 + k];
		}
		if (X) for (int i = 0; i < S.Lall; i++) for (int k = 0; k < 3; k++) X[3 * (size_t)i + k] = (double)hx[4 * (size_t)i + k];
		return CUBA_OK;
	}

	int get_chi2(double* out) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "get_chi2 before set_problem");
		CUDA_TRY(cudaMemsetAsync(chiSq.p, 0, sizeof(double) * (size_t)std::max(S.E, 1), stream));
		if (S.eLocal > 0) {
			k_chi_sqs<T><<<(S.eLocal + 255) / 256, 256, 0, stream>>>(chiArgs(cur), e_user, chiSq);
			launches++;
			CUDA_TRY(cudaGetLastError());
		}
		if (world > 1) { int rc = allreduce(chiSq.p, (size_t)S.E, false); if (rc) return rc; }
		g_d2hBytes += (long long)(sizeof(double) * (size_t)S.E);
		CUDA_TRY(cudaMemcpyAsync(out, chiSq.p, sizeof(double) * (size_t)S.E, cudaMemcpyDeviceToHost, stream));
		CUDA_TRY(cudaStreamSynchronize(stream));
		return CUBA_OK;
	}

	int get_profile(double* sec) override
	{
		resolveProfile();
		for (int i = 0; i < CUBA_PROF_NUM; i++) sec[i] = prof[i];
		return CUBA_OK;
	}

	// ---- debug getters ---------------------------------------------------------------------------------
	int dbg_hpl_structure(int32_t* colPtr, int32_t* rowInd, int32_t* e2h) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "no problem");
		{ const int rc0 = ensureHostStructure(); if (rc0) return rc0; }
		if (colPtr) memcpy(colPtr, S.hplColPtr.data(), sizeof(int) * S.hplColPtr.size());
		if (rowInd) memcpy(rowInd, S.hplRowInd.data(), sizeof(int) * S.hplRowInd.size());
		if (e2h) memcpy(e2h, S.edge2Hpl.data(), sizeof(int) * S.edge2Hpl.size());
		return CUBA_OK;
	}
	int dbg_hsc_structure(int32_t* rowPtr, int32_t* colInd) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "no problem");
		{ const int rc0 = ensureHostStructure(); if (rc0) return rc0; }
		if (rowPtr) memcpy(rowPtr, S.hscRowPtr.data(), sizeof(int) * S.hscRowPtr.size());
		if (colInd) memcpy(colInd, S.hscColInd.data(), sizeof(int) * S.hscColInd.size());
		return CUBA_OK;
	}
	int download(const T* d, size_t n, double* out)
	{
		std::vector<T> h(n);
		CUDA_TRY(cudaMemcpyAsync(h.data(), d, sizeof(T) * n, cudaMemcpyDeviceToHost, stream));
		CUDA_TRY(cudaStreamSynchronize(stream));
		for (size_t i = 0; i < n; i++) out[i] = (double)h[i];
		return CUBA_OK;
	}
	int dbg_system(double* oHpp, double* obp, double* oHll, double* obl, double* oHpl) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "no problem");
		int rc;
		if (oHpp && (rc = download(Hpp, 36 * (size_t)S.numP, oHpp))) return rc;
		if (obp && (rc = download(bp, 6 * (size_t)S.numP, obp))) return rc;
		if (oHll && (rc = download(Hll, 9 * (size_t)S.numL, oHll))) return rc;
		if (obl && (rc = download(bl, 3 * (size_t)S.numL, obl))) return rc;
		if (oHpl) {
			// local blocks land at their global positions; foreign blocks read as zero
			memset(oHpl, 0, sizeof(double) * 18 * (size_t)S.nhpl);
			if (mixed) {
				std::vector<float> hf(20 * (size_t)S.nhplLocal);
				CUDA_TRY(cudaMemcpyAsync(hf.data(), HplF.p, sizeof(float) * hf.size(), cudaMemcpyDeviceToHost, stream));
				CUDA_TRY(cudaStreamSynchronize(stream));
				for (size_t b = 0; b < (size_t)S.nhplLocal; b++) for (int e = 0; e < 18; e++) oHpl[18 * ((size_t)S.hplBase + b) + e] = (double)hf[20 * b + e];
			}
			else if ((rc = download(Hpl, 18 * (size_t)S.nhplLocal, oHpl + 18 * (size_t)S.hplBase))) return rc;
		}
		return CUBA_OK;
	}
	int dbg_schur(double* oHsc, double* obsc, double* oinv) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "no problem");
		int rc;
		if ((rc = ensureHostStructure())) return rc;
		if (oHsc) {
			std::vector<double> full(36 * (size_t)S.nfull);
			if ((rc = download(fVal, full.size(), full.data()))) return rc;
			for (int k = 0; k < S.nblk; k++) memcpy(oHsc + 36 * (size_t)k, full.data() + 36 * (size_t)S.u2f[k], sizeof(double) * 36);
		}
		if (obsc && (rc = download(bsc, 6 * (size_t)S.numP, obsc))) return rc;
		if (oinv && (rc = download(invHll, 9 * (size_t)S.numL, oinv))) return rc;
		return CUBA_OK;
	}
	int dbg_delta(double* oxp, double* oxl) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "no problem");
		int rc;
		if (oxp && (rc = download(xp, 6 * (size_t)S.numP, oxp))) return rc;
		if (oxl && (rc = download(xl, 3 * (size_t)S.numL, oxl))) return rc;
		return CUBA_OK;
	}

	int dbg_pcg_timing(long long* out, int maxCtas) override
	{
		const int n = std::min(maxCtas, pcg2Grid);
		if (!pcgTiming.p || n <= 0) return 0;
		cudaMemcpyAsync(out, pcgTiming.p, sizeof(long long) * 8 * (size_t)n, cudaMemcpyDeviceToHost, stream);
		cudaStreamSynchronize(stream);
		return n;
	}

	// ---- micro-benchmarks --------------------------------------------------------------------------------
	int bench_stage(int stage, int reps, int flush, double lambda, double* ms) override
	{
		if (!haveProblem) return fail(CUBA_ERR_STATE, "bench before set_problem");
		if (reps < 1) reps = 1;
		const size_t flushN = (size_t)40 << 20;   // 320 MB of doubles > 126 MB L2
		if (flush) CUDA_TRY(flushBuf.alloc(flushN));
		cudaEvent_t a, b;
		CUDA_TRY(cudaEventCreate(&a)); CUDA_TRY(cudaEventCreate(&b));
		double total = 0;
		const T lam = (T)lambda;
		for (int r = 0; r < reps; r++) {
			if (flush) { k_fill<<<numSMs * 8, 256, 0, stream>>>(flushBuf.p, flushN, (double)r); launches++; }
			CUDA_TRY(cudaEventRecord(a, stream));
			int rc = CUBA_OK;
			switch (stage) {
			case 0: rc = launch_linearize_landmark(); if (!rc) rc = launch_linearize_pose(); break;
			case 1: rc = launch_linearize_landmark(); break;
			case 2: rc = launch_linearize_pose(); break;
			case 3: rc = launch_schur(lam); break;
			case 4: curLambda = lambda; rc = launch_pcg(); break;
			case 5: rc = launch_backsub(lam); if (!rc) rc = stage_update_nofetch(lam); break;
			case 6: rc = launch_chi2(cur, 0); break;
			default: rc = fail(CUBA_ERR_INVALID, "bench_stage: unknown stage");
			}
			if (rc) return rc;
			CUDA_TRY(cudaEventRecord(b, stream));
			CUDA_TRY(cudaEventSynchronize(b));
			float t = 0;
			CUDA_TRY(cudaEventElapsedTime(&t, a, b));
			total += t;
		}
		cudaEventDestroy(a); cudaEventDestroy(b);
		resolveProfile();
		if (ms) *ms = total / reps;
		return CUBA_OK;
	}
	int stage_update_nofetch(T lam)
	{
		if (S.numP > 0) {
			k_update_poses<T><<<nPoseBlocks, RED_BLOCK, 0, stream>>>(xp, bp, S.numP, lam, pose[cur], pose[cur ^ 1], scalePartialP);
			launches++;
			CUDA_TRY(cudaGetLastError());
		}
		return launch_chi2(cur ^ 1, 1);
	}
};

}  // namespace cuba_b200

// ======================================================================================================
// C ABI
// ======================================================================================================
using namespace cuba_b200;

struct cuba_engine { std::unique_ptr<EngineBase> impl; };

extern "C" {

const char* cuba_last_error(void) { return g_err.c_str(); }
int cuba_version(void) { return 100; }

int cuba_engine_create(const cuba_config* cfg, cuba_engine** out)
{
	if (!out) return fail(CUBA_ERR_INVALID, "create: null out");
	cuba_config c;
	memset(&c, 0, sizeof(c));
	c.device = -1; c.deterministic = 1;
	if (cfg) c = *cfg;
	// reserved[0..3] select kernels (include/cuba_b200.h): a value that selects none is refused, never run as some other kernel
	const unsigned accepted[4] = { 0x1fdu /* 0, 2..8 */, 0x3u /* 0, 1 */, 0x11u /* 0, 4 */, 0x9u /* 0, 3 */ };
	for (int i = 0; i < 4; i++)
		if (c.reserved[i] < 0 || c.reserved[i] > 31 || !((accepted[i] >> c.reserved[i]) & 1u))
			return fail(CUBA_ERR_INVALID, "create: cuba_config.reserved[" + std::to_string(i) + "] = " + std::to_string(c.reserved[i]) + " selects no kernel");
	std::unique_ptr<EngineBase> impl;
	int rc;
	if (c.use_fp32 == 1) { auto* e = new Engine<float>(); e->cfg = c; impl.reset(e); rc = e->init(); }
	else { auto* e = new Engine<double>(); e->cfg = c; impl.reset(e); rc = e->init(); }
	if (rc) return rc;
	if (getenv("CUBA_NO_STRUCTURE_REUSE")) impl->structureReuse = false;   // like-for-like timing against the reference, which rebuilds everything
	*out = new cuba_engine{ std::move(impl) };
	return CUBA_OK;
}

int cuba_engine_destroy(cuba_engine* e) { delete e; return CUBA_OK; }   // ~Engine switches to its own device itself

#define ENGINE_OR_FAIL(e) if (!(e) || !(e)->impl) return fail(CUBA_ERR_INVALID, "null engine"); DevGuard _devGuard((e)->impl->devOrdinal)

int cuba_engine_set_robust_kernel(cuba_engine* e, int edge_type, int kernel_type, double delta)
{
	ENGINE_OR_FAIL(e);
	if (edge_type < 0 || edge_type > 1 || kernel_type < 0 || kernel_type > 2) return fail(CUBA_ERR_INVALID, "set_robust_kernel: bad type");
	e->impl->rk_type[edge_type] = kernel_type; e->impl->rk_delta[edge_type] = delta;
	return CUBA_OK;
}

int cuba_comm_unique_id(void* out128)
{
	std::string why;
	if (!g_nccl.load(why)) return fail(CUBA_ERR_COMM, why);
	Nccl::UniqueId id;
	const int rc = g_nccl.GetUniqueId(&id);
	if (rc) return fail(CUBA_ERR_COMM, "ncclGetUniqueId failed");
	memcpy(out128, &id, 128);
	return CUBA_OK;
}

int cuba_engine_set_comm(cuba_engine* e, int rank, int world, const void* uid)
{
	ENGINE_OR_FAIL(e);
	if (world < 1 || rank < 0 || rank >= world || world > PCG5_MAXWORLD) return fail(CUBA_ERR_INVALID, "set_comm: bad rank/world (at most 8 ranks)");
	if (e->impl->haveProblem) return fail(CUBA_ERR_STATE, "set_comm must precede set_problem");
	e->impl->rank = rank; e->impl->world = world;
	if (world == 1) return CUBA_OK;
	if (getenv("CUBA_DRY_SHARD")) return CUBA_OK;      // diagnosis: keep the shard, skip every collective (results are then partial sums)
	if (!uid) return fail(CUBA_ERR_INVALID, "set_comm: null unique id");
	std::string why;
	if (!g_nccl.load(why)) return fail(CUBA_ERR_COMM, why);
	Nccl::UniqueId id;
	memcpy(&id, uid, 128);
	const int rc = g_nccl.CommInitRank(&e->impl->comm, world, id, rank);
	if (rc) return fail(CUBA_ERR_COMM, std::string("ncclCommInitRank failed: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"));
	return CUBA_OK;
}

int cuba_engine_set_problem(cuba_engine* e, const cuba_problem* p) { ENGINE_OR_FAIL(e); return e->impl->set_problem(p); }
int cuba_engine_set_structure_reuse(cuba_engine* e, int enable) { ENGINE_OR_FAIL(e); e->impl->structureReuse = enable != 0; return CUBA_OK; }
int cuba_engine_get_structure_reuses(cuba_engine* e, long long* count) { ENGINE_OR_FAIL(e); if (count) *count = e->impl->structureReuses; return CUBA_OK; }
int cuba_engine_set_state(cuba_engine* e, const double* q, const double* t, const double* Xw)
{
	ENGINE_OR_FAIL(e);
	if (!q || !t || !Xw) return fail(CUBA_ERR_INVALID, "set_state: null array");
	return e->impl->set_state(q, t, Xw);
}
int cuba_engine_reset_state(cuba_engine* e) { ENGINE_OR_FAIL(e); return e->impl->reset_state(); }
int cuba_engine_get_stream(cuba_engine* e, void** s) { ENGINE_OR_FAIL(e); if (!s) return fail(CUBA_ERR_INVALID, "null out"); return e->impl->get_stream(s); }
int cuba_engine_flush_l2(cuba_engine* e) { ENGINE_OR_FAIL(e); return e->impl->flush_l2(); }
int cuba_engine_get_sizes(const cuba_engine* e, cuba_sizes* out) { ENGINE_OR_FAIL(e); if (!out) return fail(CUBA_ERR_INVALID, "null out"); return e->impl->get_sizes(out); }
int cuba_engine_optimize(cuba_engine* e, int niter, cuba_iter_stat* stats, int* nstats) { ENGINE_OR_FAIL(e); return e->impl->optimize(niter, stats, nstats); }
int cuba_engine_get_state(cuba_engine* e, double* q, double* t, double* Xw) { ENGINE_OR_FAIL(e); return e->impl->get_state(q, t, Xw); }
int cuba_engine_get_chi2(cuba_engine* e, double* per_edge) { ENGINE_OR_FAIL(e); if (!per_edge) return fail(CUBA_ERR_INVALID, "null out"); return e->impl->get_chi2(per_edge); }
int cuba_engine_get_profile(cuba_engine* e, double* sec) { ENGINE_OR_FAIL(e); if (!sec) return fail(CUBA_ERR_INVALID, "null out"); return e->impl->get_profile(sec); }
// debug: per-CTA phase timings of the last k_pcg3 launch (library built with -DCUBA_PCG_TIMING); returns the CTA count
int cuba_debug_get_pcg_timing(cuba_engine* e, long long* out, int maxCtas)
{
	if (!e || !e->impl) return -1;
	DevGuard guard(e->impl->devOrdinal);
	return e->impl->dbg_pcg_timing(out, maxCtas);
}
int cuba_get_transfer_bytes(long long* h2d, long long* d2h) { if (h2d) *h2d = g_h2dBytes; if (d2h) *d2h = g_d2hBytes; return CUBA_OK; }
int cuba_engine_get_launch_count(cuba_engine* e, long long* count) { ENGINE_OR_FAIL(e); if (count) *count = e->impl->launches; return CUBA_OK; }

int cuba_stage_linearize(cuba_engine* e, double* chi2) { ENGINE_OR_FAIL(e); return e->impl->stage_linearize(chi2); }
int cuba_stage_max_diagonal(cuba_engine* e, double* md) { ENGINE_OR_FAIL(e); return e->impl->stage_max_diagonal(md); }
int cuba_stage_solve(cuba_engine* e, double lambda, int* iters, int* ok)
{
	ENGINE_OR_FAIL(e);
	int it = 0, k = 1;
	const int rc = e->impl->stage_solve(lambda, &it, &k);
	if (iters) *iters = it;
	if (ok) *ok = k;
	return rc;
}
int cuba_stage_update(cuba_engine* e, double lambda, double* chi, double* scale) { ENGINE_OR_FAIL(e); return e->impl->stage_update(lambda, chi, scale); }
int cuba_stage_commit(cuba_engine* e, int accept) { ENGINE_OR_FAIL(e); return e->impl->stage_commit(accept); }
int cuba_stage_chi2(cuba_engine* e, double* chi) { ENGINE_OR_FAIL(e); return e->impl->stage_chi2(chi); }

int cuba_debug_get_hpl_structure(cuba_engine* e, int32_t* colPtr, int32_t* rowInd, int32_t* e2h) { ENGINE_OR_FAIL(e); return e->impl->dbg_hpl_structure(colPtr, rowInd, e2h); }
int cuba_debug_get_hsc_structure(cuba_engine* e, int32_t* rowPtr, int32_t* colInd) { ENGINE_OR_FAIL(e); return e->impl->dbg_hsc_structure(rowPtr, colInd); }
int cuba_debug_get_system(cuba_engine* e, double* Hpp, double* bp, double* Hll, double* bl, double* Hpl) { ENGINE_OR_FAIL(e); return e->impl->dbg_system(Hpp, bp, Hll, bl, Hpl); }
int cuba_debug_get_schur(cuba_engine* e, double* Hsc, double* bsc, double* invHll) { ENGINE_OR_FAIL(e); return e->impl->dbg_schur(Hsc, bsc, invHll); }
int cuba_debug_get_delta(cuba_engine* e, double* xp, double* xl) { ENGINE_OR_FAIL(e); return e->impl->dbg_delta(xp, xl); }
int cuba_debug_build_structure_host(const cuba_problem* p, int rank, int world, cuba_sizes* sizes,
	int32_t* hplColPtr, int32_t* hplRowInd, int32_t* edge2Hpl, int32_t* hscRowPtr, int32_t* hscColInd,
	int32_t* fullRowPtr, int32_t* fullColInd, int32_t* shard)
{
	if (!p) return fail(CUBA_ERR_INVALID, "null problem");
	Structure S;
	const char* err = "";
	if (!build_structure(p->Pall, p->numP, p->Lall, p->numL, p->E2, p->idx2, p->E3, p->idx3, rank, world, TILE, S, &err))
		return fail(CUBA_ERR_INVALID, err);
	if (sizes) {
		sizes->Pall = S.Pall; sizes->numP = S.numP; sizes->Lall = S.Lall; sizes->numL = S.numL; sizes->E2 = S.E2; sizes->E3 = S.E3;
		sizes->nhpl = S.nhpl; sizes->nblk = S.nblk; sizes->nmul = (int32_t)S.nmul; sizes->nblk_full = S.nfull;
	}
	auto cp = [](int32_t* dst, const std::vector<int>& v) { if (dst && !v.empty()) memcpy(dst, v.data(), sizeof(int) * v.size()); };
	cp(hplColPtr, S.hplColPtr); cp(hplRowInd, S.hplRowInd); cp(edge2Hpl, S.edge2Hpl);
	cp(hscRowPtr, S.hscRowPtr); cp(hscColInd, S.hscColInd); cp(fullRowPtr, S.fRowPtr); cp(fullColInd, S.fColInd);
	if (shard) { shard[0] = S.lmBeg; shard[1] = S.lmEnd; shard[2] = S.eLocal; shard[3] = (int32_t)S.nmulLocal; }
	// internal consistency (cheap): tiles cover the shard, products reference blocks of one landmark with row(i)<=row(j)
	if ((int)S.tileLm.size() < 1 || S.tileLm.front() != S.lmBeg || S.tileLm.back() != S.lmEnd) return fail(CUBA_ERR_INVALID, "structure self-check: tiles");
	for (size_t t = 0; t + 1 < S.tileLm.size(); t++) {
		const int nl = S.tileLm[t + 1] - S.tileLm[t];
		const int ne = S.lmPtr[S.tileLm[t + 1]] - S.lmPtr[S.tileLm[t]];
		if (nl < 1 || nl > TILE || (ne > TILE && nl != 1)) return fail(CUBA_ERR_INVALID, "structure self-check: tile size");
	}
	for (int k = 0; k < S.nblk; k++)
		for (int n = S.prodPtr[k]; n < S.prodPtr[k + 1]; n++) {
			const int i = S.prodI[n] + S.hplBase, j = S.prodJ[n] + S.hplBase;
			if (S.hplRowInd[i] != S.blkRow[k] || S.hplRowInd[j] != S.blkCol[k] || S.hplLm[S.prodI[n]] != S.hplLm[S.prodJ[n]] || i > j)
				return fail(CUBA_ERR_INVALID, "structure self-check: product list");
		}
	return CUBA_OK;
}

/* host side of the PCG setup on the CPU (no device needed): structure -> row partition over nCtas CTAs -> aggregates and coarse
 * lists with at most maxAgg aggregates; runs the invariants of check_pcg_partition.  info[8] = G, gs, A, needMax, maxRows,
 * blkMax, maxNeedAgg, size of the coarse lists. */
int cuba_debug_pcg_partition(const cuba_problem* p, int nCtas, int maxAgg, int32_t* info)
{
	if (!p || nCtas < 1 || maxAgg < 1) return fail(CUBA_ERR_INVALID, "pcg_partition: bad arguments");
	Structure S;
	const char* err = "";
	if (!build_structure(p->Pall, p->numP, p->Lall, p->numL, p->E2, p->idx2, p->E3, p->idx3, 0, 1, TILE, S, &err)) return fail(CUBA_ERR_INVALID, err);
	if (S.numP < 1) return fail(CUBA_ERR_INVALID, "pcg_partition: no free pose");
	const int G = std::max(1, std::min(nCtas, S.numP));
	PcgPartition P; CoarsePartition C;
	build_pcg_partition(S.numP, S.nfull, S.fRowPtr, S.fColInd, G, P);
	build_coarse_partition(S.numP, P, maxAgg, C);
	build_coarse_lists(S.numP, S.nfull, S.fRowPtr, S.fColInd, C);
	const char* bad = check_pcg_partition(S.numP, S.nfull, S.fRowPtr, S.fColInd, P, C);
	if (bad) return fail(CUBA_ERR_INVALID, std::string("pcg_partition self-check: ") + bad);
	if (info) { info[0] = P.G; info[1] = C.gs; info[2] = C.A; info[3] = P.needMax; info[4] = P.maxRows; info[5] = P.blkMax; info[6] = C.maxNeedAgg; info[7] = (int32_t)C.cbList.size(); }
	return CUBA_OK;
}

/* host side of the row-distributed PCG plan on the CPU (no device needed): info[8] = ok, G, gs, A, needMax, maxRows, maxNeedAgg,
 * number of rows some other rank needs (halo rows) */
int cuba_debug_pcg5_plan(const cuba_problem* p, int world, int numSMs, int maxAgg, int32_t* info)
{
	if (!p || world < 1 || world > 8 || numSMs < 1 || maxAgg < 1) return fail(CUBA_ERR_INVALID, "pcg5_plan: bad arguments");
	Structure S;
	const char* err = "";
	if (!build_structure(p->Pall, p->numP, p->Lall, p->numL, p->E2, p->idx2, p->E3, p->idx3, 0, 1, TILE, S, &err)) return fail(CUBA_ERR_INVALID, err);
	Pcg5Plan plan;
	build_pcg5_plan(S.numP, S.nfull, S.fRowPtr, S.fColInd, world, numSMs, maxAgg, 2 * PCG5_BLOCK / 6, plan);
	if (info) for (int i = 0; i < 8; i++) info[i] = 0;
	if (!plan.ok) return CUBA_OK;
	const char* bad = check_pcg5_plan(S.numP, S.nfull, S.fRowPtr, S.fColInd, plan);
	if (bad) return fail(CUBA_ERR_INVALID, std::string("pcg5_plan self-check: ") + bad);
	if (info) {
		int halo = 0;
		for (unsigned char m : plan.rowPeers) if (m) halo++;
		info[0] = 1; info[1] = plan.G; info[2] = plan.gs; info[3] = plan.A; info[4] = plan.P.needMax; info[5] = plan.P.maxRows; info[6] = plan.C.maxNeedAgg; info[7] = halo;
	}
	return CUBA_OK;
}

int cuba_bench_stage(cuba_engine* e, int stage, int reps, int flush, double lambda, double* ms) { ENGINE_OR_FAIL(e); return e->impl->bench_stage(stage, reps, flush, lambda, ms); }

}  // extern "C"
