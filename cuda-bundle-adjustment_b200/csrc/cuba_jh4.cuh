// cuba_jh4.cuh -- fourth generation of the Jacobian+Hessian landmark pass: WARP tiles.
//
// Replaces computeActiveErrorsKernel + constructQuadraticFormKernel (reference src/cuda_block_solver.cu:732-839)
// for the landmark-side outputs (Hpl, Hll, bl, chi2), like k_linearize_landmark in cuba_kernels.cuh.
//
// What the ncu source view of the third-generation pass (k_linearize_landmark3, since retired) showed (profiles/r01_ncu_jh3_*): 43 % of the samples sat in
// the per-landmark reduction loop through shared memory (branchy, 35 % of all instructions), 15 % in the
// cp.async issue code and 15 % at CTA barriers.  This kernel removes all three:
//   * the unit of work is a WARP tile: whole landmarks packed greedily into <= 32 edge slots (a landmark with
//     more than 32 edges is cut into pieces; the piece that finishes last adds the partial sums in piece order).  A
//     landmark never straddles two warps, so Hll/bl are a segmented warp-shuffle reduction -- no staging
//     array, no loop, no barrier;
//   * every warp is an independent persistent worker with its own two-stage shared-memory pipeline.  A tile's
//     edge data is ONE 1 408-byte record in HBM (built at structure time), fetched with one TMA bulk copy
//     (cp.async.bulk ... mbarrier::complete_tx); the tile's landmarks are a contiguous row range of Xw (second
//     bulk copy); its distinct poses (<= 32, listed at structure time) are staged with seven 16-byte cp.async
//     per pose.  No CTA-level barrier exists in the main loop;
//   * the Hpl blocks of a tile are staged over the (already consumed) pose area of the current stage and leave
//     with one TMA bulk store per tile.
// Everything is a fixed-order sum: bit-reproducible run to run.
#pragma once

#include "cuba_kernels.cuh"

namespace cuba_b200 {
namespace jh4 {

constexpr int WARPS = 4;         // warps per CTA (independent workers)
constexpr int CAP = 32;          // edge slots per warp tile
constexpr int PSTRIDE = 18;      // doubles per staged pose record (144 B: 16-byte granules, rows shifted by 4 banks)

// one warp tile of the landmark-major edge stream, padded to 32 slots (pad: il = -1)
struct alignas(16) Rec {
	double mx[CAP], my[CAP], mz[CAP], om[CAP];
	int ps[CAP];    // bit 31: stereo; bits 0..4: slot of the edge's pose in the tile's pose list
	int il[CAP];    // landmark index (absolute), -1 for padding slots
	int hl[CAP];    // Hpl block of the edge relative to the tile's first block, -1: no block (fixed pose / fixed landmark)
};
static_assert(sizeof(Rec) == 1408, "record layout");

// packed: nl (bits 0..7) | nd (8..15) | flags (24..31); flags bit 0: piece of a cut landmark.  nh: Hpl blocks of the tile.
// (all four words are read late in the kernel's iteration: the descriptor load two tiles ahead never blocks a register)
struct alignas(16) WTile { int l0; int h0; int packed; int nh; };

// Per-warp pipeline stage.  XW landmarks and PC distinct poses are staged; the (rare) rest of a tile is gathered from
// global memory.  After the inputs are in registers the whole stage is reused as Hpl staging (32 blocks x 144 B).
template <int XW, int PC>
struct alignas(16) StageT {
	Rec rec;
	double xw[XW * 4];
	double pose[PC * PSTRIDE];
	unsigned long long mbar;
	unsigned long long pad;
};
// (CTAs of 4 warps per SM, pipeline stages) -> landmark window, pose slots.  Shared memory per CTA = 4 * NST stages.
template <int MINB, int NST> struct Cfg;
template <> struct Cfg<4, 2> { static constexpr int XW = 32, PC = 32; };   // 7 056 B / stage
template <int MINB, int NST> using StageOf = StageT<Cfg<MINB, NST>::XW, Cfg<MINB, NST>::PC>;
static_assert(sizeof(StageOf<4, 2>) - 16 >= CAP * 144, "Hpl staging must fit the stage");

struct Args {
	const double* pose; const double* cam; const double* Xw;
	const Rec* rec; const WTile* tile; const int* tilePose;   // tilePose[t*32 + k]: k-th distinct pose of tile t
	const int* tilePieces;                                      // pieces of cut landmarks: (piece index << 16) | number of pieces
	int* pieceCount;                                            // arrival counters, one per tile (zero between launches)
	int ntiles, numL;
	double* Hpl; float* HplF;        // HplF != nullptr (kernel template HF): Hpl blocks in fp32, 20 floats (80 B) per block
	double* Hll; double* bl; double* bigPartial;  // bigPartial[t*12 ..]: partial sums of the pieces
	double* chiPartial;
	RobustParams rk;
};

__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count)
{
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned int bytes)
{
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned int parity)
{
	asm volatile(
		"{\n"
		".reg .pred p;\n"
		"WAIT_%=:\n"
		"mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
		"@p bra DONE_%=;\n"
		"bra WAIT_%=;\n"
		"DONE_%=:\n"
		"}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_load(void* smem, const void* gptr, unsigned int bytes, unsigned long long* bar)
{
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
		:: "r"(smem_u32(smem)), "l"(gptr), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// v += o where p (one predicated DADD; the select form costs two FSEL and two moves per value)
__device__ __forceinline__ void add_if(double& v, double o, int p)
{
	asm("{\n.reg .pred q;\nsetp.ne.b32 q, %2, 0;\n@q add.f64 %0, %0, %1;\n}" : "+d"(v) : "d"(o), "r"(p));
}

struct Desc { WTile ti; int pose; };    // descriptor of one tile as a lane holds it: the tile + the lane's entry of its pose list

__device__ __forceinline__ Desc load_desc(const Args& a, int t)
{
	Desc d;
	const int tc = t < a.ntiles ? t : a.ntiles - 1;     // clamped: never consumed past the end
	d.ti = a.tile[tc];
	d.pose = a.tilePose[32 * (size_t)tc + (threadIdx.x & 31)];
	return d;
}

template <int XW, int PC>
__device__ __forceinline__ void issue_loads(const Args& a, int t, const Desc& d, StageT<XW, PC>& st, int lane)
{
	int nl = d.ti.packed & 0xff, nd = (d.ti.packed >> 8) & 0xff;
	nl = nl < XW ? nl : XW; nd = nd < PC ? nd : PC;
	if (lane == 0) {
		const unsigned int xb = (unsigned int)nl * 32u;
		mbar_expect_tx(&st.mbar, (unsigned int)sizeof(Rec) + xb);
		bulk_load(&st.rec, a.rec + t, (unsigned int)sizeof(Rec), &st.mbar);
		if (xb) bulk_load(st.xw, a.Xw + 4 * (size_t)d.ti.l0, xb, &st.mbar);
	}
	if (lane < nd) {
		const double* ps = a.pose + 8 * (size_t)d.pose;
		const double* cs = a.cam + 8 * (size_t)d.pose;
		double* dst = st.pose + lane * PSTRIDE;
		cp_async16(dst, ps); cp_async16(dst + 2, ps + 2); cp_async16(dst + 4, ps + 4); cp_async16(dst + 6, ps + 6);
		cp_async16(dst + 8, cs); cp_async16(dst + 10, cs + 2); cp_async16(dst + 12, cs + 4);
	}
}

// DBG (diagnosis builds only, tools/jh4_dbg.sh): bit 0 skips the arithmetic, bit 1 the Hpl staging + bulk store,
// bit 2 the per-landmark reduction and the Hll/bl stores, bit 3 adds clock64 phase counters.  DBG == 0 is the product.
template <int MINB, int NST, int DBG = 0, bool HF = false>
__global__ void __launch_bounds__(WARPS * 32, MINB) k_linearize_landmark4(const Args a)
{
	typedef double T;
	typedef StageOf<MINB, NST> Stage;
	constexpr int XW = Cfg<MINB, NST>::XW, PC = Cfg<MINB, NST>::PC;
	constexpr int D = NST - 1;                                    // prefetch distance in tiles
	unsigned long long gt0 = 0, gt1 = 0, gt2 = 0;
	if (DBG & 8) asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt0));
	extern __shared__ __align__(16) unsigned char jh4_smem_raw[];
	__shared__ double s_red[WARPS];
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
	Stage* stg = reinterpret_cast<Stage*>(jh4_smem_raw) + NST * wid;
	const int GW = gridDim.x * WARPS;
	int t = blockIdx.x * WARPS + wid;

	if (lane == 0) {
#pragma unroll
		for (int s = 0; s < NST; s++) mbar_init(&stg[s].mbar, 1);
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
	}
	__syncwarp();

	// descriptor queue: q[0] = current tile, q[1..D-1] = issued, q[D] = the next one to issue
	Desc q[D + 1];
	if (a.ntiles > 0) {
#pragma unroll
		for (int k = 0; k <= D; k++) q[k] = load_desc(a, t + k * GW);
#pragma unroll
		for (int k = 0; k < D; k++) {
			if (t + k * GW < a.ntiles) issue_loads(a, t + k * GW, q[k], stg[k], lane);
			asm volatile("cp.async.commit_group;" ::: "memory");
		}
	}

	double chi = 0;
#define JH4_TICK(i) do { if (DBG & 8) { const long long _n = clock64(); tk[i] += _n - tlast; tlast = _n; } } while (0)
	long long tk[8] = { 0, 0, 0, 0, 0, 0, 0, 0 }, tlast = 0;
	if (DBG & 8) { tlast = clock64(); asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt1)); }
	int sidx = 0, par = 0;                 // stage of the current tile, parity of its mbarrier phase
	for (; t < a.ntiles; t += GW) {
		Stage& st = stg[sidx];
		const WTile cur = q[0].ti;
		const int poseCur = q[0].pose;
		// this tile's inputs have landed: own cp.async group, the bulk copies' mbarrier phase, other lanes' cp.async
		asm volatile("cp.async.wait_group %0;" :: "n"(D - 1) : "memory");
		JH4_TICK(0);
		mbar_wait(&st.mbar, (unsigned int)par);
		__syncwarp();
		JH4_TICK(1);

		const int psf = st.rec.ps[lane];
		const int il = st.rec.il[lane];
		const int hl = st.rec.hl[lane];
		const bool valid = il >= 0;
		const bool stereo = psf < 0;
		T qq[4], tt[3], c[5], X[3], m[3];
		T om = T(0);
		{
			const int slot = psf & 31;
			const int ipAbs = __shfl_sync(0xffffffffu, poseCur, slot);     // only the overflow path needs it
			if (PC >= CAP || slot < PC) {
				const T* sp = st.pose + slot * PSTRIDE;
				qq[0] = sp[0]; qq[1] = sp[1]; qq[2] = sp[2]; qq[3] = sp[3]; tt[0] = sp[4]; tt[1] = sp[5]; tt[2] = sp[6];
				c[0] = sp[8]; c[1] = sp[9]; c[2] = sp[10]; c[3] = sp[11]; c[4] = sp[12];
			} else load_pose(a.pose, a.cam, ipAbs, qq, tt, c);
			const int lloc = valid ? il - cur.l0 : 0;
			if (XW >= CAP || lloc < XW) { const T* sx = st.xw + 4 * lloc; X[0] = sx[0]; X[1] = sx[1]; X[2] = sx[2]; }
			else load_xw(a.Xw, il, X);
			m[0] = st.rec.mx[lane]; m[1] = st.rec.my[lane]; m[2] = st.rec.mz[lane];
			om = st.rec.om[lane];
		}
		__syncwarp();      // every lane holds its inputs: the stage may now be overwritten by Hpl blocks
		// descriptor D+1 tiles ahead.  Issued here, not at the top: cp.async.wait_group is a DEPBAR on the scoreboard the
		// compiler also gives to plain loads, so a load in flight at the top of the iteration would be waited for there.
		const Desc far = load_desc(a, t + (D + 1) * GW);
		JH4_TICK(2);

		T v[9];
#pragma unroll
		for (int i = 0; i < 9; i++) v[i] = T(0);
		if ((DBG & 1) && valid) {
			// no arithmetic: outputs are plain copies of the inputs
			chi += om;
			v[0] = qq[0]; v[1] = qq[1]; v[2] = tt[0]; v[3] = c[0]; v[4] = X[0]; v[5] = X[1]; v[6] = m[0]; v[7] = m[1];
			v[8] = m[2] + qq[2] + qq[3] + tt[1] + tt[2] + c[1] + c[2] + c[3] + c[4] + X[2];
			if (!(DBG & 2) && hl >= 0) {
				T* dst = reinterpret_cast<T*>(&st) + 18 * hl;
#pragma unroll
				for (int n = 0; n < 18; n += 2) st2(dst + n, v[n % 9], v[(n + 1) % 9]);
			}
		}
		if (!(DBG & 1) && valid) {
			T Xc[3], r[3];
			edge_residual(qq, tt, c, X, m, stereo, Xc, r);
			const T e2 = om * (r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
			T rho, drho;
			robust<T>(stereo ? a.rk.type[1] : a.rk.type[0], stereo ? a.rk.delta[1] : a.rk.delta[0], e2, rho, drho);
			chi += (double)rho;
			const T w = om * drho;
			if (il < a.numL) {
				T JP[3][6], JL[3][3];
				edge_jacobians(qq, c, Xc, stereo, JP, JL);
				T wJL[3][3], wr[3];
#pragma unroll
				for (int mm = 0; mm < 3; mm++) {
					wr[mm] = w * r[mm];
#pragma unroll
					for (int n = 0; n < 3; n++) wJL[mm][n] = w * JL[mm][n];
				}
				v[0] = JL[0][0] * wJL[0][0] + JL[1][0] * wJL[1][0] + JL[2][0] * wJL[2][0];
				v[1] = JL[0][0] * wJL[0][1] + JL[1][0] * wJL[1][1] + JL[2][0] * wJL[2][1];
				v[2] = JL[0][0] * wJL[0][2] + JL[1][0] * wJL[1][2] + JL[2][0] * wJL[2][2];
				v[3] = JL[0][1] * wJL[0][1] + JL[1][1] * wJL[1][1] + JL[2][1] * wJL[2][1];
				v[4] = JL[0][1] * wJL[0][2] + JL[1][1] * wJL[1][2] + JL[2][1] * wJL[2][2];
				v[5] = JL[0][2] * wJL[0][2] + JL[1][2] * wJL[1][2] + JL[2][2] * wJL[2][2];
				v[6] = JL[0][0] * wr[0] + JL[1][0] * wr[1] + JL[2][0] * wr[2];
				v[7] = JL[0][1] * wr[0] + JL[1][1] * wr[1] + JL[2][1] * wr[2];
				v[8] = JL[0][2] * wr[0] + JL[1][2] * wr[1] + JL[2][2] * wr[2];
				if (!(DBG & 2) && hl >= 0) {
					T* dst = reinterpret_cast<T*>(&st) + 18 * hl;
					float* dstF = reinterpret_cast<float*>(&st) + 20 * hl;      // mixed precision: 80-byte fp32 blocks
#pragma unroll
					for (int n = 0; n < 3; n++) {
#pragma unroll
						for (int l = 0; l < 6; l += 2) {
							const T h0 = JP[0][l] * wJL[0][n] + JP[1][l] * wJL[1][n] + JP[2][l] * wJL[2][n];
							const T h1 = JP[0][l + 1] * wJL[0][n] + JP[1][l + 1] * wJL[1][n] + JP[2][l + 1] * wJL[2][n];
							if constexpr (HF) *reinterpret_cast<float2*>(dstF + n * 6 + l) = make_float2((float)h0, (float)h1);
							else st2(dst + n * 6 + l, h0, h1);
						}
					}
					if constexpr (HF) *reinterpret_cast<float2*>(dstF + 18) = make_float2(0.f, 0.f);
				}
			}
		}
		// the tile's Hpl blocks: one bulk store
		JH4_TICK(3);
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
		__syncwarp();
		const int nh = cur.nh;
		if (!(DBG & 2) && lane == 0 && nh > 0) {
			if constexpr (HF) {
				float* gdst = a.HplF + 20 * (size_t)cur.h0;
				asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
					:: "l"(gdst), "r"(smem_u32(&st)), "r"((unsigned int)(nh * 20 * sizeof(float))) : "memory");
			} else {
				T* gdst = a.Hpl + 18 * (size_t)cur.h0;
				asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
					:: "l"(gdst), "r"(smem_u32(&st)), "r"((unsigned int)(nh * 18 * sizeof(T))) : "memory");
			}
		}
		if (lane == 0) asm volatile("cp.async.bulk.commit_group;" ::: "memory");
		JH4_TICK(4);

		// prefetch tile i+D into the stage tile i-1 used: its Hpl blocks (the bulk store before this one) must have left
		{
			int sn = sidx + D; sn = sn >= NST ? sn - NST : sn;
			if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
			__syncwarp();
			if (t + D * GW < a.ntiles) issue_loads(a, t + D * GW, q[D], stg[sn], lane);
			asm volatile("cp.async.commit_group;" ::: "memory");
		}
		JH4_TICK(5);

		// per-landmark sums: segmented suffix reduction over the (sorted) landmark index
		const int key = valid ? il : -1 - lane;      // padding slots never form a run
#pragma unroll
		for (int d = (DBG & 4) ? 32 : 1; d < 32; d <<= 1) {
			const int ko = __shfl_down_sync(0xffffffffu, key, d);
			const bool same = (lane + d < 32) && ko == key;
			if (!__any_sync(0xffffffffu, same)) break;      // no run of this tile is longer than d
			const T msk = same ? T(1) : T(0);                // masked add as one DFMA (a select costs two FSEL + moves per value)
#pragma unroll
			for (int i = 0; i < 9; i++) {
				const T o = __shfl_down_sync(0xffffffffu, v[i], d);
				v[i] = fma(o, msk, v[i]);
			}
		}
		const int kp = __shfl_up_sync(0xffffffffu, key, 1);
		const bool head = valid && il < a.numL && (lane == 0 || kp != key);
		if ((DBG & 4) && v[0] + v[1] + v[2] + v[3] + v[4] + v[5] + v[6] + v[7] + v[8] == 1.2345e300) a.chiPartial[0] = 1;
		if (!(DBG & 4) && head) {
			T* H; T* b;
			if ((cur.packed >> 24) & 1) { H = a.bigPartial + 12 * (size_t)t; b = H + 9; }
			else { H = a.Hll + 9 * (size_t)il; b = a.bl + 3 * (size_t)il; }
			H[0] = v[0]; H[1] = v[1]; H[2] = v[2];
			H[3] = v[1]; H[4] = v[3]; H[5] = v[4];
			H[6] = v[2]; H[7] = v[4]; H[8] = v[5];
			b[0] = v[6]; b[1] = v[7]; b[2] = v[8];
			if ((cur.packed >> 24) & 1) {
				// piece of a cut landmark (one run, so this is lane 0): the piece that arrives last adds all partial sums in
				// piece order -- fixed order whoever it is -- and re-arms the counter for the next launch
				const int pk = a.tilePieces[t], np = pk & 0xffff, first = t - (pk >> 16);
				__threadfence();
				if (atomicAdd(a.pieceCount + first, 1) == np - 1) {
					__threadfence();
					T s[12];
#pragma unroll
					for (int i = 0; i < 12; i++) s[i] = T(0);
					for (int k = 0; k < np; k++) {
						const T* pp = a.bigPartial + 12 * (size_t)(first + k);
#pragma unroll
						for (int i = 0; i < 12; i++) s[i] += __ldcg(pp + i);
					}
					T* Ho = a.Hll + 9 * (size_t)il; T* bo = a.bl + 3 * (size_t)il;
#pragma unroll
					for (int i = 0; i < 9; i++) Ho[i] = s[i];
#pragma unroll
					for (int i = 0; i < 3; i++) bo[i] = s[9 + i];
					a.pieceCount[first] = 0;
				}
			}
		}
		JH4_TICK(6);
#pragma unroll
		for (int k = 0; k < D; k++) q[k] = q[k + 1];
		q[D] = far;
		sidx = sidx + 1 == NST ? 0 : sidx + 1;
		par ^= (sidx == 0) ? 1 : 0;
		if (DBG & 8) { if (q[D].ti.l0 + q[D].pose == -12345) chi += 1; JH4_TICK(7); }
	}
	if (DBG & 8) asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt2));
	if ((DBG & 8) && lane == 0) {
		const int gw = blockIdx.x * WARPS + wid;
		double* g = a.bigPartial + 8 * (size_t)(gridDim.x * WARPS) + 3 * (size_t)gw;
		g[0] = (double)(gt0 & 0xffffffffffffull); g[1] = (double)(gt1 & 0xffffffffffffull); g[2] = (double)(gt2 & 0xffffffffffffull);
#pragma unroll
		for (int i = 0; i < 8; i++) a.bigPartial[8 * (size_t)gw + i] = (double)tk[i];
	}
	if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
	asm volatile("cp.async.wait_group 0;" ::: "memory");
	const double tot = block_sum(chi, s_red);
	if (threadIdx.x == 0) a.chiPartial[blockIdx.x] = tot;
}

// ---- structure: greedy packing of whole landmarks into warp tiles, fully parallel (binary lifting) ---------------
// lmPtr: run pointers of the shard's landmarks [lb, le) into the local edge stream; j below is l - lb, N = le - lb.

// next[j]: first landmark of the tile after the one that starts at j.  next[N] = N.
__global__ void k_next(const int* __restrict__ lmPtr, int lb, int N, int* next)
{
	const int j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j > N) return;
	if (j == N) { next[j] = N; return; }
	const int* p = lmPtr + lb;
	const int base = p[j];
	int lo = j, hi = (j + CAP < N) ? j + CAP : N;      // largest m in [j, min(N, j+CAP)] with p[m] - base <= CAP (<= CAP landmarks per tile)
	while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (p[mid] - base <= CAP) lo = mid; else hi = mid - 1; }
	next[j] = lo == j ? j + 1 : lo;
}

__global__ void k_lift(const int* __restrict__ in, int N, int* out)
{
	const int j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j > N) return;
	out[j] = in[in[j]];
}

// start[s] = next^s(0) for s in [0, N]; piece count of every step (0 past the end / for an edge-less tail)
__global__ void k_starts(const int* __restrict__ levels, int K, int N, const int* __restrict__ lmPtr, int lb, int* start, int* pieces, int* anyCut)
{
	const int s = blockIdx.x * blockDim.x + threadIdx.x;
	if (s > N) return;
	int j = 0;
	for (int k = 0; k < K && j < N; k++) if ((s >> k) & 1) j = levels[(size_t)k * (N + 1) + j];
	if ((s >> K) != 0) j = N;
	start[s] = j;
	int np = 0;
	if (j < N) {
		const int* p = lmPtr + lb;
		const int jn = levels[j];                      // level 0 = next
		const int cnt = p[jn] - p[j];
		np = cnt == 0 ? 0 : (cnt + CAP - 1) / CAP;    // a tile of several landmarks has cnt <= CAP -> 1
		if (np > 1) atomicMax(anyCut, 1);
	}
	pieces[s] = np;
}

// one warp per greedy step: fills the descriptors, the padded records and the pose lists of its warp tiles
__global__ void k_emit(const int* __restrict__ start, const int* __restrict__ pieces, const int* __restrict__ base, int N,
	const int* __restrict__ lmPtr, int lb, const int* __restrict__ next,
	const double* __restrict__ mx, const double* __restrict__ my, const double* __restrict__ mz, const double* __restrict__ om,
	const int* __restrict__ e_ip, const int* __restrict__ e_il, const int* __restrict__ e_hpl,
	WTile* tile, Rec* rec, int* tilePose, int* tilePieces)
{
	const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
	if (s >= N) return;
	const int np = pieces[s];
	if (np == 0) return;
	const int j = start[s], jn = next[j];
	const int* p = lmPtr + lb;
	const int e0 = p[j], e1 = p[jn];
	for (int k = 0; k < np; k++) {
		const int t = base[s] + k;
		const int b = e0 + k * CAP;
		const int cnt = (e1 - b) < CAP ? (e1 - b) : CAP;
		const int e = b + lane;
		const bool valid = lane < cnt;
		const int ipf = valid ? e_ip[e] : 0;
		const int ip = ipf & 0x7fffffff;
		const int il = valid ? e_il[e] : -1;
		const int hp = valid ? e_hpl[e] : -1;
		// distinct poses of the tile in lane order
		const unsigned int vm = __ballot_sync(0xffffffffu, valid);
		unsigned int same = 0;
		if (valid) same = __match_any_sync(vm, ip);
		const bool leader = valid && (__ffs(same) - 1) == lane;
		const unsigned int lm = __ballot_sync(0xffffffffu, leader);
		int slot = 0;
		if (valid) slot = __popc(lm & ((1u << (__ffs(same) - 1)) - 1u));
		if (leader) tilePose[32 * (size_t)t + slot] = ip;
		const int nd = __popc(lm);
		if (lane >= nd) tilePose[32 * (size_t)t + lane] = 0;
		// Hpl blocks of the tile: consecutive ranks
		const unsigned int hm = __ballot_sync(0xffffffffu, hp >= 0);
		const int first = e_hpl[b];
		const int h0 = first >= 0 ? first : -1 - first;
		Rec& r = rec[t];
		r.mx[lane] = valid ? mx[e] : 0.0; r.my[lane] = valid ? my[e] : 0.0; r.mz[lane] = valid ? mz[e] : 0.0; r.om[lane] = valid ? om[e] : 0.0;
		r.ps[lane] = (ipf & (int)0x80000000u) | slot;
		r.il[lane] = il;
		r.hl[lane] = hp >= 0 ? hp - h0 : -1;
		if (lane == 0) {
			WTile ti;
			ti.l0 = lb + j;
			ti.h0 = h0;
			const int nl = np > 1 ? 1 : jn - j;
			ti.packed = nl | (nd << 8) | ((np > 1 ? 1 : 0) << 24);
			ti.nh = __popc(hm);
			tile[t] = ti;
			tilePieces[t] = np > 1 ? ((k << 16) | np) : 0;
		}
	}
}

}  // namespace jh4
}  // namespace cuba_b200
