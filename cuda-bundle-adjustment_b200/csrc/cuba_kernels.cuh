// cuba_kernels.cuh -- sm_100a kernels of the LM inner loop (templated on the scalar type).
//
// Data layout in HBM (DESIGN.md section 3):
//   pose  [Pall][8]  q(x,y,z,w) t(x,y,z) pad      cam [Pall][8] fx fy cx cy bf pad pad pad
//   Xw    [Lall][4]  X Y Z pad
//   landmark-major edge stream (sorted by (iL,iP)), SoA: mx,my,mz,om (T), ip (bit31 = stereo), il, hpl
//   pose-major edge stream (sorted by (iP,iL), free poses only), SoA: mx,my,mz,om (T), il (bit31 = stereo)
//   Hpp [numP][36] bp [numP][6] Hll [numL][9] bl [numL][3] Hpl [nhpl][18]   (blocks column-major)
//   Hsc: symmetric-full BSR (fRowPtr,fColInd,fVal[nfull][36]) for the PCG; upper view for parity.
#pragma once

#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "cuba_math.cuh"

namespace cuba_b200 {

constexpr int TILE = 256;        // tile bound of the host structure builder in the cuba_debug_* entry points
// Landmark tiles of the J+H landmark pass and the back-substitution: CTAs of LM_TILE edges, cut by the structure builder into
// windows of LM_WINDOW edges so that the tail of a tile's last landmark usually still fits the same chunk.  Changing either
// regroups the per-tile sums (Hll/bl, chi2 partials, back-substitution) and so changes the results in the last bits.
constexpr int LM_TILE = 128;
constexpr int LM_WINDOW = 112;

constexpr int POSE_BLOCK = 128;  // threads per CTA of the pose pass
constexpr int RED_BLOCK = 256;

template <typename T> struct V2;
template <> struct V2<double> { using type = double2; };
template <> struct V2<float> { using type = float2; };

template <typename T>
__device__ __forceinline__ void ld2(const T* __restrict__ p, T& a, T& b)
{
	const typename V2<T>::type v = __ldg(reinterpret_cast<const typename V2<T>::type*>(p));
	a = v.x; b = v.y;
}
template <typename T>
__device__ __forceinline__ void st2(T* p, T a, T b)
{
	typename V2<T>::type v; v.x = a; v.y = b;
	*reinterpret_cast<typename V2<T>::type*>(p) = v;
}

template <typename T>
__device__ __forceinline__ void load_pose(const T* __restrict__ pose, const T* __restrict__ cam, int ip, T q[4], T t[3], T c[5])
{
	const T* p = pose + 8 * (size_t)ip;
	T pad;
	ld2(p, q[0], q[1]); ld2(p + 2, q[2], q[3]); ld2(p + 4, t[0], t[1]); ld2(p + 6, t[2], pad);
	const T* k = cam + 8 * (size_t)ip;
	ld2(k, c[0], c[1]); ld2(k + 2, c[2], c[3]); ld2(k + 4, c[4], pad);
}

template <typename T>
__device__ __forceinline__ void load_xw(const T* __restrict__ Xw, int il, T X[3])
{
	T pad;
	ld2(Xw + 4 * (size_t)il, X[0], X[1]); ld2(Xw + 4 * (size_t)il + 2, X[2], pad);
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
	return v;
}
__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
	return v;
}

// deterministic block sum (fixed tree); result valid in thread 0. s_red must hold blockDim/32 doubles.
__device__ __forceinline__ double block_sum(double v, double* s_red)
{
	v = warp_sum(v);
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
	if (lane == 0) s_red[wid] = v;
	__syncthreads();
	double r = 0;
	if (threadIdx.x == 0) for (int i = 0; i < (int)(blockDim.x >> 5); i++) r += s_red[i];
	__syncthreads();
	return r;
}

struct RobustParams { int type[2]; double delta[2]; };

// ------------------------------------------------------------------------------------------------
// Landmark pass of the Jacobian+Hessian stage: one CTA per tile of whole landmarks (<= TILE edges,
// or one giant landmark).  Thread per edge: residual, robust weight, JP/JL, Hpl block (global store),
// Hll/bl contributions staged in shared memory and summed per landmark run -- no atomics.
// Also emits the robustified chi2 partial of the tile.
// Replaces computeActiveErrorsKernel + constructQuadraticFormKernel (reference cu:732-839) for the
// landmark-side outputs.
// ------------------------------------------------------------------------------------------------
template <typename T>
struct LinLmArgs {
	const T* pose; const T* cam; const T* Xw;
	const T* mx; const T* my; const T* mz; const T* om;
	const int* ip; const int* il; const int* hpl;
	const int* lmPtr; const int* tileLm;
	int numP, numL;
	T* Hpl; T* Hll; T* bl;
	double* chiPartial;
	RobustParams rk;
};

template <typename T, int TL, int MINB>
__global__ void __launch_bounds__(TL, MINB) k_linearize_landmark(const LinLmArgs<T> a)
{
	__shared__ T s_val[9][TL + 1];
	__shared__ T s_acc[TL * 9];
	__shared__ int s_ptr[TL + 1];
	__shared__ double s_red[TL / 32];

	const int tid = threadIdx.x;
	const int l0 = a.tileLm[blockIdx.x], l1 = a.tileLm[blockIdx.x + 1];
	const int nl = l1 - l0;
	for (int i = tid; i <= nl; i += TL) s_ptr[i] = a.lmPtr[l0 + i];
	for (int i = tid; i < nl * 9; i += TL) s_acc[i] = T(0);
	__syncthreads();
	const int e0 = s_ptr[0], e1 = s_ptr[nl];

	double chi = 0;
	for (int cs = e0; cs < e1; cs += TL) {
		const int e = cs + tid;
		T v[9];
#pragma unroll
		for (int i = 0; i < 9; i++) v[i] = T(0);
		if (e < e1) {
			const int ipf = a.ip[e];
			const bool stereo = ipf < 0;
			const int ip = ipf & 0x7fffffff;
			const int il = a.il[e];
			T q[4], t[3], c[5], X[3], m[3], Xc[3], r[3];
			load_pose(a.pose, a.cam, ip, q, t, c);
			load_xw(a.Xw, il, X);
			m[0] = a.mx[e]; m[1] = a.my[e]; m[2] = stereo ? a.mz[e] : T(0);
			const T om = a.om[e];
			edge_residual(q, t, c, X, m, stereo, Xc, r);
			const T e2 = om * (r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
			T rho, drho;
			robust<T>(a.rk.type[stereo ? 1 : 0], (T)a.rk.delta[stereo ? 1 : 0], e2, rho, drho);
			chi += (double)rho;
			const T w = om * drho;
			if (il < a.numL) {
				T JP[3][6], JL[3][3];
				edge_jacobians(q, c, Xc, stereo, JP, JL);
				T wJL[3][3], wr[3];
#pragma unroll
				for (int mm = 0; mm < 3; mm++) {
					wr[mm] = w * r[mm];
#pragma unroll
					for (int n = 0; n < 3; n++) wJL[mm][n] = w * JL[mm][n];
				}
				// unique Hll entries 00,01,02,11,12,22 then bl
				v[0] = JL[0][0] * wJL[0][0] + JL[1][0] * wJL[1][0] + JL[2][0] * wJL[2][0];
				v[1] = JL[0][0] * wJL[0][1] + JL[1][0] * wJL[1][1] + JL[2][0] * wJL[2][1];
				v[2] = JL[0][0] * wJL[0][2] + JL[1][0] * wJL[1][2] + JL[2][0] * wJL[2][2];
				v[3] = JL[0][1] * wJL[0][1] + JL[1][1] * wJL[1][1] + JL[2][1] * wJL[2][1];
				v[4] = JL[0][1] * wJL[0][2] + JL[1][1] * wJL[1][2] + JL[2][1] * wJL[2][2];
				v[5] = JL[0][2] * wJL[0][2] + JL[1][2] * wJL[1][2] + JL[2][2] * wJL[2][2];
				v[6] = JL[0][0] * wr[0] + JL[1][0] * wr[1] + JL[2][0] * wr[2];
				v[7] = JL[0][1] * wr[0] + JL[1][1] * wr[1] + JL[2][1] * wr[2];
				v[8] = JL[0][2] * wr[0] + JL[1][2] * wr[1] + JL[2][2] * wr[2];
				const int hp = a.hpl[e];
				if (hp >= 0) {
					T* dst = a.Hpl + 18 * (size_t)hp;
#pragma unroll
					for (int n = 0; n < 3; n++) {
#pragma unroll
						for (int l = 0; l < 6; l += 2) {
							const T h0 = JP[0][l] * wJL[0][n] + JP[1][l] * wJL[1][n] + JP[2][l] * wJL[2][n];
							const T h1 = JP[0][l + 1] * wJL[0][n] + JP[1][l + 1] * wJL[1][n] + JP[2][l + 1] * wJL[2][n];
							st2(dst + n * 6 + l, h0, h1);
						}
					}
				}
			}
		}
#pragma unroll
		for (int i = 0; i < 9; i++) s_val[i][tid] = v[i];
		__syncthreads();
		for (int wi = tid; wi < nl * 9; wi += TL) {
			const int j = wi / 9, cc = wi - 9 * j;
			int s = s_ptr[j], t = s_ptr[j + 1];
			s = (s > cs ? s : cs) - cs;
			t = (t < cs + TL ? t : cs + TL) - cs;
			if (t > s) {
				T sum = T(0);
				for (int k = s; k < t; k++) sum += s_val[cc][k];
				s_acc[wi] += sum;
			}
		}
		__syncthreads();
	}
	// write Hll (full symmetric 3x3, column-major) and bl of the tile's free landmarks, coalesced
	{
		const int map9[9] = { 0, 1, 2, 1, 3, 4, 2, 4, 5 };
		for (int wi = tid; wi < nl * 9; wi += TL) {
			const int j = wi / 9, cc = wi - 9 * j;
			if (l0 + j < a.numL) a.Hll[9 * (size_t)l0 + wi] = s_acc[j * 9 + map9[cc]];
		}
		for (int wi = tid; wi < nl * 3; wi += TL) {
			const int j = wi / 3, cc = wi - 3 * j;
			if (l0 + j < a.numL) a.bl[3 * (size_t)l0 + wi] = s_acc[j * 9 + 6 + cc];
		}
	}
	const double tot = block_sum(chi, s_red);
	if (tid == 0) a.chiPartial[blockIdx.x] = tot;
}

__device__ __forceinline__ unsigned int smem_u32(const void* p) { return (unsigned int)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void cp_async16(void* smem, const void* gptr)
{
	asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(smem_u32(smem)), "l"(gptr) : "memory");
}

// ------------------------------------------------------------------------------------------------
// Pose pass of the Jacobian+Hessian stage: one CTA per free pose over its pose-major edge list.
// Each thread accumulates the 21 upper entries of JP^T w JP and the 6 of JP^T w r in registers;
// one fixed-order block reduction per pose -- no atomics.  (reference cu:815-824)
// ------------------------------------------------------------------------------------------------
template <typename T>
struct LinPoseArgs {
	const T* pose; const T* cam; const T* Xw;
	const T* mx; const T* my; const T* mz; const T* om; const int* il;
	const int* posePtr;
	T* Hpp; T* bp;
	RobustParams rk;
};

template <typename T>
__global__ void __launch_bounds__(POSE_BLOCK) k_linearize_pose(const LinPoseArgs<T> a)
{
	__shared__ T s_part[POSE_BLOCK / 32][27];
	__shared__ T s_fin[27];
	const int p = blockIdx.x, tid = threadIdx.x;
	const int e0 = a.posePtr[p], e1 = a.posePtr[p + 1];
	T q[4], t[3], c[5];
	load_pose(a.pose, a.cam, p, q, t, c);
	T acc[27];
#pragma unroll
	for (int i = 0; i < 27; i++) acc[i] = T(0);
	// software pipeline: the inputs of the thread's next edge (stream entries, then the gathered landmark) are in flight
	// while the current edge is computed -- the gather through il is a dependent L2 access
	int e = e0 + tid;
	int ilfN = 0; T XN[3] = { T(0), T(0), T(0) }, mN[3] = { T(0), T(0), T(0) }, omN = T(0);
	if (e < e1) {
		ilfN = a.il[e]; mN[0] = a.mx[e]; mN[1] = a.my[e]; mN[2] = ilfN < 0 ? a.mz[e] : T(0); omN = a.om[e];
		load_xw(a.Xw, ilfN & 0x7fffffff, XN);
	}
	for (; e < e1; e += POSE_BLOCK) {
		const int ilf = ilfN;
		const bool stereo = ilf < 0;
		T X[3], m[3], Xc[3], r[3];
#pragma unroll
		for (int i = 0; i < 3; i++) { X[i] = XN[i]; m[i] = mN[i]; }
		const T om = omN;
		const int en = e + POSE_BLOCK;
		if (en < e1) {
			ilfN = a.il[en]; mN[0] = a.mx[en]; mN[1] = a.my[en]; mN[2] = ilfN < 0 ? a.mz[en] : T(0); omN = a.om[en];
			load_xw(a.Xw, ilfN & 0x7fffffff, XN);
		}
		edge_residual(q, t, c, X, m, stereo, Xc, r);
		const T e2 = om * (r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
		T rho, drho;
		robust<T>(stereo ? a.rk.type[1] : a.rk.type[0], (T)(stereo ? a.rk.delta[1] : a.rk.delta[0]), e2, rho, drho);
		const T w = om * drho;
		T JP[3][6], JL[3][3];
		edge_jacobians(q, c, Xc, stereo, JP, JL);
		T wJP[3][6];
#pragma unroll
		for (int mm = 0; mm < 3; mm++)
#pragma unroll
			for (int l = 0; l < 6; l++) wJP[mm][l] = w * JP[mm][l];
		int k = 0;
#pragma unroll
		for (int n = 0; n < 6; n++)
#pragma unroll
			for (int l = 0; l <= n; l++) {
				acc[k] += JP[0][l] * wJP[0][n] + JP[1][l] * wJP[1][n] + JP[2][l] * wJP[2][n];
				k++;
			}
#pragma unroll
		for (int l = 0; l < 6; l++) acc[21 + l] += wJP[0][l] * r[0] + wJP[1][l] * r[1] + wJP[2][l] * r[2];
	}
	const int lane = tid & 31, wid = tid >> 5;
#pragma unroll
	for (int i = 0; i < 27; i++) {
		const T s = warp_sum(acc[i]);
		if (lane == 0) s_part[wid][i] = s;
	}
	__syncthreads();
	if (tid < 27) {
		T s = T(0);
#pragma unroll
		for (int w = 0; w < POSE_BLOCK / 32; w++) s += s_part[w][tid];
		s_fin[tid] = s;
	}
	__syncthreads();
	if (tid < 36) {
		const int n = tid / 6, l = tid - 6 * n;   // column n, row l
		const int lo = l < n ? l : n, hi = l < n ? n : l;
		a.Hpp[36 * (size_t)p + tid] = s_fin[hi * (hi + 1) / 2 + lo];
	} else if (tid < 42) {
		a.bp[6 * (size_t)p + (tid - 36)] = s_fin[21 + (tid - 36)];
	}
}

// max over the diagonals of Hpp and Hll, starting from 0 (reference cu:877-904).
template <typename T>
__global__ void k_max_diagonal(const T* Hpp, int numP, const T* Hll, int numL, unsigned long long* out)
{
	double m = 0;
	const int n1 = numP * 6, n2 = numL * 3;
	for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n1 + n2; i += gridDim.x * blockDim.x) {
		double v;
		if (i < n1) { const int j = i / 6, k = i - 6 * j; v = (double)Hpp[36 * (size_t)j + 7 * k]; }
		else { const int ii = i - n1; const int j = ii / 3, k = ii - 3 * j; v = (double)Hll[9 * (size_t)j + 4 * k]; }
		m = v > m ? v : m;
	}
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) { const double x = __shfl_xor_sync(0xffffffffu, m, o); m = x > m ? x : m; }
	if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(out, (unsigned long long)__double_as_longlong(m));
}

// invHll = (Hll + lambda I)^-1, closed form (reference cu:417-452, 941-942)
template <typename T>
__global__ void k_inv_hll(const T* __restrict__ Hll, int numL, T lambda, T* __restrict__ invHll)
{
	const int l = blockIdx.x * blockDim.x + threadIdx.x;
	if (l >= numL) return;
	const T* H = Hll + 9 * (size_t)l;
	T B[6];
	sym3_inverse<T>(H[0] + lambda, H[3], H[6], H[4] + lambda, H[7], H[8] + lambda, B);
	T* o = invHll + 9 * (size_t)l;
	o[0] = B[0]; o[1] = B[1]; o[2] = B[2];
	o[3] = B[1]; o[4] = B[3]; o[5] = B[4];
	o[6] = B[2]; o[7] = B[4]; o[8] = B[5];
}

// result of every PCG kernel (cuba_pcg2/3/4/5/5t.cuh)
struct PcgStatus { int iters; int status; double rz0; double rz; };  // status: 0 converged, 1 max iters, 2 breakdown

// ------------------------------------------------------------------------------------------------
// Back-substitution + landmark update + landmark part of the LM scale, landmark tiles again:
//   xl = invHll (bl - sum_i Hpl_i^T xp[row_i]) ; Xw_trial = Xw + xl ; scale += xl.(lambda xl + bl)
// (reference cu:1029-1043, 1057-1068, 1070-1091)
// ------------------------------------------------------------------------------------------------
// Mixed precision (SURVEY.md 8 f-4): an fp64 engine may keep the Hpl blocks -- the dominant 144 B/edge stream, written once by the
// J+H pass and read by the Schur and back-substitution kernels -- in fp32, 18 values padded to 20 (80-byte blocks: a multiple
// of the 16-byte granule of the bulk store).  Everything is still computed and accumulated in fp64.
template <typename T, typename TH> struct HplStride { static constexpr int value = sizeof(TH) < sizeof(T) ? 20 : 18; };
template <typename T, typename TH>
__device__ __forceinline__ void ldh2(const TH* __restrict__ p, T& a, T& b)
{
	if constexpr (sizeof(TH) == sizeof(T)) ld2(p, a, b);
	else { const float2 v = __ldg(reinterpret_cast<const float2*>(p)); a = (T)v.x; b = (T)v.y; }
}
template <typename T, typename TH>
__device__ __forceinline__ T ldh(const TH* __restrict__ p) { return (T)__ldg(p); }

template <typename T, typename TH = T>
struct BacksubArgs {
	const TH* Hpl; const T* invHll; const T* bl; const T* xp;
	const int* ip; const int* hpl; const int* lmPtr; const int* tileLm;
	int numL;
	T lambda;
	const T* XwCur; T* XwTrial; T* xl;
	double* scalePartial;
};

template <typename T, int TL, typename TH = T>
__global__ void __launch_bounds__(TL) k_backsub(const BacksubArgs<T, TH> a)
{
	__shared__ T s_val[3][TL + 1];
	__shared__ T s_acc[TL * 3];
	__shared__ int s_ptr[TL + 1];
	__shared__ double s_red[TL / 32];
	const int tid = threadIdx.x;
	const int l0 = a.tileLm[blockIdx.x], l1 = a.tileLm[blockIdx.x + 1];
	const int nl = l1 - l0;
	double sc = 0;
	if (l0 < a.numL) {   // tiles of fixed landmarks have nothing to solve (uniform branch)
		for (int i = tid; i <= nl; i += TL) s_ptr[i] = a.lmPtr[l0 + i];
		for (int i = tid; i < nl * 3; i += TL) s_acc[i] = T(0);
		__syncthreads();
		const int e0 = s_ptr[0], e1 = s_ptr[nl];
		for (int cs = e0; cs < e1; cs += TL) {
			const int e = cs + tid;
			T v0 = T(0), v1 = T(0), v2 = T(0);
			if (e < e1) {
				const int hp = a.hpl[e];
				if (hp >= 0) {
					const int ip = a.ip[e] & 0x7fffffff;
					const TH* A = a.Hpl + HplStride<T, TH>::value * (size_t)hp;
					const T* x = a.xp + 6 * (size_t)ip;
					T xr[6];
					ld2(x, xr[0], xr[1]); ld2(x + 2, xr[2], xr[3]); ld2(x + 4, xr[4], xr[5]);
					T A0[6], A1[6], A2[6];
#pragma unroll
					for (int r = 0; r < 6; r += 2) { ldh2<T, TH>(A + r, A0[r], A0[r + 1]); ldh2<T, TH>(A + 6 + r, A1[r], A1[r + 1]); ldh2<T, TH>(A + 12 + r, A2[r], A2[r + 1]); }
#pragma unroll
					for (int r = 0; r < 6; r++) { v0 += A0[r] * xr[r]; v1 += A1[r] * xr[r]; v2 += A2[r] * xr[r]; }
				}
			}
			s_val[0][tid] = v0; s_val[1][tid] = v1; s_val[2][tid] = v2;
			__syncthreads();
			for (int wi = tid; wi < nl * 3; wi += TL) {
				const int j = wi / 3, cc = wi - 3 * j;
				int s = s_ptr[j], t = s_ptr[j + 1];
				s = (s > cs ? s : cs) - cs;
				t = (t < cs + TL ? t : cs + TL) - cs;
				if (t > s) {
					T sum = T(0);
					for (int k = s; k < t; k++) sum += s_val[cc][k];
					s_acc[wi] += sum;
				}
			}
			__syncthreads();
		}
		for (int j = tid; j < nl; j += TL) {
			const int l = l0 + j;
			if (l < a.numL) {
				const T* bl = a.bl + 3 * (size_t)l;
				const T c0 = bl[0] - s_acc[3 * j], c1 = bl[1] - s_acc[3 * j + 1], c2 = bl[2] - s_acc[3 * j + 2];
				const T* iv = a.invHll + 9 * (size_t)l;
				const T x0 = iv[0] * c0 + iv[3] * c1 + iv[6] * c2;
				const T x1 = iv[1] * c0 + iv[4] * c1 + iv[7] * c2;
				const T x2 = iv[2] * c0 + iv[5] * c1 + iv[8] * c2;
				a.xl[3 * (size_t)l] = x0; a.xl[3 * (size_t)l + 1] = x1; a.xl[3 * (size_t)l + 2] = x2;
				const T* X = a.XwCur + 4 * (size_t)l;
				T* Y = a.XwTrial + 4 * (size_t)l;
				Y[0] = X[0] + x0; Y[1] = X[1] + x1; Y[2] = X[2] + x2; Y[3] = T(0);
				sc += (double)(x0 * (a.lambda * x0 + bl[0]) + x1 * (a.lambda * x1 + bl[1]) + x2 * (a.lambda * x2 + bl[2]));
			}
		}
	}
	const double tot = block_sum(sc, s_red);
	if (tid == 0) a.scalePartial[blockIdx.x] = tot;
}

// landmark-only BA (no free pose): xl = (Hll + lambda I)^-1 bl  (reference cu:1124-1131)
template <typename T>
__global__ void k_solve_landmarks_only(const T* invHll, const T* bl, int numL, T lambda, const T* XwCur, T* XwTrial, T* xl, double* scalePartial)
{
	__shared__ double s_red[RED_BLOCK / 32];
	const int l = blockIdx.x * blockDim.x + threadIdx.x;
	double sc = 0;
	if (l < numL) {
		const T* iv = invHll + 9 * (size_t)l; const T* b = bl + 3 * (size_t)l;
		const T x0 = iv[0] * b[0] + iv[3] * b[1] + iv[6] * b[2];
		const T x1 = iv[1] * b[0] + iv[4] * b[1] + iv[7] * b[2];
		const T x2 = iv[2] * b[0] + iv[5] * b[1] + iv[8] * b[2];
		xl[3 * (size_t)l] = x0; xl[3 * (size_t)l + 1] = x1; xl[3 * (size_t)l + 2] = x2;
		const T* X = XwCur + 4 * (size_t)l; T* Y = XwTrial + 4 * (size_t)l;
		Y[0] = X[0] + x0; Y[1] = X[1] + x1; Y[2] = X[2] + x2; Y[3] = T(0);
		sc = (double)(x0 * (lambda * x0 + b[0]) + x1 * (lambda * x1 + b[1]) + x2 * (lambda * x2 + b[2]));
	}
	const double tot = block_sum(sc, s_red);
	if (threadIdx.x == 0) scalePartial[blockIdx.x] = tot;
}

// pose-only BA (no free landmark): xp = (Hpp + lambda I)^-1 bp  (reference cu:1133-1140 solves the
// 6x6 by a 3+3 Schur split; we use the Cholesky inverse -- same solution up to rounding)
template <typename T>
__global__ void k_solve_poses_only(const T* Hpp, const T* bp, int numP, T lambda, T* xp)
{
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	if (p >= numP) return;
	T M[36];
	for (int e = 0; e < 36; e++) M[e] = Hpp[36 * (size_t)p + e] + ((e % 7) == 0 ? lambda : T(0));
	if (!spd6_inverse(M)) { for (int e = 0; e < 6; e++) xp[6 * (size_t)p + e] = T(0); return; }
	for (int r = 0; r < 6; r++) {
		T s = T(0);
		for (int c = 0; c < 6; c++) s += M[c * 6 + r] * bp[6 * (size_t)p + c];
		xp[6 * (size_t)p + r] = s;
	}
}

// SE(3) update of the free poses into the trial buffer + pose part of the LM scale (cu:1045-1055,1070-1091)
template <typename T>
__global__ void k_update_poses(const T* xp, const T* bp, int numP, T lambda, const T* poseCur, T* poseTrial, double* scalePartial)
{
	__shared__ double s_red[RED_BLOCK / 32];
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	double sc = 0;
	if (p < numP) {
		T u[6], q[4], t[3];
		for (int i = 0; i < 6; i++) u[i] = xp[6 * (size_t)p + i];
		const T* s = poseCur + 8 * (size_t)p;
		for (int i = 0; i < 4; i++) q[i] = s[i];
		for (int i = 0; i < 3; i++) t[i] = s[4 + i];
		se3_update(u, q, t);
		T* d = poseTrial + 8 * (size_t)p;
		for (int i = 0; i < 4; i++) d[i] = q[i];
		for (int i = 0; i < 3; i++) d[4 + i] = t[i];
		d[7] = T(0);
		T acc = T(0);
		for (int i = 0; i < 6; i++) acc += u[i] * (lambda * u[i] + bp[6 * (size_t)p + i]);
		sc = (double)acc;
	}
	const double tot = block_sum(sc, s_red);
	if (threadIdx.x == 0) scalePartial[blockIdx.x] = tot;
}

// Residual-only pass: robustified chi2 of a state (trial evaluation) -- reference cu:732-786 without
// the errors/Xcs side outputs.  Grid-stride over the landmark-major edge stream, block partials.
template <typename T>
struct ChiArgs {
	const T* pose; const T* cam; const T* Xw;
	const T* mx; const T* my; const T* mz; const T* om; const int* ip; const int* il;
	int E;
	RobustParams rk;
	double* chiPartial;
};

template <typename T>
__global__ void __launch_bounds__(RED_BLOCK) k_chi2(const ChiArgs<T> a)
{
	__shared__ double s_red[RED_BLOCK / 32];
	double chi = 0;
	for (int e = blockIdx.x * RED_BLOCK + threadIdx.x; e < a.E; e += gridDim.x * RED_BLOCK) {
		const int ipf = a.ip[e];
		const bool stereo = ipf < 0;
		T q[4], t[3], c[5], X[3], m[3], Xc[3], r[3];
		load_pose(a.pose, a.cam, ipf & 0x7fffffff, q, t, c);
		load_xw(a.Xw, a.il[e], X);
		m[0] = a.mx[e]; m[1] = a.my[e]; m[2] = stereo ? a.mz[e] : T(0);
		edge_residual(q, t, c, X, m, stereo, Xc, r);
		const T e2 = a.om[e] * (r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
		T rho, drho;
		robust<T>(a.rk.type[stereo ? 1 : 0], (T)a.rk.delta[stereo ? 1 : 0], e2, rho, drho);
		chi += (double)rho;
	}
	const double tot = block_sum(chi, s_red);
	if (threadIdx.x == 0) a.chiPartial[blockIdx.x] = tot;
}

// per-edge non-robust omega*|r|^2 in edge-id order (reference cu:841-875)
template <typename T>
__global__ void k_chi_sqs(const ChiArgs<T> a, const int* userId, double* out)
{
	const int e = blockIdx.x * blockDim.x + threadIdx.x;
	if (e >= a.E) return;
	const int ipf = a.ip[e];
	const bool stereo = ipf < 0;
	T q[4], t[3], c[5], X[3], m[3], Xc[3], r[3];
	load_pose(a.pose, a.cam, ipf & 0x7fffffff, q, t, c);
	load_xw(a.Xw, a.il[e], X);
	m[0] = a.mx[e]; m[1] = a.my[e]; m[2] = stereo ? a.mz[e] : T(0);
	edge_residual(q, t, c, X, m, stereo, Xc, r);
	out[userId[e]] = (double)(a.om[e] * (r[0] * r[0] + r[1] * r[1] + r[2] * r[2]));
}

// Fixed-order sum of up to three partial arrays into out[0..2] (single CTA).
__global__ void __launch_bounds__(RED_BLOCK) k_sum_partials(const double* p0, int n0, const double* p1, int n1, const double* p2, int n2, double* out)
{
	__shared__ double s_red[RED_BLOCK / 32];
	const double* ps[3] = { p0, p1, p2 };
	const int ns[3] = { n0, n1, n2 };
	for (int k = 0; k < 3; k++) {
		double s = 0;
		for (int i = threadIdx.x; i < ns[k]; i += RED_BLOCK) s += ps[k][i];
		const double tot = block_sum(s, s_red);
		if (threadIdx.x == 0) out[k] = tot;
	}
}

// L2 flush helper for the micro-benchmarks: overwrite a buffer larger than L2.
// flat fp64 state of the caller -> padded records of the engine's scalar type (initial copy + both working buffers)
template <typename T>
__global__ void k_pack_state(const double* __restrict__ q, const double* __restrict__ t, const double* __restrict__ c, const double* __restrict__ X,
	int Pall, int Lall, T* pose0, T* poseA, T* poseB, T* cam, T* Xw0, T* XwA, T* XwB)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < Pall) {
		T r[8];
		for (int k = 0; k < 4; k++) r[k] = (T)q[4 * (size_t)i + k];
		for (int k = 0; k < 3; k++) r[4 + k] = (T)t[3 * (size_t)i + k];
		r[7] = T(0);
		for (int k = 0; k < 8; k++) { pose0[8 * (size_t)i + k] = r[k]; poseA[8 * (size_t)i + k] = r[k]; poseB[8 * (size_t)i + k] = r[k]; }
		if (cam) {
			for (int k = 0; k < 5; k++) cam[8 * (size_t)i + k] = (T)c[5 * (size_t)i + k];
			for (int k = 5; k < 8; k++) cam[8 * (size_t)i + k] = T(0);
		}
	}
	if (i < Lall) {
		T r[4];
		for (int k = 0; k < 3; k++) r[k] = (T)X[3 * (size_t)i + k];
		r[3] = T(0);
		for (int k = 0; k < 4; k++) { Xw0[4 * (size_t)i + k] = r[k]; XwA[4 * (size_t)i + k] = r[k]; XwB[4 * (size_t)i + k] = r[k]; }
	}
}

__global__ void k_fill(double* p, size_t n, double v)
{
	for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

}  // namespace cuba_b200
