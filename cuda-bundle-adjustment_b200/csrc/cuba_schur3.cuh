// cuba_schur3.cuh -- Schur complement, third kernel: one warp per destination block like the first kernel, k_schur (since retired; products
// sorted by destination at structure time -> every block is a fixed-order sum, no fp64 atomics; reference
// src/cuda_block_solver.cu:955-977 does 36 atomics per product), but SIX lanes per product instead of one.
//
// Why (ncu of k_schur, profiles/r01_ncu_schur_*): a lane per product needs 36+6 accumulators and two whole blocks
// in registers (196 registers -> 8 warps per SM, 5.5 achieved), the loop is a chain of three dependent L2 gathers
// (product -> landmark -> inverse), and destinations with fewer than 32 products leave lanes idle: issue-active 14 %.
// Here lane = (product slot s = lane / 6, row r = lane % 6): a lane owns one row of the 6x6 product (6 + 1
// accumulators), the landmark of a product comes with the product list (no dependent lookup), the indices of
// the next step are fetched while the current one is computed, and five products are in flight per warp step.
//   Hsc(a,b) = [a==b](Hpp_a + lambda I) - sum_products (Hpl_i invHll_l) Hpl_j^T      bsc(a) = bp_a - sum (Hpl_i invHll_l) bl_l
#pragma once

#include "cuba_kernels.cuh"

namespace cuba_b200 {
namespace schur3 {

constexpr int WARPS = 8;      // warps per CTA == destination blocks per CTA
constexpr int SLOTS = 5;      // products per warp step (6 lanes each; lanes 30, 31 idle in the loop)

__global__ void k_prod_landmark(const int* __restrict__ prodI, const int* __restrict__ hplLm, int n, int* prodL)
{
	const int k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= n) return;
	const int i = prodI[k];
	prodL[k] = i >= 0 ? hplLm[i] : -1;
}

template <typename T, typename TH = T>
struct Args {
	const TH* Hpl; const T* invHll; const T* bl; const T* Hpp; const T* bp;
	const int* prodPtr; const int* prodI; const int* prodJ; const int* prodL;
	const int* blkRow; const int* blkCol; const int* u2f; const int* u2fT;
	int nblk;
	T lambda;
	int addDiag;
	T* fVal; T* bsc;
	T* uVal;     // landmark-sharded runs: the UPPER blocks only, [nblk][36] in block order (half the all-reduce; k_expand_upper mirrors them)
};

template <typename T, typename TH = T>
__global__ void __launch_bounds__(WARPS * 32, 3) k_schur3(const Args<T, TH> a)
{
	__shared__ T s_red[WARPS][SLOTS][6][8];     // [slot][row][6 entries of the row + bsc + pad]
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
	const int k = blockIdx.x * WARPS + wid;
	if (k >= a.nblk) return;
	const int ra = a.blkRow[k], cb = a.blkCol[k];
	const bool diag = ra == cb;
	const int n0 = a.prodPtr[k], n1 = a.prodPtr[k + 1];
	const int slot = lane / 6, r = lane - 6 * slot;
	const bool worker = slot < SLOTS;
	T C[6], vr = T(0);
#pragma unroll
	for (int c = 0; c < 6; c++) C[c] = T(0);

	int n = n0 + slot;
	int pi = -1, pj = -1, pl = -1;
	if (worker && n < n1) { pi = a.prodI[n]; pj = a.prodJ[n]; pl = a.prodL[n]; }
	for (; n0 < n1; ) {            // uniform loop: every lane runs ceil((n1-n0)/SLOTS) steps
		const int ci = pi, cj = pj, cl = pl;
		const bool have = worker && n < n1 && ci >= 0;
		// indices of the next step while this one computes
		const int nn = n + SLOTS;
		pi = -1; pj = -1; pl = -1;
		if (worker && nn < n1) { pi = a.prodI[nn]; pj = a.prodJ[nn]; pl = a.prodL[nn]; }
		if (have) {
			const TH* Ai = a.Hpl + HplStride<T, TH>::value * (size_t)ci;
			const TH* Aj = a.Hpl + HplStride<T, TH>::value * (size_t)cj;
			const T* iv = a.invHll + 9 * (size_t)cl;
			const T a0 = ldh<T, TH>(Ai + r), a1 = ldh<T, TH>(Ai + 6 + r), a2 = ldh<T, TH>(Ai + 12 + r);
			const T i0 = __ldg(iv), i1 = __ldg(iv + 3), i2 = __ldg(iv + 6), i3 = __ldg(iv + 4), i4 = __ldg(iv + 7), i5 = __ldg(iv + 8);
			T B[18];
#pragma unroll
			for (int x = 0; x < 18; x += 2) ldh2<T, TH>(Aj + x, B[x], B[x + 1]);
			const T w0 = a0 * i0 + a1 * i1 + a2 * i2;
			const T w1 = a0 * i1 + a1 * i3 + a2 * i4;
			const T w2 = a0 * i2 + a1 * i4 + a2 * i5;
#pragma unroll
			for (int c = 0; c < 6; c++) C[c] += w0 * B[c] + w1 * B[6 + c] + w2 * B[12 + c];
			if (diag) {
				const T* b3 = a.bl + 3 * (size_t)cl;
				vr += w0 * __ldg(b3) + w1 * __ldg(b3 + 1) + w2 * __ldg(b3 + 2);
			}
		}
		n = nn;
		if (__all_sync(0xffffffffu, !(worker && n < n1))) break;
	}
	// fixed-order sum over the five slots
	if (worker) {
#pragma unroll
		for (int c = 0; c < 6; c++) s_red[wid][slot][r][c] = C[c];
		s_red[wid][slot][r][6] = vr;
	}
	__syncwarp();
	for (int e = lane; e < 42; e += 32) {
		const int c = e < 36 ? e / 6 : 6, rr = e < 36 ? e - 6 * c : e - 36;
		T s = T(0);
#pragma unroll
		for (int q = 0; q < SLOTS; q++) s += s_red[wid][q][rr][c];
		if (e < 36) {
			T val = -s;
			if (diag && a.addDiag) val += a.Hpp[36 * (size_t)ra + e] + (rr == c ? a.lambda : T(0));
			if (a.uVal) a.uVal[36 * (size_t)k + e] = val;
			else {
				a.fVal[36 * (size_t)a.u2f[k] + e] = val;
				if (!diag) a.fVal[36 * (size_t)a.u2fT[k] + rr * 6 + c] = val;
			}
		} else if (diag) {
			a.bsc[6 * (size_t)ra + rr] = (a.addDiag ? a.bp[6 * (size_t)ra + rr] : T(0)) - s;
		}
	}
}

// upper blocks (summed over the ranks) -> both triangles of the symmetric-full BSR
template <typename T>
__global__ void k_expand_upper(const T* __restrict__ uVal, const int* __restrict__ u2f, const int* __restrict__ u2fT, const int* __restrict__ blkRow,
	const int* __restrict__ blkCol, int nblk, T* fVal)
{
	const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
	if (w >= 36LL * nblk) return;
	const int k = (int)(w / 36), e = (int)(w - 36LL * k), c = e / 6, r = e - 6 * c;
	const T v = uVal[w];
	fVal[36 * (size_t)u2f[k] + e] = v;
	if (blkRow[k] != blkCol[k]) fVal[36 * (size_t)u2fT[k] + r * 6 + c] = v;
}

}  // namespace schur3
}  // namespace cuba_b200
