// cuba_pcg2.cuh -- persistent, shared-memory-resident block-Jacobi PCG (second generation).
//
// Same mathematics as the first-generation k_pcg (since retired; block-Jacobi preconditioned CG on the reduced pose system) but organised
// for B200 latency instead of generality:
//   * split preconditioning: with M_i = L_i L_i^T (Cholesky of the 6x6 diagonal blocks) the kernel forms
//     A^ = L^-1 S L^-T once per solve (diagonal blocks become I) and runs plain CG on A^ y = L^-1 b,
//     x = L^-T y.  r^.r^ = r' M^-1 r, so the stopping rule is the same as k_pcg's.
//   * one CTA per SM, each owning a contiguous range of block rows whose A^ blocks live in shared memory
//     for the whole solve (227 KB/CTA, 33 MB across the chip -- ba_kitti_00's Schur matrix is 23 MB);
//     rows that do not fit are streamed from the global copy.
//   * Chronopoulos-Gear single-reduction CG: both inner products of an iteration are reduced behind ONE
//     grid barrier; the updated residual of the neighbouring rows is recomputed on the fly from the
//     owner-published vectors (r, s, w) instead of waiting for a second barrier.
//   * hand-rolled sense-reversing grid barrier (one atomic per CTA, acquire spin), partial sums combined
//     in a fixed order => bit-reproducible.
#pragma once

#include "cuba_kernels.cuh"

namespace cuba_b200 {

constexpr int PCG2_BLOCK = 512;

struct GridBar { unsigned int count; unsigned int gen; };

__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p)
{
	unsigned int v;
	asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
	return v;
}
__device__ __forceinline__ unsigned int atom_add_acqrel_u32(unsigned int* p, unsigned int v)
{
	unsigned int old;
	asm volatile("atom.add.acq_rel.gpu.global.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
	return old;
}
__device__ __forceinline__ void st_release_u32(unsigned int* p, unsigned int v)
{
	asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

// Sense-reversing barrier over all CTAs of a cooperative launch: one acq_rel atomic per CTA, acquire spin.
// bar.sync orders the CTA's earlier writes before thread 0's release (PTX causality order), so no separate
// __threadfence() is needed; data written by other CTAs must afterwards be read with __ldcg (L1 may be stale).
__device__ __forceinline__ void grid_barrier(GridBar* b, unsigned int nblocks, unsigned int& gen)
{
	__syncthreads();
	if (threadIdx.x == 0) {
		const unsigned int prev = atom_add_acqrel_u32(&b->count, 1u);
		if (prev == nblocks - 1) {
			b->count = 0;
			st_release_u32(&b->gen, gen + 1);
		} else {
			while (ld_acquire_u32(&b->gen) == gen) { }
		}
	}
	gen++;
	__syncthreads();
}

template <typename T>
struct Pcg2Args {
	const int* fRowPtr; const int* fColInd; const int* fLocal;   // fLocal: index of each block's column in the CTA's need list
	const T* fVal; T* fHat;                                       // S blocks in, A^ blocks out (global copy)
	const int* ctaRow;      // [G+1] row range per CTA
	const int* needPtr;     // [G+1]
	const int* needCol;     // needed columns per CTA (sorted)
	const T* b;             // bsc
	int numP;
	T* Linv;                // [numP][36]
	T* R0; T* R1; T* S0; T* S1; T* W0; T* W1; T* P; T* Y;   // vectors [6 numP]
	T* x;                   // out: xp
	double* partial;        // [2][G][2]
	GridBar* bar;
	int capBlocks;          // blocks of A^ a CTA can keep in shared memory
	int needMax;            // max need-list length over CTAs
	int maxRows;            // max rows per CTA
	int maxIters; double tol2;
	PcgStatus* status;
};

// inverse of the lower Cholesky factor of a 6x6 SPD block (column-major); false if not positive definite
template <typename T>
__device__ bool chol6_inverse_factor(const T* A, T* Li)
{
	T L[36];
	for (int i = 0; i < 36; i++) { L[i] = T(0); Li[i] = T(0); }
	for (int j = 0; j < 6; j++) {
		T d = A[j * 6 + j];
		for (int k = 0; k < j; k++) d -= L[k * 6 + j] * L[k * 6 + j];
		if (!(d > T(0))) return false;
		d = t_sqrt(d);
		L[j * 6 + j] = d;
		const T id = 1 / d;
		for (int i = j + 1; i < 6; i++) {
			T s = A[j * 6 + i];
			for (int k = 0; k < j; k++) s -= L[k * 6 + i] * L[k * 6 + j];
			L[j * 6 + i] = s * id;
		}
	}
	for (int j = 0; j < 6; j++) {
		Li[j * 6 + j] = 1 / L[j * 6 + j];
		for (int i = j + 1; i < 6; i++) {
			T s = T(0);
			for (int k = j; k < i; k++) s -= L[k * 6 + i] * Li[j * 6 + k];
			Li[j * 6 + i] = s / L[i * 6 + i];
		}
	}
	return true;
}

template <typename T>
__global__ void __launch_bounds__(PCG2_BLOCK, 1) k_pcg2(const Pcg2Args<T> a)
{
	extern __shared__ __align__(16) unsigned char smem_raw[];
	T* s_blk = reinterpret_cast<T*>(smem_raw);                          // [36][capBlocks]  cached A^ blocks, element-major:
	                                                                    // lane-per-block reads are bank-conflict free
	T* s_rj = s_blk + (size_t)a.capBlocks * 36;                         // [needMax][6]     gathered residual
	int* s_loc = reinterpret_cast<int*>(s_rj + (size_t)a.needMax * 6);  // [capBlocks]      need index of a block's column (<0: diagonal)
	int* s_rowPtr = s_loc + a.capBlocks;                                // [maxRows+1]      local block offsets of the own rows
	int* s_need = s_rowPtr + a.maxRows + 1;                             // [needMax]        global column of each need entry
	__shared__ double s_red[PCG2_BLOCK / 32][2];
	__shared__ double s_bc[2];
	__shared__ unsigned int s_gen;

	const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
	const int G = gridDim.x, cta = blockIdx.x;
	const int row0 = a.ctaRow[cta], row1 = a.ctaRow[cta + 1], nrows = row1 - row0;
	const int need0 = a.needPtr[cta], nneed = a.needPtr[cta + 1] - need0;
	const int blk0 = a.fRowPtr[row0], nblkCta = a.fRowPtr[row1] - blk0;
	const int ncached = nblkCta < a.capBlocks ? nblkCta : a.capBlocks;
	if (tid == 0) s_gen = ld_acquire_u32(&a.bar->gen);
	for (int i = tid; i <= nrows; i += PCG2_BLOCK) s_rowPtr[i] = a.fRowPtr[row0 + i] - blk0;
	for (int i = tid; i < nneed; i += PCG2_BLOCK) s_need[i] = a.needCol[need0 + i];
	__syncthreads();
	unsigned int gen = s_gen;

	// ---- S1: factor the diagonal blocks of the own rows, b^ = L^-1 b, initial vectors --------------
	int bad = 0;
	for (int i = row0 + tid; i < row1; i += PCG2_BLOCK) {
		int d = -1;
		for (int n = a.fRowPtr[i]; n < a.fRowPtr[i + 1]; n++) if (a.fColInd[n] == i) { d = n; break; }
		T Li[36];
		bool ok = d >= 0 && chol6_inverse_factor(a.fVal + 36 * (size_t)d, Li);
		if (!ok) { bad = 1; for (int e = 0; e < 36; e++) Li[e] = (e % 7) == 0 ? T(1) : T(0); }
		for (int e = 0; e < 36; e++) a.Linv[36 * (size_t)i + e] = Li[e];
		for (int r = 0; r < 6; r++) {
			T s = T(0);
			for (int c = 0; c <= r; c++) s += Li[c * 6 + r] * a.b[6 * (size_t)i + c];
			const size_t o = 6 * (size_t)i + r;
			a.R0[o] = s; a.S1[o] = T(0); a.S0[o] = T(0); a.P[o] = T(0); a.Y[o] = T(0); a.W0[o] = T(0); a.W1[o] = T(0); a.R1[o] = T(0);
		}
	}
	{
		const int anyBad = __syncthreads_or(bad);
		if (tid == 0) a.partial[(size_t)cta * 2] = (double)anyBad;
	}
	grid_barrier(a.bar, G, gen);
	double nbad = 0;
	if (tid < 32) {
		for (int i = tid; i < G; i += 32) nbad += __ldcg(a.partial + (size_t)i * 2);
		nbad = warp_sum(nbad);
		if (tid == 0) s_bc[0] = nbad;
	}
	__syncthreads();
	nbad = s_bc[0];
	__syncthreads();

	// ---- S2: A^_ij = L_i^-1 S_ij L_j^-T for the own rows -> shared memory (+ global for the overflow) ----
	for (int n = tid; n < nblkCta; n += PCG2_BLOCK) {
		const int g = blk0 + n;
		int lo = 0, hi = nrows - 1;       // row of block n: largest i with s_rowPtr[i] <= n
		while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (s_rowPtr[mid] <= n) lo = mid; else hi = mid - 1; }
		const int i = row0 + lo, j = a.fColInd[g];
		const T* B = a.fVal + 36 * (size_t)g;
		const T* Li = a.Linv + 36 * (size_t)i;
		const T* Lj = a.Linv + 36 * (size_t)j;
		T tmp[36], out[36];
		for (int c = 0; c < 6; c++)
			for (int r = 0; r < 6; r++) {
				T s = T(0);
				for (int k = 0; k <= r; k++) s += Li[k * 6 + r] * B[c * 6 + k];
				tmp[c * 6 + r] = s;
			}
		for (int c = 0; c < 6; c++)
			for (int r = 0; r < 6; r++) {
				T s = T(0);
				for (int k = 0; k <= c; k++) s += tmp[k * 6 + r] * __ldcg(Lj + k * 6 + c);
				out[c * 6 + r] = s;
			}
		if (n < ncached) {
			for (int e = 0; e < 36; e++) s_blk[(size_t)e * a.capBlocks + n] = out[e];
			s_loc[n] = a.fLocal[g];
		} else {
			for (int e = 0; e < 36; e++) a.fHat[36 * (size_t)g + e] = out[e];
		}
	}
	__syncthreads();

	int status = 1, it = 0;
	double gamma = 0, gamma0 = 0, alpha = 0, beta = 0;
	if (nbad > 0) status = 2;
	else {
		// pass k = -1 computes w0 = A^ r0 and the first inner products; pass k >= 0 is CG iteration k.
		// The inner products of pass k-1 are read at the top of pass k, together with the vector prefetch,
		// so one iteration costs one grid barrier and one round of L2 reads.
		for (int k = -1;; k++) {
			const int par = (k + 2) & 1;
			const T* Rin = (par == 0) ? a.R0 : a.R1;           // r_k
			T* Rout = (par == 0) ? a.R1 : a.R0;                // r_{k+1}
			const T* Win = (par == 0) ? a.W0 : a.W1;           // w_k
			T* Wout = (par == 0) ? a.W1 : a.W0;                // w_{k+1}
			const T* Sprev = (par == 0) ? a.S1 : a.S0;         // s_{k-1}
			T* Scur = (par == 0) ? a.S0 : a.S1;                // s_k
			// ---- prefetch the first gather item of every thread (independent of alpha/beta) ----
			T g_r = T(0), g_w = T(0), g_s = T(0);
			if (tid < nneed * 6) {
				const int c = tid / 6, comp = tid - 6 * c;
				const size_t o = 6 * (size_t)s_need[c] + comp;
				if (k < 0) g_r = __ldcg(a.R0 + o);
				else { g_r = __ldcg(Rin + o); g_w = __ldcg(Win + o); g_s = __ldcg(Sprev + o); }
			}
			// ---- scalars of this pass from the partial sums of the previous one ----
			if (k >= 0) {
				if (tid < 32) {
					double g2 = 0, d2 = 0;
					const double* src = a.partial + (size_t)(1 - par) * G * 2;   // written in pass k-1
					for (int i = tid; i < G; i += 32) { g2 += __ldcg(src + 2 * i); d2 += __ldcg(src + 2 * i + 1); }
					g2 = warp_sum(g2); d2 = warp_sum(d2);
					if (tid == 0) { s_bc[0] = g2; s_bc[1] = d2; }
				}
				__syncthreads();
				const double gnew = s_bc[0], delta = s_bc[1];
				if (!(gnew == gnew) || !(delta == delta)) { status = 2; break; }
				if (k == 0) {
					gamma0 = gamma = gnew;
					if (gamma0 <= 0) { status = 0; break; }
					if (!(delta > 0)) { status = 2; break; }
					alpha = gamma / delta; beta = 0;
				} else {
					it = k;
					if (gnew <= a.tol2 * gamma0) { gamma = gnew; status = 0; break; }
					beta = gnew / gamma;
					const double den = delta - beta * gnew / alpha;
					gamma = gnew;
					if (!(den > 0)) { status = 2; break; }
					alpha = gnew / den;
				}
				if (k >= a.maxIters) { status = 1; break; }
			}
			// ---- gather: updated residual r_{k+1} of every needed column into shared memory ----
			if (tid < nneed * 6) s_rj[tid] = (k < 0) ? g_r : g_r - (T)alpha * (g_w + (T)beta * g_s);
			for (int wi = tid + PCG2_BLOCK; wi < nneed * 6; wi += PCG2_BLOCK) {
				const int c = wi / 6, comp = wi - 6 * c;
				const size_t o = 6 * (size_t)s_need[c] + comp;
				s_rj[wi] = (k < 0) ? __ldcg(a.R0 + o) : __ldcg(Rin + o) - (T)alpha * (__ldcg(Win + o) + (T)beta * __ldcg(Sprev + o));
			}
			// ---- owners: p, y, s, r updates for the own rows ----
			if (k >= 0) {
				for (int wi = tid; wi < nrows * 6; wi += PCG2_BLOCK) {
					const size_t o = 6 * (size_t)row0 + wi;
					const T rk = __ldcg(Rin + o);
					const T s = __ldcg(Win + o) + (T)beta * __ldcg(Sprev + o);
					const T p = rk + (T)beta * a.P[o];
					a.P[o] = p;
					a.Y[o] += (T)alpha * p;
					Scur[o] = s;
					Rout[o] = rk - (T)alpha * s;
				}
			}
			__syncthreads();
			// ---- w_{k+1} = A^ r_{k+1} for the own rows (warp per row), partial gamma', delta ----
			double pg = 0, pd = 0;
			for (int li = wid; li < nrows; li += PCG2_BLOCK / 32) {
				T acc[6] = { T(0), T(0), T(0), T(0), T(0), T(0) };
				const int n0 = s_rowPtr[li], n1 = s_rowPtr[li + 1];
				int selfLoc = -1;
				for (int n = n0 + lane; n < n1; n += 32) {
					const bool cached = n < ncached;
					const int loc = cached ? s_loc[n] : a.fLocal[blk0 + n];
					if (loc < 0) { selfLoc = -1 - loc; continue; }
					const T* rj = s_rj + 6 * (size_t)loc;
					if (cached) {
						const T* B = s_blk + n;
						const size_t st = (size_t)a.capBlocks;
#pragma unroll
						for (int c = 0; c < 6; c++) {
							const T rc = rj[c];
#pragma unroll
							for (int r = 0; r < 6; r++) acc[r] += B[(c * 6 + r) * st] * rc;
						}
					} else {
						const T* B = a.fHat + 36 * (size_t)(blk0 + n);
#pragma unroll
						for (int c = 0; c < 6; c++) {
							const T rc = rj[c];
#pragma unroll
							for (int r = 0; r < 6; r++) acc[r] += B[c * 6 + r] * rc;
						}
					}
				}
#pragma unroll
				for (int c = 0; c < 6; c++) acc[c] = warp_sum(acc[c]);
				selfLoc = __reduce_max_sync(0xffffffffu, selfLoc);
				if (lane < 6) {
					T wv = acc[0];
#pragma unroll
					for (int c = 1; c < 6; c++) if (lane == c) wv = acc[c];
					const T ri = s_rj[6 * (size_t)selfLoc + lane];
					wv += ri;                                   // A^_ii = I
					Wout[6 * (size_t)(row0 + li) + lane] = wv;
					pg += (double)ri * (double)ri;
					pd += (double)wv * (double)ri;
				}
			}
			// ---- publish the two inner products, one grid barrier ----
			pg = warp_sum(pg); pd = warp_sum(pd);
			if (lane == 0) { s_red[wid][0] = pg; s_red[wid][1] = pd; }
			__syncthreads();
			if (tid == 0) {
				double g2 = 0, d2 = 0;
				for (int w = 0; w < PCG2_BLOCK / 32; w++) { g2 += s_red[w][0]; d2 += s_red[w][1]; }
				double* dst = a.partial + ((size_t)par * G + cta) * 2;
				dst[0] = g2; dst[1] = d2;
			}
			grid_barrier(a.bar, G, gen);
		}
	}
	// ---- x = L^-T y for the own rows ----
	for (int wi = tid; wi < nrows * 6; wi += PCG2_BLOCK) {
		const int i = row0 + wi / 6, r = wi % 6;
		const T* Li = a.Linv + 36 * (size_t)i;
		T s = T(0);
		for (int c = r; c < 6; c++) s += Li[r * 6 + c] * a.Y[6 * (size_t)i + c];   // (L^-T)(r,c) = Li(c,r)
		a.x[6 * (size_t)i + r] = s;
	}
	if (cta == 0 && tid == 0) { a.status->iters = it; a.status->status = status; a.status->rz0 = gamma0; a.status->rz = gamma; }
}

}  // namespace cuba_b200
