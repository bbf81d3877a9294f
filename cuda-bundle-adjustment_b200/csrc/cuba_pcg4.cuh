// cuba_pcg4.cuh -- TWO-LEVEL preconditioned CG on the reduced pose system: block-Jacobi (6x6 blocks, as in k_pcg2/3)
// plus an additive coarse-grid correction over rigid-body motions of pose aggregates.
//
// Why: with block-Jacobi alone the iteration count of ba_kitti_00-shaped graphs grows from ~25 to ~2000-4000 as the LM
// damping falls (DESIGN.md 4.2) -- the slow modes are smooth drifts of whole stretches of the trajectory, which a
// block-diagonal preconditioner cannot see.  Let the free poses be cut into A aggregates of consecutive poses and let
// Z (6P x 6A) map a world-frame twist xi_a of aggregate a to the pose increments it induces, delta_i = Ad(T_i) xi_a
// (poses are updated as T <- Exp(delta) T, reference cu:551-592, so the adjoint of T_i = (R_i, t_i) is the exact
// tangent of a rigid motion of the aggregate).  The preconditioner is
//      M^-1 = D^-1 + Z (Z^T S Z)^-1 Z^T            D = blockdiag(S)
// i.e. two-level additive Schwarz with the block-Jacobi "smoother".  Measured on the CPU prototype
// (kitti00_shaped, tol 1e-11): lambda 2.9e3 / 2.9 / 0.029 -> 23 / 301 / 1948 iterations with block-Jacobi,
// 26 / 114 / 222 with 42 aggregates.  The solution is the same to the CG tolerance: only the path differs.
//
// Organisation = k_pcg2 (cuba_pcg2.cuh): split preconditioning (A^ = L^-1 S L^-T resident in shared memory, hat space),
// Chronopoulos-Gear single-reduction CG, ONE grid barrier per iteration.  The coarse level costs no extra barrier:
//   * hat-space basis Z^_i = L_i^T Z_i; every CTA owns one aggregate share and publishes, next to its inner-product
//     partials, the six numbers Z^_own^T w -- so every CTA can advance the coarse residual rc = Z^^T r by the same
//     recurrences as r itself (sc = wc + beta sc, rc -= alpha sc);
//   * c = Ac^-1 rc is needed only for the aggregates of a CTA's own and neighbouring rows: a few 6-row slices of the
//     explicit inverse (computed per solve by k_coarse_invert) times rc;
//   * u_j = r_j + Z^_j c_a(j) for every needed column j, then w = A^ u from shared memory as before.
// All sums are in fixed order: bit-reproducible.
// Replaces convertBSRToCSR + cuSOLVER csrchol (reference cuda_linear_solver.cpp:301-335) like the other PCG kernels.
#pragma once

#include "cuba_pcg3.cuh"

namespace cuba_b200 {

constexpr int PCG4_BLOCK = 512;
constexpr int PCG4_PSTRIDE = 12;    // doubles per CTA on the partial board: gamma, delta, rho, -, wc[6], -, -
constexpr int PCG4_MAXAGG = 74;     // k_coarse_invert_cluster: the packed block triangle lives in the shared memory of an 8-CTA cluster
constexpr int PCG4_MAXAGG1 = 37;    // k_coarse_invert: ... of one CTA
constexpr int PCG4_CL = 8;          // CTAs per cluster of k_coarse_invert_cluster
constexpr int PCG4_TPR = 16;        // threads per row of the coarse slice product

template <typename T>
struct Pcg4Args {
	Pcg2Args<T> base;
	const T* Zx;          // [numP][36] Ad(T_i), column-major
	T* Zhat;              // [numP][36] L_i^T Z_i, written by the row's owner before the first barrier
	const float* AcInv;   // [nc][nc] row-major (symmetric), SINGLE precision: it only shapes the preconditioner -- every CTA
	                      // applies the same rounded operator, so M^-1 stays one fixed symmetric matrix and CG stays exact
	const int* aggRow;    // [A+1] first row of every aggregate (aggregates are groups of gs consecutive CTAs)
	const int* naPtr;     // [G+1]
	const int* naList;    // aggregates a CTA needs (sorted)
	const int* needAgg;   // per need entry (indexing of needCol): position of its aggregate in the CTA's list
	int A, gs, maxNeedAgg;
	int sliceInSmem;      // 1: the CTA's slices of AcInv live in shared memory for the whole solve
	int zhInSmem;         // 1: Z^ of the needed columns lives in shared memory (else it is read from L2 every pass)
	double* cpart;        // [2][G][PCG4_PSTRIDE]
	long long* timing;    // [G][8] per-phase clock64 sums of thread 0 (only with -DCUBA_PCG_TIMING)
};

// lower Cholesky factor L and its inverse of a 6x6 SPD block (column-major); false if not positive definite
template <typename T>
__device__ bool chol6_factor_and_inverse(const T* A, T* L, T* Li)
{
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
__global__ void __launch_bounds__(PCG4_BLOCK, 1) k_pcg4(const Pcg4Args<T> aa)
{
	const Pcg2Args<T>& a = aa.base;
	const int nc = 6 * aa.A;
	extern __shared__ __align__(16) unsigned char smem_raw[];
	T* s_blk = reinterpret_cast<T*>(smem_raw);                          // [36][capBlocks] cached A^ blocks, element-major
	T* s_r = s_blk + (size_t)a.capBlocks * 36;                          // [needMax][6] residual of the needed columns
	T* s_u = s_r + (size_t)a.needMax * 6;                               // [needMax][6] preconditioned residual u = M^-1 r
	T* s_uown = s_u + (size_t)a.needMax * 6;                            // [maxRows][6] u_k of the own rows (previous pass)
	T* s_rc = s_uown + (size_t)a.maxRows * 6;                           // [nc] coarse residual Z^^T r
	T* s_sc = s_rc + nc;                                                // [nc] Z^^T s
	T* s_c = s_sc + nc;                                                 // [maxNeedAgg][6] coarse correction of the needed aggregates
	T* s_zh = s_c + (size_t)aa.maxNeedAgg * 6;                          // [needMax][36] Z^ of the needed columns (if zhInSmem)
	float* s_ai = reinterpret_cast<float*>(s_zh + (aa.zhInSmem ? (size_t)a.needMax * 36 : 0));   // [maxNeedAgg*6][nc] slices of AcInv (if sliceInSmem)
	int* s_loc = reinterpret_cast<int*>(s_ai + (aa.sliceInSmem ? (((size_t)aa.maxNeedAgg * 6 * nc + 1) & ~(size_t)1) : 0));  // [capBlocks]
	int* s_rowPtr = s_loc + a.capBlocks;                                // [maxRows+1]
	int* s_need = s_rowPtr + a.maxRows + 1;                             // [needMax] global column of each need entry
	int* s_nagg = s_need + a.needMax;                                   // [needMax] position of the column's aggregate in s_alist
	int* s_alist = s_nagg + a.needMax;                                  // [maxNeedAgg]
	int* s_diag = s_alist + aa.maxNeedAgg;                              // [maxRows] need index of each own row
	__shared__ double s_red[PCG4_BLOCK / 32][9];
	__shared__ double s_bc[4];
	__shared__ unsigned int s_gen;

	const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
	const int G = gridDim.x, cta = blockIdx.x;
	const int row0 = a.ctaRow[cta], row1 = a.ctaRow[cta + 1], nrows = row1 - row0;
	const int need0 = a.needPtr[cta], nneed = a.needPtr[cta + 1] - need0;
	const int na0 = aa.naPtr[cta], nagg = aa.naPtr[cta + 1] - na0;
	const int blk0 = a.fRowPtr[row0], nblkCta = a.fRowPtr[row1] - blk0;
	const int ncached = nblkCta < a.capBlocks ? nblkCta : a.capBlocks;
	if (tid == 0) s_gen = ld_acquire_u32(&a.bar->gen);
	for (int i = tid; i <= nrows; i += PCG4_BLOCK) s_rowPtr[i] = a.fRowPtr[row0 + i] - blk0;
	for (int i = tid; i < nneed; i += PCG4_BLOCK) {
		const int j = a.needCol[need0 + i];
		s_need[i] = j;
		s_nagg[i] = aa.needAgg[need0 + i];
		if (j >= row0 && j < row1) s_diag[j - row0] = i;
	}
	for (int i = tid; i < nagg; i += PCG4_BLOCK) s_alist[i] = aa.naList[na0 + i];
	for (int i = tid; i < nc; i += PCG4_BLOCK) { s_rc[i] = T(0); s_sc[i] = T(0); }
	for (int i = tid; i < nrows * 6; i += PCG4_BLOCK) s_uown[i] = T(0);
	__syncthreads();
	unsigned int gen = s_gen;

	// ---- S1: factor the diagonal blocks of the own rows, b^ = L^-1 b, Z^_i = L_i^T Z_i, partial of rc0 = Z^^T b^ --------
	int bad = 0;
	for (int i = row0 + tid; i < row1; i += PCG4_BLOCK) {
		int d = -1;
		for (int n = a.fRowPtr[i]; n < a.fRowPtr[i + 1]; n++) if (a.fColInd[n] == i) { d = n; break; }
		T L[36], Li[36];
		bool ok = d >= 0 && chol6_factor_and_inverse(a.fVal + 36 * (size_t)d, L, Li);
		if (!ok) { bad = 1; for (int e = 0; e < 36; e++) { Li[e] = (e % 7) == 0 ? T(1) : T(0); L[e] = Li[e]; } }
		for (int e = 0; e < 36; e++) a.Linv[36 * (size_t)i + e] = Li[e];
		T bh[6];
		for (int r = 0; r < 6; r++) {
			T s = T(0);
			for (int c = 0; c <= r; c++) s += Li[c * 6 + r] * a.b[6 * (size_t)i + c];
			bh[r] = s;
			const size_t o = 6 * (size_t)i + r;
			a.R0[o] = s; a.S1[o] = T(0); a.S0[o] = T(0); a.P[o] = T(0); a.Y[o] = T(0); a.W0[o] = T(0); a.W1[o] = T(0); a.R1[o] = T(0);
		}
		// Z^(r,q) = sum_{k>=r} L(k,r) Z(k,q); staged per row in s_u (free until the first pass) for the rc0 partial
		const T* Z = aa.Zx + 36 * (size_t)i;
		for (int q = 0; q < 6; q++) {
			T rcq = T(0);
			for (int r = 0; r < 6; r++) {
				T s = T(0);
				for (int k = r; k < 6; k++) s += L[r * 6 + k] * Z[q * 6 + k];
				aa.Zhat[36 * (size_t)i + q * 6 + r] = s;
				rcq += s * bh[r];
			}
			s_u[6 * (size_t)(i - row0) + q] = rcq;
		}
	}
	{
		const int anyBad = __syncthreads_or(bad);
		double* dst = aa.cpart + (size_t)cta * PCG4_PSTRIDE;              // slot 0: read by pass -1
		if (tid == 0) dst[0] = (double)anyBad;
		if (tid < 6) {
			double s = 0;
			for (int li = 0; li < nrows; li++) s += (double)s_u[6 * (size_t)li + tid];
			dst[4 + tid] = s;
		}
	}
	grid_barrier(a.bar, G, gen);
	double nbad = 0;
	if (tid < 32) {
		for (int i = tid; i < G; i += 32) nbad += __ldcg(aa.cpart + (size_t)i * PCG4_PSTRIDE);
		nbad = warp_sum(nbad);
		if (tid == 0) s_bc[0] = nbad;
	}
	__syncthreads();
	nbad = s_bc[0];
	// Z^ of the needed columns (published by their owners before the barrier) and the CTA's slices of AcInv
	if (aa.zhInSmem)
		for (int wi = tid; wi < nneed * 36; wi += PCG4_BLOCK) s_zh[wi] = __ldcg(aa.Zhat + 36 * (size_t)s_need[wi / 36] + (wi % 36));
	if (aa.sliceInSmem)
		for (int wi = tid; wi < nagg * 6 * nc; wi += PCG4_BLOCK) {
			const int rowi = wi / nc, q = wi - rowi * nc;
			s_ai[wi] = __ldg(aa.AcInv + (size_t)(s_alist[rowi / 6] * 6 + (rowi % 6)) * nc + q);
		}
	__syncthreads();

	// ---- S2: A^_ij = L_i^-1 S_ij L_j^-T for the own rows -> shared memory (+ global for the overflow) ----
	for (int n = tid; n < nblkCta; n += PCG4_BLOCK) {
		const int g = blk0 + n;
		int lo = 0, hi = nrows - 1;
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
	double gamma = 0, rho0 = 0, rho = 0, alpha = 0, beta = 0;
#ifdef CUBA_PCG_TIMING
	long long tacc[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
#endif
	if (nbad > 0) status = 2;
	else {
		// pass k = -1: u0 = M^-1 r0, w0 = A^ u0 and the first inner products; pass k >= 0: CG iteration k
		for (int k = -1;; k++) {
			const int par = (k + 2) & 1;
			const T* Rin = (par == 0) ? a.R0 : a.R1;
			T* Rout = (par == 0) ? a.R1 : a.R0;
			const T* Win = (par == 0) ? a.W0 : a.W1;
			T* Wout = (par == 0) ? a.W1 : a.W0;
			const T* Sprev = (par == 0) ? a.S1 : a.S0;
			T* Scur = (par == 0) ? a.S0 : a.S1;
			const double* src = aa.cpart + (size_t)(1 - par) * G * PCG4_PSTRIDE;   // written in pass k-1 (S1 for k = -1)
			PCG_T(t0);
			// ---- prefetch the first gather item of every thread (independent of alpha/beta) ----
			T g_r = T(0), g_w = T(0), g_s = T(0);
			if (tid < nneed * 6) {
				const int c = tid / 6, comp = tid - 6 * c;
				const size_t o = 6 * (size_t)s_need[c] + comp;
				if (k < 0) g_r = __ldcg(a.R0 + o);
				else { g_r = __ldcg(Rin + o); g_w = __ldcg(Win + o); g_s = __ldcg(Sprev + o); }
			}
			// ---- coarse partials of the previous pass, summed per aggregate in CTA order (threads 64 .. 64+nc) ----
			T wcv = T(0);
			if (tid >= 64 && tid < 64 + nc) {
				const int q = tid - 64, ag = q / 6, comp = q - 6 * ag;
				const int c0 = ag * aa.gs, c1 = (c0 + aa.gs < G) ? c0 + aa.gs : G;
				double s = 0;
				for (int c = c0; c < c1; c++) s += __ldcg(src + (size_t)c * PCG4_PSTRIDE + 4 + comp);
				wcv = (T)s;
			}
			// ---- scalars of this pass ----
			if (k >= 0) {
				if (tid < 32) {
					double g2 = 0, d2 = 0, r2 = 0;
					for (int i = tid; i < G; i += 32) {
						g2 += __ldcg(src + (size_t)i * PCG4_PSTRIDE); d2 += __ldcg(src + (size_t)i * PCG4_PSTRIDE + 1); r2 += __ldcg(src + (size_t)i * PCG4_PSTRIDE + 2);
					}
					g2 = warp_sum(g2); d2 = warp_sum(d2); r2 = warp_sum(r2);
					if (tid == 0) { s_bc[0] = g2; s_bc[1] = d2; s_bc[2] = r2; }
				}
				__syncthreads();
				const double gnew = s_bc[0], delta = s_bc[1], rnew = s_bc[2];
				if (!(gnew == gnew) || !(delta == delta) || !(rnew == rnew)) { status = 2; break; }
				if (k == 0) {
					gamma = gnew; rho0 = rho = rnew;
					if (rho0 <= 0) { status = 0; break; }
					if (!(delta > 0) || !(gamma > 0)) { status = 2; break; }
					alpha = gamma / delta; beta = 0;
				} else {
					it = k;
					rho = rnew;
					if (rnew <= a.tol2 * rho0) { status = 0; break; }       // the block-Jacobi norm r' D^-1 r, as in k_pcg2/3
					if (!(gnew > 0)) { status = 2; break; }
					beta = gnew / gamma;
					const double den = delta - beta * gnew / alpha;
					gamma = gnew;
					if (!(den > 0)) { status = 2; break; }
					alpha = gnew / den;
				}
				if (k >= a.maxIters) { status = 1; break; }
			}
			PCG_T(t1);
			// ---- coarse residual: rc0 = sum of the S1 partials; later sc = wc + beta sc, rc -= alpha sc ----
			if (tid >= 64 && tid < 64 + nc) {
				const int q = tid - 64;
				if (k < 0) s_rc[q] = wcv;
				else {
					const T sc = wcv + (T)beta * s_sc[q];
					s_sc[q] = sc;
					s_rc[q] -= (T)alpha * sc;
				}
			}
			// ---- owners: p, y, s, r updates for the own rows (u_k is still in s_uown) ----
			if (k >= 0) {
				for (int wi = tid; wi < nrows * 6; wi += PCG4_BLOCK) {
					const size_t o = 6 * (size_t)row0 + wi;
					const T rk = __ldcg(Rin + o);
					const T s = __ldcg(Win + o) + (T)beta * __ldcg(Sprev + o);
					const T p = s_uown[wi] + (T)beta * a.P[o];
					a.P[o] = p;
					a.Y[o] += (T)alpha * p;
					Scur[o] = s;
					Rout[o] = rk - (T)alpha * s;
				}
			}
			// ---- gather: updated residual r_{k+1} of every needed column ----
			if (tid < nneed * 6) s_r[tid] = (k < 0) ? g_r : g_r - (T)alpha * (g_w + (T)beta * g_s);
			for (int wi = tid + PCG4_BLOCK; wi < nneed * 6; wi += PCG4_BLOCK) {
				const int c = wi / 6, comp = wi - 6 * c;
				const size_t o = 6 * (size_t)s_need[c] + comp;
				s_r[wi] = (k < 0) ? __ldcg(a.R0 + o) : __ldcg(Rin + o) - (T)alpha * (__ldcg(Win + o) + (T)beta * __ldcg(Sprev + o));
			}
			__syncthreads();
			PCG_T(t2);
			// ---- c_a = (Ac^-1 rc)_a for the needed aggregates: PCG4_TPR threads per row, fixed-order butterfly ----
			for (int rb = 0; rb < nagg * 6; rb += PCG4_BLOCK / PCG4_TPR) {
				const int rowi = rb + tid / PCG4_TPR, sub = tid % PCG4_TPR;
				T s = T(0);
				if (rowi < nagg * 6) {
					if (aa.sliceInSmem) {
						const float* Arow = s_ai + (size_t)rowi * nc;
						for (int q = sub; q < nc; q += PCG4_TPR) s += (T)Arow[q] * s_rc[q];
					} else {
						const int la = rowi / 6, comp = rowi - 6 * la;
						const float* Arow = aa.AcInv + (size_t)(s_alist[la] * 6 + comp) * nc;
						for (int q = sub; q < nc; q += PCG4_TPR) s += (T)__ldg(Arow + q) * s_rc[q];
					}
				}
#pragma unroll
				for (int o = 1; o < PCG4_TPR; o <<= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
				if (rowi < nagg * 6 && sub == 0) s_c[rowi] = s;
			}
			__syncthreads();
			PCG_T(t3);
			// ---- u_j = r_j + Z^_j c_a(j) for every needed column ----
			for (int wi = tid; wi < nneed * 6; wi += PCG4_BLOCK) {
				const int c = wi / 6, comp = wi - 6 * c;
				const T* cc = s_c + 6 * (size_t)s_nagg[c];
				T u = s_r[wi];
				if (aa.zhInSmem) {
					const T* Zh = s_zh + 36 * (size_t)c + comp;
#pragma unroll
					for (int q = 0; q < 6; q++) u += Zh[6 * q] * cc[q];
				} else {
					const T* Zh = aa.Zhat + 36 * (size_t)s_need[c] + comp;
#pragma unroll
					for (int q = 0; q < 6; q++) u += __ldcg(Zh + 6 * q) * cc[q];
				}
				s_u[wi] = u;
			}
			__syncthreads();
			PCG_T(t4);
			// ---- w_{k+1} = A^ u_{k+1} for the own rows (warp per row), partials of gamma', delta, rho', Z^^T w ----
			double pg = 0, pd = 0, pr = 0, pw[6] = { 0, 0, 0, 0, 0, 0 };
			for (int li = wid; li < nrows; li += PCG4_BLOCK / 32) {
				T acc[6] = { T(0), T(0), T(0), T(0), T(0), T(0) };
				const int n0 = s_rowPtr[li], n1 = s_rowPtr[li + 1];
				for (int n = n0 + lane; n < n1; n += 32) {
					const bool cached = n < ncached;
					const int loc = cached ? s_loc[n] : a.fLocal[blk0 + n];
					if (loc < 0) continue;                       // diagonal block: A^_ii = I, added below
					const T* uj = s_u + 6 * (size_t)loc;
					if (cached) {
						const T* B = s_blk + n;
						const size_t st = (size_t)a.capBlocks;
#pragma unroll
						for (int c = 0; c < 6; c++) {
							const T uc = uj[c];
#pragma unroll
							for (int r = 0; r < 6; r++) acc[r] += B[(c * 6 + r) * st] * uc;
						}
					} else {
						const T* B = a.fHat + 36 * (size_t)(blk0 + n);
#pragma unroll
						for (int c = 0; c < 6; c++) {
							const T uc = uj[c];
#pragma unroll
							for (int r = 0; r < 6; r++) acc[r] += B[c * 6 + r] * uc;
						}
					}
				}
#pragma unroll
				for (int c = 0; c < 6; c++) acc[c] = warp_sum(acc[c]);
				const int dl = s_diag[li];
				T wv = T(0), ui = T(0);
				if (lane < 6) {
					wv = acc[0];
#pragma unroll
					for (int c = 1; c < 6; c++) if (lane == c) wv = acc[c];
					const T ri = s_r[6 * (size_t)dl + lane];
					ui = s_u[6 * (size_t)dl + lane];
					wv += ui;
					Wout[6 * (size_t)(row0 + li) + lane] = wv;
					s_uown[6 * (size_t)li + lane] = ui;
					pg += (double)ri * (double)ui;
					pd += (double)wv * (double)ui;
					pr += (double)ri * (double)ri;
				}
				// Z^_i^T w_i: lane comp holds w_i[comp]; (Z^^T w)(q) = sum_comp Z^(comp,q) w(comp)
				const T* Zh = aa.zhInSmem ? s_zh + 36 * (size_t)dl : aa.Zhat + 36 * (size_t)(row0 + li);
#pragma unroll
				for (int q = 0; q < 6; q++) {
					double t = lane < 6 ? (double)((aa.zhInSmem ? Zh[6 * q + lane] : __ldcg(Zh + 6 * q + lane)) * wv) : 0.0;
					t += __shfl_xor_sync(0xffffffffu, t, 1); t += __shfl_xor_sync(0xffffffffu, t, 2); t += __shfl_xor_sync(0xffffffffu, t, 4);
					pw[q] += t;                                  // lanes 0..7 hold the sum of lanes 0..7
				}
			}
			// ---- publish the partials, one grid barrier ----
			PCG_T(t5);
			pg = warp_sum(pg); pd = warp_sum(pd); pr = warp_sum(pr);
			if (lane == 0) {
				s_red[wid][0] = pg; s_red[wid][1] = pd; s_red[wid][2] = pr;
#pragma unroll
				for (int q = 0; q < 6; q++) s_red[wid][3 + q] = pw[q];
			}
			__syncthreads();
			if (tid < 9) {
				double v = 0;
				for (int w = 0; w < PCG4_BLOCK / 32; w++) v += s_red[w][tid];
				double* dst = aa.cpart + ((size_t)par * G + cta) * PCG4_PSTRIDE;
				dst[tid < 3 ? tid : tid + 1] = v;                // 0,1,2 = gamma, delta, rho; 4..9 = wc
			}
			PCG_T(t6);
			grid_barrier(a.bar, G, gen);
			PCG_T(t7);
			PCG_ACC(0, t0, t1); PCG_ACC(1, t1, t2); PCG_ACC(2, t2, t3); PCG_ACC(3, t3, t4); PCG_ACC(4, t4, t5); PCG_ACC(5, t5, t6); PCG_ACC(6, t6, t7);
		}
	}
	// ---- x = L^-T y for the own rows ----
	for (int wi = tid; wi < nrows * 6; wi += PCG4_BLOCK) {
		const int i = row0 + wi / 6, r = wi % 6;
		const T* Li = a.Linv + 36 * (size_t)i;
		T s = T(0);
		for (int c = r; c < 6; c++) s += Li[r * 6 + c] * a.Y[6 * (size_t)i + c];
		a.x[6 * (size_t)i + r] = s;
	}
#ifdef CUBA_PCG_TIMING
	if (tid == 0 && aa.timing) { for (int i = 0; i < 7; i++) aa.timing[(size_t)cta * 8 + i] = tacc[i]; aa.timing[(size_t)cta * 8 + 7] = it; }
#endif
	if (cta == 0 && tid == 0) { a.status->iters = it; a.status->status = status; a.status->rz0 = rho0; a.status->rz = rho; }
}

// ---- coarse-level setup ------------------------------------------------------------------------------------------

// Z_i = Ad(T_i) for every free pose: delta = [omega; upsilon], Ad = [[R, 0], [[t]x R, R]] (column-major 6x6)
template <typename T>
__global__ void k_coarse_basis(const T* __restrict__ pose, int numP, T* Zx)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= numP) return;
	const T* p = pose + 8 * (size_t)i;
	const T x = p[0], y = p[1], z = p[2], w = p[3], tx = p[4], ty = p[5], tz = p[6];
	T R[3][3];
	R[0][0] = 1 - 2 * (y * y + z * z); R[0][1] = 2 * (x * y - z * w); R[0][2] = 2 * (x * z + y * w);
	R[1][0] = 2 * (x * y + z * w); R[1][1] = 1 - 2 * (x * x + z * z); R[1][2] = 2 * (y * z - x * w);
	R[2][0] = 2 * (x * z - y * w); R[2][1] = 2 * (y * z + x * w); R[2][2] = 1 - 2 * (x * x + y * y);
	const T K[3][3] = { { T(0), -tz, ty }, { tz, T(0), -tx }, { -ty, tx, T(0) } };
	T* Z = Zx + 36 * (size_t)i;
	for (int c = 0; c < 3; c++)
		for (int r = 0; r < 3; r++) {
			Z[c * 6 + r] = R[r][c];                              // top-left R
			Z[(c + 3) * 6 + r] = T(0);                           // top-right 0
			Z[(c + 3) * 6 + r + 3] = R[r][c];                    // bottom-right R
			Z[c * 6 + r + 3] = K[r][0] * R[0][c] + K[r][1] * R[1][c] + K[r][2] * R[2][c];   // bottom-left [t]x R
		}
}

// U_n = Z_i^T S_n Z_j for every block n = (i,j) of the symmetric-full BSR: one thread per (block, entry)
template <typename T>
__global__ void k_coarse_project(const T* __restrict__ fVal, const int* __restrict__ fRowOf, const int* __restrict__ fColInd, int nfull,
	const T* __restrict__ Zx, double* U)
{
	const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
	if (e >= 36LL * nfull) return;
	const int n = (int)(e / 36), rc = (int)(e - 36LL * n), c = rc / 6, r = rc - 6 * c;
	const T* Sb = fVal + 36 * (size_t)n;
	const T* Zi = Zx + 36 * (size_t)fRowOf[n] + r * 6;        // column r of Z_i
	const T* Zj = Zx + 36 * (size_t)fColInd[n] + c * 6;       // column c of Z_j
	double zj[6];
#pragma unroll
	for (int m = 0; m < 6; m++) zj[m] = (double)Zj[m];
	double s = 0;
#pragma unroll
	for (int k = 0; k < 6; k++) {
		double t = 0;
#pragma unroll
		for (int m = 0; m < 6; m++) t += (double)Sb[m * 6 + k] * zj[m];      // (S Z_j)(k,c)
		s += (double)Zi[k] * t;
	}
	U[e] = s;
}

// Ac = Z^T S Z, lower block triangle, packed: block (ib >= jb) at (ib (ib+1)/2 + jb) * 36, column-major 6x6.
// cbPtr/cbList: the fine blocks of every coarse block in ascending order (built on the host) -> fixed-order sums.
__global__ void k_coarse_assemble(const int* __restrict__ cbPtr, const int* __restrict__ cbList, const double* __restrict__ U, int nblkP, double* AcP)
{
	const int e = blockIdx.x * blockDim.x + threadIdx.x;
	if (e >= nblkP * 36) return;
	const int bp = e / 36, rc = e - 36 * bp;
	double s0 = 0, s1 = 0;
	int k = cbPtr[bp];
	const int k1 = cbPtr[bp + 1];
	for (; k + 1 < k1; k += 2) { s0 += U[36 * (size_t)cbList[k] + rc]; s1 += U[36 * (size_t)cbList[k + 1] + rc]; }
	if (k < k1) s0 += U[36 * (size_t)cbList[k] + rc];
	AcP[e] = s0 + s1;
}

// AcInv = Ac^-1 by block Cholesky (6x6 blocks) of the packed lower triangle in shared memory: ONE CTA.
// On a non-positive pivot the inverse is zeroed (the preconditioner degrades to block-Jacobi, still valid).
template <typename T>
__global__ void __launch_bounds__(1024, 1) k_coarse_invert(const double* __restrict__ AcP, int A, float* AcInv, int* info)
{
	extern __shared__ __align__(16) unsigned char smem_raw[];
	double* B = reinterpret_cast<double*>(smem_raw);             // [nblkP][36] packed blocks
	const int nblkP = A * (A + 1) / 2, nc = 6 * A;
	double* sLi = B + (size_t)nblkP * 36;                        // [A][36] inverses of the diagonal factors
	double* sRow = sLi + (size_t)A * 36;                         // [A][36] scratch row
	__shared__ int s_fail;
	__shared__ unsigned char s_ib[PCG4_MAXAGG1 * (PCG4_MAXAGG1 + 1) / 2], s_jb[PCG4_MAXAGG1 * (PCG4_MAXAGG1 + 1) / 2];   // packed index -> (ib, jb)
	__shared__ double s_L[36], s_id[6];
	const int tid = threadIdx.x, NT = blockDim.x;
	auto idx = [](int ib, int jb) { return (size_t)(ib * (ib + 1) / 2 + jb) * 36; };
	for (int e = tid; e < nblkP * 36; e += NT) B[e] = AcP[e];
	for (int ib = tid; ib < A; ib += NT) for (int jb = 0; jb <= ib; jb++) { s_ib[ib * (ib + 1) / 2 + jb] = (unsigned char)ib; s_jb[ib * (ib + 1) / 2 + jb] = (unsigned char)jb; }
	if (tid == 0) s_fail = 0;
	__syncthreads();
	// ---- phase 1: block Cholesky, L overwrites the triangle ----
	for (int kb = 0; kb < A; kb++) {
		if (tid < 32) {
			// 6x6 Cholesky of the diagonal block in place (lane r owns row r), then L^-1 column by column (lane q owns column q)
			double* D = B + idx(kb, kb);
			const int r = tid;
			for (int j = 0; j < 6; j++) {
				const double d = D[j * 6 + j];
				if (!(d > 0)) { if (r == 0) s_fail = 1; break; }
				const double sq = sqrt(d);
				__syncwarp();
				if (r == j) D[j * 6 + j] = sq;
				else if (r > j && r < 6) D[j * 6 + r] = D[j * 6 + r] / sq;
				__syncwarp();
				if (r > j && r < 6)
					for (int c = j + 1; c <= r; c++) D[c * 6 + r] -= D[j * 6 + r] * D[j * 6 + c];
				__syncwarp();
			}
			__syncwarp();
			if (r < 6) {
				for (int c = r + 1; c < 6; c++) D[c * 6 + r] = 0.0;       // the strict upper part is not part of L
				s_id[r] = 1.0 / D[r * 6 + r];
			}
			__syncwarp();
			if (r < 6) {
				const int q = r;                                           // column q of Li = L^-1
				double col[6];
				for (int i = 0; i < 6; i++) col[i] = 0.0;
				col[q] = s_id[q];
				for (int i = q + 1; i < 6; i++) {
					double sum = 0;
					for (int k = q; k < i; k++) sum += D[k * 6 + i] * col[k];
					col[i] = -sum * s_id[i];
				}
				for (int i = 0; i < 6; i++) sLi[(size_t)kb * 36 + q * 6 + i] = col[i];
			}
		}
		__syncthreads();
		if (s_fail) break;
		// panel: B(ib,kb) <- B(ib,kb) L_kk^-T, one thread per (block, row)
		const double* Li = sLi + (size_t)kb * 36;
		for (int w = tid; w < (A - kb - 1) * 6; w += NT) {
			const int ib = kb + 1 + w / 6, r = w % 6;
			double* X = B + idx(ib, kb);
			double x[6], y[6];
			for (int k = 0; k < 6; k++) x[k] = X[k * 6 + r];
			for (int c = 0; c < 6; c++) { double s = 0; for (int k = 0; k <= c; k++) s += x[k] * Li[k * 6 + c]; y[c] = s; }   // (X Li^T)(r,c) = sum_k X(r,k) Li(c,k)
			for (int c = 0; c < 6; c++) X[c * 6 + r] = y[c];
		}
		__syncthreads();
		// trailing update: B(ib,jb) -= B(ib,kb) B(jb,kb)^T for kb < jb <= ib
		const int m = A - kb - 1;
		const int nent = m * (m + 1) / 2 * 36;
		for (int w = tid; w < nent; w += NT) {
			const int bq = w / 36, rc = w - 36 * bq, c = rc / 6, r = rc - 6 * c;
			const int ib = kb + 1 + s_ib[bq], jb = kb + 1 + s_jb[bq];
			const double* P = B + idx(ib, kb);
			const double* Q = B + idx(jb, kb);
			double s = 0;
			for (int k = 0; k < 6; k++) s += P[k * 6 + r] * Q[k * 6 + c];
			B[idx(ib, jb) + c * 6 + r] -= s;
		}
		__syncthreads();
	}
	if (s_fail) {
		for (int e = tid; e < nc * nc; e += NT) AcInv[e] = 0.f;
		if (tid == 0 && info) *info = 1;
		return;
	}
	// ---- phase 2: W = L^-1 (block lower triangular), row by row: W(ib,jb) = -L_ii^-1 sum_{k=jb}^{ib-1} L(ib,k) W(k,jb) ----
	for (int ib = 0; ib < A; ib++) {
		for (int w = tid; w < ib * 36; w += NT) {
			const int jb = w / 36, rc = w - 36 * jb, c = rc / 6, r = rc - 6 * c;
			double s = 0;
			for (int k = jb; k < ib; k++) {
				const double* Lb = B + idx(ib, k);
				const double* Wb = B + idx(k, jb);               // rows < ib already hold W (diagonal blocks: W(k,k) = L_kk^-1)
				for (int mm = 0; mm < 6; mm++) s += Lb[mm * 6 + r] * Wb[c * 6 + mm];
			}
			sRow[(size_t)jb * 36 + c * 6 + r] = s;
		}
		__syncthreads();
		const double* Li = sLi + (size_t)ib * 36;
		for (int w = tid; w < (ib + 1) * 36; w += NT) {
			const int jb = w / 36, rc = w - 36 * jb, c = rc / 6, r = rc - 6 * c;
			double v;
			if (jb == ib) v = Li[c * 6 + r];
			else {
				double s = 0;
				for (int k = 0; k <= r; k++) s += Li[k * 6 + r] * sRow[(size_t)jb * 36 + c * 6 + k];   // Li lower: Li(r,k), k <= r
				v = -s;
			}
			B[idx(ib, jb) + c * 6 + r] = v;
		}
		__syncthreads();
	}
	// ---- phase 3: Ac^-1 = W^T W; block (ib,jb), ib >= jb: sum_{k >= ib} W(k,ib)^T W(k,jb) ----
	for (int w = tid; w < nblkP * 36; w += NT) {
		const int bq = w / 36, rc = w - 36 * bq, c = rc / 6, r = rc - 6 * c;
		const int ib = s_ib[bq], jb = s_jb[bq];
		double s = 0;
		for (int k = ib; k < A; k++) {
			const double* Wa = B + idx(k, ib);
			const double* Wb = B + idx(k, jb);
			for (int mm = 0; mm < 6; mm++) s += Wa[r * 6 + mm] * Wb[c * 6 + mm];
		}
		AcInv[(size_t)(ib * 6 + r) * nc + jb * 6 + c] = (float)s;
		AcInv[(size_t)(jb * 6 + c) * nc + ib * 6 + r] = (float)s;
	}
	if (tid == 0 && info) *info = 0;
}


// ------------------------------------------------------------------------------------------------------------------
// The same inversion for up to PCG4_MAXAGG aggregates: the packed triangle (74 aggregates: 2 775 blocks, 800 KB) is
// spread over the shared memory of an 8-CTA thread-block cluster, block b in CTA b % 8 (distributed shared memory);
// every CTA updates the blocks it owns and reads the others' through cluster.map_shared_rank.  cluster.sync() between
// phases.  Same arithmetic and summation order as k_coarse_invert.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __cluster_dims__(PCG4_CL, 1, 1) __launch_bounds__(1024, 1)
k_coarse_chol_cluster(const double* __restrict__ AcP, int A, double* Lp, double* Ld, float* AcInv, int* info)
{
	namespace cgx = cooperative_groups;
	cgx::cluster_group cluster = cgx::this_cluster();
	extern __shared__ __align__(16) unsigned char smem_raw[];
	const int nblkP = A * (A + 1) / 2, nc = 6 * A;
	const int nloc = (nblkP + PCG4_CL - 1) / PCG4_CL;              // blocks per CTA
	double* Bl = reinterpret_cast<double*>(smem_raw);              // [nloc][36] own blocks: local slot lb holds block lb * 8 + rank
	double* sLiL = Bl + (size_t)nloc * 36;                         // [A][36] inverses of the diagonal factors (rank 0's copy is the one in use)
	double* sScr = sLiL + (size_t)A * 36;                          // [A][36] scratch (phase 2), [36] scratch of the diagonal factorisation
	unsigned char* s_ib = reinterpret_cast<unsigned char*>(sScr + (size_t)A * 36);   // [nblkP] packed index -> (ib, jb)
	unsigned char* s_jb = s_ib + nblkP;
	__shared__ int s_fail;
	const int rank = (int)cluster.block_rank(), tid = threadIdx.x, NT = blockDim.x;
	double* base[PCG4_CL];
#pragma unroll
	for (int r = 0; r < PCG4_CL; r++) base[r] = cluster.map_shared_rank(Bl, r);
	double* sLi0 = cluster.map_shared_rank(sLiL, 0);
	int* fail0 = cluster.map_shared_rank(&s_fail, 0);
	auto blk = [&](int ib, int jb) -> double* { const int b = ib * (ib + 1) / 2 + jb; return base[b & (PCG4_CL - 1)] + (size_t)(b / PCG4_CL) * 36; };
	for (int e = tid; e < nloc * 36; e += NT) {
		const int b = (e / 36) * PCG4_CL + rank;
		Bl[e] = b < nblkP ? AcP[(size_t)b * 36 + (e % 36)] : 0.0;
	}
	for (int ib = tid; ib < A; ib += NT) for (int jb = 0; jb <= ib; jb++) { s_ib[ib * (ib + 1) / 2 + jb] = (unsigned char)ib; s_jb[ib * (ib + 1) / 2 + jb] = (unsigned char)jb; }
	if (tid == 0) s_fail = 0;
	cluster.sync();
	// ---- phase 1: block Cholesky.  Every CTA factors the (already final) diagonal block itself -- two cluster barriers per
	//      block column instead of three, and the panel reads its own copy of L_kk^-1 ----
	for (int kb = 0; kb < A; kb++) {
		if (tid < 32) {
			double* D = sScr;
			const double* Dg = blk(kb, kb);                     // raw diagonal block: nobody writes it any more
			for (int e = tid; e < 36; e += 32) D[e] = Dg[e];
			__syncwarp();
			const int r = tid;
			for (int j = 0; j < 6; j++) {
				const double d = D[j * 6 + j];
				if (!(d > 0)) { if (r == 0) s_fail = 1; break; }
				const double sq = sqrt(d);
				__syncwarp();
				if (r == j) D[j * 6 + j] = sq;
				else if (r > j && r < 6) D[j * 6 + r] = D[j * 6 + r] / sq;
				__syncwarp();
				if (r > j && r < 6)
					for (int c = j + 1; c <= r; c++) D[c * 6 + r] -= D[j * 6 + r] * D[j * 6 + c];
				__syncwarp();
			}
			__syncwarp();
			__shared__ double s_id[6];
			if (r < 6) {
				for (int c = r + 1; c < 6; c++) D[c * 6 + r] = 0.0;
				s_id[r] = 1.0 / D[r * 6 + r];
			}
			__syncwarp();
			if (r < 6) {
				const int q = r;
				double col[6];
				for (int i = 0; i < 6; i++) col[i] = 0.0;
				col[q] = s_id[q];
				for (int i = q + 1; i < 6; i++) {
					double sum = 0;
					for (int k = q; k < i; k++) sum += D[k * 6 + i] * col[k];
					col[i] = -sum * s_id[i];
				}
				for (int i = 0; i < 6; i++) sLiL[(size_t)kb * 36 + q * 6 + i] = col[i];
			}
			__syncwarp();
			// the factor of the diagonal block goes straight to the output (its shared-memory copy stays raw)
			if (rank == (((kb * (kb + 1)) / 2 + kb) & (PCG4_CL - 1))) for (int e = tid; e < 36; e += 32) Lp[((size_t)kb * (kb + 1) / 2 + kb) * 36 + e] = D[e];
		}
		__syncthreads();
		if (s_fail) { *fail0 = 1; }                                // every CTA computes the same verdict; rank 0's flag is the shared one
		// panel of the blocks this CTA owns
		const double* Li = sLiL + (size_t)kb * 36;
		if (!s_fail)
		for (int w = tid; w < nloc * 6; w += NT) {            // panel: one thread per (own block, row)
			const int lb = w / 6, r = w - 6 * lb, b = lb * PCG4_CL + rank;
			if (b >= nblkP) continue;
			const int ib = s_ib[b], jb = s_jb[b];
			if (jb != kb || ib <= kb) continue;
			double* X = Bl + (size_t)lb * 36;
			double x[6], y[6];
			for (int k = 0; k < 6; k++) x[k] = X[k * 6 + r];
			for (int c = 0; c < 6; c++) { double sm = 0; for (int k = 0; k <= c; k++) sm += x[k] * Li[k * 6 + c]; y[c] = sm; }
			for (int c = 0; c < 6; c++) X[c * 6 + r] = y[c];
		}
		cluster.sync();
		if (*fail0) break;
		for (int w = tid; w < nloc * 36; w += NT) {           // trailing: one thread per (own block, entry)
			const int lb = w / 36, rc = w - 36 * lb, c = rc / 6, r = rc - 6 * c, b = lb * PCG4_CL + rank;
			if (b >= nblkP) continue;
			const int ib = s_ib[b], jb = s_jb[b];
			if (jb <= kb) continue;                            // ib >= jb > kb
			const double* P = blk(ib, kb);
			const double* Q = blk(jb, kb);
			double sm = 0;
			for (int k = 0; k < 6; k++) sm += P[k * 6 + r] * Q[k * 6 + c];
			Bl[(size_t)lb * 36 + rc] -= sm;
		}
		cluster.sync();
	}
	if (*fail0) {
		for (int e = rank * NT + tid; e < nc * nc; e += PCG4_CL * NT) AcInv[e] = 0.f;
		if (rank == 0 && tid == 0 && info) *info = 1;
		cluster.sync();
		return;
	}
	// ---- the factor L (packed, block b at Lp + 36 b) and the inverses of its diagonal blocks leave for k_coarse_trinv ----
	for (int e = tid; e < nloc * 36; e += NT) {
		const int b = (e / 36) * PCG4_CL + rank;
		if (b < nblkP && s_ib[b] != s_jb[b]) Lp[(size_t)b * 36 + (e % 36)] = Bl[e];     // diagonal factors were written in phase 1
	}
	if (rank == 0) for (int e = tid; e < A * 36; e += NT) Ld[e] = sLiL[e];
	if (rank == 0 && tid == 0 && info) *info = 0;
	cluster.sync();                                            // nobody leaves while its shared memory may still be read
}


// at most one coarse aggregate per CTA of k_pcg5 (about nine poses each)
constexpr int PCG5_MAXAGG = 148;

// W = L^-1 (block lower triangular), one CTA per block column jb: W(jb,jb) = L_jj^-1,
// W(ib,jb) = -L_ii^-1 sum_{k=jb}^{ib-1} L(ib,k) W(k,jb).  The columns are independent; a column is sequential in ib.
constexpr int PCG4_KS = 7;      // k-slices of the inner sum (36 entries x 7 slices = 252 threads)
__global__ void __launch_bounds__(256) k_coarse_trinv(const double* __restrict__ Lp, const double* __restrict__ Ld, int A, double* Wp, const int* __restrict__ info)
{
	extern __shared__ __align__(16) unsigned char smem_raw[];
	double* Wcol = reinterpret_cast<double*>(smem_raw);          // [A][36] this column of W (rows < jb unused)
	__shared__ double s_part[PCG4_KS][36], s_S[36];
	if (*info != 0) return;
	const int jb = blockIdx.x, tid = threadIdx.x;
	const int e = tid % 36, sl = tid / 36, c = e / 6, r = e - 6 * c;
	auto pidx = [](int ib, int kb) { return (size_t)(ib * (ib + 1) / 2 + kb) * 36; };
	if (tid < 36) { const double v = Ld[(size_t)jb * 36 + tid]; Wcol[(size_t)jb * 36 + tid] = v; Wp[pidx(jb, jb) + tid] = v; }
	__syncthreads();
	for (int ib = jb + 1; ib < A; ib++) {
		if (sl < PCG4_KS) {
			double sm = 0;
			for (int k = jb + sl; k < ib; k += PCG4_KS) {
				const double* Lb = Lp + pidx(ib, k);
				const double* Wb = Wcol + (size_t)k * 36;
#pragma unroll
				for (int mm = 0; mm < 6; mm++) sm += Lb[mm * 6 + r] * Wb[c * 6 + mm];
			}
			s_part[sl][e] = sm;
		}
		__syncthreads();
		if (tid < 36) {
			double sm = 0;
#pragma unroll
			for (int q = 0; q < PCG4_KS; q++) sm += s_part[q][tid];
			s_S[tid] = sm;
		}
		__syncthreads();
		if (tid < 36) {
			const double* Li = Ld + (size_t)ib * 36;
			double sm = 0;
			for (int k = 0; k <= r; k++) sm += Li[k * 6 + r] * s_S[c * 6 + k];
			Wcol[(size_t)ib * 36 + tid] = -sm;
			Wp[pidx(ib, jb) + tid] = -sm;
		}
		__syncthreads();
	}
}

// Ac^-1 = W^T W: one thread per entry of the lower block triangle, written to both triangles of the full fp32 matrix
__global__ void k_coarse_wtw(const double* __restrict__ Wp, int A, float* AcInv, const int* __restrict__ info)
{
	const int w = blockIdx.x * blockDim.x + threadIdx.x;
	const int nblkP = A * (A + 1) / 2, nc = 6 * A;
	if (w >= nblkP * 36 || *info != 0) return;
	const int bq = w / 36, rc = w - 36 * bq, c = rc / 6, r = rc - 6 * c;
	int ib = (int)((sqrt(8.0 * bq + 1.0) - 1.0) * 0.5);
	while ((ib + 1) * (ib + 2) / 2 <= bq) ib++;
	while (ib * (ib + 1) / 2 > bq) ib--;
	const int jb = bq - ib * (ib + 1) / 2;
	double s0 = 0, s1 = 0;
	int k = ib;
	for (; k + 1 < A; k += 2) {
		const double* Wa = Wp + (size_t)(k * (k + 1) / 2 + ib) * 36, *Wb = Wp + (size_t)(k * (k + 1) / 2 + jb) * 36;
		const double* Wa1 = Wp + (size_t)((k + 1) * (k + 2) / 2 + ib) * 36, *Wb1 = Wp + (size_t)((k + 1) * (k + 2) / 2 + jb) * 36;
#pragma unroll
		for (int mm = 0; mm < 6; mm++) { s0 += Wa[r * 6 + mm] * Wb[c * 6 + mm]; s1 += Wa1[r * 6 + mm] * Wb1[c * 6 + mm]; }
	}
	if (k < A) {
		const double* Wa = Wp + (size_t)(k * (k + 1) / 2 + ib) * 36, *Wb = Wp + (size_t)(k * (k + 1) / 2 + jb) * 36;
#pragma unroll
		for (int mm = 0; mm < 6; mm++) s0 += Wa[r * 6 + mm] * Wb[c * 6 + mm];
	}
	const float v = (float)(s0 + s1);
	AcInv[(size_t)(ib * 6 + r) * nc + jb * 6 + c] = v;
	AcInv[(size_t)(jb * 6 + c) * nc + ib * 6 + r] = v;
}

}  // namespace cuba_b200
