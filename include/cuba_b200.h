/*
 * cuba_b200.h -- C ABI of the B200-native Levenberg-Marquardt bundle-adjustment engine.
 *
 * This is the drop-in boundary for the ONE hot path of fixstars/cuda-bundle-adjustment:
 * everything the reference's CudaBlockSolver does below `optimize()` (paths relative to the reference
 * checkout):
 *
 *   what this ABI replaces                                   reference interface
 *   ------------------------------------------------------   -------------------------------------------------
 *   cuba_engine_set_problem   (flat arrays -> device, + all   CudaBlockSolver::initialize/buildStructure,
 *                              sparsity structures)           src/cuda_bundle_adjustment.cpp:115-366;
 *                                                             gpu::buildHplStructure / findHschureMulBlockIndices,
 *                                                             src/cuda_block_solver.h:36-41;
 *                                                             HschurSparseBlockMatrix, src/sparse_block_matrix.h:81-98
 *   cuba_engine_optimize      (whole LM loop)                 CudaBundleAdjustmentImpl::optimize, cpp:793-857
 *   cuba_stage_linearize      (residual+Jacobian+Hessian)     gpu::computeActiveErrors + gpu::constructQuadraticForm,
 *                                                             src/cuda_block_solver.h:43-57
 *   cuba_stage_max_diagonal                                   gpu::maxDiagonal, h:65-67
 *   cuba_stage_solve          (Schur + PCG + back-subst.)     gpu::addLambda/computeBschure/computeHschure/
 *                                                             convertHschureBSRToCSR/schurComplementPost, h:69-88 and
 *                                                             SparseLinearSolver::solve, src/cuda_linear_solver.h:28-39
 *   cuba_stage_update         (SE3 exp update + trial chi2)   gpu::updatePoses/updateLandmarks/computeScale, h:90-94
 *   cuba_engine_get_state / _get_chi2 / _get_profile          CudaBlockSolver::finalize/getChiSqs/getTimeProfile,
 *                                                             cpp:512-562
 *
 * Plain C types only: pointers and sizes, no torch / Eigen / STL types.  All host arrays are fp64 and
 * column-major where they hold blocks (reference MatView, src/cuda_block_solver.cu:79-85); an engine
 * configured for fp32 narrows at this boundary like the reference's ScalarCast (cpp:54-69).
 *
 * Every function returns CUBA_OK (0) or a negative error code; cuba_last_error() gives the message.
 * The library has NO CPU fallback: without a usable CUDA device every compute entry point fails with
 * CUBA_ERR_CUDA.
 */
#ifndef CUBA_B200_H
#define CUBA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CUBA_OK 0
#define CUBA_ERR_INVALID (-1)  /* bad argument / inconsistent problem                */
#define CUBA_ERR_CUDA (-2)     /* CUDA runtime failure or no device                  */
#define CUBA_ERR_STATE (-3)    /* call order violated (e.g. optimize before problem) */
#define CUBA_ERR_COMM (-4)     /* NCCL failure                                       */

/* robust kernels: reference include/cuda_bundle_adjustment_types.h:213-218, cu:692-727 */
#define CUBA_ROBUST_NONE 0
#define CUBA_ROBUST_HUBER 1
#define CUBA_ROBUST_TUKEY 2

/* edge types: reference include/cuda_bundle_adjustment_types.h:143-148 */
#define CUBA_EDGE_MONOCULAR 0
#define CUBA_EDGE_STEREO 1

/* time-profile buckets: same 8 items as the reference, cpp:77-88,547-557 */
#define CUBA_PROF_INITIALIZE 0
#define CUBA_PROF_BUILD_STRUCTURE 1
#define CUBA_PROF_COMPUTE_ERROR 2
#define CUBA_PROF_BUILD_SYSTEM 3
#define CUBA_PROF_SCHUR_COMPLEMENT 4
#define CUBA_PROF_DECOMP_SYMBOLIC 5   /* always 0: PCG has no symbolic phase */
#define CUBA_PROF_DECOMP_NUMERICAL 6  /* the PCG solve                        */
#define CUBA_PROF_UPDATE 7
#define CUBA_PROF_NUM 8

typedef struct cuba_config {
	int device;            /* CUDA device ordinal, -1 = current device                            */
	int use_fp32;          /* 0 = fp64 (default); 1 = reference's USE_FLOAT32 behaviour; 2 = mixed precision: fp64 engine whose Hpl
	                          blocks -- the dominant 144 B/edge stream -- are STORED in fp32 (80-byte blocks), everything computed
	                          and accumulated in fp64, PCG in fp64 (SURVEY.md 8 f-4)                                        */
	int pcg_max_iters;     /* <=0: default (see DESIGN.md)                                         */
	double pcg_tol;        /* stop when sqrt(r'z / r0'z0) <= pcg_tol; <=0: default 1e-11 (fp64)    */
	int deterministic;     /* kept for layout compatibility; every kernel sums in a fixed order: results are bit-reproducible run to run */
	int reserved[7];       /* reserved[0]: reduced-system solver.  0 (default) = automatic: block-Jacobi PCG while a solve converges within
	                          reserved[5] iterations (k_pcg3 on one GPU: shared-memory resident, flag-synchronised exchange, no barrier
	                          in the iteration), two-level PCG afterwards (k_pcg5, cuba_pcg5.cuh: block-Jacobi + coarse correction
	                          over rigid motions of pose aggregates in the same flag-synchronised protocol).  With several ranks and
	                          >= 2048 free poses k_pcg5 runs with the block rows DISTRIBUTED over the ranks (NVLink peer boards);
	                          7 = never distribute (replicated solve), 8 = always distribute.  5 = always two-level k_pcg5,
	                          6 = always block-Jacobi k_pcg5, 3 = always k_pcg4 (two-level, one grid barrier per iteration),
	                          4 = always k_pcg3, 2 = k_pcg2 (one grid barrier per iteration)
	                          reserved[1]: 1 = build the index structures on the host (cuba_structure.cpp) instead of
	                          on the device (cuba_structure_gpu.cuh, default); both give identical structures
	                          reserved[2]: J+H landmark kernel, 0 = k_linearize_landmark4 (warp tiles, default; fp32: first generation),
	                          4 = first generation (k_linearize_landmark, 128-edge tiles)
	                          reserved[3]: Schur kernel, 0 or 3 = k_schur3 (six lanes per product)
	                          Any other value of reserved[0..3] makes cuba_engine_create fail with CUBA_ERR_INVALID.
	                          reserved[4]: two-level PCG: solves between rebuilds of the coarse matrix (<=0: 8)
	                          reserved[5]: automatic solver: block-Jacobi iteration count that switches to two-level (<=0: 100)
	                          reserved[6]: two-level PCG: upper bound on the number of pose aggregates (<=0: 74; <= 37 uses the one-CTA inverse) */
} cuba_config;

/* Flat problem: exactly what CudaBlockSolver::initialize produces (cpp:115-261).
 * Vertices are indexed by iP / iL: free vertices first (iP < numP, iL < numL), fixed ones appended.
 * Edges with both ends fixed must not be present.  Edge ids: monocular 0..E2-1, stereo E2..E2+E3-1. */
typedef struct cuba_problem {
	int32_t Pall, numP;
	int32_t Lall, numL;
	const double* q;       /* [4*Pall] unit quaternions, coefficient order x,y,z,w                */
	const double* t;       /* [3*Pall]                                                            */
	const double* cam;     /* [5*Pall] fx,fy,cx,cy,bf per pose                                    */
	const double* Xw;      /* [3*Lall]                                                            */
	int32_t E2;
	const int32_t* idx2;   /* [2*E2] (iP,iL) per monocular edge                                   */
	const double* meas2;   /* [2*E2] (u,v)                                                        */
	const double* omega2;  /* [E2] scalar information                                             */
	int32_t E3;
	const int32_t* idx3;   /* [2*E3]                                                              */
	const double* meas3;   /* [3*E3] (u_left, v, u_right)                                         */
	const double* omega3;  /* [E3]                                                                */
} cuba_problem;

/* reference BatchInfo (include/cuda_bundle_adjustment_types.h:226-232) plus solver diagnostics */
typedef struct cuba_iter_stat {
	int32_t iteration;
	int32_t trials;        /* LM trials spent in this outer iteration (1 = first trial accepted)   */
	double chi2;           /* objective after the iteration (robustified, like the reference)      */
	double lambda;         /* damping after the iteration                                          */
	int32_t pcg_iters;     /* PCG iterations summed over the trials                                */
	int32_t pcg_failed;    /* number of trials whose PCG did not converge / broke down             */
} cuba_iter_stat;

typedef struct cuba_sizes {
	int32_t Pall, numP, Lall, numL, E2, E3;
	int32_t nhpl;          /* free-free edges = Hpl blocks                                         */
	int32_t nblk;          /* upper-triangular Hsc blocks                                          */
	int32_t nmul;          /* Schur block products                                                 */
	int32_t nblk_full;     /* blocks of the symmetric-full BSR used by the PCG                     */
} cuba_sizes;

typedef struct cuba_engine cuba_engine;

const char* cuba_last_error(void);
int cuba_version(void);

int cuba_engine_create(const cuba_config* cfg /* NULL = defaults */, cuba_engine** out);
int cuba_engine_destroy(cuba_engine* e);

/* setRobustKernels (include/cuda_bundle_adjustment.h:93): one kernel per edge type */
int cuba_engine_set_robust_kernel(cuba_engine* e, int edge_type, int kernel_type, double delta);

/* Landmark sharding for multi-GPU runs (one process per GPU).  Must precede set_problem.
 * `nccl_unique_id` = 128 bytes produced by cuba_comm_unique_id() on rank 0 and broadcast by the host
 * (torch.distributed / MPI / a file).  world == 1 disables it. */
int cuba_comm_unique_id(void* out128);
int cuba_engine_set_comm(cuba_engine* e, int rank, int world, const void* nccl_unique_id);

/* Upload the problem and build every index structure (initialize + buildStructure). */
int cuba_engine_set_problem(cuba_engine* e, const cuba_problem* p);
/* Structure reuse (SURVEY.md 8 f-2; on by default): a set_problem whose sizes, fixed/free split and (iP,iL) lists equal those of the
 * problem the engine already holds keeps every device structure (index lists, tiles, product lists, PCG partition) and only
 * uploads the numbers -- repeated local-BA calls on an unchanged graph, e.g. the reference protocol's second initialize()
 * (samples/sample_ba_from_file.cpp:159-161).  The reference rebuilds everything (cpp:263-366).  Results are identical either way. */
int cuba_engine_set_structure_reuse(cuba_engine* e, int enable);
int cuba_engine_get_structure_reuses(cuba_engine* e, long long* count);
/* Replace only the estimate (q,t,Xw), keeping structure -- repeated optimize() on the same graph. */
int cuba_engine_set_state(cuba_engine* e, const double* q, const double* t, const double* Xw);

/* Restore the estimate last given by set_problem / set_state from its device-resident copy (no host
 * traffic): lets a benchmark time optimize() repeatedly with all inputs already in HBM. */
int cuba_engine_reset_state(cuba_engine* e);

int cuba_engine_get_sizes(const cuba_engine* e, cuba_sizes* out);
/* The CUDA stream (cudaStream_t) every kernel of this engine is launched on -- for CUDA-event timing. */
int cuba_engine_get_stream(cuba_engine* e, void** stream);
/* Overwrite a buffer larger than L2 on the engine's stream (benchmark hygiene between timed steps). */
int cuba_engine_flush_l2(cuba_engine* e);

/* optimize(niterations): stats[niterations]; *nstats = number of entries written (cpp:848-851). */
int cuba_engine_optimize(cuba_engine* e, int niterations, cuba_iter_stat* stats, int* nstats);

/* finalize(): current estimate, [4*Pall], [3*Pall], [3*Lall]; any pointer may be NULL */
int cuba_engine_get_state(cuba_engine* e, double* q, double* t, double* Xw);
/* getChiSqs(): non-robust omega*|r|^2 per edge, edge-id order, [E2+E3] */
int cuba_engine_get_chi2(cuba_engine* e, double* per_edge);
/* seconds per profile bucket accumulated since set_problem, [CUBA_PROF_NUM] */
int cuba_engine_get_profile(cuba_engine* e, double* seconds);
/* number of kernels this library launched since create (for bench.py's gpu_launches) */
int cuba_engine_get_launch_count(cuba_engine* e, long long* count);

/* cumulative host->device / device->host bytes copied by this thread's engines (for bench.py's e2e record) */
int cuba_get_transfer_bytes(long long* h2d, long long* d2h);

/* ---- stage-wise entry points (used by optimize(); exported for stage parity tests) ---- */
int cuba_stage_linearize(cuba_engine* e, double* chi2);
int cuba_stage_max_diagonal(cuba_engine* e, double* maxdiag);
/* Schur complement with damping lambda, PCG, back-substitution.  *ok = 0 when PCG failed. */
int cuba_stage_solve(cuba_engine* e, double lambda, int* pcg_iters, int* ok);
/* trial update into the spare state buffer + its chi2 and the LM scale (without the +1e-3) */
int cuba_stage_update(cuba_engine* e, double lambda, double* chi2_trial, double* scale);
/* accept (swap buffers) or reject (keep) the trial state */
int cuba_stage_commit(cuba_engine* e, int accept);
/* residual-only pass on the current state */
int cuba_stage_chi2(cuba_engine* e, double* chi2);

/* ---- debug getters (host copies; blocks column-major; any pointer may be NULL) ---- */
/* Hpl CSC sorted by (iL,iP): colPtr[numL+1], rowInd[nhpl], edge2Hpl[E2+E3] (-1 = no block) */
int cuba_debug_get_hpl_structure(cuba_engine* e, int32_t* colPtr, int32_t* rowInd, int32_t* edge2Hpl);
/* Hsc upper-triangular BSR: rowPtr[numP+1], colInd[nblk] */
int cuba_debug_get_hsc_structure(cuba_engine* e, int32_t* rowPtr, int32_t* colInd);
int cuba_debug_get_system(cuba_engine* e, double* Hpp /*36*numP*/, double* bp /*6*numP*/, double* Hll /*9*numL*/,
	double* bl /*3*numL*/, double* Hpl /*18*nhpl*/);
int cuba_debug_get_schur(cuba_engine* e, double* Hsc /*36*nblk, upper*/, double* bsc /*6*numP*/, double* invHll /*9*numL*/);
int cuba_debug_get_delta(cuba_engine* e, double* xp /*6*numP*/, double* xl /*3*numL*/);

/* Host-only (no CUDA call): builds the index structures from the (iP,iL) lists exactly as
 * cuba_engine_set_problem does and copies them out -- the not-gpu tests check them against the oracle.
 * Sizes are returned first with all array pointers NULL, then the arrays on a second call. */
int cuba_debug_build_structure_host(const cuba_problem* p, int rank, int world, cuba_sizes* sizes,
	int32_t* hplColPtr /*numL+1*/, int32_t* hplRowInd /*nhpl*/, int32_t* edge2Hpl /*E2+E3*/,
	int32_t* hscRowPtr /*numP+1*/, int32_t* hscColInd /*nblk*/,
	int32_t* fullRowPtr /*numP+1*/, int32_t* fullColInd /*nblk_full*/,
	int32_t* shard /*[4]: lmBeg, lmEnd, edges, local products*/);

/* CPU-only check of the host side of the PCG setup (row partition over nCtas persistent CTAs, need lists, pose aggregates and
 * coarse lists of the two-level PCG, csrc/cuba_structure.cpp): builds them for the problem and verifies their invariants.
 * info[8] = G, gs, A, needMax, maxRows, blkMax, maxNeedAgg, size of the coarse lists.  No device needed. */
int cuba_debug_pcg_partition(const cuba_problem* p, int nCtas, int maxAgg, int32_t* info);

/* CPU-only check of the plan of the row-distributed two-level PCG (k_pcg5; csrc/cuba_structure.cpp): rows over world x G virtual
 * CTAs, aggregates aligned with the ranks, halo masks.  info[8] = ok (0: system too small for this kernel), G, gs, A, needMax,
 * maxRows, maxNeedAgg, number of halo rows.  No device needed. */
int cuba_debug_pcg5_plan(const cuba_problem* p, int world, int numSMs, int maxAgg, int32_t* info);
/* The flat arrays the drop-in class (cuba::CudaBundleAdjustment, csrc/cuba_api.cpp) built in its last initialize(): what optimize()
 * hands to cuba_engine_set_problem.  `dropin` is the object's address; the pointers stay valid until the next initialize().
 * Needs no GPU (tests of the graph container: tombstones, re-added edges, fixed vertices, vertices without edges). */
int cuba_debug_dropin_problem(void* dropin, cuba_problem* out);

/* ---- micro-benchmark hooks for bench.py / profiles (device-resident data, CUDA-event timed) ---- */
/* Runs the named stage `reps` times back to back and returns the average device milliseconds per
 * repetition.  stage: 0 linearize (landmark pass + pose pass), 1 landmark pass only, 2 pose pass only,
 * 3 schur, 4 pcg, 5 backsub+update+residual, 6 residual only.  flush_l2 != 0 writes a >L2 buffer
 * between repetitions (outside the timed interval). */
int cuba_bench_stage(cuba_engine* e, int stage, int reps, int flush_l2, double lambda, double* avg_ms);

#ifdef __cplusplus
}
#endif
#endif /* CUBA_B200_H */
