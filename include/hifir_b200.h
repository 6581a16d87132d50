/*
 * hifir_b200.h -- C-ABI of the B200 (sm_100a) device backend for HIFIR's
 * preconditioner-application hot path.
 *
 * A device context is ATTACHED to an already factorized multilevel
 * preconditioner (hif::HIF, reference src/hif/builder.hpp:109-585).  The Crout
 * factorization stays on the host and is not part of this library; its
 * per-level factors (hif::Prec, reference src/hif/alg/Prec.hpp:309-323) are
 * described with plain pointers/sizes in LhfdGpuLevel and uploaded once.
 *
 * Naming/typing follows libhifir (reference libhifir/include/libhifir.h):
 * "lhf" + value-type letter ("d" = double) + "Gpu" + Verb, LhfInt = int32,
 * LhfIndPtr = ptrdiff_t (libhifir.h:47-83), LhfStatus / LhfOperationType are the
 * same enums with the same values (libhifir.h:148-165).
 *
 * Every entry point returns LhfStatus and never throws; the message of the last
 * failure on the calling thread is returned by lhfGpuGetErrorMsg().
 *
 * Threading: one handle = one CUDA stream + one workspace; calls on a handle are
 * serialized by the caller (same rule as hif::HIF::solve, which shares a mutable
 * work buffer, builder.hpp:579).  Distinct handles may be driven concurrently.
 */
#ifndef HIFIR_B200_H_
#define HIFIR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- types shared with libhifir (same values; guarded so both headers can be
 * included in one translation unit) ---------------------------------------- */
#ifndef _LIBHIFIR_H
typedef int32_t   LhfInt;    /* libhifir.h:62-66 */
typedef ptrdiff_t LhfIndPtr; /* libhifir.h:81-85 */
typedef enum LhfStatus {     /* libhifir.h:148-154 */
  LHF_SUCCESS = 0,
  LHF_NULL_OBJ,
  LHF_MISMATCHED_SIZES,
  LHF_BAD_PREC,
  LHF_HIFIR_ERROR,
} LhfStatus;
typedef enum LhfOperationType { /* libhifir.h:160-165 */
  LHF_S = 0,
  LHF_SH,
  LHF_M,
  LHF_MH,
} LhfOperationType;
static const int LHF_DEFAULT_RANK = -2; /* libhifir.h:167 */
#endif

/* Opaque device-backend handle (the analogue of LhfdHifHdl, libhifir.h:560-575) */
typedef struct LhfdGpu *LhfdGpuHdl;

/* One compressed-column block exactly as hif::CCS stores it
 * (reference src/hif/ds/CompressedStorage.hpp:55-93, 1810-1915):
 * col_start[ncols+1] (0-based), row_ind[nnz] ascending within a column, vals[nnz].
 * An empty block may pass NULL pointers with nnz == 0. */
typedef struct LhfdGpuCcs {
  size_t           nrows, ncols;
  const LhfIndPtr *col_start;
  const LhfInt *   row_ind;
  const double *   vals;
} LhfdGpuCcs;

/* One level = one hif::Prec (reference src/hif/alg/Prec.hpp:309-323).
 * All pointers are HOST pointers borrowed for the duration of the attach call. */
typedef struct LhfdGpuLevel {
  size_t        m;     /* leading block size              (Prec::m) */
  size_t        n;     /* level system size               (Prec::n) */
  LhfdGpuCcs    L_B;   /* m x m, strictly lower, unit diagonal implicit */
  const double *d_B;   /* m, diagonal of the leading block */
  LhfdGpuCcs    U_B;   /* m x m, strictly upper, unit diagonal implicit */
  LhfdGpuCcs    E;     /* (n-m) x m */
  LhfdGpuCcs    F;     /* m x (n-m) */
  const double *s;     /* n, row scaling */
  const double *t;     /* n, column scaling */
  const LhfInt *p;     /* n, row permutation */
  const LhfInt *p_inv; /* n (only needed by transpose ops; may be NULL) */
  const LhfInt *q;     /* n (only needed by transpose ops; may be NULL) */
  const LhfInt *q_inv; /* n, inverse column permutation */
  /* Dense last level: state of hif::QRCP<double> after factorize()
   * (reference src/hif/small_scale/QRCP.hpp:107-179, members :544-555).
   * dense_n == 0 on every level but the last. */
  size_t        dense_n;    /* order of the final Schur complement (n-m of last level) */
  size_t        dense_rank; /* numerical rank found by QRCP (_rank) */
  const double *qr_mat;     /* dense_n x dense_n column-major: R on/above diag, Householder vectors below (_mat) */
  const double *qr_tau;     /* dense_n (_tau) */
  const LhfInt *qr_jpvt;    /* dense_n, 1-BASED column pivots verbatim (_jpvt) */
  int           has_symm_dense; /* non-zero if Prec::symm_dense_solver is in use -> attach refuses (LHF_BAD_PREC) */
} LhfdGpuLevel;

/* ---- life cycle ---------------------------------------------------------- */

/* Upload the factors of an already factorized preconditioner to `device` and
 * build the device-side schedule.  Replaces nothing in the reference: it is the
 * new boundary between hif::HIF (L3) and prec_solve (L2a), SURVEY.md section 1.
 * Refuses (LHF_BAD_PREC) symmetric dense factors (SYEIG), >2^31-1 nnz per block.
 * The host object may be destroyed after the call returns. */
LhfStatus lhfdGpuAttachLevels(int device, size_t nlevels, const LhfdGpuLevel *levels,
                              LhfdGpuHdl *out);

/* cf. lhfdDestroy (libhifir.h:619) */
LhfStatus lhfdGpuDestroy(LhfdGpuHdl hdl);

/* Give the handle the user matrix A needed by iterative refinement and the
 * Krylov drivers -- the role of lhfdCreateMatrix + the A argument of lhfdSetup
 * (libhifir.h:327-331, 634-636).  is_rowmajor != 0: CRS, else CCS (converted to
 * CRS at upload).  Arrays are copied to the device. */
LhfStatus lhfdGpuSetMatrix(LhfdGpuHdl hdl, int is_rowmajor, size_t n, const LhfIndPtr *indptr,
                           const LhfInt *indices, const double *vals);

/* hif::HIF::nsp = create_nsp_filter(start, end) in constant mode
 * (reference src/hif/NspFilter.hpp:139-175, 190).  end == (size_t)-1 -> n. */
LhfStatus lhfdGpuSetNspConst(LhfdGpuHdl hdl, size_t start, size_t end);
/* The same for the TRANSPOSED solve (LHF_SH): hif::HIF::nsp_tran, applied by hif::HIF::solve(b, x, true)
 * instead of nsp (builder.hpp:421-422).  Without it a transposed solve is not filtered, as in the
 * reference. */
LhfStatus lhfdGpuSetNspTranConst(LhfdGpuHdl hdl, size_t start, size_t end);
LhfStatus lhfdGpuClearNsp(LhfdGpuHdl hdl);

/* Run all work of this handle on `cuda_stream` (a cudaStream_t passed as void*; NULL is
 * the legacy default stream) or, with use_own_stream != 0, on the handle's own
 * non-blocking stream (the state after attach).  Lets a host framework (e.g. torch)
 * time the kernels with events on its current stream. */
LhfStatus lhfdGpuSetStream(LhfdGpuHdl hdl, void *cuda_stream, int use_own_stream);
/* block until all work queued on the handle's stream finished */
LhfStatus lhfdGpuSynchronize(LhfdGpuHdl hdl);

/* ---- the hot path, HOST buffers (drop-in for libhifir) --------------------- */

/* x = M^{-1} b. Drop-in for lhfdSolve (libhifir.h:698, libhifir.cpp:151-158)
 * = hif::HIF::solve(b, x) (builder.hpp:409-423), last-level rank = numerical. */
LhfStatus lhfdGpuSolve(LhfdGpuHdl hdl, const double *b, double *x);

/* lhfdGpuSolve without the wait: the copy of b to the device, the apply and the copy of x back are
 * enqueued as a three-stage pipeline over two staging slots, so that consecutive calls overlap
 * (H2D of call k+1, apply of call k, D2H of call k-1).  b and x (pinned host memory for true
 * overlap) must stay valid, and x must not be read, until lhfdGpuSynchronize(hdl) returns.
 * Same arithmetic and result as lhfdGpuSolve (libhifir.cpp:151-158 semantics); errors of the
 * enqueued work surface at lhfdGpuSynchronize. */
LhfStatus lhfdGpuSolveAsync(LhfdGpuHdl hdl, const double *b, double *x);

/* Drop-in for lhfdApply (libhifir.h:685-688, libhifir.cpp:447-472): same `op`,
 * `nirs`, `betas`, `rank`, `ir_status` meaning, including the rank-defaulting
 * rule (libhifir.cpp:453-455) and the fact that the plain solve path ignores
 * `rank`.  All four operations run on the device: LHF_S = prec_solve, LHF_SH =
 * prec_solve_tran (prec_solve.hpp:541-612), LHF_M / LHF_MH = prec_prod / prec_prod_tran
 * (prec_prod.hpp:54-230).  The transposed operations are served by a transposed twin of
 * the preconditioner built on first use (needs p_inv and q of every level).
 * nirs > 1 needs lhfdGpuSetMatrix. */
LhfStatus lhfdGpuApply(LhfdGpuHdl hdl, LhfOperationType op, const double *b, int nirs,
                       const double *betas, int rank, double *x, int *ir_status);

/* X = M^{-1} B for nrhs right-hand sides stored ROW-INTERLEAVED, B[i*nrhs + k]
 * (the Array<std::array<T,Nrhs>> layout of hif::HIF::solve_mrhs,
 * builder.hpp:433-445).  Semantics = nrhs independent HIF::solve calls (the
 * reference's own multilevel mrhs driver is defective, SURVEY.md App. B-1). */
LhfStatus lhfdGpuSolveMrhs(LhfdGpuHdl hdl, size_t nrhs, const double *B, double *X);

/* Right-preconditioned restarted FGMRES with HIFIR inner refinement, and GMRES
 * with the plain HIF apply: the signatures of fgmres_hifir / gmres_hif
 * (reference examples/advanced/gmres.hpp:126-130, 18-21) flattened.
 * flag: 0 success, 1 stagnated, 2 diverged/maxit (gmres.hpp:12-14). */
LhfStatus lhfdGpuFgmres(LhfdGpuHdl hdl, const double *b, int restart, double rtol, int maxit,
                        int full_rank, double *x, int *flag, int *iters, int *num_mv);
LhfStatus lhfdGpuGmres(LhfdGpuHdl hdl, const double *b, int restart, double rtol, int maxit,
                       double *x, int *flag, int *iters);

/* nrhs independent fgmres_hifir / gmres_hif solves with one matrix and one preconditioner.
 * B and X are row-interleaved, B[i*nrhs + k].  flag / iters / num_mv are arrays of nrhs
 * entries, or NULL.  The per-column meaning is that of lhfdGpuFgmres / lhfdGpuGmres.
 * The columns run in lockstep on the batched apply; nrhs == 1 is lhfdGpuFgmres / lhfdGpuGmres.
 * nrhs == 0 is a no-op; a null-space filter is refused (as lhfdGpuSolveMrhs). */
LhfStatus lhfdGpuFgmresMrhs(LhfdGpuHdl hdl, size_t nrhs, const double *B, int restart, double rtol,
                            int maxit, int full_rank, double *X, int *flag, int *iters, int *num_mv);
LhfStatus lhfdGpuGmresMrhs(LhfdGpuHdl hdl, size_t nrhs, const double *B, int restart, double rtol,
                           int maxit, double *X, int *flag, int *iters);

/* ---- single-precision factors: hif::HIF<float> (libhifir's lhfs* family, libhifir.h:775-872)
 * and the mixed-precision lhfsd* family (float factors, double vectors; libhifir.h:1231-1280,
 * libhifir.cpp:1192-1229, examples/intermediate/demo_mixedprecision.cpp) ------------------------
 *
 * The level description is LhfdGpuLevel with float value arrays.  On the device the values of
 * the triangular sweeps -- the bulk of an apply's traffic -- are STORED in single precision
 * (8 instead of 12 bytes per streamed entry); every accumulation and every vector of the apply
 * is double, i.e. at least as accurate as the reference's float work vector (builder.hpp:125-131,
 * prec_solve.hpp:341-342).  Parity gate against the reference's single-precision apply: relative
 * 1e-5 (BASELINE.json north_star). */
typedef struct LhfsGpu *LhfsGpuHdl;

typedef struct LhfsGpuCcs { /* hif::CCS<float,int> */
  size_t           nrows, ncols;
  const LhfIndPtr *col_start;
  const LhfInt *   row_ind;
  const float *    vals;
} LhfsGpuCcs;

typedef struct LhfsGpuLevel { /* hif::Prec<float,int,ptrdiff_t>; fields as LhfdGpuLevel */
  size_t        m, n;
  LhfsGpuCcs    L_B;
  const float * d_B;
  LhfsGpuCcs    U_B, E, F;
  const float * s, *t;
  const LhfInt *p, *p_inv, *q, *q_inv;
  size_t        dense_n, dense_rank;
  const float * qr_mat, *qr_tau; /* hif::QRCP<float>: _mat, _tau */
  const LhfInt *qr_jpvt;
  int           has_symm_dense;
} LhfsGpuLevel;

LhfStatus lhfsGpuAttachLevels(int device, size_t nlevels, const LhfsGpuLevel *levels, LhfsGpuHdl *out);
LhfStatus lhfsGpuDestroy(LhfsGpuHdl hdl); /* cf. lhfsDestroy, libhifir.h:775 */

/* The same handle viewed as an LhfdGpuHdl: every lhfdGpu* entry point that takes DOUBLE vectors
 * (SolveDev, ApplyDev, SolveMrhs, Fgmres, SetNspConst, SetStream, GetStats, ...) serves a
 * single-precision preconditioner through it.  Destroy with either lhfsGpuDestroy or
 * lhfdGpuDestroy, once. */
LhfdGpuHdl lhfsGpuAsDouble(LhfsGpuHdl hdl);

/* user matrix for refinement: single precision (lhfsSetup/lhfsUpdate, libhifir.h:790-800; widened at
 * upload) or double (lhfsdUpdate, libhifir.h:1231 -- the mixed-precision refinement computes its
 * residuals with the double matrix) */
LhfStatus lhfsGpuSetMatrix(LhfsGpuHdl hdl, int is_rowmajor, size_t n, const LhfIndPtr *indptr,
                           const LhfInt *indices, const float *vals);
LhfStatus lhfsdGpuUpdate(LhfsGpuHdl hdl, int is_rowmajor, size_t n, const LhfIndPtr *indptr,
                         const LhfInt *indices, const double *vals);

/* drop-ins for lhfsSolve / lhfsApply (libhifir.h:841-854): float vectors (widened / narrowed on
 * the device) and for lhfsdSolve / lhfsdApply (libhifir.h:1267-1280): double vectors.  Same op /
 * nirs / betas / rank / ir_status semantics as lhfdGpuApply. */
LhfStatus lhfsGpuSolve(LhfsGpuHdl hdl, const float *b, float *x);
LhfStatus lhfsGpuApply(LhfsGpuHdl hdl, LhfOperationType op, const float *b, int nirs, const double *betas,
                       int rank, float *x, int *ir_status);
LhfStatus lhfsdGpuSolve(LhfsGpuHdl hdl, const double *b, double *x);
LhfStatus lhfsdGpuApply(LhfsGpuHdl hdl, LhfOperationType op, const double *b, int nirs, const double *betas,
                        int rank, double *x, int *ir_status);

/* ---- factor arena files (SURVEY.md 8f: the reference has matrix IO, utils/io.hpp:76-303, but no
 * on-disk form of a factorized preconditioner) ----------------------------------------------
 *
 * lhf?GpuSaveLevels writes the level description -- what lhf?GpuAttachLevels consumes, integers
 * verbatim, values in the precision of the preconditioner -- and, with with_plans != 0, the result
 * of the attach-time analysis of every L_B / U_B (sweep form + algebraic level merging).  It is plain
 * host code: no GPU is needed to write a file.  lhf?GpuAttachFile = lhf?GpuAttachLevels on the arrays
 * read back (results are bit-identical to attaching the live object), skipping the analysis when the
 * file carries plans; a later process needs neither the hif::HIF object nor its factorization.
 * Files end in a checksum; a corrupt or foreign file is refused (LHF_BAD_PREC / LHF_HIFIR_ERROR). */
LhfStatus lhfdGpuSaveLevels(size_t nlevels, const LhfdGpuLevel *levels, int with_plans, const char *path);
LhfStatus lhfsGpuSaveLevels(size_t nlevels, const LhfsGpuLevel *levels, int with_plans, const char *path);
LhfStatus lhfdGpuAttachFile(int device, const char *path, LhfdGpuHdl *out);
LhfStatus lhfsGpuAttachFile(int device, const char *path, LhfsGpuHdl *out);
/* info = {format version, single precision, levels, n, nnz of all blocks, has plans, entries of the
 * stored plans, their total dependency depth}; reads and verifies the whole file (host only) */
LhfStatus lhfGpuFileInfo(const char *path, size_t info[8]);
/* ---- the hot path, DEVICE buffers (asynchronous on the handle's stream) ---- */

/* lhfdGpuApply on device buffers (no residual bounds): op in {LHF_S, LHF_SH, LHF_M, LHF_MH} */
LhfStatus lhfdGpuApplyDev(LhfdGpuHdl hdl, LhfOperationType op, const double *d_b, int nirs, int rank,
                          double *d_x);

/* as lhfdGpuSolve with an explicit last-level rank: 0 = numerical rank,
 * (size_t)-1 = full (QRCP.hpp:376-377).  b and x may not alias. */
LhfStatus lhfdGpuSolveDev(LhfdGpuHdl hdl, const double *d_b, double *d_x, size_t rank);
LhfStatus lhfdGpuSolveMrhsDev(LhfdGpuHdl hdl, size_t nrhs, const double *d_B, double *d_X,
                              size_t rank);
/* hif::HIF::hifir fixed-count variant (builder.hpp:458-465, IterRefine.hpp:77-105) */
LhfStatus lhfdGpuHifirDev(LhfdGpuHdl hdl, const double *d_b, size_t nirs, double *d_x,
                          size_t rank);
/* hif::HIF::hifir, fixed count (as lhfdGpuHifirDev), on a row-interleaved device block */
LhfStatus lhfdGpuHifirMrhsDev(LhfdGpuHdl hdl, size_t nrhs, const double *d_B, size_t nirs,
                              double *d_X, size_t rank);
/* y = A x with the matrix given to lhfdGpuSetMatrix (mt::multiply_nt, mt_mv.hpp:57-73) */
LhfStatus lhfdGpuSpmvDev(LhfdGpuHdl hdl, const double *d_x, double *d_y);

/* ---- introspection -------------------------------------------------------- */

enum {
  LHF_GPU_STAT_LEVELS = 0,      /* number of hif::Prec levels */
  LHF_GPU_STAT_N,               /* system size of level 0 */
  LHF_GPU_STAT_NNZ,             /* nnz(L_B)+nnz(U_B)+nnz(E)+nnz(F) over levels + m (diag) */
  LHF_GPU_STAT_DENSE_N,         /* order of the dense Schur block */
  LHF_GPU_STAT_DENSE_RANK,      /* its numerical rank */
  LHF_GPU_STAT_BYTES_FACTORS,   /* algorithmic factor bytes per apply (SURVEY.md 8d) */
  LHF_GPU_STAT_BYTES_VEC_PER_RHS, /* algorithmic vector bytes per apply per rhs */
  LHF_GPU_STAT_BYTES_DENSE,     /* algorithmic dense-level bytes per apply */
  LHF_GPU_STAT_DEVICE_BYTES,    /* bytes of HBM held by the handle */
  LHF_GPU_STAT_KERNELS_PER_APPLY, /* kernels launched by one nrhs=1 apply */
  LHF_GPU_STAT_DEPTH_TOTAL,     /* sum of dependency depths of all triangular sweeps in one apply */
  LHF_GPU_STAT_LAUNCH_COUNT,    /* kernels launched by this handle since attach */
  LHF_GPU_STAT_DEPTH_MERGED,    /* the same sum after the algebraic level merging done at attach */
  LHF_GPU_STAT_SWEEP_BYTES,     /* bytes of the merged, packed factors streamed by the sweeps of one apply */
  LHF_GPU_STAT_SWEEP_ENTRIES,   /* entries (= gathers of one solution value) of those sweeps per apply */
  LHF_GPU_NUMBER_STATS
};
LhfStatus lhfdGpuGetStats(LhfdGpuHdl hdl, size_t stats[/* LHF_GPU_NUMBER_STATS */]);

/* Instrumented apply: as lhfdGpuSolveDev, but records a CUDA event after every kernel of
 * the schedule, synchronizes, and reports each kernel's duration (milliseconds) with a
 * label such as "lv0.down.L".  names receives the '\n'-separated labels.  For bench /
 * roofline reporting only -- the events serialize nothing but cost launch overhead. */
LhfStatus lhfdGpuProfileSolveDev(LhfdGpuHdl hdl, const double *d_b, double *d_x, size_t rank,
                                 size_t max_entries, float *ms, size_t *count, char *names,
                                 size_t names_len);

/* per-level dependency depth of the L and U sweeps: depth[2*l], depth[2*l+1] */
LhfStatus lhfdGpuGetDepths(LhfdGpuHdl hdl, size_t nlevels, size_t *depth);

/* cf. lhfGetErrorMsg (libhifir.h:203) -- thread-local here, pointer valid until
 * the next failing call on this thread */
const char *lhfGpuGetErrorMsg(void);

/* library version string */
const char *lhfGpuVersion(void);

#ifdef __cplusplus
}
#endif

#endif /* HIFIR_B200_H_ */
