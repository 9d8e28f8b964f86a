/*
 * include/conflux_b200.h -- C ABI of the B200-native CONFLUX LU hot path (libconflux_b200.so).
 *
 * This is the drop-in boundary for ONE path of eth-cscs/conflux: conflux::LU_rep<double> and the parts of
 * conflux::lu_params<double> it needs.  Plain pointers and sizes only; every function returns 0 on success or
 * a negative status code (never throws, never aborts); cflx_last_error() gives the message of the last failure
 * on the calling thread.  SPMD like the reference: one host thread (or process) per rank = per GPU; every
 * entry point that is marked COLLECTIVE must be called by all ranks of the grid in the same order.
 *
 * Reference interfaces replaced (file:line relative to the reference repository):
 *   MPI_Comm / MPI_Init / MPI_Cart_create ............ src/conflux/lu/lu_params.hpp:85-108   -> cflx_comm_*
 *   lu_params<T>::initialize (sizes, grid, comms) .... src/conflux/lu/lu_params.hpp:49-138   -> cflx_lu_create
 *   lu_params<T>::get_p_grid ......................... src/conflux/lu/lu_params.hpp:21-47    -> cflx_auto_grid
 *   lu_params<T>::InitMatrix (seeded generator) ...... src/conflux/lu/lu_params.hpp:364-375  -> cflx_init_matrix_host
 *   lu_params<T>::data (local tiles, ld = Nl) ........ src/conflux/lu/layout.cpp:95-109      -> cflx_lu_set_local
 *   LU_rep<T>(gv, C, permutation) main loop .......... src/conflux/lu/conflux_opt.hpp:343-1827 -> cflx_lu_factor
 *   validation outputs C / permutation ............... src/conflux/lu/conflux_opt.hpp:1660-1771,1822 -> cflx_lu_get_factors
 * Beyond the reference: cflx_lu_solve solves A X = B with the factors where they lie, on the same grid.
 * There is no CPU fallback: without a CUDA device every device entry point returns CFLX_ERR_NO_DEVICE.
 */
#ifndef CONFLUX_B200_H
#define CONFLUX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    CFLX_OK = 0,
    CFLX_ERR_ARG = -1,         /* invalid argument */
    CFLX_ERR_CUDA = -2,        /* CUDA runtime failure */
    CFLX_ERR_NCCL = -3,        /* NCCL failure */
    CFLX_ERR_UNSUPPORTED = -4, /* shape/grid outside the supported envelope (Px != Py, v % 4, ...) */
    CFLX_ERR_STATE = -5,       /* call order violated (e.g. get_factors before factor) */
    CFLX_ERR_NO_DEVICE = -6    /* no CUDA device visible: the library refuses to run (no CPU fallback) */
} cflx_status;

typedef struct cflx_comm cflx_comm; /* process grid handle: one per rank, owns the NCCL communicators */
typedef struct cflx_lu cflx_lu;     /* one factorisation plan: sizes, device buffers, pivot history */

#define CFLX_UNIQUE_ID_BYTES 128

const char* cflx_last_error(void);
const char* cflx_version(void);
int cflx_device_count(int* count);

/* ---- process grid (replaces MPI_COMM_WORLD + MPI_Cart_create/sub) ------------------------------------ */
/* rank 0 creates an id and ships it to the other ranks by any host channel (MPI, torch.distributed, a file) */
int cflx_get_unique_id(void* id_out /* CFLX_UNIQUE_ID_BYTES */);
/* COLLECTIVE.  world_size == 1 needs no id (may be NULL).  device = CUDA ordinal this rank drives. */
int cflx_comm_create(int world_size, int world_rank, const void* unique_id, int device, cflx_comm** out);
int cflx_comm_barrier(cflx_comm*); /* COLLECTIVE: device-side barrier + host synchronisation */
void cflx_comm_destroy(cflx_comm*);

/* page-locked host staging buffers for cflx_lu_set_local (cudaHostAlloc / cudaFreeHost) */
int cflx_host_alloc(size_t bytes, void** out);
int cflx_host_free(void* p);

/* ---- sizes (pure host arithmetic, no device needed) ---------------------------------------------------- */
/* lu_params::get_p_grid for a square matrix: P = 1 -> 1x1x1, 2 -> 1x1x2, 4 -> 2x2x1, 8 -> 2x2x2, ... */
int cflx_auto_grid(int M, int N, int P, int* Px, int* Py, int* Pz);
/* dims_out[8] = {M, N, Ml, Nl, Nt, nlayr, Mt, P} after padding, exactly as lu_params::initialize */
int cflx_lu_dims(int M, int N, int v, int Px, int Py, int Pz, int* dims_out);
/* lu_params::InitMatrix, random branch: fills the Ml x Nl row-major local array of `rank` (layers pk != 0 zero) */
int cflx_init_matrix_host(int M, int N, int v, int Px, int Py, int Pz, int rank, int seed, double* local_out);

/* ---- the factorisation ----------------------------------------------------------------------------------- */
/* COLLECTIVE.  Px <= 0 selects cflx_auto_grid(world_size).  Requires Px == Py, Px*Py*Pz == world_size,
 * v % 4 == 0, (v / Pz) % 4 == 0.  Allocates all device memory of the plan. */
int cflx_lu_create(cflx_comm*, int M, int N, int v, int Px, int Py, int Pz, cflx_lu** out);
/* info_out[16] = {M, N, Ml, Nl, Nt, nlayr, P, Px, Py, Pz, pi, pj, pk, rank, v, 0} */
int cflx_lu_info(const cflx_lu*, int* info_out);
/* host -> device copy of this rank's local matrix (conflux tile layout, row-major, ld = Nl); kept pristine */
int cflx_lu_set_local(cflx_lu*, const double* host_local);
/* Input streaming for back-to-back factorisations (no counterpart in the reference, whose input already sits in host
 * memory): the NEXT cflx_lu_factor uploads `host_next` (page-locked; free again when that call returns) into the input
 * buffer behind its own working copy, on a copy stream, so the transfer overlaps the factorisation; the factorisation
 * after that consumes it without a cflx_lu_set_local.  cflx_lu_validate of a run whose input buffer was handed on is
 * refused (CFLX_ERR_STATE). */
int cflx_lu_queue_next_local(cflx_lu*, const double* host_next);
/* COLLECTIVE.  Runs steps 0..Nt-1 on the GPU(s).  ms_out = device time of the main loop only (CUDA events on
 * this rank's stream, after a grid barrier) -- the region the reference times (conflux_opt.hpp:531-532,1805). */
int cflx_lu_factor(cflx_lu*, double* ms_out);
/* COLLECTIVE.  C_host (Ml x Nl, may be NULL on layers pk != 0): L\U of P*A in the conflux layout, row
 * (k/Px)*v + i of rank (k%Px, pj, 0) = pivoted row k*v + i; permutation_out[M] = pivotIndsBuff. */
int cflx_lu_get_factors(cflx_lu*, double* C_host, int* permutation_out);
/* device -> host copy of the permutation only (the cheap "result" of a run) */
int cflx_lu_get_permutation(cflx_lu*, int* permutation_out);
/* COLLECTIVE.  The reference's validation (examples/conflux_miniapp.cpp:349-500: L = unit-lower(C), U = upper(C),
 * P from the pivots, P*A - L*U with pdgemm on the Px x Py grid, Frobenius norm reduced over the grid) on the GPU grid:
 * frob_abs_out = ||P*A - L*U||_F (what the reference prints), frob_rel_out = that / ||A||_F.  Either may be NULL.
 * Uses the library's own GEMM and NCCL; allocates ~4 local matrices temporarily; identical result on every rank. */
int cflx_lu_validate(cflx_lu*, double* frob_abs_out, double* frob_rel_out);
/* COLLECTIVE.  = cflx_lu_validate(lu, NULL, rel_out) */
int cflx_lu_residual(cflx_lu*, double* rel_out);
/* COLLECTIVE.  Solves A X = B with the factors of the last cflx_lu_factor (P A = L U, A is the padded M x M matrix),
 * nrhs >= 1 right-hand sides, the same nrhs on every rank.
 * B_local: Ml x nrhs, row-major, ld = nrhs -- B in A's ROW distribution: global row g lives on grid row (g / v) % Px
 *          at local row (g / (v*Px))*v + g % v.  Read on ranks with pj == 0 && pk == 0; ignored (may be NULL) elsewhere.
 * X_local: Nl x nrhs, row-major -- X in A's COLUMN distribution: global row g on every rank with pj == (g / v) % Py
 *          (all pi, all pk) at local row (g / (v*Py))*v + g % v.  Written on every rank.
 * ms_out (may be NULL): device time of the solve proper (grid barrier .. last X tile), excluding the upload of B, the
 * read-back of X and the one-time preparation after each factorisation.
 * Does not modify the factors: cflx_lu_get_factors / cflx_lu_validate afterwards return what they returned before.
 * CFLX_ERR_STATE before any cflx_lu_factor or after a cflx_lu_set_local no factorisation has consumed (a streamed
 * factorisation, cflx_lu_queue_next_local, keeps its factors solvable).  As in dgetrs, there is no singularity check. */
int cflx_lu_solve(cflx_lu*, int nrhs, const double* B_local, double* X_local, double* ms_out);
/* 1 when this plan's trailing update runs on the int8 tcgen05 path (ozaki.cu), 0 for the FP64 DMMA kernel (gemm.cu) */
int cflx_lu_uses_tcgen05(const cflx_lu*);
/* number of kernels this plan launched since the last call (for bench.py's gpu_launches) */
int cflx_lu_launch_count(cflx_lu*, int64_t* count_out, int reset);
/* per-phase device time of the last cflx_lu_factor when profiling was enabled: ms_out[8] =
 * {panel, tournament+bcast, row moves, reduce+gather, trsm, gemm, stores, other} */
/* mode 0 off; 1 serialising timers (per-phase device time without overlap); 2 non-serialising timeline: CUDA event
 * pairs on the launching streams, resolved after the run -- the timeline of the real, overlapped execution.  Every region
 * is also an NVTX range named like the reference's semiprof regions (src/conflux/lu/profiler.hpp:5-19: step0_copy,
 * step1_lup, step2_pushingpivots, step4_dtrsm, step6_dgemm, ...). */
int cflx_lu_set_profiling(cflx_lu*, int mode);
int cflx_lu_phase_ms(cflx_lu*, double* ms_out);
/* JSON text {"main": {"step6_dgemm": [ms, count], ...}, "side": {...}} of the last profiled cflx_lu_factor (main stream /
 * look-ahead stream).  Returns 0, or the buffer length needed when buf is NULL or too small. */
int cflx_lu_timeline(cflx_lu*, char* buf, int buf_len);
/* CUDA-event timing of the dominant kernel (the trailing-update DGEMM launches of the last cflx_lu_factor, events
 * recorded on the launching stream): summed device ms and the algorithmic flops 2*m*n*k of those launches */
int cflx_lu_set_kernel_timing(cflx_lu*, int enabled);
int cflx_lu_trailing_stats(cflx_lu*, double* ms_out, double* flops_out);
void cflx_lu_destroy(cflx_lu*);

/* ---- CONFCHOX: Cholesky factorisation A = L L^T (lower) on the same process grid (BASELINE config C5) -----------------
 * Reference interfaces replaced (src/conflux/cholesky):
 *   initialize(argc, argv, N, v, grid)  Cholesky.cpp:60-160 (grid / tile choice :75-134)  -> cflx_chol_auto_grid/_tile, cflx_chol_create
 *   CholeskyIO::generateInputMatrixDistributed  CholeskyIO.cpp:100-172                   -> cflx_chol_init_matrix_host
 *   parallelCholesky()                  Cholesky.cpp:760-921                              -> cflx_chol_factor
 *   finalize(clean)                     Cholesky.cpp:160-175                              -> cflx_chol_destroy
 * Local data: row-major Ml x Nl, tile (gi, gj) of the v x v tiling on rank (gi % Px, gj % Py) at local tile (gi / Px,
 * gj / Py); ranks are numbered (pi * Py + pj) * Pz + pk like the LU path; only the lower triangle is referenced. */
typedef struct cflx_chol cflx_chol;
int cflx_chol_auto_grid(int P, int N, int* grid3_out);
int cflx_chol_auto_tile(int N, int P, int Pz);
/* dims_out[6] = {N padded to a multiple of v, Kappa (tiles per dimension), Ml, Nl, v / Pz, P} */
int cflx_chol_dims(int N, int v, int Px, int Py, int Pz, int* dims_out);
int cflx_chol_init_matrix_host(int N, int v, int Px, int Py, int Pz, int rank, double* local_out);
/* COLLECTIVE.  Px <= 0 / v <= 0 select the reference's automatic choices.  Requires v % 4 == 0, (v / Pz) % 4 == 0, v <= 512. */
int cflx_chol_create(cflx_comm*, int N, int v, int Px, int Py, int Pz, cflx_chol** out);
/* info_out[16] = {N, v, Kappa, Ml, Nl, v / Pz, P, Px, Py, Pz, pi, pj, pk, rank, 0, 0} */
int cflx_chol_info(const cflx_chol*, int* info_out);
int cflx_chol_set_local(cflx_chol*, const double* host_local);
/* COLLECTIVE.  ms_out = device time of the factorisation loop (the region the reference's miniapp times).  A matrix that
 * is not positive definite returns CFLX_ERR_STATE on EVERY rank, and cflx_last_error() names the first failing column,
 * 1-based, like LAPACK dpotrf's info ("... not positive definite ... column <c> ..."); the factor is then not available. */
int cflx_chol_factor(cflx_chol*, double* ms_out);
int cflx_chol_get_local(cflx_chol*, double* L_host);
/* COLLECTIVE.  ||A - L L^T||_F over the lower triangle, absolute and relative to ||A||_F, computed on the GPU grid. */
int cflx_chol_validate(cflx_chol*, double* frob_abs_out, double* frob_rel_out);
int cflx_chol_launch_count(cflx_chol*, int64_t* count_out, int reset);
void cflx_chol_destroy(cflx_chol*);

/* ---- single-device building blocks exposed for tests and micro-benchmarks (host buffers in, host out) ----- */
/* D = beta*C + alpha * AT^T * B with AT [K x M], B [K x N], C/D [M x N], all row-major, dense */
int cflx_dbg_gemm_tn(int M, int N, int K, const double* AT, const double* B, const double* C, double alpha, double beta,
                     double* D, int reps, double* ms_out);
/* partial-pivot LU of an n x v row-major panel: perm_out[v], A00_out[v*v] (L00\U00), LU_out[n*v] rows unpermuted */
int cflx_dbg_panel(int n, int v, const double* panel, int* perm_out, double* A00_out, double* LU_out, int reps,
                   double* ms_out);
/* X = B * U^-1 (right, upper, non-unit; B n x v) and Y = L^-1 * R (left, lower, unit; R v x n), A00 = L\U packed */
int cflx_dbg_trsm(int n, int v, const double* A00, const double* B, double* X_out, const double* R, double* Y_out);
/* X = U^-1 * R (left, upper, non-unit; R v x n row-major), U = upper(A00) -- the diagonal-tile solve of cflx_lu_solve */
int cflx_dbg_trsm_left_upper(int v, int n, const double* A00, const double* R, double* X_out);
/* the diagonal-tile Cholesky of cflx_chol_factor: A v x v row-major (lower triangle referenced), L_out = L (zeros above the
 * diagonal), LT_out = L^T, info_out = dpotrf's info (1-based first non-positive pivot, 0 = success).  blocked = 0: the
 * one-CTA kernel (v % 4 == 0, v <= 512); blocked = 1: 128-wide block columns on the GEMMs (v % 128 == 0, v >= 256), what
 * the factorisation uses for those v. */
int cflx_dbg_potrf_tile(int v, int blocked, const double* A, double* L_out, double* LT_out, int* info_out);
/* D = C - AT^T * B on the int8 tcgen05 path (error-free digit planes, ozaki.cu); K % 128 == 0, N even.  Optional test
 * outputs: digit planes [8][M][K] / [8][N][K], exponents [M] / [N].  ms_out / split_ms_out: mean device time of the GEMM
 * kernel / of the two digit-plane kernels. */
int cflx_dbg_ozaki_gemm(int M, int N, int K, const double* AT, const double* B, const double* C, double* D,
                        signed char* planesA_out, signed char* planesB_out, int* ea_out, int* eb_out, int reps,
                        double* ms_out, double* split_ms_out);
/* raw tensor-pipe rate of back-to-back tcgen05.mma (128 x n x 32 bytes of K, operands resident in shared memory, one
 * CTA per SM): which = 0 kind::i8, 1 kind::f16 on bf16.  tmacs_out = tera-MACs/s (x2 = TOP/s). */
int cflx_dbg_umma_peak(int which, int n, double* tmacs_out);
/* plan_moves + push_phase1..3 + gri bookkeeping on one rank: the npiv pivot rows (local indices >= fnpr, tournament
 * order) are pushed to rows [fnpr, fnpr+npiv) exactly like push_pivots_up (conflux_opt.hpp:176-218, tests/unit/
 * test_utils.cpp:8-84).  n_cols even.  gri_out[n_rows] = new row -> old row, a01_out[npiv*n_cols] = extracted rows. */
int cflx_dbg_push_pivots(int n_rows, int n_cols, double* A_inout, int npiv, const int* pivot_rows, int fnpr, int* gri_out,
                         double* a01_out);
/* cycle counters of CTA 0 of the last cflx_dbg_panel launch: {candidate+argmax, exchange, argmax2, row fetch,
 * eliminate, load/write-back, U12 gather+solve, rank update} */
int cflx_dbg_last_panel_cycles(long long* out8);
/* raw FP64 pipe micro-benchmarks: which = 0 DMMA (mma.sync m8n8k4 f64), 1 DFMA; returns TFLOP/s */
int cflx_dbg_fp64_peak(int which, double* tflops_out);
/* same probe: burst (best of ~2 ms launches) and sustained (one ~0.5 s launch, power-capped) TFLOP/s */
int cflx_dbg_fp64_peak_ex(int which, double* burst_out, double* sustained_out);

#ifdef __cplusplus
}
#endif
#endif /* CONFLUX_B200_H */
