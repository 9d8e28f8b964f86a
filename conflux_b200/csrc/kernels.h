// conflux_b200/csrc/kernels.h -- host-callable launchers of the sm_100a kernels (internal; the public boundary is
// include/conflux_b200.h).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace cflx {

// ---------------------------------------------------------------- gemm.cu
struct GemmArgs {
    int M, N, K;
    const double* AT;  // [K][ldat]  (A transposed: AT[k][m])
    int64_t ldat;
    const double* B;  // [K][ldb]
    int64_t ldb;
    const double* C;  // [M][ldc]   (read only when beta != 0)
    int64_t ldc;
    double* D;  // [M][ldd]   (may alias C)
    int64_t ldd;
    double alpha, beta;
};
int gemm_tn_setup();
int launch_gemm_tn(const GemmArgs& g, cudaStream_t stream);

// ---------------------------------------------------------------- ozaki.cu
// FP64 trailing update on the int8 tcgen05 path (error-free digit planes): C -= L * U with L^T, U K-major in HBM.
struct OzakiWorkspace {
    struct Maps;              // the two CUtensorMap objects (kept out of this header)
    int8_t* planesA = nullptr;  // [8][cap_a][K]
    int8_t* planesB = nullptr;  // [8][cap_b][K]
    int* ea = nullptr;          // [cap_a]
    int* eb = nullptr;          // [cap_b]
    long long* dbg = nullptr;   // [16] cycle counters of CTA 0 (CFLX_OZAKI_DBG=1)
    Maps* maps = nullptr;
    int K = 0, cap_a = 0, cap_b = 0, sms = 0;
};
int ozaki_workspace_create(OzakiWorkspace* ws, int max_rows, int max_cols, int K);
void ozaki_workspace_destroy(OzakiWorkspace* ws);
int ozaki_split_a(OzakiWorkspace* ws, const double* LT, int64_t ld, int n, cudaStream_t s);
int ozaki_split_b(OzakiWorkspace* ws, const double* U, int64_t ld, int col0, int n, cudaStream_t s);
int umma_peak_probe(int n, int use_f16, double* tmacs_out);
int launch_ozaki_gemm(OzakiWorkspace* ws, int M, int N, int row0, int col0, double* C, int64_t ldc, int max_ctas, cudaStream_t s);

// ---------------------------------------------------------------- panel.cu
// Partial-pivot LU of the n x v panel stored TRANSPOSED in W (W[c][r], ld = ldw), in place, rows never move:
// afterwards W[:, r] holds row r of L\U (multipliers left of its pivot column, U from it on, for pivot rows;
// multipliers only for the others).  perm_out[0..v) = LAPACK-equivalent winners (row index chosen at step j,
// identity beyond min(n, v)); see panel.cu for the tie-breaking contract.
struct PanelWorkspace {
    void* slot_hdr;     // [2][148][4]  LL words (payload32, epoch)
    void* slot_rows;    // [2][148][64] LL words
    long long* dbg;     // [8] cycle counters of CTA 0 of the last launch (profiling aid)
    int epoch;          // host-side running epoch (monotonic across launches)
    int max_ctas;       // co-resident CTA budget (<= 148)
    int cta_cap;        // optional cap on the grid (look-ahead: leave SMs to the trailing update); 0 = none
    // column-owner kernel for panels of <= 1024 rows (tournament stacks)
    unsigned* sk_flags;  // [1024] epoch of the last publication of column block b
    int* sk_ppos;        // [v] LAPACK position of every pivot when it was chosen
    unsigned* sk_ticket; // logical CTA ids in start order
    unsigned sk_epoch, sk_ticket_count;
    int sk_enabled;
};
int panel_workspace_create(PanelWorkspace* ws);
void panel_workspace_destroy(PanelWorkspace* ws);
int launch_panel_getrf(double* W, int64_t ldw, int n, int v, int* perm_out, PanelWorkspace* ws, cudaStream_t stream);
// same, and CTA 0 also emits into A00 (v x v) the columns >= (i / nb) * nb of pivot i's L\U row; *nb_used = nb
int launch_panel_getrf_a00(double* W, int64_t ldw, int n, int v, int* perm_out, double* A00, int* nb_used,
                           PanelWorkspace* ws, cudaStream_t stream);

// ---------------------------------------------------------------- rows.cu
// PT[c][r] = A[(row0 + r) * lda + col0 + c]  for r < n, c < v     (transposing strided copy, K8/a3)
int launch_extract_panel_T(const double* A, int64_t lda, int64_t row0, int64_t col0, int n, int v, double* PT,
                           int64_t ldp, cudaStream_t stream);
// A[(row0 + r) * lda + col0 + c] = LT[c][r]                        (L written back in place)
int launch_store_panel_T(double* A, int64_t lda, int64_t row0, int64_t col0, int n, int v, const double* LT,
                         int64_t ldp, cudaStream_t stream);
// winners of a pivot search: out_vals[c][dst0 + i] = PT[c][perm[i]] (0 when perm[i] >= n_valid),
// out_tags[dst0 + i] = tags[perm[i]] (0 when padded)               (inverse_permute_rows, utils.hpp:85-116)
int launch_gather_winners(const double* PT, int64_t ldp, const int* tags, int n_valid, const int* perm, int v,
                          double* out_vals, int64_t ldo, int* out_tags, int dst0, cudaStream_t stream);
// A00[i][c] = W[c][perm[i]], A00T[c][i] = same                      (top v x v of the factored panel)
// (completes the L prefix c < (i / nb) * nb of the rows emitted by launch_panel_getrf_a00, and writes A00T)
int launch_gather_a00(const double* W, int64_t ldw, const int* perm, int v, int nb, double* A00, double* A00T,
                      cudaStream_t stream);

// One-CTA planner of step 2 (g2lnoTile + igri lookup + analyze_pivots, conflux_opt.cpp:74-148):
struct MovePlan {
    int* npiv;     // [1]
    int* cur_piv;  // [v] local rows of my pivots, tournament order
    int* order;    // [v] tournament position of my i-th pivot
    int* slot2piv; // [v] tournament position -> my pivot index, -1 if not mine
    int* early;    // [v]
    int* late;     // [v]
    int* nel;      // [1]
    int* rowsrc;   // [Ml] new local row -> old local row (identity outside the active range)
};
int launch_plan_moves(const int* gpivots, int v, int Px, int pi, int fnpr, int Ml, const int* igri, MovePlan plan,
                      cudaStream_t stream);
// push_pivots_up phases (conflux_opt.hpp:176-218), 128-bit row moves over columns [col_lo, ncols)
int launch_push_phase1(const double* A, int64_t lda, int ncols, int col_lo, MovePlan plan, int v, double* tmp,
                       double* a01raw, int64_t ld01, int c0, cudaStream_t stream);
int launch_push_phase2(double* A, int64_t lda, int ncols, int col_lo, MovePlan plan, int v, cudaStream_t stream);
int launch_push_phase3(double* A, int64_t lda, int ncols, int col_lo, int fnpr, MovePlan plan, int v,
                       const double* tmp, cudaStream_t stream);
// gri/igri bookkeeping after the push (conflux_opt.hpp:1083-1124)
int launch_update_gri(int* gri, int* gri_tmp, int* igri, const int* rowsrc, int fnpr, int Ml, int v, int Px,
                      cudaStream_t stream);
// PT2[c][r'] = PT[c][rowsrc[fnpr_new + r'] - fnpr_old], fnpr_new = fnpr_old + *npiv   (A10Buff push, :1067)
int launch_compact_panel(const double* PT, int64_t ldp, double* PT2, int64_t ldp2, const int* rowsrc, int fnpr_old,
                         const int* npiv, int Ml, int v, cudaStream_t stream);
// my pivot rows receive their U values / diagonal block:  A[(fnpr_old+i)*lda + c0 + c] = U[order[i]][c]
int launch_store_u_rows(double* A, int64_t lda, int fnpr_old, MovePlan plan, const double* U, int64_t ldu, int c0,
                        int ncols, int v, cudaStream_t stream);
int launch_store_diag(double* A, int64_t lda, int fnpr_old, MovePlan plan, const double* A00, int loff, int v,
                      cudaStream_t stream);
// residual helpers (validation only)
int launch_split_factors(const double* F, int64_t ldf, int n, double* LT, double* U, cudaStream_t stream);
int launch_gather_perm_rows(const double* A, int64_t lda, const int* perm, int n, double* out, cudaStream_t stream);
int launch_sumsq(const double* X, int64_t count, double* out, cudaStream_t stream);
// misc
int launch_fill(double* p, int64_t n, double val, cudaStream_t stream);
int launch_iota_gri(int* gri, int* igri, int Ml, int v, int Px, int pi, cudaStream_t stream);
int launch_pack_bcast(const double* A00, const int* tags, int v, double* buf, cudaStream_t stream);
int launch_unpack_bcast(const double* buf, int v, double* A00, double* A00T, int* gpivots, cudaStream_t stream);
int launch_record_pivots(const int* gpivots, int v, int* hist, int k, cudaStream_t stream);

// ---------------------------------------------------------------- trsm.cu
// inverses of the nb x nb diagonal blocks of A00 = L00\U00: Uinv[j] (row-major; inv(U_jj)^T when u_transposed) and
// LinvT[j] (= inv(L_jj)^T)
int launch_diag_inverses(const double* A00, int v, int nb, double* Uinv, double* LinvT, cudaStream_t stream,
                         bool u_transposed = false);
// LT = (PT * U00^-1)^T : PT, LT are [v][ld] transposed panels with n columns; PT is destroyed
int trsm_right_upper_T(const double* A00, const double* Uinv, int v, int nb, double* PT, double* LT, int64_t ld,
                       int n, cudaStream_t stream);
// U = L00^-1 * R : R, U are [v][ld] with n columns; R is destroyed
int trsm_left_lower_unit(const double* A00T, const double* LinvT, int v, int nb, double* R, double* U, int64_t ld,
                         int n, cudaStream_t stream);
// X = U00^-1 * R (left, upper, non-unit) : R, X are [v][ld] with n columns (n even); R is destroyed.  A00T = U00^T
// (lower part ignored), UinvT = the transposed diagonal-block inverses (launch_diag_inverses, u_transposed)
int trsm_left_upper(const double* A00T, const double* UinvT, int v, int nb, double* R, double* X, int64_t ld, int n,
                    cudaStream_t stream);

// ---------------------------------------------------------------- solve.cu
// W[r][c] -= sum_k AT[k][r] * Y[k][c] for r < M, c < n (n <= 16): the few-right-hand-side trailing update of the
// distributed triangular solves, bandwidth-bound on the AT panel (K = v rows of ldat doubles)
int launch_solve_update_skinny(const double* AT, int64_t ldat, int M, int K, const double* Y, int64_t ldy, int n,
                               double* W, int64_t ldw, cudaStream_t stream);
constexpr int SOLVE_SKINNY_MAX = 16;  // widest right-hand-side block of the skinny update

}  // namespace cflx
