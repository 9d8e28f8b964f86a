// conflux_b200/csrc/lu_state.h -- internal state of a process-grid handle and of one factorisation plan, shared by the
// orchestration (lu.cu), the validation path (validate.cu) and the Cholesky path (chol.cu).  Not part of the C ABI.
#pragma once
#include <nccl.h>

#include <algorithm>
#include <vector>

#include "../../include/conflux_b200.h"
#include "common.cuh"
#include "kernels.h"

#define CFLX_NCCL(call)                                                                                    \
    do {                                                                                                   \
        ncclResult_t r__ = (call);                                                                         \
        if (r__ != ncclSuccess) {                                                                          \
            ::cflx::set_last_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, ncclGetErrorString(r__)); \
            return CFLX_ERR_NCCL;                                                                          \
        }                                                                                                  \
    } while (0)

struct cflx_comm {
    int world_size = 1, world_rank = 0, device = 0;
    ncclComm_t world = nullptr;
    cudaStream_t stream = nullptr;
    double* d_scratch = nullptr;  // 1 double for barriers
};

namespace cflx {
struct SubComm {
    ncclComm_t c = nullptr;
    int size = 1, rank = 0;
};

enum Phase { PH_PANEL = 0, PH_TOURN, PH_MOVES, PH_REDUCE, PH_TRSM, PH_GEMM, PH_STORE, PH_OTHER, PH_COUNT };

// Profiling regions, named like the reference's semiprof regions (PE(...) in conflux_opt.hpp; profiler.hpp:5-19) so
// that an Nsight Systems timeline (NVTX ranges) or cflx_lu_timeline() reads like the reference's profiler summary.
enum Region {
    RG_init = 0, RG_step0_copy, RG_step0_reduce, RG_step1_A10copy, RG_step1_lup, RG_step1_rowpermute, RG_step1_pivoting,
    RG_step1_A00Buff_bcast, RG_step2_pushingpivots, RG_step2_reduce, RG_step4_reshuffling, RG_step4_dtrsm, RG_step4_comm,
    RG_step5_dtrsm, RG_step5_comm, RG_step6_dgemm, RG_storingresults, RG_COUNT
};
inline const char* region_name(int r) {
    static const char* n[RG_COUNT] = {"init", "step0_copy", "step0_reduce", "step1_A10copy", "step1_lup", "step1_rowpermute",
                                      "step1_pivoting", "step1_A00Buff_bcast", "step2_pushingpivots", "step2_reduce",
                                      "step4_reshuffling", "step4_dtrsm", "step4_comm", "step5_dtrsm", "step5_comm",
                                      "step6_dgemm", "storingresults"};
    return n[r];
}
inline int region_phase(int r) {
    static const int p[RG_COUNT] = {PH_OTHER, PH_PANEL, PH_PANEL, PH_PANEL, PH_PANEL, PH_PANEL, PH_TOURN, PH_TOURN, PH_MOVES,
                                    PH_REDUCE, PH_MOVES, PH_TRSM, PH_REDUCE, PH_TRSM, PH_REDUCE, PH_GEMM, PH_STORE};
    return p[r];
}

template <class T>
inline int dmalloc(T** p, size_t n) {
    CFLX_CUDA(cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(T) + 4096));  // tail pad: bulk copies may over-read
    return CFLX_OK;
}
int make_sub(cflx_comm* c, int color, int key, int size, SubComm* out);
int grid_barrier(cflx_comm* c);

// State of cflx_lu_solve (solve.cu): the factors re-laid out for the triangular sweeps, built on the first solve after
// each factorisation, and the right-hand-side work buffers, grown to the widest solve so far.
struct SolveState {
    bool ready = false;             // CT / diagonal blocks describe the current factors
    std::vector<int> hist;          // pivot history of those factors (row of global id hist[q] is pivoted row q)
    std::vector<int> diag_slot;     // [Nt] index of diagonal tile t among this rank's diagonal tiles, -1 if not mine
    double* CT = nullptr;           // [Nl][Ml] (layer 0): CT[lc][r] = C[r][lc], C the factors in the conflux layout
    double* diag = nullptr;         // per owned diagonal tile: DT [v][v] (transposed tile), LinvT [v*nb], UinvT [v*nb]
    double *W = nullptr, *X = nullptr, *B = nullptr, *stage = nullptr;  // Ml x ldr, Nl x ldr, Ml x ldr, 2 Ml x ldr
    int ldr_cap = 0;
};
}  // namespace cflx

struct cflx_lu {
    cflx_comm* comm = nullptr;
    int M = 0, N = 0, v = 0, Px = 1, Py = 1, Pz = 1, P = 1, Ml = 0, Nl = 0, Nt = 0, Mt = 0, nlayr = 0;
    int pi = 0, pj = 0, pk = 0, rank = 0, nb = 0;
    cflx::SubComm k_comm, i_comm, jk_comm, ik_comm;
    // device memory
    double *A0 = nullptr, *A11 = nullptr, *PT = nullptr, *PT2 = nullptr, *W = nullptr, *LT = nullptr, *A01raw = nullptr,
           *U = nullptr, *tmp = nullptr, *A00 = nullptr, *A00T = nullptr, *Uinv = nullptr, *LinvT = nullptr,
           *candH = nullptr, *S = nullptr, *W2 = nullptr, *bcast = nullptr, *Cbuf = nullptr, *xbuf = nullptr;
    int *gri = nullptr, *gri_tmp = nullptr, *igri = nullptr, *perm = nullptr, *gpivots = nullptr, *tagsH = nullptr,
        *tagsS = nullptr, *hist = nullptr, *plan_mem = nullptr, *idx_buf = nullptr;
    cflx::MovePlan plan{};
    cflx::PanelWorkspace pws{};
    cflx::OzakiWorkspace oz{};   // digit planes of the int8 tcgen05 trailing update (CFLX_GEMM=ozaki)
    bool use_ozaki = false;
    int64_t ldp_max = 0;
    int* h_npiv = nullptr;  // pinned
    std::vector<int> h_hist;
    bool have_input = false, factored = false, time_gemm = false;
    // double-buffered input streaming (cflx_lu_queue_next_local): the upload of the NEXT matrix overlaps this factorisation
    const double* next_host = nullptr;
    bool a0_is_next = false;  // A0 already holds (or is receiving) the next input: validation of the last run is refused
    cudaStream_t copy = nullptr;
    cudaEvent_t ev_a0_read = nullptr, ev_upload = nullptr;
    double gemm_ms = 0, gemm_flops = 0;
    int64_t launches = 0;
    double phase_ms[cflx::PH_COUNT] = {0};
    // non-serialising timeline (profiling mode 2): event pairs recorded on the launching stream, resolved after the run
    struct TlRec { int region, side, ev; };
    std::vector<cudaEvent_t> tl_pool;
    std::vector<TlRec> tl_recs;
    double region_ms[2][cflx::RG_COUNT] = {{0}};   // [main / side stream][region]
    int region_cnt[2][cflx::RG_COUNT] = {{0}};
    int prof_mode = 0;                              // 0 off, 1 serialising phase timers, 2 timeline
    std::vector<cudaEvent_t> ev;
    std::vector<char> ev_used;
    cudaStream_t side = nullptr;  // high-priority look-ahead stream (null: no overlap)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_npiv = nullptr;
    cflx::SolveState sv;  // cflx_lu_solve (marked stale by cflx_lu_set_local / cflx_lu_factor)
};

namespace cflx {
// validate.cu
int redistribute_pivoted_rows(cflx_lu* lu, const std::vector<int>& hist, bool factors, const double* src, double* dst);
int redistribute_pivoted_rows(cflx_lu* lu, const std::vector<int>& hist, bool factors, const double* src, double* dst,
                              int ncols, int64_t ld, double* stage);
int lu_residual_grid(cflx_lu* lu, const std::vector<int>& hist, double* abs_out, double* rel_out);
// solve.cu
void solve_state_free(SolveState* sv);
}  // namespace cflx
