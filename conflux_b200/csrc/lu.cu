// conflux_b200/csrc/lu.cu -- host orchestration of the CONFLUX LU step loop on B200 + the C ABI.
//
// One rank = one GPU = one host thread/process (SPMD, like the reference's MPI ranks).  The step order follows
// conflux::LU_rep<T> (/root/reference/src/conflux/lu/conflux_opt.hpp:535-1803, blueprint in SURVEY.md appendix A)
// but the data layout and the division of labour are B200-first:
//   * A11 stays resident in HBM (row-major Ml x Nl, 64-bit indexing); L and U are written IN PLACE into it
//     (the reference keeps a second Ml x Nl array A10resultBuff + a caller-owned C and MPI_Puts into it);
//   * panels are kept transposed/K-major (see gemm.cu, panel.cu) so every kernel streams contiguous rows;
//   * pivot rows are gathered by ONE sum-reduction over the (i,k) plane of zero-padded v x ncols buffers
//     (exact: every row has exactly one non-zero contributor per layer) instead of reduce + p2p gather
//     (conflux_opt.hpp:1164-1173,1226-1258,1474-1511); A00 and the pivot ids travel in one broadcast
//     (conflux_opt.hpp:818-850,872);
//   * all communication is NCCL on the rank's stream; at Px == 1 the whole factorisation is enqueued without a
//     single host synchronisation, at Px > 1 the host reads back one int (this rank's pivot count) per step.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "lu_state.h"

namespace cflx {
static thread_local char g_err[1024] = "";
void set_last_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
}  // namespace cflx

using namespace cflx;

namespace {
int flipbit(int n, int k) { return n ^ (1 << k); }
int butterfly_pair(int pi, int r, int Px) {  // conflux_opt.cpp:59-72
    int src = flipbit(pi, r);
    if (src >= Px) {
        if (r == 0) src = pi;
        else {
            src = flipbit(src, r - 1);
            if (src >= Px) src = Px - 1;
        }
    }
    return src;
}
#include "init_tables.inc"
// decodes the fixed input matrix of size n x n (row-major) if the reference has one
bool fixed_input_matrix(int n, std::vector<double>* out) {
    for (const InitTable& t : kInitTables) {
        if (t.n != n) continue;
        out->clear();
        out->reserve((size_t)n * n);
        if (t.kind == 0) {
            for (const char* p = t.text; *p; ++p) out->push_back((double)(*p - '0'));
        } else {
            const char* p = t.text;
            while (*p) {
                char* e = nullptr;
                out->push_back(std::strtod(p, &e));
                p = (*e == ',') ? e + 1 : e;
            }
        }
        return out->size() == (size_t)n * n;
    }
    return false;
}
int pick_nb(int v) {  // block size of the diagonal inverses / TRSM sweeps (template instances: 128, 64, 32, 16, 8, 4)
    static int cap = -1;  // CFLX_TRSM_NB caps the block size (A/B switch; default 128)
    if (cap < 0) {
        const char* e = getenv("CFLX_TRSM_NB");
        cap = e ? atoi(e) : 128;
    }
    for (int nb : {128, 64, 32, 16, 8, 4})
        if (nb <= cap && v % nb == 0) return nb;
    return 0;
}
}  // namespace

namespace cflx {
int make_sub(cflx_comm* c, int color, int key, int size, SubComm* out) {
    out->size = size;
    out->rank = key;
    out->c = nullptr;
    if (c->world_size == 1) return CFLX_OK;
    // every rank takes part in every split (collective over the world communicator)
    CFLX_NCCL(ncclCommSplit(c->world, color, key, &out->c, nullptr));
    int r = -1, s = -1;
    CFLX_NCCL(ncclCommUserRank(out->c, &r));
    CFLX_NCCL(ncclCommCount(out->c, &s));
    if (r != key || s != size) {
        set_last_error("sub-communicator mismatch: rank %d/%d expected %d/%d", r, s, key, size);
        return CFLX_ERR_NCCL;
    }
    return CFLX_OK;
}
int grid_barrier(cflx_comm* c) {
    if (c->world_size > 1)
        CFLX_NCCL(ncclAllReduce(c->d_scratch, c->d_scratch, 1, ncclDouble, ncclSum, c->world, c->stream));
    CFLX_CUDA(cudaStreamSynchronize(c->stream));
    return CFLX_OK;
}
}  // namespace cflx

namespace {
// One profiling region: always an NVTX range named like the reference's semiprof region; with profiling mode 1 a
// serialising CUDA-event timer (accurate per-phase device time, no overlap), with mode 2 an event pair on the launching
// stream that is resolved after the factorisation (no synchronisation: the timeline of the real, overlapped run).
struct PhaseTimer {
    cflx_lu* lu;
    int rg;
    cudaStream_t st;
    cudaEvent_t a = nullptr, b = nullptr;
    int ev = -1;
    PhaseTimer(cflx_lu* l, int region, cudaStream_t stream) : lu(l), rg(region), st(stream) {
        nvtxRangePushA(region_name(rg));
        if (lu->prof_mode == 1) {
            cudaEventCreate(&a);
            cudaEventCreate(&b);
            cudaEventRecord(a, st);
        } else if (lu->prof_mode == 2) {
            ev = (int)lu->tl_recs.size() * 2;
            while ((int)lu->tl_pool.size() < ev + 2) {
                cudaEvent_t e;
                cudaEventCreate(&e);
                lu->tl_pool.push_back(e);
            }
            lu->tl_recs.push_back({rg, st == lu->comm->stream ? 0 : 1, ev});
            cudaEventRecord(lu->tl_pool[ev], st);
        }
    }
    ~PhaseTimer() {
        if (lu->prof_mode == 1) {
            cudaEventRecord(b, st);
            cudaEventSynchronize(b);
            float ms = 0;
            cudaEventElapsedTime(&ms, a, b);
            lu->phase_ms[region_phase(rg)] += ms;
            lu->region_ms[st == lu->comm->stream ? 0 : 1][rg] += ms;
            lu->region_cnt[st == lu->comm->stream ? 0 : 1][rg]++;
            cudaEventDestroy(a);
            cudaEventDestroy(b);
        } else if (lu->prof_mode == 2) {
            cudaEventRecord(lu->tl_pool[ev + 1], st);
        }
        nvtxRangePop();
    }
};

// exchange of tournament candidates with the butterfly partner(s) of round r (conflux_opt.hpp:242-280)
int tournament_exchange(cflx_lu* lu, int r, int my_half, cudaStream_t s) {
    const int v = lu->v, Px = lu->Px, pi = lu->pi;
    const int src = butterfly_pair(pi, r, Px);
    const int other = 1 - my_half;
    const size_t hv = (size_t)v * v;
    double* mine = lu->candH + my_half * hv;
    double* recv = lu->candH + other * hv;
    int* mine_t = lu->tagsH + my_half * v;
    int* recv_t = lu->tagsH + other * v;
    const bool self = (src == pi);
    if (self) {  // MPI_Sendrecv with itself: the own half is duplicated into the other half (conflux_opt.hpp:258-266)
        CFLX_CUDA(cudaMemcpyAsync(recv, mine, hv * sizeof(double), cudaMemcpyDeviceToDevice, s));
        CFLX_CUDA(cudaMemcpyAsync(recv_t, mine_t, v * sizeof(int), cudaMemcpyDeviceToDevice, s));
    }
    // a self-paired rank still serves one-sided requesters (the reference's extra Isend, conflux_opt.hpp:271-279)
    bool any = !self;
    for (int ppi = 0; ppi < Px && !any; ++ppi) any = (ppi != pi && butterfly_pair(ppi, r, Px) == pi);
    if (!any) return CFLX_OK;
    CFLX_NCCL(ncclGroupStart());
    for (int ppi = 0; ppi < Px; ++ppi) {
        if (ppi == pi || butterfly_pair(ppi, r, Px) != pi) continue;
        // mutual partner gets my own half; a one-sided requester gets the lower half
        const bool mutual = (!self && ppi == src);
        const double* sv = mutual ? mine : lu->candH + hv;
        const int* st = mutual ? mine_t : lu->tagsH + v;
        CFLX_NCCL(ncclSend(sv, hv, ncclDouble, ppi, lu->i_comm.c, s));
        CFLX_NCCL(ncclSend(st, v, ncclInt, ppi, lu->i_comm.c, s));
    }
    if (!self) {
        CFLX_NCCL(ncclRecv(recv, hv, ncclDouble, src, lu->i_comm.c, s));
        CFLX_NCCL(ncclRecv(recv_t, v, ncclInt, src, lu->i_comm.c, s));
    }
    CFLX_NCCL(ncclGroupEnd());
    return CFLX_OK;
}

// S[c][h*v + i] = candH[h][c][i]; tagsS likewise
__global__ void stack_kernel(const double* __restrict__ candH, const int* __restrict__ tagsH, int v, double* __restrict__ S,
                             double* __restrict__ W2, int* __restrict__ tagsS) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t tot = (int64_t)2 * v * v;
    if (e < tot) {
        const int c = (int)(e / (2 * v)), hi = (int)(e % (2 * v));
        const int h = hi / v, i = hi % v;
        const double x = candH[(size_t)h * v * v + (size_t)c * v + i];
        S[e] = x;
        W2[e] = x;
    }
    if (e < 2 * v) tagsS[e] = tagsH[e];
}
// ---- steps 0 + 1 of iteration k: panel extract (+ layer reduce), local pivot search, tournament.  Runs on stream
// `s`; with look-ahead that is the high-priority side stream and overlaps the trailing update of iteration k-1.
// Touches only: PT, W, perm, candH/tagsH/S/W2/tagsS, A00/A00T (outputs consumed by finish_step(k) after the join).
int panel_phase(cflx_lu* lu, int k, int fnpr, cudaStream_t s) {
    const int v = lu->v, Px = lu->Px, Py = lu->Py, Pz = lu->Pz, Ml = lu->Ml, Nl = lu->Nl;
    const int pi = lu->pi, pj = lu->pj, pk = lu->pk;
    const int loff = (k / Py) * v, pjk = k % Py;
    if (pj != pjk) return CFLX_OK;
    // A00 / A00T are double-buffered by step parity: the look-ahead search of step k+1 must not overwrite the block
    // that the U solve and the factor stores of step k are still reading on the main stream
    double* A00 = lu->A00 + (size_t)(k & 1) * v * v;
    double* A00T = lu->A00T + (size_t)(k & 1) * v * v;
    const int n_old = Ml - fnpr;
    const int64_t ldk = std::max<int64_t>(2, round_up(n_old, 2));
    int nR = 0;
    while ((1 << nR) < Px) ++nR;
    // ---- step 0: panel extract (+ reduce over layers onto pk = 0)            conflux_opt.hpp:618-648
    {
        PhaseTimer t(lu, RG_step0_copy, s);
        CFLX_TRY(launch_extract_panel_T(lu->A11, Nl, fnpr, loff, n_old, v, lu->PT, ldk, s));
        lu->launches++;
    }
    if (Pz > 1 && n_old > 0) {
        PhaseTimer t(lu, RG_step0_reduce, s);
        CFLX_NCCL(ncclReduce(lu->PT, lu->PT, (size_t)v * ldk, ncclDouble, ncclSum, 0, lu->k_comm.c, s));
    }
    if (pk != 0) return CFLX_OK;
    // ---- step 1: local pivot search + tournament on column pj == k % Py, layer 0   conflux_opt.hpp:693-816
    int my_half = 0;
    {
        PhaseTimer t(lu, RG_step1_A10copy, s);
        CFLX_CUDA(cudaMemcpyAsync(lu->W, lu->PT, (size_t)v * ldk * sizeof(double), cudaMemcpyDeviceToDevice, s));
    }
    {
        PhaseTimer t(lu, RG_step1_lup, s);
        int nb_used = 0;
        if (nR == 0) {  // the local search already is the tournament: A00 comes from it (SURVEY.md fact 7)
            CFLX_TRY(launch_panel_getrf_a00(lu->W, ldk, n_old, v, lu->perm, A00, &nb_used, &lu->pws, s));
            CFLX_TRY(launch_gather_a00(lu->W, ldk, lu->perm, v, nb_used, A00, A00T, s));
            lu->launches += 2;
        } else {
            CFLX_TRY(launch_panel_getrf(lu->W, ldk, n_old, v, lu->perm, &lu->pws, s));
            lu->launches++;
        }
    }
    {
        PhaseTimer t(lu, RG_step1_rowpermute, s);
        int first_partner = flipbit(pi, 0);
        if (first_partner > Px - 1) first_partner = Px - 1;
        my_half = first_partner < pi ? 1 : 0;  // "higher rank puts his candidates below" (conflux_opt.hpp:717-750)
        CFLX_TRY(launch_gather_winners(lu->PT, ldk, lu->gri + fnpr, n_old, lu->perm, v,
                                       lu->candH + (size_t)my_half * v * v, v, lu->tagsH + my_half * v, 0, s));
        lu->launches++;
    }
    PhaseTimer t(lu, RG_step1_pivoting, s);
    for (int r = 0; r < nR; ++r) {
        CFLX_TRY(tournament_exchange(lu, r, my_half, s));
        const int64_t tot = (int64_t)2 * v * v;
        stack_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(lu->candH, lu->tagsH, v, lu->S, lu->W2, lu->tagsS);
        CFLX_CUDA(cudaGetLastError());
        const bool last = (r == nR - 1);
        int nb_used = 0;
        if (last) {
            CFLX_TRY(launch_panel_getrf_a00(lu->W2, 2 * v, 2 * v, v, lu->perm, A00, &nb_used, &lu->pws, s));
            CFLX_TRY(launch_gather_a00(lu->W2, 2 * v, lu->perm, v, nb_used, A00, A00T, s));
            lu->launches++;
            my_half = 0;
        } else {
            CFLX_TRY(launch_panel_getrf(lu->W2, 2 * v, 2 * v, v, lu->perm, &lu->pws, s));
            my_half = butterfly_pair(pi, r + 1, Px) < pi ? 1 : 0;
        }
        CFLX_TRY(launch_gather_winners(lu->S, 2 * v, lu->tagsS, 2 * v, lu->perm, v, lu->candH + (size_t)my_half * v * v,
                                       v, lu->tagsH + my_half * v, 0, s));
        lu->launches += 3;
    }
    // winners now sit in the upper half: tagsH[0..v) = global pivot rows (conflux_opt.hpp:810-815)
    return CFLX_OK;
}

// digit planes of the operands of this step's trailing update (int8 tcgen05 path): L^T slab of this layer, U slab columns
int ozaki_planes_a(cflx_lu* lu, int n_act, int64_t ld2, cudaStream_t s) {
    if (!lu->use_ozaki || n_act <= 0) return CFLX_OK;
    PhaseTimer t(lu, RG_step6_dgemm, s);
    lu->launches++;
    return ozaki_split_a(&lu->oz, lu->LT + (int64_t)lu->pk * lu->nlayr * ld2, ld2, n_act, s);
}
int ozaki_planes_b(cflx_lu* lu, int col0, int n, int64_t ldu, cudaStream_t s) {
    if (!lu->use_ozaki || n <= 0) return CFLX_OK;
    PhaseTimer t(lu, RG_step6_dgemm, s);
    lu->launches++;
    return ozaki_split_b(&lu->oz, lu->U + (int64_t)lu->pk * lu->nlayr * ldu, ldu, col0, n, s);
}

int trailing_gemm(cflx_lu* lu, int k, int part, int fnpr, int n_act, int col_lo, int ncols, int64_t ld2, int64_t ldu,
                  int u_col_off, cudaStream_t s, int max_ctas = 0) {
    if (n_act <= 0 || ncols <= 0) return CFLX_OK;
    PhaseTimer t(lu, RG_step6_dgemm, s);
    GemmArgs g{};
    g.M = n_act;
    g.N = ncols;
    g.K = lu->nlayr;
    g.AT = lu->LT + (int64_t)lu->pk * lu->nlayr * ld2;
    g.ldat = ld2;
    g.B = lu->U + (int64_t)lu->pk * lu->nlayr * ldu + u_col_off;
    g.ldb = ldu;
    g.C = lu->A11 + (int64_t)fnpr * lu->Nl + col_lo;
    g.ldc = lu->Nl;
    g.D = lu->A11 + (int64_t)fnpr * lu->Nl + col_lo;
    g.ldd = lu->Nl;
    g.alpha = -1.0;
    g.beta = 1.0;
    const int e = 4 * k + 2 * part;
    if (lu->time_gemm) CFLX_CUDA(cudaEventRecord(lu->ev[e], s));
    if (lu->use_ozaki) CFLX_TRY(launch_ozaki_gemm(&lu->oz, g.M, g.N, 0, u_col_off, g.D, g.ldd, max_ctas, s));
    else CFLX_TRY(launch_gemm_tn(g, s));
    if (lu->time_gemm) CFLX_CUDA(cudaEventRecord(lu->ev[e + 1], s));
    lu->ev_used[e / 2] = lu->time_gemm;
    lu->gemm_flops += 2.0 * g.M * (double)g.N * g.K;
    lu->launches++;
    return CFLX_OK;
}

// ---- everything of iteration k after the pivot search: pivot broadcast, row moves, solves, stores, trailing update
// (with the columns of panel k+1 updated first so that panel_phase(k+1) can start on the side stream).
int finish_step(cflx_lu* lu, int k, int& fnpr) {
    cudaStream_t s = lu->comm->stream;
    const int v = lu->v, Px = lu->Px, Py = lu->Py, Pz = lu->Pz, Ml = lu->Ml, Nl = lu->Nl;
    const int pi = lu->pi, pj = lu->pj, pk = lu->pk;
    const int loff = (k / Py) * v, pjk = k % Py, pik = k % Px;
    const bool on_col = (pj == pjk), on_row = (pi == pik), layer0 = (pk == 0);
    const int c0 = loff + (pj <= pjk ? v : 0);  // first live column of this rank after step k
    const int ncols = Nl - c0;
    const int fnpr_old = fnpr;
    const int n_old = Ml - fnpr_old;
    const int64_t ldk = std::max<int64_t>(2, round_up(n_old, 2));
    int nR = 0;
    while ((1 << nR) < Px) ++nR;
    double* A00 = lu->A00 + (size_t)(k & 1) * v * v;
    double* A00T = lu->A00T + (size_t)(k & 1) * v * v;
    // ---- A00 + pivot ids to everybody (one broadcast)                     conflux_opt.hpp:818-850,872
    {
        PhaseTimer t(lu, RG_step1_A00Buff_bcast, s);
        if (lu->P > 1) {
            const int root = (pik * Py + pjk) * Pz;  // rank of (k % Px, k % Py, 0)
            if (lu->rank == root) {
                CFLX_TRY(launch_pack_bcast(A00, lu->tagsH, v, lu->bcast, s));
                lu->launches++;
            }
            CFLX_NCCL(ncclBroadcast(lu->bcast, lu->bcast, (size_t)v * v + v, ncclDouble, root, lu->comm->world, s));
            CFLX_TRY(launch_unpack_bcast(lu->bcast, v, A00, A00T, lu->gpivots, s));
            lu->launches++;
        } else {
            CFLX_CUDA(cudaMemcpyAsync(lu->gpivots, lu->tagsH, v * sizeof(int), cudaMemcpyDeviceToDevice, s));
        }
        CFLX_TRY(launch_record_pivots(lu->gpivots, v, lu->hist, k, s));
        lu->launches++;
    }
    // ---- step 2: localise pivots, push them up, extract pivot rows        conflux_opt.hpp:876-1147
    // At Px > 1 the host needs this rank's pivot count (it sizes the L-panel work).  Everything that does NOT depend
    // on it -- row moves, pivot-row reduce, the U solve, its broadcast, the factor stores -- is enqueued first, and
    // the host only then waits for the 4-byte read-back, so the GPU stays busy while the rest is enqueued.
    {
        PhaseTimer t(lu, RG_step2_pushingpivots, s);
        CFLX_TRY(launch_plan_moves(lu->gpivots, v, Px, pi, fnpr_old, Ml, lu->igri, lu->plan, s));
        lu->launches++;
        if (Px > 1) {
            CFLX_CUDA(cudaMemcpyAsync(lu->h_npiv, lu->plan.npiv, sizeof(int), cudaMemcpyDeviceToHost, s));
            CFLX_CUDA(cudaEventRecord(lu->ev_npiv, s));
        }
        const int col_lo = layer0 ? 0 : loff;
        const int64_t ldu0 = std::max(2, ncols);
        CFLX_TRY(launch_push_phase1(lu->A11, Nl, Nl, col_lo, lu->plan, v, lu->tmp, ncols > 0 ? lu->A01raw : nullptr, ldu0, c0,
                                    s));
        CFLX_TRY(launch_push_phase2(lu->A11, Nl, Nl, col_lo, lu->plan, v, s));
        CFLX_TRY(launch_push_phase3(lu->A11, Nl, Nl, col_lo, fnpr_old, lu->plan, v, lu->tmp, s));
        CFLX_TRY(launch_update_gri(lu->gri, lu->gri_tmp, lu->igri, lu->plan.rowsrc, fnpr_old, Ml, v, Px, s));
        lu->launches += 5;
    }
    const int64_t ldu = std::max(2, ncols);
    // At Px == 1 the local pivot search IS the panel factorisation: its multipliers are the L panel (same values a
    // LAPACK getrf leaves behind; the reference recomputes them with dtrsm against A00, conflux_opt.hpp:1347).
    const bool fused_l = (nR == 0);
    // ---- steps 2b/3: pivot rows summed over layers and gathered on row pi == k % Px   conflux_opt.hpp:1164-1260
    if (ncols > 0 && Px * Pz > 1) {
        PhaseTimer t(lu, RG_step2_reduce, s);
        CFLX_NCCL(ncclReduce(lu->A01raw, lu->A01raw, (size_t)v * ldu, ncclDouble, ncclSum, pik * Pz, lu->ik_comm.c, s));
    }
    // ---- step 5 first: U = L00^-1 * (pivot rows)                            conflux_opt.hpp:1522-1593
    if (layer0 && ((on_col && !fused_l) || on_row)) {
        PhaseTimer t(lu, RG_step5_dtrsm, s);
        CFLX_TRY(launch_diag_inverses(A00, v, lu->nb, lu->Uinv, lu->LinvT, s));
        lu->launches++;
    }
    // The U solve is split in two column windows: the first v columns (= the next panel) are solved before the
    // look-ahead fork, the rest after it, off the pivot search's critical path (single-rank grids only: with more
    // ranks the U panel is broadcast whole).
    const bool split_u = (lu->P == 1) && (k + 1 < lu->Nt) && ncols > v;
    const int ncols_a = split_u ? v : ncols;
    if (on_row && layer0 && ncols > 0) {
        PhaseTimer t(lu, RG_step5_dtrsm, s);
        CFLX_TRY(trsm_left_lower_unit(A00T, lu->LinvT, v, lu->nb, lu->A01raw, lu->U, ldu, ncols_a, s));
        lu->launches += 2 * (v / lu->nb) - 1;
    }
    if (Px * Pz > 1 && ncols > 0) {  // U panel to every (pi', pk') of my grid column   conflux_opt.hpp:1567-1593
        PhaseTimer t(lu, RG_step5_comm, s);
        CFLX_NCCL(ncclBroadcast(lu->U, lu->U, (size_t)v * ldu, ncclDouble, pik * Pz, lu->ik_comm.c, s));
    }
    auto store_factors = [&]() -> int {  // my promoted rows receive their U part and diagonal block   :1721-1754
        if (!layer0) return CFLX_OK;
        PhaseTimer t(lu, RG_storingresults, s);
        if (ncols > 0) {
            CFLX_TRY(launch_store_u_rows(lu->A11, Nl, fnpr_old, lu->plan, lu->U, ldu, c0, ncols, v, s));
            lu->launches++;
        }
        if (on_col) {
            CFLX_TRY(launch_store_diag(lu->A11, Nl, fnpr_old, lu->plan, A00, loff, v, s));
            lu->launches++;
        }
        return CFLX_OK;
    };
    if (!split_u) CFLX_TRY(store_factors());
    // ---- now the pivot count: sizes of the L panel and of the trailing update
    int npiv = v;
    if (Px > 1) {
        CFLX_CUDA(cudaEventSynchronize(lu->ev_npiv));
        npiv = *lu->h_npiv;
    }
    if (npiv < 0 || npiv > v || fnpr_old + npiv > Ml) {
        set_last_error("step %d: inconsistent pivot count %d (fnpr %d, Ml %d)", k, npiv, fnpr_old, Ml);
        return CFLX_ERR_STATE;
    }
    fnpr = fnpr_old + npiv;
    const int n_act = Ml - fnpr;
    const int64_t ld2 = std::max<int64_t>(2, round_up(n_act, 2));
    // ---- step 4: L = A10 * U00^-1 on the panel column                       conflux_opt.hpp:1329-1434
    if (on_col && layer0 && n_act > 0) {
        {
            PhaseTimer t(lu, RG_step4_reshuffling, s);
            CFLX_TRY(launch_compact_panel(fused_l ? lu->W : lu->PT, ldk, fused_l ? lu->LT : lu->PT2, ld2, lu->plan.rowsrc,
                                          fnpr_old, lu->plan.npiv, Ml, v, s));
            lu->launches++;
        }
        if (!fused_l) {
            PhaseTimer t(lu, RG_step4_dtrsm, s);
            CFLX_TRY(trsm_right_upper_T(A00, lu->Uinv, v, lu->nb, lu->PT2, lu->LT, ld2, n_act, s));
            lu->launches += 2 * (v / lu->nb) - 1;
        }
        PhaseTimer t(lu, RG_storingresults, s);
        CFLX_TRY(launch_store_panel_T(lu->A11, Nl, fnpr, loff, n_act, v, lu->LT, ld2, s));  // L in place
        lu->launches++;
    }
    if (Py * Pz > 1 && n_act > 0) {  // L panel to every (pj', pk') of my grid row    conflux_opt.hpp:1404-1434
        PhaseTimer t(lu, RG_step4_comm, s);
        CFLX_NCCL(ncclBroadcast(lu->LT, lu->LT, (size_t)v * ld2, ncclDouble, pjk * Pz, lu->jk_comm.c, s));
    }
    // ---- step 6: trailing update on every rank and layer                    conflux_opt.hpp:1628-1632
    // Look-ahead: the rank that owns panel k+1 updates those v columns first (they are its first live block), forks
    // the pivot search of iteration k+1 onto the side stream, and only then updates the remaining columns.
    const bool next_col = (k + 1 < lu->Nt) && (pj == (k + 1) % Py);
    CFLX_TRY(ozaki_planes_a(lu, n_act, ld2, s));
    if (n_act > 0) CFLX_TRY(ozaki_planes_b(lu, 0, split_u ? std::min(v, ncols) : ncols, ldu, s));
    if (next_col) {
        const int w = std::min(v, ncols);
        CFLX_TRY(trailing_gemm(lu, k, 0, fnpr, n_act, c0, w, ld2, ldu, 0, s));
        cudaStream_t side = (lu->prof_mode == 1) ? nullptr : lu->side;  // phase profiling serialises everything
        cudaStream_t sp = side ? side : s;
        if (side) {
            CFLX_CUDA(cudaEventRecord(lu->ev_fork, s));
            CFLX_CUDA(cudaStreamWaitEvent(sp, lu->ev_fork, 0));
        }
        CFLX_TRY(panel_phase(lu, k + 1, fnpr, sp));
        if (side) CFLX_CUDA(cudaEventRecord(lu->ev_join, sp));
        if (split_u) {
            PhaseTimer t(lu, RG_step5_dtrsm, s);
            CFLX_TRY(trsm_left_lower_unit(A00T, lu->LinvT, v, lu->nb, lu->A01raw + v, lu->U + v, ldu, ncols - v, s));
            lu->launches += 2 * (v / lu->nb) - 1;
        }
        if (split_u) CFLX_TRY(store_factors());
        if (split_u && n_act > 0) CFLX_TRY(ozaki_planes_b(lu, w, ncols - w, ldu, s));
        // the persistent tcgen05 kernel leaves the SMs of the concurrent pivot search alone
        const int leave = (side && lu->use_ozaki) ? lu->pws.cta_cap : 0;
        CFLX_TRY(trailing_gemm(lu, k, 1, fnpr, n_act, c0 + w, ncols - w, ld2, ldu, w, s, leave > 0 ? lu->oz.sms - leave : 0));
        if (side) CFLX_CUDA(cudaStreamWaitEvent(s, lu->ev_join, 0));
    } else {
        CFLX_TRY(trailing_gemm(lu, k, 0, fnpr, n_act, c0, ncols, ld2, ldu, 0, s));
    }
    return CFLX_OK;
}

void free_lu(cflx_lu* lu) {
    if (!lu) return;
    cudaSetDevice(lu->comm->device);
    double* dbl[] = {lu->A0, lu->A11, lu->PT, lu->PT2, lu->W, lu->LT, lu->A01raw, lu->U, lu->tmp, lu->A00, lu->A00T,
                     lu->Uinv, lu->LinvT, lu->candH, lu->S, lu->W2, lu->bcast, lu->Cbuf, lu->xbuf};
    for (double* p : dbl) cudaFree(p);
    int* ints[] = {lu->gri, lu->gri_tmp, lu->igri, lu->perm, lu->gpivots, lu->tagsH, lu->tagsS, lu->hist, lu->plan_mem,
                   lu->idx_buf};
    for (int* p : ints) cudaFree(p);
    if (lu->h_npiv) cudaFreeHost(lu->h_npiv);
    if (lu->pws.slot_hdr) panel_workspace_destroy(&lu->pws);
    if (lu->use_ozaki) ozaki_workspace_destroy(&lu->oz);
    for (auto& e : lu->ev) cudaEventDestroy(e);
    for (auto& e : lu->tl_pool) cudaEventDestroy(e);
    if (lu->side) cudaStreamDestroy(lu->side);
    if (lu->ev_fork) cudaEventDestroy(lu->ev_fork);
    if (lu->ev_join) cudaEventDestroy(lu->ev_join);
    if (lu->ev_npiv) cudaEventDestroy(lu->ev_npiv);
    if (lu->copy) cudaStreamDestroy(lu->copy);
    if (lu->ev_a0_read) cudaEventDestroy(lu->ev_a0_read);
    if (lu->ev_upload) cudaEventDestroy(lu->ev_upload);
    solve_state_free(&lu->sv);
    for (SubComm* sc : {&lu->k_comm, &lu->i_comm, &lu->jk_comm, &lu->ik_comm})
        if (sc->c) ncclCommDestroy(sc->c);
    delete lu;
}
}  // namespace

// ======================================================================================================== C ABI
extern "C" {

const char* cflx_last_error(void) { return g_err; }
const char* cflx_version(void) { return "conflux_b200 0.1 (sm_100a)"; }

int cflx_device_count(int* count) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        n = 0;
        cudaGetLastError();
    }
    *count = n;
    return CFLX_OK;
}

int cflx_get_unique_id(void* id_out) {
    static_assert(sizeof(ncclUniqueId) == CFLX_UNIQUE_ID_BYTES, "unique id size");
    ncclUniqueId id;
    CFLX_NCCL(ncclGetUniqueId(&id));
    std::memcpy(id_out, &id, sizeof(id));
    return CFLX_OK;
}

int cflx_comm_create(int world_size, int world_rank, const void* unique_id, int device, cflx_comm** out) {
    if (!out || world_size < 1 || world_rank < 0 || world_rank >= world_size) return CFLX_ERR_ARG;
    int ndev = 0;
    cflx_device_count(&ndev);
    if (ndev == 0) {
        set_last_error("no CUDA device visible: conflux_b200 has no CPU fallback");
        return CFLX_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= ndev) {
        set_last_error("device %d out of range (%d visible)", device, ndev);
        return CFLX_ERR_ARG;
    }
    CFLX_CUDA(cudaSetDevice(device));
    auto* c = new cflx_comm;
    c->world_size = world_size;
    c->world_rank = world_rank;
    c->device = device;
    CFLX_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CFLX_CUDA(cudaMalloc((void**)&c->d_scratch, sizeof(double)));
    CFLX_CUDA(cudaMemset(c->d_scratch, 0, sizeof(double)));
    if (world_size > 1) {
        if (!unique_id) {
            set_last_error("unique_id required for world_size > 1");
            return CFLX_ERR_ARG;
        }
        ncclUniqueId id;
        std::memcpy(&id, unique_id, sizeof(id));
        CFLX_NCCL(ncclCommInitRank(&c->world, world_size, id, world_rank));
    }
    *out = c;
    return CFLX_OK;
}

int cflx_comm_barrier(cflx_comm* c) {
    if (!c) return CFLX_ERR_ARG;
    CFLX_CUDA(cudaSetDevice(c->device));
    return grid_barrier(c);
}

void cflx_comm_destroy(cflx_comm* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->world) ncclCommDestroy(c->world);
    if (c->stream) cudaStreamDestroy(c->stream);
    cudaFree(c->d_scratch);
    delete c;
}

int cflx_auto_grid(int M, int N, int P, int* Px, int* Py, int* Pz) {  // lu_params.hpp:21-47
    if (M <= 0 || N <= 0 || P <= 0) return CFLX_ERR_ARG;
    const double ratio = 1.0 * std::max(M, N) / std::min(M, N);
    const int p1 = (int)std::cbrt(P / ratio);
    const int psq = (int)std::sqrt(P / ratio);
    const int phs = (int)std::sqrt(P / (2 * ratio));
    if (P == psq * psq) {
        *Px = psq; *Py = psq; *Pz = 1;
        return CFLX_OK;
    }
    if (phs * phs == P / 2) {
        *Px = phs; *Py = phs; *Pz = 2;
        return CFLX_OK;
    }
    int d[3] = {p1, (int)(ratio * p1), 0};
    d[2] = P / (d[0] * d[1]);
    std::sort(d, d + 3, [](int a, int b) { return a > b; });
    *Px = d[0]; *Py = d[1]; *Pz = d[2];
    return CFLX_OK;
}

int cflx_lu_dims(int M, int N, int v, int Px, int Py, int Pz, int* o) {  // lu_params.hpp:67-82
    if (M <= 0 || N <= 0 || v <= 0 || Px <= 0 || Py <= 0 || Pz <= 0 || !o) return CFLX_ERR_ARG;
    const int tx = (int)std::ceil((double)M / (v * Px)), ty = (int)std::ceil((double)N / (v * Py));
    const int Mp = v * Px * tx, Np = v * Py * ty;
    const int Nt = (int)std::ceil((double)Np / v), Mt = (int)std::ceil((double)Mp / v);
    o[0] = Mp; o[1] = Np;
    o[2] = (int)std::ceil((double)Mt / Px) * v;
    o[3] = (int)std::ceil((double)Nt / Py) * v;
    o[4] = Nt; o[5] = (v + Pz - 1) / Pz; o[6] = Mt; o[7] = Px * Py * Pz;
    return CFLX_OK;
}

int cflx_init_matrix_host(int M, int N, int v, int Px, int Py, int Pz, int rank, int seed, double* out) {
    int d[8];
    CFLX_TRY(cflx_lu_dims(M, N, v, Px, Py, Pz, d));
    const int Ml = d[2], Nl = d[3];
    if (rank < 0 || rank >= d[7] || !out) return CFLX_ERR_ARG;
    std::fill(out, out + (size_t)Ml * Nl, 0.0);
    if (rank % Pz != 0) return CFLX_OK;  // layers pk != 0 start at zero (lu_params.hpp:149-155)
    // lu_params.hpp:157-363: for (padded) M == N in {8, 9, 16, 20, 27, 32} the reference fills a FIXED matrix,
    // element (gi, gj) of the table at the tile-layout slot of this rank
    if (d[0] == d[1]) {
        std::vector<double> tab;
        if (fixed_input_matrix(d[0], &tab)) {
            const int n = d[0], pi = rank / (Py * Pz), pj = (rank / Pz) % Py;
            for (int lr = 0; lr < Ml; ++lr) {
                const int gi = ((lr / v) * Px + pi) * v + lr % v;
                for (int lc = 0; lc < Nl; ++lc) {
                    const int gj = ((lc / v) * Py + pj) * v + lc % v;
                    out[(size_t)lr * Nl + lc] = tab[(size_t)gi * n + gj];
                }
            }
            return CFLX_OK;
        }
    }
    // lu_params.hpp:364-375: mt19937_64(seed + rank), values 5 + U[0,1), tile by tile (lti outer, ltj inner),
    // row-major inside a tile (libs/costa/src/costa/grid2grid/grid_layout.hpp:68-92)
    std::mt19937_64 eng((unsigned long long)(seed + rank));
    std::uniform_real_distribution<double> dist;
    for (int lti = 0; lti < Ml / v; ++lti)
        for (int ltj = 0; ltj < Nl / v; ++ltj)
            for (int li = 0; li < v; ++li)
                for (int lj = 0; lj < v; ++lj) out[(size_t)(lti * v + li) * Nl + ltj * v + lj] = 5 + dist(eng);
    return CFLX_OK;
}

int cflx_lu_create(cflx_comm* c, int M, int N, int v, int Px, int Py, int Pz, cflx_lu** out) {
    if (!c || !out || M <= 0 || N <= 0 || v <= 0) return CFLX_ERR_ARG;
    CFLX_CUDA(cudaSetDevice(c->device));
    if (Px <= 0 || Py <= 0 || Pz <= 0) CFLX_TRY(cflx_auto_grid(M, N, c->world_size, &Px, &Py, &Pz));
    if (Px != Py) {
        set_last_error("grid %dx%dx%d: the CONFLUX LU path requires Px == Py (SURVEY.md fact 6)", Px, Py, Pz);
        return CFLX_ERR_UNSUPPORTED;
    }
    if (Px * Py * Pz != c->world_size) {
        set_last_error("grid %dx%dx%d does not match the %d ranks of the communicator", Px, Py, Pz, c->world_size);
        return CFLX_ERR_ARG;
    }
    if (v % 4 != 0 || v % Pz != 0 || (v / Pz) % 4 != 0 || pick_nb(v) == 0) {
        set_last_error("tile size v=%d unsupported: need v %% 4 == 0 and (v / Pz) %% 4 == 0", v);
        return CFLX_ERR_UNSUPPORTED;
    }
    int d[8];
    CFLX_TRY(cflx_lu_dims(M, N, v, Px, Py, Pz, d));
    auto* lu = new cflx_lu;
    lu->comm = c;
    lu->M = d[0]; lu->N = d[1]; lu->Ml = d[2]; lu->Nl = d[3]; lu->Nt = d[4]; lu->nlayr = d[5]; lu->Mt = d[6]; lu->P = d[7];
    lu->v = v; lu->Px = Px; lu->Py = Py; lu->Pz = Pz;
    lu->rank = c->world_rank;  // row-major cart numbering: rank = (pi*Py + pj)*Pz + pk
    lu->pi = lu->rank / (Py * Pz);
    lu->pj = (lu->rank / Pz) % Py;
    lu->pk = lu->rank % Pz;
    lu->nb = pick_nb(v);
    if (lu->M != lu->N) {
        set_last_error("only square matrices are supported (the miniapp passes M = N)");
        delete lu;
        return CFLX_ERR_UNSUPPORTED;
    }
    int rc = CFLX_OK;
    auto fail = [&](int code) {
        free_lu(lu);
        return code;
    };
    // sub-communicators (all ranks call all splits, same order)
    if ((rc = make_sub(c, lu->pi * Py + lu->pj, lu->pk, Pz, &lu->k_comm))) return fail(rc);
    if ((rc = make_sub(c, lu->pj * Pz + lu->pk, lu->pi, Px, &lu->i_comm))) return fail(rc);
    if ((rc = make_sub(c, lu->pi, lu->pj * Pz + lu->pk, Py * Pz, &lu->jk_comm))) return fail(rc);
    if ((rc = make_sub(c, lu->pj, lu->pi * Pz + lu->pk, Px * Pz, &lu->ik_comm))) return fail(rc);

    const size_t loc = (size_t)lu->Ml * lu->Nl;
    const int64_t ldp = round_up(lu->Ml, 2) + 2;
    lu->ldp_max = ldp;
    const size_t pan = (size_t)v * ldp, upan = (size_t)v * (lu->Nl + 2), vv = (size_t)v * v;
#define ALLOC(ptr, n) if ((rc = dmalloc(&(ptr), (n)))) return fail(rc)
    ALLOC(lu->A0, loc); ALLOC(lu->A11, loc);
    ALLOC(lu->PT, pan); ALLOC(lu->PT2, pan); ALLOC(lu->W, pan); ALLOC(lu->LT, pan);
    ALLOC(lu->A01raw, upan); ALLOC(lu->U, upan); ALLOC(lu->tmp, (size_t)v * lu->Nl);
    ALLOC(lu->A00, 2 * vv); ALLOC(lu->A00T, 2 * vv); ALLOC(lu->Uinv, vv); ALLOC(lu->LinvT, vv);
    ALLOC(lu->candH, 2 * vv); ALLOC(lu->S, 2 * vv); ALLOC(lu->W2, 2 * vv); ALLOC(lu->bcast, vv + v);
    ALLOC(lu->gri, lu->Ml); ALLOC(lu->gri_tmp, lu->Ml); ALLOC(lu->igri, lu->Ml); ALLOC(lu->perm, 2 * v);
    ALLOC(lu->gpivots, v); ALLOC(lu->tagsH, 2 * v); ALLOC(lu->tagsS, 2 * v); ALLOC(lu->hist, lu->M);
    ALLOC(lu->plan_mem, 6 * (size_t)v + 8 + lu->Ml);
#undef ALLOC
    int* pm = lu->plan_mem;
    lu->plan.npiv = pm; lu->plan.nel = pm + 4; pm += 8;
    lu->plan.cur_piv = pm; pm += v;
    lu->plan.order = pm; pm += v;
    lu->plan.slot2piv = pm; pm += v;
    lu->plan.early = pm; pm += v;
    lu->plan.late = pm; pm += v;
    pm += v;
    lu->plan.rowsrc = pm;
    if (cudaMallocHost((void**)&lu->h_npiv, sizeof(int)) != cudaSuccess) return fail(CFLX_ERR_CUDA);
    if (cudaEventCreateWithFlags(&lu->ev_npiv, cudaEventDisableTiming) != cudaSuccess) return fail(CFLX_ERR_CUDA);
    if ((rc = panel_workspace_create(&lu->pws))) return fail(rc);
    if ((rc = gemm_tn_setup())) return fail(rc);
    {
        // Trailing update on the int8 tcgen05 path (ozaki.cu) whenever the layer's contraction length is a whole number
        // of 128-element k chunks (v = 256 / 512 of the BASELINE configs); CFLX_GEMM=dmma selects the FP64 DMMA anchor.
        const char* e = getenv("CFLX_GEMM");
        const bool want = !(e && !strcmp(e, "dmma"));
        if (want && lu->nlayr % 128 == 0 && lu->nlayr <= 512) {
            if ((rc = ozaki_workspace_create(&lu->oz, lu->Ml, lu->Nl, lu->nlayr))) return fail(rc);
            lu->use_ozaki = true;
        }
    }
    lu->h_hist.assign(lu->M, -1);
    {
        // look-ahead: pivot search of iteration k+1 (extract, layer reduce, local search, tournament exchanges) on a
        // high-priority side stream, on a capped number of SMs, while the trailing update of iteration k runs on the
        // rest.  A rank never has NCCL work in flight on both streams: the side stream's collectives (k- and
        // i-communicator) sit between the fork after GEMM_next and the join before the next world broadcast.
        const char* e = getenv("CFLX_LOOKAHEAD");
        const char* em = getenv("CFLX_LOOKAHEAD_MULTI");  // multi-rank grids: on by default (validated on 2x2x1 / 1x1x2)
        const bool want = (e ? atoi(e) != 0 : true) && (lu->P == 1 || !em || atoi(em) != 0);
        if (want) {
            int lo = 0, hi = 0;
            cudaDeviceGetStreamPriorityRange(&lo, &hi);
            if (cudaStreamCreateWithPriority(&lu->side, cudaStreamNonBlocking, hi) != cudaSuccess) return fail(CFLX_ERR_CUDA);
            if (cudaEventCreateWithFlags(&lu->ev_fork, cudaEventDisableTiming) != cudaSuccess) return fail(CFLX_ERR_CUDA);
            if (cudaEventCreateWithFlags(&lu->ev_join, cudaEventDisableTiming) != cudaSuccess) return fail(CFLX_ERR_CUDA);
            const char* c = getenv("CFLX_PANEL_CTAS");
            // measured: 1x1x1 (C2) 32 -> 96.9 ms, 48 -> 96.7, 64 -> 102.6; 2x2x1 (C3) 48 -> 308 ms, 64 -> 283, 96 -> 309;
            // 1x1x2 was measured at 48 only (no tournament there, the trailing update is twice as large per rank)
            lu->pws.cta_cap = c ? atoi(c) : (lu->P == 1 ? 32 : (lu->Px == 1 ? 48 : 64));
        }
    }
    // zero the panels once: padded columns are read (and masked) by the GEMM producer
    cudaMemsetAsync(lu->PT, 0, pan * sizeof(double), c->stream);
    cudaMemsetAsync(lu->PT2, 0, pan * sizeof(double), c->stream);
    cudaMemsetAsync(lu->LT, 0, pan * sizeof(double), c->stream);
    cudaMemsetAsync(lu->W, 0, pan * sizeof(double), c->stream);
    cudaMemsetAsync(lu->A01raw, 0, upan * sizeof(double), c->stream);
    cudaMemsetAsync(lu->U, 0, upan * sizeof(double), c->stream);
    cudaMemsetAsync(lu->A0, 0, loc * sizeof(double), c->stream);
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) return fail(CFLX_ERR_CUDA);
    *out = lu;
    return CFLX_OK;
}

int cflx_lu_info(const cflx_lu* lu, int* o) {
    if (!lu || !o) return CFLX_ERR_ARG;
    const int vals[16] = {lu->M, lu->N, lu->Ml, lu->Nl, lu->Nt, lu->nlayr, lu->P, lu->Px, lu->Py, lu->Pz, lu->pi, lu->pj,
                          lu->pk, lu->rank, lu->v, 0};
    std::memcpy(o, vals, sizeof(vals));
    return CFLX_OK;
}

int cflx_lu_set_local(cflx_lu* lu, const double* host_local) {
    if (!lu || !host_local) return CFLX_ERR_ARG;
    CFLX_CUDA(cudaSetDevice(lu->comm->device));
    const size_t loc = (size_t)lu->Ml * lu->Nl;
    CFLX_CUDA(cudaMemcpyAsync(lu->A0, host_local, loc * sizeof(double), cudaMemcpyHostToDevice, lu->comm->stream));
    CFLX_CUDA(cudaStreamSynchronize(lu->comm->stream));
    lu->have_input = true;
    lu->factored = false;
    lu->sv.ready = false;
    lu->a0_is_next = false;
    lu->next_host = nullptr;
    return CFLX_OK;
}

// Input streaming for back-to-back factorisations: the NEXT cflx_lu_factor call uploads `host_next` (page-locked memory,
// valid until that call returns) into the input buffer on a copy stream as soon as it has taken its own working copy of
// the current input, so the 8*Ml*Nl-byte transfer overlaps the factorisation; the factorisation after that consumes it
// without a cflx_lu_set_local.  The residual of a run whose input buffer was handed to the next matrix is refused.
int cflx_lu_queue_next_local(cflx_lu* lu, const double* host_next) {
    if (!lu || !host_next) return CFLX_ERR_ARG;
    if (!lu->have_input) {
        set_last_error("cflx_lu_queue_next_local needs a current input (cflx_lu_set_local) first");
        return CFLX_ERR_STATE;
    }
    CFLX_CUDA(cudaSetDevice(lu->comm->device));
    if (!lu->copy) {
        CFLX_CUDA(cudaStreamCreateWithFlags(&lu->copy, cudaStreamNonBlocking));
        CFLX_CUDA(cudaEventCreateWithFlags(&lu->ev_a0_read, cudaEventDisableTiming));
        CFLX_CUDA(cudaEventCreateWithFlags(&lu->ev_upload, cudaEventDisableTiming));
    }
    lu->next_host = host_next;
    return CFLX_OK;
}

int cflx_lu_factor(cflx_lu* lu, double* ms_out) {
    if (!lu) return CFLX_ERR_ARG;
    if (!lu->have_input) {
        set_last_error("cflx_lu_factor before cflx_lu_set_local");
        return CFLX_ERR_STATE;
    }
    lu->sv.ready = false;  // the solve's copy of the factors describes the previous factorisation
    cflx_comm* c = lu->comm;
    cudaStream_t s = c->stream;
    CFLX_CUDA(cudaSetDevice(c->device));
    const size_t loc = (size_t)lu->Ml * lu->Nl;
    // "init" region of the reference (conflux_opt.hpp:347-515): A11Buff = copy of gv.data, gri, counters
    {
        PhaseTimer t(lu, RG_init, s);
        if (lu->a0_is_next) CFLX_CUDA(cudaStreamWaitEvent(s, lu->ev_upload, 0));  // this run's input was streamed in
        CFLX_CUDA(cudaMemcpyAsync(lu->A11, lu->A0, loc * sizeof(double), cudaMemcpyDeviceToDevice, s));
    }
    lu->a0_is_next = false;
    if (lu->next_host) {  // queued next input: overwrite A0 behind the working copy, concurrently with everything below
        CFLX_CUDA(cudaEventRecord(lu->ev_a0_read, s));
        CFLX_CUDA(cudaStreamWaitEvent(lu->copy, lu->ev_a0_read, 0));
        CFLX_CUDA(cudaMemcpyAsync(lu->A0, lu->next_host, loc * sizeof(double), cudaMemcpyHostToDevice, lu->copy));
        CFLX_CUDA(cudaEventRecord(lu->ev_upload, lu->copy));
        lu->next_host = nullptr;
        lu->a0_is_next = true;
    }
    CFLX_TRY(launch_iota_gri(lu->gri, lu->igri, lu->Ml, lu->v, lu->Px, lu->pi, s));
    for (double& x : lu->phase_ms) x = 0;
    for (int sd = 0; sd < 2; ++sd)
        for (int r = 0; r < RG_COUNT; ++r) lu->region_ms[sd][r] = 0, lu->region_cnt[sd][r] = 0;
    lu->tl_recs.clear();
    CFLX_TRY(grid_barrier(c));  // MPI_Barrier(lu_comm) before t1 (conflux_opt.hpp:531)
    cudaEvent_t e0, e1;
    CFLX_CUDA(cudaEventCreate(&e0));
    CFLX_CUDA(cudaEventCreate(&e1));
    CFLX_CUDA(cudaEventRecord(e0, s));
    int fnpr = 0;
    lu->gemm_flops = 0;
    lu->gemm_ms = 0;
    if (lu->time_gemm && (int)lu->ev.size() < 4 * lu->Nt) {
        for (auto& e : lu->ev) cudaEventDestroy(e);
        lu->ev.assign(4 * lu->Nt, nullptr);
        for (auto& e : lu->ev) CFLX_CUDA(cudaEventCreate(&e));
    }
    lu->ev_used.assign(2 * lu->Nt, 0);
    {
        cudaStream_t side = (lu->prof_mode == 1) ? nullptr : lu->side;
        if (side) {
            CFLX_CUDA(cudaEventRecord(lu->ev_fork, s));
            CFLX_CUDA(cudaStreamWaitEvent(side, lu->ev_fork, 0));
        }
        int rc0 = panel_phase(lu, 0, 0, side ? side : s);
        if (rc0 != CFLX_OK) return rc0;
        if (side) {
            CFLX_CUDA(cudaEventRecord(lu->ev_join, side));
            CFLX_CUDA(cudaStreamWaitEvent(s, lu->ev_join, 0));
        }
    }
    for (int k = 0; k < lu->Nt; ++k) {
        int rc = finish_step(lu, k, fnpr);
        if (rc != CFLX_OK) {
            cudaEventDestroy(e0);
            cudaEventDestroy(e1);
            return rc;
        }
    }
    CFLX_CUDA(cudaEventRecord(e1, s));
    CFLX_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    CFLX_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    CFLX_CUDA(cudaGetLastError());
    if (ms_out) *ms_out = ms;
    if (lu->prof_mode == 2) {  // resolve the timeline: every event has completed (e1 was synchronised, the side stream joined)
        if (lu->side) cudaStreamSynchronize(lu->side);
        for (const auto& r : lu->tl_recs) {
            float g = 0;
            if (cudaEventElapsedTime(&g, lu->tl_pool[r.ev], lu->tl_pool[r.ev + 1]) == cudaSuccess) {
                lu->region_ms[r.side][r.region] += g;
                lu->region_cnt[r.side][r.region]++;
                lu->phase_ms[region_phase(r.region)] += g;
            } else {
                cudaGetLastError();
            }
        }
    }
    if (lu->time_gemm) {
        for (int i = 0; i < 2 * lu->Nt; ++i) {
            if (!lu->ev_used[i]) continue;
            float g = 0;
            if (cudaEventElapsedTime(&g, lu->ev[2 * i], lu->ev[2 * i + 1]) == cudaSuccess) lu->gemm_ms += g;
            else cudaGetLastError();
        }
    }
    if (lu->a0_is_next) CFLX_CUDA(cudaStreamSynchronize(lu->copy));  // the caller's staging buffer is free again
    lu->factored = true;
    return CFLX_OK;
}

int cflx_lu_get_permutation(cflx_lu* lu, int* perm_out) {
    if (!lu || !perm_out) return CFLX_ERR_ARG;
    if (!lu->factored) {
        set_last_error("permutation requested before cflx_lu_factor");
        return CFLX_ERR_STATE;
    }
    CFLX_CUDA(cudaSetDevice(lu->comm->device));
    CFLX_CUDA(cudaMemcpyAsync(lu->h_hist.data(), lu->hist, sizeof(int) * lu->M, cudaMemcpyDeviceToHost, lu->comm->stream));
    CFLX_CUDA(cudaStreamSynchronize(lu->comm->stream));
    std::memcpy(perm_out, lu->h_hist.data(), sizeof(int) * lu->M);
    return CFLX_OK;
}

// Rows of the finished factors live where their original row lives (local rows are in the order they were
// promoted).  The reference's validation layout wants pivoted row q = k*v + i on rank (k % Px, pj, 0) at local
// row (k / Px)*v + i (conflux_opt.hpp:1673-1699,1721-1754): an all-to-all of whole rows inside each grid column.
int cflx_lu_get_factors(cflx_lu* lu, double* C_host, int* perm_out) {
    if (!lu) return CFLX_ERR_ARG;
    if (!lu->factored) {
        set_last_error("factors requested before cflx_lu_factor");
        return CFLX_ERR_STATE;
    }
    cflx_comm* c = lu->comm;
    cudaStream_t s = c->stream;
    CFLX_CUDA(cudaSetDevice(c->device));
    std::vector<int> hist(lu->M);
    CFLX_TRY(cflx_lu_get_permutation(lu, hist.data()));
    if (perm_out) std::memcpy(perm_out, hist.data(), sizeof(int) * lu->M);
    if (lu->pk != 0) return CFLX_OK;  // only layer 0 holds factors
    const size_t loc = (size_t)lu->Ml * lu->Nl;
    if (!lu->Cbuf) CFLX_TRY(dmalloc(&lu->Cbuf, loc));
    CFLX_TRY(redistribute_pivoted_rows(lu, hist, true, lu->A11, lu->Cbuf));
    if (C_host) CFLX_CUDA(cudaMemcpyAsync(C_host, lu->Cbuf, loc * sizeof(double), cudaMemcpyDeviceToHost, s));
    CFLX_CUDA(cudaStreamSynchronize(s));
    return CFLX_OK;
}

// ||P A - L U||_F (absolute, what the reference's validation build prints, conflux_miniapp.cpp:494-500) and the same
// relative to ||A||_F, computed on the device grid with the library's own GEMM + NCCL (validate.cu).  COLLECTIVE.
int cflx_lu_validate(cflx_lu* lu, double* frob_abs_out, double* frob_rel_out) {
    if (!lu) return CFLX_ERR_ARG;
    if (!lu->factored) {
        set_last_error("residual requested before cflx_lu_factor");
        return CFLX_ERR_STATE;
    }
    if (lu->a0_is_next) {
        set_last_error("residual refused: the input buffer of the last run was handed to the queued next matrix");
        return CFLX_ERR_STATE;
    }
    CFLX_CUDA(cudaSetDevice(lu->comm->device));
    std::vector<int> hist(lu->M);
    CFLX_TRY(cflx_lu_get_permutation(lu, hist.data()));
    return lu_residual_grid(lu, hist, frob_abs_out, frob_rel_out);
}
int cflx_lu_residual(cflx_lu* lu, double* rel_out) {
    if (!rel_out) return CFLX_ERR_ARG;
    return cflx_lu_validate(lu, nullptr, rel_out);
}

int cflx_host_alloc(size_t bytes, void** out) {
    if (!out) return CFLX_ERR_ARG;
    int n = 0;
    cflx_device_count(&n);
    if (n == 0) {
        set_last_error("no CUDA device visible: conflux_b200 has no CPU fallback");
        return CFLX_ERR_NO_DEVICE;
    }
    CFLX_CUDA(cudaHostAlloc(out, bytes, cudaHostAllocPortable));
    return CFLX_OK;
}
int cflx_host_free(void* p) {
    if (p) CFLX_CUDA(cudaFreeHost(p));
    return CFLX_OK;
}

int cflx_lu_uses_tcgen05(const cflx_lu* lu) { return lu && lu->use_ozaki ? 1 : 0; }
int cflx_lu_launch_count(cflx_lu* lu, int64_t* count_out, int reset) {
    if (!lu || !count_out) return CFLX_ERR_ARG;
    *count_out = lu->launches;
    if (reset) lu->launches = 0;
    return CFLX_OK;
}
int cflx_lu_set_profiling(cflx_lu* lu, int mode) {  // 0 off, 1 serialising phase timers, 2 non-serialising timeline
    if (!lu || mode < 0 || mode > 2) return CFLX_ERR_ARG;
    lu->prof_mode = mode;
    return CFLX_OK;
}
// JSON text {"main": {region: [ms, count], ...}, "side": {...}} of the last profiled cflx_lu_factor; region names are the
// reference's semiprof regions.  Returns the length needed (incl. the terminator) when buf is too small.
int cflx_lu_timeline(cflx_lu* lu, char* buf, int buf_len) {
    if (!lu) return CFLX_ERR_ARG;
    std::string o = "{";
    for (int sd = 0; sd < 2; ++sd) {
        o += sd ? ", \"side\": {" : "\"main\": {";
        bool first = true;
        for (int r = 0; r < RG_COUNT; ++r) {
            if (!lu->region_cnt[sd][r]) continue;
            char tmp[160];
            snprintf(tmp, sizeof(tmp), "%s\"%s\": [%.4f, %d]", first ? "" : ", ", region_name(r), lu->region_ms[sd][r], lu->region_cnt[sd][r]);
            o += tmp;
            first = false;
        }
        o += "}";
    }
    o += "}";
    if (!buf || buf_len <= (int)o.size()) return (int)o.size() + 1;
    std::memcpy(buf, o.c_str(), o.size() + 1);
    return CFLX_OK;
}
int cflx_lu_phase_ms(cflx_lu* lu, double* ms_out) {
    if (!lu || !ms_out) return CFLX_ERR_ARG;
    for (int i = 0; i < PH_COUNT; ++i) ms_out[i] = lu->phase_ms[i];
    return CFLX_OK;
}
int cflx_lu_set_kernel_timing(cflx_lu* lu, int enabled) {
    if (!lu) return CFLX_ERR_ARG;
    lu->time_gemm = enabled != 0;
    return CFLX_OK;
}
int cflx_lu_trailing_stats(cflx_lu* lu, double* ms_out, double* flops_out) {
    if (!lu || !ms_out || !flops_out) return CFLX_ERR_ARG;
    *ms_out = lu->gemm_ms;
    *flops_out = lu->gemm_flops;
    return CFLX_OK;
}
void cflx_lu_destroy(cflx_lu* lu) { free_lu(lu); }

}  // extern "C"
