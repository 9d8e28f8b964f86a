// conflux_b200/csrc/solve.cu -- A X = B with the factors of the last cflx_lu_factor (P A = L U), on the same grid.
//
// No counterpart in the reference (its LU stops at the factors).  The factors stay where the factorisation left them,
// re-laid out once per factorisation on the first solve:
//   C  = L\U in the conflux pivoted layout (redistribute_pivoted_rows, as cflx_lu_get_factors);
//   CT = C transposed per local column tile, CT[lc][r] = C[r][lc]: the K-major operand gemm_tn and the skinny update
//        stream, the same array serving the L part (rows below the diagonal tile) and the U part (rows above it);
//   on each diagonal-tile owner (t % Px, t % Py): the transposed diagonal tile and its nb x nb block inverses.
// The solve is a fan-in tile schedule over the Px x Py grid.  W (Ml x ldr, tile row t on grid row t % Px) holds the
// partial sums of the right-hand side still to be reduced:
//   P B    W = P B on grid column 0 (one copy per grid row), 0 elsewhere
//   L Y = P B, t = 0 .. Nt-1:  reduce tile row t over the grid row to (pr, pc, 0); Y_t = L_tt^-1 W_t there and kept in
//          its W_t slot (zeroed on the other ranks); Y_t broadcast over grid column pc; W[tiles > t] -= L[., t] Y_t
//   U X = Y, t = Nt-1 .. 0:    the same reduce; X_t = U_tt^-1 W_t; X_t broadcast over grid column pc (every layer:
//          that is the output layout); W[tiles < t] -= U[., t] X_t
// Layers pk != 0 contribute zeros to the reductions and receive the broadcasts; every rank issues its collectives in
// the same global order (t, reduce before broadcast), like the residual sweep in validate.cu.
#include <cstring>

#include "lu_state.h"

namespace cflx {
namespace {

// W[r][j] -= sum_k AT[k][r] * Y[k][j]: 64 rows per CTA, the K range split over 4 slices of 64 threads (one row per
// thread: every warp load is 32 consecutive doubles of one AT row).  Y is staged in shared memory in chunks of KC rows;
// each thread keeps NR FP64 FMA accumulators; the four slice partials are summed in a fixed order and subtracted once.
template <int NR>
__global__ void __launch_bounds__(256) solve_update_skinny_kernel(const double* __restrict__ AT, int64_t ldat, int M, int K,
                                                                  const double* __restrict__ Y, int64_t ldy, int n,
                                                                  double* __restrict__ W, int64_t ldw) {
    constexpr int RB = 64, KS = 4, KC = 128, KPS = KC / KS;
    __shared__ double sm[KS * RB * NR];  // Y chunk [KC][NR] during the sweep, then the slice partials [KS][RB][NR]
    const int row = threadIdx.x % RB, ks = threadIdx.x / RB;
    const int r = blockIdx.x * RB + row;
    double acc[NR];
#pragma unroll
    for (int j = 0; j < NR; ++j) acc[j] = 0.0;
    for (int k0 = 0; k0 < K; k0 += KC) {
        const int kn = min(KC, K - k0);
        __syncthreads();
        for (int e = threadIdx.x; e < KC * NR; e += blockDim.x) {
            const int k = e / NR, j = e % NR;
            sm[e] = (k < kn && j < n) ? Y[(int64_t)(k0 + k) * ldy + j] : 0.0;
        }
        __syncthreads();
        if (r < M) {
            const int kb = ks * KPS;
            const double* a = AT + (int64_t)(k0 + kb) * ldat + r;
            const double* y = sm + kb * NR;
#pragma unroll 8
            for (int k = 0; k < KPS; ++k) {
                const double x = (kb + k < kn) ? a[(int64_t)k * ldat] : 0.0;
#pragma unroll
                for (int j = 0; j < NR; ++j) acc[j] = fma(x, y[k * NR + j], acc[j]);
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < NR; ++j) sm[(ks * RB + row) * NR + j] = acc[j];
    __syncthreads();
    for (int e = threadIdx.x; e < RB * NR; e += blockDim.x) {
        const int rr = e / NR, j = e % NR, gr = blockIdx.x * RB + rr;
        if (gr < M && j < n) {
            double x = sm[rr * NR + j];
#pragma unroll
            for (int s = 1; s < KS; ++s) x += sm[(s * RB + rr) * NR + j];
            W[(int64_t)gr * ldw + j] -= x;
        }
    }
}

template <int NR>
int launch_skinny(const double* AT, int64_t ldat, int M, int K, const double* Y, int64_t ldy, int n, double* W, int64_t ldw,
                  cudaStream_t s) {
    solve_update_skinny_kernel<NR><<<(M + 63) / 64, 256, 0, s>>>(AT, ldat, M, K, Y, ldy, n, W, ldw);
    CFLX_CUDA(cudaGetLastError());
    return CFLX_OK;
}

// W[r][.] -= sum_k AT[k][r] * Y[k][.] for r < M: the skinny kernel up to SOLVE_SKINNY_MAX right-hand sides (ldr is the
// padded width; the padding columns are zero throughout), FP64 DMMA (gemm_tn) beyond.
int solve_update(const double* AT, int64_t ldat, int M, int K, const double* Y, int nrhs, int ldr, double* W,
                 cudaStream_t s) {
    if (M <= 0) return CFLX_OK;
    if (ldr <= SOLVE_SKINNY_MAX) return launch_solve_update_skinny(AT, ldat, M, K, Y, ldr, nrhs, W, ldr, s);
    GemmArgs g{};
    g.M = M; g.N = ldr; g.K = K;
    g.AT = AT; g.ldat = ldat;
    g.B = Y; g.ldb = ldr;
    g.C = W; g.ldc = ldr;
    g.D = W; g.ldd = ldr;
    g.alpha = -1.0; g.beta = 1.0;
    return launch_gemm_tn(g, s);
}

// One-time re-layout of the factors after a factorisation (layer 0; collective over the i-communicator when Px > 1).
int solve_prepare(cflx_lu* lu) {
    SolveState& sv = lu->sv;
    cflx_comm* c = lu->comm;
    cudaStream_t s = c->stream;
    const int v = lu->v, nb = lu->nb, Ml = lu->Ml, Nl = lu->Nl, Nt = lu->Nt;
    sv.hist.assign(lu->M, -1);
    CFLX_TRY(cflx_lu_get_permutation(lu, sv.hist.data()));
    sv.diag_slot.assign(Nt, -1);
    int ndiag = 0;
    for (int t = 0; t < Nt; ++t)
        if (t % lu->Px == lu->pi && t % lu->Py == lu->pj) sv.diag_slot[t] = ndiag++;
    if (lu->pk != 0) {
        sv.ready = true;
        return CFLX_OK;
    }
    const size_t loc = (size_t)Ml * Nl, per_diag = (size_t)v * v + 2 * (size_t)v * nb;
    if (!sv.CT) CFLX_TRY(dmalloc(&sv.CT, loc));
    if (!sv.diag && ndiag) CFLX_TRY(dmalloc(&sv.diag, ndiag * per_diag + (size_t)v * v));
    const bool own_cbuf = lu->Cbuf == nullptr, own_xbuf = lu->xbuf == nullptr;
    if (own_cbuf) CFLX_TRY(dmalloc(&lu->Cbuf, loc));
    int rc = redistribute_pivoted_rows(lu, sv.hist, true, lu->A11, lu->Cbuf);
    for (int lt = 0; lt < Nl / v && !rc; ++lt)
        rc = launch_extract_panel_T(lu->Cbuf, Nl, 0, (int64_t)lt * v, Ml, v, sv.CT + (size_t)lt * v * Ml, Ml, s);
    double* tile = sv.diag + ndiag * per_diag;  // row-major staging of one diagonal tile
    for (int t = 0; t < Nt && !rc; ++t) {
        const int d = sv.diag_slot[t];
        if (d < 0) continue;
        const int64_t lr = (int64_t)(t / lu->Px) * v, lc = (int64_t)(t / lu->Py) * v;
        double* DT = sv.diag + d * per_diag;
        if (cudaMemcpy2DAsync(tile, v * sizeof(double), lu->Cbuf + lr * Nl + lc, Nl * sizeof(double), v * sizeof(double), v,
                              cudaMemcpyDeviceToDevice, s) != cudaSuccess ||
            cudaMemcpy2DAsync(DT, v * sizeof(double), sv.CT + lc * Ml + lr, Ml * sizeof(double), v * sizeof(double), v,
                              cudaMemcpyDeviceToDevice, s) != cudaSuccess) {
            set_last_error("solve: diagonal tile copy: %s", cudaGetErrorString(cudaGetLastError()));
            rc = CFLX_ERR_CUDA;
            break;
        }
        rc = launch_diag_inverses(tile, v, nb, DT + (size_t)v * v + (size_t)v * nb, DT + (size_t)v * v, s, true);
    }
    if (!rc && cudaStreamSynchronize(s) != cudaSuccess) {
        set_last_error("solve: preparation: %s", cudaGetErrorString(cudaGetLastError()));
        rc = CFLX_ERR_CUDA;
    }
    if (own_cbuf) {  // a whole local matrix of staging: do not keep it alive for the solves
        cudaFree(lu->Cbuf);
        lu->Cbuf = nullptr;
    }
    if (own_xbuf) {
        cudaFree(lu->xbuf);
        lu->xbuf = nullptr;
    }
    if (!rc) sv.ready = true;
    return rc;
}

int solve_buffers(cflx_lu* lu, int ldr, bool reads_b) {
    SolveState& sv = lu->sv;
    if (ldr > sv.ldr_cap) {
        for (double** p : {&sv.W, &sv.X, &sv.B, &sv.stage}) {
            cudaFree(*p);
            *p = nullptr;
        }
        sv.ldr_cap = ldr;
    }
    const size_t cap = (size_t)lu->Ml * sv.ldr_cap;
    if (!sv.W) CFLX_TRY(dmalloc(&sv.W, cap));
    if (!sv.X) CFLX_TRY(dmalloc(&sv.X, (size_t)lu->Nl * sv.ldr_cap));
    if (reads_b && !sv.B) CFLX_TRY(dmalloc(&sv.B, cap));
    if (reads_b && lu->Px > 1 && !sv.stage) CFLX_TRY(dmalloc(&sv.stage, 2 * cap));
    return CFLX_OK;
}

int nccl_check(ncclResult_t r, const char* what, int t) {
    if (r == ncclSuccess) return CFLX_OK;
    set_last_error("solve: %s at tile %d -> %s", what, t, ncclGetErrorString(r));
    return CFLX_ERR_NCCL;
}

// the two sweeps; W holds P B (grid column 0, layer 0) and zeros elsewhere on entry, X receives the solution
int solve_sweeps(cflx_lu* lu, int nrhs, int ldr) {
    SolveState& sv = lu->sv;
    cudaStream_t s = lu->comm->stream;
    const int v = lu->v, nb = lu->nb, Px = lu->Px, Py = lu->Py, Pz = lu->Pz, Ml = lu->Ml, Nt = lu->Nt;
    const int pi = lu->pi, pj = lu->pj;
    const bool layer0 = lu->pk == 0;
    const bool row_comm = Py * Pz > 1, col_comm = Px * Pz > 1;
    const size_t per_diag = (size_t)v * v + 2 * (size_t)v * nb, tile = (size_t)v * ldr;
    for (int pass = 0; pass < 2; ++pass) {
        const bool fwd = pass == 0;
        for (int i = 0; i < Nt; ++i) {
            const int t = fwd ? i : Nt - 1 - i;
            const int pr = t % Px, pc = t % Py;
            const bool in_row = pi == pr, in_col = pj == pc, root = in_row && in_col && layer0;
            double* Wt = sv.W + (size_t)(t / Px) * tile;
            double* Xt = sv.X + (size_t)(t / Py) * tile;  // Y_t in the forward sweep, X_t in the backward one
            if (in_row && row_comm)
                CFLX_TRY(nccl_check(ncclReduce(Wt, Wt, tile, ncclDouble, ncclSum, pc * Pz, lu->jk_comm.c, s), "ncclReduce", t));
            if (root) {
                const double* DT = sv.diag + sv.diag_slot[t] * per_diag;
                if (fwd) {
                    CFLX_TRY(trsm_left_lower_unit(DT, DT + (size_t)v * v, v, nb, Wt, Xt, ldr, ldr, s));
                    CFLX_CUDA(cudaMemcpyAsync(Wt, Xt, tile * sizeof(double), cudaMemcpyDeviceToDevice, s));
                } else {
                    CFLX_TRY(trsm_left_upper(DT, DT + (size_t)v * v + (size_t)v * nb, v, nb, Wt, Xt, ldr, ldr, s));
                }
            } else if (in_row && fwd) {
                CFLX_CUDA(cudaMemsetAsync(Wt, 0, tile * sizeof(double), s));
            }
            if (in_col && col_comm)
                CFLX_TRY(nccl_check(ncclBroadcast(Xt, Xt, tile, ncclDouble, pr * Pz, lu->ik_comm.c, s), "ncclBroadcast", t));
            if (in_col && layer0) {
                const double* AT = sv.CT + (size_t)(t / Py) * v * Ml;
                if (fwd) {  // local rows of the tiles below t
                    const int lo = std::min(Ml, (t + 1 - pi + Px - 1) / Px * v);
                    CFLX_TRY(solve_update(AT + lo, Ml, Ml - lo, v, Xt, nrhs, ldr, sv.W + (size_t)lo * ldr, s));
                } else {    // local rows of the tiles above t
                    const int hi = std::min(Ml, (t - pi + Px - 1) / Px * v);
                    CFLX_TRY(solve_update(AT, Ml, hi, v, Xt, nrhs, ldr, sv.W, s));
                }
            }
        }
    }
    return CFLX_OK;
}
}  // namespace

int launch_solve_update_skinny(const double* AT, int64_t ldat, int M, int K, const double* Y, int64_t ldy, int n,
                               double* W, int64_t ldw, cudaStream_t s) {
    if (M <= 0 || K <= 0 || n <= 0) return CFLX_OK;
    if (n <= 2) return launch_skinny<2>(AT, ldat, M, K, Y, ldy, n, W, ldw, s);
    if (n <= 4) return launch_skinny<4>(AT, ldat, M, K, Y, ldy, n, W, ldw, s);
    if (n <= 8) return launch_skinny<8>(AT, ldat, M, K, Y, ldy, n, W, ldw, s);
    if (n <= 16) return launch_skinny<16>(AT, ldat, M, K, Y, ldy, n, W, ldw, s);
    set_last_error("solve_update_skinny: %d right-hand sides exceed %d", n, SOLVE_SKINNY_MAX);
    return CFLX_ERR_UNSUPPORTED;
}

void solve_state_free(SolveState* sv) {
    for (double* p : {sv->CT, sv->diag, sv->W, sv->X, sv->B, sv->stage}) cudaFree(p);
    *sv = SolveState{};
}

}  // namespace cflx

using namespace cflx;

extern "C" int cflx_lu_solve(cflx_lu* lu, int nrhs, const double* B_local, double* X_local, double* ms_out) {
    if (!lu || nrhs < 1 || !X_local) return CFLX_ERR_ARG;
    const bool reads_b = lu->pj == 0 && lu->pk == 0;
    if (reads_b && !B_local) {
        set_last_error("cflx_lu_solve: B_local is NULL on rank %d, which holds right-hand-side rows", lu->rank);
        return CFLX_ERR_ARG;
    }
    if (!lu->factored) {
        set_last_error("cflx_lu_solve needs the factors of a cflx_lu_factor on the current input");
        return CFLX_ERR_STATE;
    }
    cflx_comm* c = lu->comm;
    cudaStream_t s = c->stream;
    CFLX_CUDA(cudaSetDevice(c->device));
    if (!lu->sv.ready) CFLX_TRY(solve_prepare(lu));
    SolveState& sv = lu->sv;
    const int ldr = (int)round_up(nrhs, 2), Ml = lu->Ml, Nl = lu->Nl;
    CFLX_TRY(solve_buffers(lu, ldr, reads_b));
    CFLX_CUDA(cudaMemsetAsync(sv.W, 0, (size_t)Ml * ldr * sizeof(double), s));
    if (reads_b) {
        CFLX_CUDA(cudaMemsetAsync(sv.B, 0, (size_t)Ml * ldr * sizeof(double), s));
        CFLX_CUDA(cudaMemcpy2DAsync(sv.B, ldr * sizeof(double), B_local, nrhs * sizeof(double), nrhs * sizeof(double), Ml,
                                    cudaMemcpyHostToDevice, s));
    }
    CFLX_TRY(grid_barrier(c));
    cudaEvent_t e0, e1;
    CFLX_CUDA(cudaEventCreate(&e0));
    CFLX_CUDA(cudaEventCreate(&e1));
    int rc = cudaEventRecord(e0, s) == cudaSuccess ? CFLX_OK : CFLX_ERR_CUDA;
    if (!rc && reads_b) rc = redistribute_pivoted_rows(lu, sv.hist, false, sv.B, sv.W, ldr, ldr, sv.stage);
    if (!rc) rc = solve_sweeps(lu, nrhs, ldr);
    if (!rc && cudaEventRecord(e1, s) != cudaSuccess) rc = CFLX_ERR_CUDA;
    if (!rc && cudaMemcpy2DAsync(X_local, nrhs * sizeof(double), sv.X, ldr * sizeof(double), nrhs * sizeof(double), Nl,
                                 cudaMemcpyDeviceToHost, s) != cudaSuccess)
        rc = CFLX_ERR_CUDA;
    if (cudaStreamSynchronize(s) != cudaSuccess && !rc) {
        set_last_error("cflx_lu_solve: %s", cudaGetErrorString(cudaGetLastError()));
        rc = CFLX_ERR_CUDA;
    }
    float ms = 0;
    if (!rc && cudaEventElapsedTime(&ms, e0, e1) != cudaSuccess) rc = CFLX_ERR_CUDA;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (!rc && ms_out) *ms_out = ms;
    return rc;
}
