// conflux_b200/csrc/chol.cu -- CONFCHOX: the reference's communication-avoiding Cholesky factorisation (A = L L^T, lower),
// re-designed for a grid of B200s.  BASELINE config C5: cholesky_miniapp --dim=32768 --tile=512 on 8 GPUs.
//
// Reference (relative to /root/reference/src/conflux/cholesky):
//   Cholesky.cpp:60-160        initialize(): grid / tile-size choice, buffers, input generation      -> cflx_chol_create,
//                                                                                                      cflx_chol_auto_grid/_tile
//   CholeskyIO.cpp:100-172     generateInputMatrixDistributed(): every v x v tile = lower(R^T R), srand(1),
//                              diagonal := 2 * Kappa * max row sum                                   -> cflx_chol_init_matrix_host
//   Cholesky.cpp:188-193       choleskyA00: LAPACKE_dpotrf on the diagonal tile                      -> potrf_tile_kernel
//   Cholesky.cpp:280-281,450   updateA10: cblas_dtrsm(Right, Lower, Trans, NonUnit) tile by tile     -> trsm_right_upper_T on L_kk^T
//   Cholesky.cpp:345-351,512+  computeA11: cblas_dgemm(N, T) tile by tile, k-slab of the z layer     -> gemm_tn on K-major panels
//   Cholesky.cpp:580-612       reduceA11: the next tile column is summed over the z layers            -> ncclReduce (k-communicator)
//   Cholesky.cpp:620-700       scatterA11 / A00 broadcast                                            -> ncclBroadcast of L_kk^T and of the
//                                                                                                      panel pieces
// B200-first layout instead of the reference's tile objects (TileMatrix.h): every rank keeps its 2-D block-cyclic share
// of the matrix as ONE row-major Ml x Nl array in HBM (tile (gi, gj) on rank (gi % Px, gj % Py) at local tile (gi / Px,
// gj / Py); the lower triangle is meaningful), the tile column of a step is handled as a transposed (K-major) panel like
// in the LU path, so the TRSM and the rank-v update run on the same FP64 tensor-core GEMM (gemm.cu) on long contiguous
// operands instead of v x v tile calls.  The "A10 -> A01 representative" exchange of the reference (every rank needs the
// panel rows of its tile rows AND of its tile columns) is one grouped broadcast of the Px panel pieces to all ranks.
#include <climits>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "lu_state.h"

using namespace cflx;

struct cflx_chol {
    cflx_comm* comm = nullptr;
    int N = 0, v = 0, Kappa = 0, Px = 1, Py = 1, Pz = 1, P = 1, Ml = 0, Nl = 0, nlayr = 0, nb = 0;
    int pi = 0, pj = 0, pk = 0, rank = 0;
    SubComm k_comm, i_comm;
    double *A0 = nullptr, *A11 = nullptr, *PT = nullptr, *LT = nullptr, *G = nullptr /* [2] */, *Bc = nullptr /* [2] */, *D = nullptr, *A00 = nullptr,
           *W = nullptr, *Uinv = nullptr, *LinvT = nullptr, *acc = nullptr, *Q = nullptr /* scratch of the blocked tile Cholesky */;
    int* info = nullptr;
    int64_t ldp = 0, ldb = 0;
    OzakiWorkspace oz{};                    // digit planes of the int8 tcgen05 rank-v update (default when v / Pz is 128..512)
    bool use_ozaki = false;
    cudaStream_t side = nullptr;            // panel pipeline of step k+1 (all NCCL traffic lives here) under the update of step k
    cudaEvent_t ev_col[2] = {nullptr, nullptr}, ev_panel[2] = {nullptr, nullptr};
    bool have_input = false, factored = false;
    int64_t launches = 0;
};

namespace {

// ---------------------------------------------------------------------------------------------- diagonal tile
// Cholesky of one v x v tile (row-major, lower triangle referenced) by ONE CTA: right-looking, 32-column blocks.
//   D   in: the tile; out: L in the lower triangle, zeros above
//   UT  out: L^T (upper triangular, row-major) -- the operand of the panel TRSM and what is broadcast
// info[0] = global column + 1 of the first non-positive pivot, like LAPACK's dpotrf on the whole matrix.  A kernel writes
// it only while it is still 0: after a failure NaN reaches every later block and tile, and on one stream the first
// failure must win.
constexpr int PB = 32;
// D: v x v window (leading dimension ldd) of the tile, UT: the same window of L^T (leading dimension ldu); Uc (optional): a
// contiguous v x v copy of the factored block's L^T; col_off: global column of the window's first column (for *info)
__global__ void __launch_bounds__(1024) potrf_tile_kernel(double* __restrict__ D, int v, int ldd, double* __restrict__ UT, int ldu,
                                                          double* __restrict__ Uc, int* __restrict__ info, int col_off) {
    extern __shared__ double sm[];
    double* Ld = sm;                 // [PB][PB + 1] factored diagonal block
    double* Xs = sm + PB * (PB + 1);  // [v][PB + 1] panel below it
    __shared__ int s_bad;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) s_bad = 0;
    for (int jb = 0; jb < v; jb += PB) {
        const int nb = min(PB, v - jb), m = v - jb - nb;
        for (int e = t; e < nb * nb; e += blockDim.x) Ld[(e / nb) * (PB + 1) + e % nb] = D[(size_t)(jb + e / nb) * ldd + jb + e % nb];
        __syncthreads();
        if (warp == 0) {  // lane = row of the block, the row lives in registers
            double a[PB];
#pragma unroll
            for (int c = 0; c < PB; ++c) a[c] = (lane < nb && c <= lane && c < nb) ? Ld[lane * (PB + 1) + c] : 0.0;
#pragma unroll
            for (int c = 0; c < PB; ++c) {
                if (c < nb) {
                    const double d = __shfl_sync(0xffffffffu, a[c], c);
                    if (!(d > 0.0) && lane == 0 && s_bad == 0) s_bad = col_off + jb + c + 1;
                    const double sq = sqrt(d);
                    if (lane == c) a[c] = sq;
                    else if (lane > c) a[c] = a[c] / sq;
#pragma unroll
                    for (int c2 = c + 1; c2 < PB; ++c2) {
                        const double l2 = __shfl_sync(0xffffffffu, a[c], c2);  // L[c2][c]
                        if (lane >= c2) a[c2] = fma(-a[c], l2, a[c2]);
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < PB; ++c)
                if (lane < nb && c < nb) Ld[lane * (PB + 1) + c] = (c <= lane) ? a[c] : 0.0;
        }
        __syncthreads();
        // the factored block goes back (zeros above its diagonal) and into UT transposed
        for (int e = t; e < nb * nb; e += blockDim.x) {
            const int r = e / nb, c = e % nb;
            const double x = Ld[r * (PB + 1) + c];
            D[(size_t)(jb + r) * ldd + jb + c] = x;
            UT[(size_t)(jb + c) * ldu + jb + r] = x;          // UT[c][r] = L[r][c] (zero for c > r)
        }
        // panel below: X = P * L_d^-T, one thread per row (forward substitution against the block in shared memory)
        for (int i = t; i < m; i += blockDim.x) {
            double* prow = D + (size_t)(jb + nb + i) * ldd + jb;
            double x[PB];
#pragma unroll
            for (int c = 0; c < PB; ++c) x[c] = c < nb ? prow[c] : 0.0;
#pragma unroll
            for (int c = 0; c < PB; ++c) {
                if (c < nb) {
                    double s = x[c];
#pragma unroll
                    for (int q = 0; q < c; ++q) s = fma(-x[q], Ld[c * (PB + 1) + q], s);
                    x[c] = s / Ld[c * (PB + 1) + c];
                }
            }
#pragma unroll
            for (int c = 0; c < PB; ++c) {
                if (c < nb) {
                    prow[c] = x[c];
                    Xs[i * (PB + 1) + c] = x[c];
                    UT[(size_t)(jb + c) * ldu + jb + nb + i] = x[c];   // L^T
                }
            }
        }
        __syncthreads();
        // trailing block (lower triangle, row i >= column j): T[i][j] -= X[i][:] . X[j][:]
        const int tiles = (m + 31) / 32;
        for (int tt = warp; tt < tiles * tiles; tt += (blockDim.x >> 5)) {
            const int ti = tt / tiles, tj = tt % tiles;
            if (tj > ti) continue;
            const int j = tj * 32 + lane;
            // 8 rows per iteration: the 8 loads of T are issued together (they are L2 round trips of a single SM), then
            // the dot products against the shared-memory panel, then the 8 stores
#pragma unroll 1
            for (int i0 = 0; i0 < 32; i0 += 8) {
                double tv[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int i = ti * 32 + i0 + q;
                    tv[q] = (i < m && j < m && j <= i) ? D[(size_t)(jb + nb + i) * ldd + jb + nb + j] : 0.0;
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int i = ti * 32 + i0 + q;
                    if (i < m && j < m && j <= i) {
                        double s = 0.0;
#pragma unroll
                        for (int c = 0; c < PB; ++c) s = fma(Xs[i * (PB + 1) + c], Xs[j * (PB + 1) + c], s);
                        tv[q] -= s;
                    }
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int i = ti * 32 + i0 + q;
                    if (i < m && j < m && j <= i) D[(size_t)(jb + nb + i) * ldd + jb + nb + j] = tv[q];
                }
            }
        }
        __syncthreads();
    }
    // zeros above the diagonal of D / below the diagonal of UT
    for (int e = t; e < v * v; e += blockDim.x) {
        const int r = e / v, c = e % v;
        if (c > r) {
            D[(size_t)r * ldd + c] = 0.0;
            UT[(size_t)c * ldu + r] = 0.0;
        }
    }
    if (Uc != nullptr) {
        __syncthreads();
        for (int e = t; e < v * v; e += blockDim.x) Uc[e] = UT[(size_t)(e / v) * ldu + e % v];
    }
    if (t == 0 && s_bad && info[0] == 0) info[0] = s_bad;
}

// Cholesky of ONE 128 x 128 diagonal block held entirely in shared memory (the building block of potrf_tile): all 512
// threads take part in every phase -- 32-column diagonal blocks on warp 0 (row per lane), the rows below
// by forward substitution (one row per thread), the trailing part one element per thread from shared memory.  D / UT are
// windows of the tile (leading dimensions ldd / ldu), Uc a contiguous copy of L^T for the block-column solve.
constexpr int QBK = 128;
constexpr int QPITCH = QBK + 1;
constexpr int QTHREADS = 512;
__global__ void __launch_bounds__(QTHREADS) potrf128_kernel(double* __restrict__ D, int ldd, double* __restrict__ UT, int ldu,
                                                        double* __restrict__ Uc, int* __restrict__ info, int col_off) {
    extern __shared__ double As[];  // [QBK][QPITCH], lower triangle
    __shared__ int s_bad;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) s_bad = 0;
    for (int e = t; e < QBK * QBK; e += QTHREADS) {
        const int r = e / QBK, c = e % QBK;
        As[r * QPITCH + c] = (c <= r) ? D[(size_t)r * ldd + c] : 0.0;
    }
    __syncthreads();
    for (int jb = 0; jb < QBK; jb += PB) {
        const int m = QBK - jb - PB;
        if (warp == 0) {  // 32 x 32 diagonal block in place, lane = row (shared memory: a register array of 32 doubles that is
                          // indexed by the unrolled column loop ends up in local memory, which is what made the old kernel slow)
            double* B = As + jb * QPITCH + jb;
            for (int c = 0; c < PB; ++c) {
                const double d = B[c * QPITCH + c];
                if (!(d > 0.0) && lane == 0 && s_bad == 0) s_bad = col_off + jb + c + 1;
                const double sq = sqrt(d);
                double l = 0.0;
                if (lane == c) B[c * QPITCH + c] = sq;
                else if (lane > c) {
                    l = B[lane * QPITCH + c] / sq;
                    B[lane * QPITCH + c] = l;
                }
                __syncwarp();
#pragma unroll 4
                for (int c2 = c + 1; c2 < PB; ++c2) {
                    const double l2 = B[c2 * QPITCH + c];  // L[c2][c], broadcast
                    if (lane >= c2) B[lane * QPITCH + c2] = fma(-l, l2, B[lane * QPITCH + c2]);
                }
                __syncwarp();
            }
        }
        __syncthreads();
        if (m <= 0) break;
        // rows below: X = P * L_d^-T, one row per thread, in place in shared memory (L_d is a broadcast read)
        if (t < m) {
            double* prow = As + (jb + PB + t) * QPITCH + jb;
            const double* Ld = As + jb * QPITCH + jb;
#pragma unroll 4
            for (int c = 0; c < PB; ++c) {
                double sacc = prow[c];
                for (int q = 0; q < c; ++q) sacc = fma(-prow[q], Ld[c * QPITCH + q], sacc);
                prow[c] = sacc / Ld[c * QPITCH + c];
            }
        }
        __syncthreads();
        // trailing part (lower triangle): T[i][k] -= X[i][:] . X[k][:], one element per thread and pass
        for (int e = t; e < m * m; e += QTHREADS) {
            const int i = e / m, k = e % m;
            if (k > i) continue;
            const double* xi = As + (jb + PB + i) * QPITCH + jb;
            const double* xk = As + (jb + PB + k) * QPITCH + jb;
            double sacc = 0.0;
#pragma unroll
            for (int c = 0; c < PB; ++c) sacc = fma(xi[c], xk[c], sacc);
            As[(jb + PB + i) * QPITCH + jb + PB + k] -= sacc;
        }
        __syncthreads();
    }
    // L into the tile (zeros above its diagonal), L^T into UT and into the contiguous copy
    for (int e = t; e < QBK * QBK; e += QTHREADS) {
        const int r = e / QBK, c = e % QBK;
        D[(size_t)r * ldd + c] = As[r * QPITCH + c];            // (zeros above the diagonal were loaded as zeros)
        const double lt = As[c * QPITCH + r];                    // L^T[r][c] = L[c][r]
        UT[(size_t)r * ldu + c] = lt;
        Uc[e] = lt;
    }
    if (t == 0 && s_bad && info[0] == 0) info[0] = s_bad;   // the first failure wins (see potrf_tile_kernel)
}

// zeros above the diagonal of D (= L) and below the diagonal of UT (= L^T)
__global__ void tri_clean_kernel(double* __restrict__ D, double* __restrict__ UT, int v) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= v * v) return;
    const int r = e / v, c = e % v;
    if (c > r) {
        D[e] = 0.0;
        UT[(size_t)c * v + r] = 0.0;
    }
}

// D[r][c] = PT[c][r] (diagonal tile out of the transposed panel) / A11 tile <- D
__global__ void tile_from_panel_kernel(const double* __restrict__ PT, int64_t ldp, int v, double* __restrict__ D) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < v * v) D[e] = PT[(int64_t)(e % v) * ldp + e / v];
}
__global__ void tile_store_kernel(const double* __restrict__ D, int v, double* __restrict__ A, int64_t lda) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < v * v) A[(int64_t)(e / v) * lda + e % v] = D[e];
}
// Bc[c][t * v + x] = G_piece(j % Px)[c][(j / Px) * v - row1(j % Px) + x] for the local column tiles t (global j = (lj0 + t) * Py + pj)
struct GatherArgs {
    const double* G;       // Px pieces, piece p = [v][ld_p] with ld_p = its active rows rounded up to even
    int64_t piece_stride;
    double* Bc;
    int64_t ldb;
    int v, Px, Py, pj, lj0, ntiles, gfirst, Ml;
};
__global__ void gather_cols_kernel(GatherArgs a) {
    const int t = blockIdx.x, c = blockIdx.y;
    const int j = (a.lj0 + t) * a.Py + a.pj;            // global tile index of this local column tile
    const int p = j % a.Px;
    const int d = a.gfirst - p;
    const int first = d <= 0 ? 0 : (d + a.Px - 1) / a.Px;   // first local tile row of piece p that holds a tile >= gfirst
    const int rows = a.Ml - first * a.v;
    const int64_t ldg = max(2, (rows + 1) & ~1);
    const double* src = a.G + (int64_t)p * a.piece_stride + (int64_t)c * ldg + (int64_t)(j / a.Px - first) * a.v;
    double* dst = a.Bc + (int64_t)c * a.ldb + (int64_t)t * a.v;
    for (int x = threadIdx.x; x < a.v; x += blockDim.x) dst[x] = src[x];
}
// sum of squares of the lower triangle (global row >= global column) of a local block-cyclic array
__global__ void sumsq_lower_kernel(const double* __restrict__ X, int Ml, int Nl, int v, int Px, int Py, int pi, int pj,
                                   double* __restrict__ out) {
    double s = 0.0;
    const int64_t total = (int64_t)Ml * Nl;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int lr = (int)(e / Nl), lc = (int)(e % Nl);
        const int64_t gr = ((int64_t)(lr / v) * Px + pi) * v + lr % v, gc = ((int64_t)(lc / v) * Py + pj) * v + lc % v;
        if (gr >= gc) s = fma(X[e], X[e], s);
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ double w[32];
    if ((threadIdx.x & 31) == 0) w[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        s = threadIdx.x < (blockDim.x >> 5) ? w[threadIdx.x] : 0.0;
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (threadIdx.x == 0) atomicAdd(out, s);
    }
}
// validation: transposed panel of column block t out of the stored factor, the diagonal tile masked to its lower triangle
__global__ void extract_l_panel_T_kernel(const double* __restrict__ A, int64_t lda, int row0, int col0, int n, int v, int Px,
                                         int pi, int t, double* __restrict__ PT, int64_t ldp) {
    __shared__ double tile[32][33];
    const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int dy = threadIdx.y; dy < 32; dy += blockDim.y) {
        const int r = r0 + dy, c = c0 + threadIdx.x;
        double x = 0.0;
        if (r < n && c < v) {
            const int lr = row0 + r;
            const int64_t gr = ((int64_t)(lr / v) * Px + pi) * v + lr % v, gc = (int64_t)t * v + c;
            x = gr >= gc ? A[(int64_t)lr * lda + col0 + c] : 0.0;
        }
        tile[dy][threadIdx.x] = x;
    }
    __syncthreads();
    for (int dy = threadIdx.y; dy < 32; dy += blockDim.y) {
        const int c = c0 + dy, r = r0 + threadIdx.x;
        if (r < n && c < v) PT[(int64_t)c * ldp + r] = tile[threadIdx.x][dy];
    }
}

int ceil_div_pos(int a, int b) { return a <= 0 ? 0 : (a + b - 1) / b; }
// first local tile row / column whose global tile index is >= g
int first_local_tile(int g, int p, int P) { return ceil_div_pos(g - p, P); }

int chol_pick_nb(int v) {
    for (int nb : {128, 64, 32, 16, 8, 4})
        if (v % nb == 0) return nb;
    return 0;
}

void free_chol(cflx_chol* ch) {
    if (!ch) return;
    cudaSetDevice(ch->comm->device);
    for (double* p : {ch->A0, ch->A11, ch->PT, ch->LT, ch->W, ch->G, ch->Bc, ch->D, ch->A00, ch->Uinv, ch->LinvT, ch->acc, ch->Q}) cudaFree(p);
    cudaFree(ch->info);
    if (ch->use_ozaki) ozaki_workspace_destroy(&ch->oz);
    if (ch->side) cudaStreamDestroy(ch->side);
    for (int i = 0; i < 2; ++i) {
        if (ch->ev_col[i]) cudaEventDestroy(ch->ev_col[i]);
        if (ch->ev_panel[i]) cudaEventDestroy(ch->ev_panel[i]);
    }
    for (SubComm* sc : {&ch->k_comm, &ch->i_comm})
        if (sc->c) ncclCommDestroy(sc->c);
    delete ch;
}

// Broadcast the Px pieces of the (transposed) panel of column block t to every rank and apply
//   X[i][j] -= L[i][t] * L[j][t]^T   to the local tiles with global tile row i >= tile column j >= jmin (lower triangle),
// each z layer with its own slab of the v contraction indices.  piece_rows0(p) = first local row of piece p.
int piece_ld(const cflx_chol* ch, int gfirst, int p) {  // leading dimension of piece p: its active rows, even, >= 2
    const int rows = ch->Ml - first_local_tile(gfirst, p, ch->Px) * ch->v;
    return (int)std::max<int64_t>(2, round_up(std::max(rows, 0), 2));
}
// Broadcast the Px pieces of the (transposed) panel of column block t (rows of global tiles >= gfirst) to every rank into
// buffer set `buf`, and assemble the column operand for the local column tiles with global index >= jmin.
int broadcast_pieces(cflx_chol* ch, int t, int gfirst, int jmin, int buf, cudaStream_t s) {
    const int v = ch->v, Px = ch->Px, Py = ch->Py, Pz = ch->Pz, Ml = ch->Ml, Nl = ch->Nl;
    const int pjt = t % Py;
    const int64_t piece_stride = (int64_t)v * ch->ldp;
    double* G = ch->G + (int64_t)buf * Px * piece_stride;
    double* Bc = ch->Bc + (int64_t)buf * v * ch->ldb;
    if (ch->P > 1) {
        CFLX_NCCL(ncclGroupStart());
        for (int p = 0; p < Px; ++p) {
            const int rows = Ml - first_local_tile(gfirst, p, Px) * v;
            if (rows <= 0) continue;
            const int root = (p * Py + pjt) * Pz;
            double* dst = G + (int64_t)p * piece_stride;
            const double* src = (ch->rank == root) ? ch->LT : dst;
            CFLX_NCCL(ncclBroadcast(src, dst, (size_t)v * piece_ld(ch, gfirst, p), ncclDouble, root, ch->comm->world, s));
        }
        CFLX_NCCL(ncclGroupEnd());
    } else {
        CFLX_CUDA(cudaMemcpyAsync(G, ch->LT, (size_t)v * piece_ld(ch, gfirst, 0) * sizeof(double), cudaMemcpyDeviceToDevice, s));
    }
    const int lj0 = first_local_tile(jmin, ch->pj, Py);
    const int ntc = Nl / v - lj0;
    if (ntc <= 0) return CFLX_OK;
    GatherArgs ga{G, piece_stride, Bc, ch->ldb, v, Px, Py, ch->pj, lj0, ntc, gfirst, Ml};
    gather_cols_kernel<<<dim3(ntc, v), 128, 0, s>>>(ga);
    CFLX_CUDA(cudaGetLastError());
    ch->launches++;
    return CFLX_OK;
}
// X[i][j] -= L[i][t] * L[j][t]^T on the local tiles with global tile row i >= tile column j, j in the local column tiles
// [lj_lo, lj_hi) (global index >= jmin; lower triangle), each z layer with its own slab of the v contraction indices.
// SMs the persistent tcgen05 update leaves to the look-ahead panel pipeline on the side stream (CFLX_CHOL_LEAVE)
static int chol_leave_sms() {
    static int leave = -1;
    if (leave < 0) {
        const char* e = getenv("CFLX_CHOL_LEAVE");
        leave = e ? atoi(e) : 8;
        if (leave < 0) leave = 0;
        if (leave > 100) leave = 100;
    }
    return leave;
}

int update_columns(cflx_chol* ch, int gfirst, int jmin, int buf, double* X, int lj_lo, int lj_hi, cudaStream_t s, int planes_buf = -1) {
    const int v = ch->v, Px = ch->Px, Py = ch->Py, Ml = ch->Ml, Nl = ch->Nl;
    const int pi = ch->pi, pj = ch->pj, pk = ch->pk;
    const int64_t piece_stride = (int64_t)v * ch->ldp;
    const double* G = ch->G + (int64_t)buf * Px * piece_stride;
    const double* Bc = ch->Bc + (int64_t)buf * v * ch->ldb;
    const int lj0 = first_local_tile(jmin, pj, Py);              // Bc column 0 corresponds to this local tile
    const int my_first = first_local_tile(gfirst, pi, Px);        // first local tile row of MY piece
    const int64_t ldg = piece_ld(ch, gfirst, pi);
    // One launch per GROUP of local tile columns: wide enough (>= ~8192 rows x columns of v) to fill the machine; the rows
    // start at the diagonal of the group's first column, so later columns of a group also update a few tiles above their
    // own diagonal (upper triangle: never read) -- a few per cent of extra flops instead of many half-empty launches.
    const int lj_end = std::min(lj_hi, Nl / v);
    const int my_rows = Ml - my_first * v;                          // rows of my piece = rows of the A planes
    for (int lj = std::max(lj_lo, lj0); lj < lj_end;) {
        const int j = lj * Py + pj;                               // global tile column of the group's first column
        const int li = first_local_tile(j, pi, Px);               // first local tile row with global index >= j
        const int M = Ml - li * v;
        if (M <= 0) break;                                        // later columns have even fewer rows
        int gcols = std::max(1, (8192 + M - 1) / M);
        gcols = std::min(gcols, lj_end - lj);
        GemmArgs g{};
        g.M = M; g.N = gcols * v; g.K = ch->nlayr;
        g.AT = G + (int64_t)pi * piece_stride + (int64_t)pk * ch->nlayr * ldg + (int64_t)(li - my_first) * v;
        g.ldat = ldg;
        g.B = Bc + (int64_t)pk * ch->nlayr * ch->ldb + (int64_t)(lj - lj0) * v;
        g.ldb = ch->ldb;
        g.C = X + (int64_t)li * v * Nl + (int64_t)lj * v;
        g.ldc = Nl;
        g.D = const_cast<double*>(g.C);
        g.ldd = Nl;
        g.alpha = -1.0; g.beta = 1.0;
        if (ch->use_ozaki && planes_buf == buf)   // planes of this buffer set are current (see split_planes)
            CFLX_TRY(launch_ozaki_gemm(&ch->oz, M, g.N, (li - my_first) * v, (lj - lj0) * v, g.D, Nl, ch->oz.sms - chol_leave_sms(), s));
        else
            CFLX_TRY(launch_gemm_tn(g, s));
        ch->launches++;
        lj += gcols;
    }
    (void)my_rows;
    return CFLX_OK;
}
// digit planes of the operands of one update sweep: my piece (rows) and the gathered column operand, this layer's slab
int split_planes(cflx_chol* ch, int gfirst, int jmin, int buf, cudaStream_t s);
int split_planes(cflx_chol* ch, int gfirst, int jmin, int buf, cudaStream_t s) {
    if (!ch->use_ozaki) return CFLX_OK;
    const int v = ch->v, Px = ch->Px;
    const int64_t piece_stride = (int64_t)v * ch->ldp;
    const double* G = ch->G + (int64_t)buf * Px * piece_stride;
    const double* Bc = ch->Bc + (int64_t)buf * v * ch->ldb;
    const int my_first = first_local_tile(gfirst, ch->pi, Px);
    const int rows = ch->Ml - my_first * v;
    const int ncols = ch->Nl - first_local_tile(jmin, ch->pj, ch->Py) * v;
    const int64_t ldg = piece_ld(ch, gfirst, ch->pi);
    if (rows > 0) CFLX_TRY(ozaki_split_a(&ch->oz, G + (int64_t)ch->pi * piece_stride + (int64_t)ch->pk * ch->nlayr * ldg, ldg, rows, s));
    if (ncols > 0) CFLX_TRY(ozaki_split_b(&ch->oz, Bc + (int64_t)ch->pk * ch->nlayr * ch->ldb, ch->ldb, 0, ncols, s));
    ch->launches += 2;
    return CFLX_OK;
}
int broadcast_and_update(cflx_chol* ch, int t, int jmin, bool below_only, double* X, cudaStream_t s) {
    const int gfirst = below_only ? t + 1 : t;
    CFLX_TRY(broadcast_pieces(ch, t, gfirst, jmin, 0, s));
    return update_columns(ch, gfirst, jmin, 0, X, 0, ch->Nl / ch->v, s);
}

// Panel pipeline of step k on stream s: z-reduce of tile column k, Cholesky of the diagonal tile, L_kk^T down the grid
// column, the panel solve, the stores, and (k < Kappa - 1) the broadcast of the panel pieces into buffer set k & 1.
// (1) Cholesky of the v x v diagonal tile.  One CTA needs 2.2 ms for a 512 x 512 tile (measured: 2/3 of a whole 16384^2
// factorisation), so the tile is itself factored in 128-wide block columns: the 128 x 128 diagonal block on one CTA, the
// block column below it by ONE GEMM with the inverted block, the trailing part of the tile by one rank-128 GEMM -- both on
// the whole GPU (FP64 DMMA kernel).  Tiles that are not a multiple of 128 (tests) keep the one-CTA kernel.
//   D [v][v] in: the tile, out: L (zeros above the diagonal);  UT [v][v] out: L^T;  Q: scratch of the blocked path
//   (potrf_tile_scratch(v) doubles; nullptr selects the one-CTA kernel);  info: see potrf_tile_kernel;  col0: global column
//   of the tile's first column.  Adds its kernel launches to *launches.  The factorisation and cflx_dbg_potrf_tile both
//   run this.
constexpr int QB = 128;
size_t potrf_tile_smem(int v) { return ((size_t)PB * (PB + 1) + (size_t)v * (PB + 1)) * sizeof(double); }
size_t potrf_tile_scratch(int v) { return (size_t)3 * QB * QB + (size_t)2 * QB * v; }
bool potrf_tile_blocked(int v) { return v % QB == 0 && v >= 2 * QB; }
int potrf_tile_setup(int v) {   // shared memory limits of both kernels (per device)
    CFLX_CUDA(cudaFuncSetAttribute(potrf_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)potrf_tile_smem(v)));
    CFLX_CUDA(cudaFuncSetAttribute(potrf128_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(QBK * QPITCH * sizeof(double))));
    return CFLX_OK;
}
int potrf_tile(int v, double* D, double* UT, double* Q, int* info, int col0, cudaStream_t s, int64_t* launches) {
    if (!potrf_tile_blocked(v) || Q == nullptr) {
        potrf_tile_kernel<<<1, 1024, potrf_tile_smem(v), s>>>(D, v, v, UT, v, nullptr, info, col0);
        CFLX_CUDA(cudaGetLastError());
        *launches += 1;
        return CFLX_OK;
    }
    double* U128 = Q;                          // [QB][QB]  L_d^T of the current diagonal block, contiguous
    double* Ui = U128 + QB * QB;               // [QB][QB]  its inverse
    double* Li = Ui + QB * QB;                 // [QB][QB]  (unit-lower companion of launch_diag_inverses, unused)
    double* XT0 = Li + QB * QB;                // [QB][v]   block column below the diagonal block, transposed
    double* XT = XT0 + (size_t)QB * v;         // [QB][v]   ... after the solve
    static_assert(QB == QBK, "block width of the tile Cholesky");
    for (int jb = 0; jb < v; jb += QB) {
        const int m = v - jb - QB;
        potrf128_kernel<<<1, QTHREADS, QBK * QPITCH * sizeof(double), s>>>(D + (size_t)jb * v + jb, v, UT + (size_t)jb * v + jb, v, U128,
                                                                        info, col0 + jb);
        CFLX_CUDA(cudaGetLastError());
        *launches += 1;
        if (m <= 0) break;
        const int64_t ldx = m;
        CFLX_TRY(launch_extract_panel_T(D, v, jb + QB, jb, m, QB, XT0, ldx, s));
        CFLX_TRY(launch_diag_inverses(U128, QB, QB, Ui, Li, s));
        CFLX_TRY(trsm_right_upper_T(U128, Ui, QB, QB, XT0, XT, ldx, m, s));          // X^T = L_d^-1 P^T
        CFLX_TRY(launch_store_panel_T(D, v, jb + QB, jb, m, QB, XT, ldx, s));
        CFLX_CUDA(cudaMemcpy2DAsync(UT + (size_t)jb * v + jb + QB, (size_t)v * sizeof(double), XT, ldx * sizeof(double),
                                    (size_t)m * sizeof(double), QB, cudaMemcpyDeviceToDevice, s));
        GemmArgs g{};                                                                 // T -= X X^T
        g.M = m; g.N = m; g.K = QB;
        g.AT = XT; g.ldat = ldx;
        g.B = XT; g.ldb = ldx;
        g.C = D + (size_t)(jb + QB) * v + jb + QB; g.ldc = v;
        g.D = D + (size_t)(jb + QB) * v + jb + QB; g.ldd = v;
        g.alpha = -1.0; g.beta = 1.0;
        CFLX_TRY(launch_gemm_tn(g, s));
        *launches += 6;
    }
    tri_clean_kernel<<<(v * v + 255) / 256, 256, 0, s>>>(D, UT, v);
    CFLX_CUDA(cudaGetLastError());
    *launches += 1;
    return CFLX_OK;
}

int panel_step(cflx_chol* ch, int k, cudaStream_t s) {
    const int v = ch->v, Px = ch->Px, Py = ch->Py, Pz = ch->Pz, Ml = ch->Ml, Nl = ch->Nl;
    const int pi = ch->pi, pj = ch->pj, pk = ch->pk;
    const int pik = k % Px, pjk = k % Py;
    const int loff = (k / Py) * v;
    const int row0 = first_local_tile(k, pi, Px) * v;        // my first row at or below tile k
    const int row1 = first_local_tile(k + 1, pi, Px) * v;    // ... strictly below tile k
    const int n0 = Ml - row0, n1 = Ml - row1;
    const int64_t ld = std::max<int64_t>(2, round_up(n0, 2));    // panel from the diagonal tile down
    const int64_t ld1 = piece_ld(ch, k + 1, pi);                 // rows strictly below tile k (what is broadcast)
    const bool on_col = (pj == pjk);
    const bool owner = on_col && pi == pik && pk == 0;
    // (4 of the previous step) tile column k summed over the z layers                  Cholesky.cpp:580-612
    if (on_col && n0 > 0) {
        CFLX_TRY(launch_extract_panel_T(ch->A11, Nl, row0, loff, n0, v, ch->PT, ld, s));
        ch->launches++;
        if (Pz > 1) CFLX_NCCL(ncclReduce(ch->PT, ch->PT, (size_t)v * ld, ncclDouble, ncclSum, 0, ch->k_comm.c, s));
    }
    // (1) Cholesky of the diagonal tile                                                 Cholesky.cpp:188-193
    if (owner) {
        tile_from_panel_kernel<<<(v * v + 255) / 256, 256, 0, s>>>(ch->PT, ld, v, ch->D);
        CFLX_TRY(potrf_tile(v, ch->D, ch->A00, ch->Q, ch->info + 1, k * v, s, &ch->launches));
        tile_store_kernel<<<(v * v + 255) / 256, 256, 0, s>>>(ch->D, v, ch->A11 + (int64_t)row0 * Nl + loff, Nl);
        CFLX_CUDA(cudaGetLastError());
        ch->launches += 2;
    }
    if (k == ch->Kappa - 1) return CFLX_OK;
    // L_kk^T to the ranks that hold the tile column (layer 0)                           Cholesky.cpp:680-690
    if (on_col && pk == 0 && Px > 1)
        CFLX_NCCL(ncclBroadcast(ch->A00, ch->A00, (size_t)v * v, ncclDouble, pik, ch->i_comm.c, s));
    // (2) tile column: A10 <- A10 * L_kk^-T                                              Cholesky.cpp:280-281,450-451
    if (on_col && pk == 0 && n1 > 0) {
        CFLX_TRY(launch_diag_inverses(ch->A00, v, ch->nb, ch->Uinv, ch->LinvT, s));
        // PT rows are relative to row0 (ld); the solve works on the window below the diagonal tile and the result is
        // repacked with the leading dimension of the broadcast piece (ld1)
        CFLX_TRY(trsm_right_upper_T(ch->A00, ch->Uinv, v, ch->nb, ch->PT + (row1 - row0), ch->W, ld, n1, s));
        CFLX_CUDA(cudaMemcpy2DAsync(ch->LT, ld1 * sizeof(double), ch->W, ld * sizeof(double), (size_t)n1 * sizeof(double), v,
                                    cudaMemcpyDeviceToDevice, s));
        CFLX_TRY(launch_store_panel_T(ch->A11, Nl, row1, loff, n1, v, ch->LT, ld1, s));
        ch->launches += 2 * (v / ch->nb) + 1;
    }
    // the reference's A10 -> A01 representative exchange                                 Cholesky.cpp:205-330
    return broadcast_pieces(ch, k, k + 1, k + 1, k & 1, s);
}

}  // namespace

// ======================================================================================================== C ABI
extern "C" {

// Cholesky.cpp:75-111: grid chosen for the user when grid == {0,0,0}
int cflx_chol_auto_grid(int P, int N, int* grid3) {
    if (P <= 0 || !grid3) return CFLX_ERR_ARG;
    if (P == 8 && N < 16384) { grid3[0] = 2; grid3[1] = 2; grid3[2] = 2; }
    else if (P == 32 && N < 8192) { grid3[0] = 4; grid3[1] = 4; grid3[2] = 2; }
    else if (P == 128 && N <= 16384) { grid3[0] = 8; grid3[1] = 8; grid3[2] = 2; }
    else if (P == 512) { grid3[0] = 16; grid3[1] = 16; grid3[2] = 2; }
    else {
        const unsigned pw = (unsigned)std::log2((double)P);
        grid3[0] = pw % 2 == 0 ? 1 << (pw / 2) : (1 << (pw / 2)) * 2;
        grid3[1] = 1 << (pw / 2);
        grid3[2] = 1;
    }
    return CFLX_OK;
}
// Cholesky.cpp:113-134: tile size chosen for the user when v == 0
int cflx_chol_auto_tile(int N, int P, int Pz) {
    const double ratio = ((double)N * N * Pz / P) / 1000000.0;
    return ratio < 2.5 ? 128 : (ratio < 30 ? 256 : (ratio < 250 ? 512 : 1024));
}

// dims_out[6] = {N padded to a multiple of v, Kappa, Ml, Nl, nlayr, P}
int cflx_chol_dims(int N, int v, int Px, int Py, int Pz, int* o) {
    if (N <= 0 || v <= 0 || Px <= 0 || Py <= 0 || Pz <= 0 || !o) return CFLX_ERR_ARG;
    const int Kappa = (N + v - 1) / v;
    o[0] = Kappa * v; o[1] = Kappa;
    o[2] = ((Kappa + Px - 1) / Px) * v;
    o[3] = ((Kappa + Py - 1) / Py) * v;
    o[4] = v / Pz; o[5] = Px * Py * Pz;
    return CFLX_OK;
}

// CholeskyIO.cpp:100-172: T = lower triangle of R^T R with R = v x v uniform(-1, 1) from rand() after srand(1) (same on
// every rank); every tile of the (lower triangle of the) matrix is T, the global diagonal is 2 * Kappa * max_i sum_j |T_ij|.
// Layers pz != 0 start at zero.  (The reference leaves the upper triangle of its tile buffer unwritten; zeros here.)
int cflx_chol_init_matrix_host(int N, int v, int Px, int Py, int Pz, int rank, double* out) {
    int d[6];
    CFLX_TRY(cflx_chol_dims(N, v, Px, Py, Pz, d));
    if (rank < 0 || rank >= d[5] || !out) return CFLX_ERR_ARG;
    const int Ml = d[2], Nl = d[3], Kappa = d[1];
    std::fill(out, out + (size_t)Ml * Nl, 0.0);
    if (rank % Pz != 0) return CFLX_OK;
    const int pi = rank / (Py * Pz), pj = (rank / Pz) % Py;
    std::vector<double> R((size_t)v * v), T((size_t)v * v, 0.0);
    srand(1);
    for (size_t i = 0; i < (size_t)v * v; ++i) R[i] = (double)rand() / RAND_MAX * 2 - 1;
    for (int i = 0; i < v; ++i)                 // T = lower(R^T R)  (cblas_dsyrk RowMajor, Lower, Trans)
        for (int j = 0; j <= i; ++j) {
            double s = 0.0;
            for (int k = 0; k < v; ++k) s += R[(size_t)k * v + i] * R[(size_t)k * v + j];
            T[(size_t)i * v + j] = s;
        }
    double mx = -1;
    for (int i = 0; i < v; ++i) {
        double cur = 0.0;
        for (int j = 0; j < v; ++j) cur += std::fabs(T[(size_t)i * v + j]);
        mx = std::max(mx, cur);
    }
    mx = mx * Kappa * 2;
    for (int lti = 0; lti < Ml / v; ++lti)
        for (int ltj = 0; ltj < Nl / v; ++ltj) {
            const int gi = lti * Px + pi, gj = ltj * Py + pj;
            if (gi >= Kappa || gj >= Kappa) continue;
            for (int r = 0; r < v; ++r) std::memcpy(out + (size_t)(lti * v + r) * Nl + (size_t)ltj * v, T.data() + (size_t)r * v, sizeof(double) * v);
            if (gi == gj)
                for (int r = 0; r < v; ++r) out[(size_t)(lti * v + r) * Nl + (size_t)ltj * v + r] = mx;
        }
    return CFLX_OK;
}

int cflx_chol_create(cflx_comm* c, int N, int v, int Px, int Py, int Pz, cflx_chol** out) {
    if (!c || !out || N <= 0) return CFLX_ERR_ARG;
    CFLX_CUDA(cudaSetDevice(c->device));
    if (Px <= 0 || Py <= 0 || Pz <= 0) {
        int g[3];
        CFLX_TRY(cflx_chol_auto_grid(c->world_size, N, g));
        Px = g[0]; Py = g[1]; Pz = g[2];
    }
    if (v <= 0) v = cflx_chol_auto_tile(N, c->world_size, Pz);
    if (Px * Py * Pz != c->world_size) {
        set_last_error("cholesky grid %dx%dx%d does not match the %d ranks of the communicator", Px, Py, Pz, c->world_size);
        return CFLX_ERR_ARG;
    }
    if (v % 4 != 0 || v % Pz != 0 || (v / Pz) % 4 != 0 || v > 512 || chol_pick_nb(v) == 0) {
        set_last_error("cholesky tile size v=%d unsupported: need v %% 4 == 0, (v / Pz) %% 4 == 0, v <= 512", v);
        return CFLX_ERR_UNSUPPORTED;
    }
    int d[6];
    CFLX_TRY(cflx_chol_dims(N, v, Px, Py, Pz, d));
    auto* ch = new cflx_chol;
    ch->comm = c;
    ch->N = d[0]; ch->Kappa = d[1]; ch->Ml = d[2]; ch->Nl = d[3]; ch->nlayr = d[4]; ch->P = d[5];
    ch->v = v; ch->Px = Px; ch->Py = Py; ch->Pz = Pz;
    ch->rank = c->world_rank;  // like the LU path: rank = (pi * Py + pj) * Pz + pk
    ch->pi = ch->rank / (Py * Pz);
    ch->pj = (ch->rank / Pz) % Py;
    ch->pk = ch->rank % Pz;
    ch->nb = chol_pick_nb(v);
    int rc = CFLX_OK;
    auto fail = [&](int code) {
        free_chol(ch);
        return code;
    };
    if ((rc = make_sub(c, ch->pi * Py + ch->pj, ch->pk, Pz, &ch->k_comm))) return fail(rc);
    if ((rc = make_sub(c, ch->pj * Pz + ch->pk, ch->pi, Px, &ch->i_comm))) return fail(rc);
    const size_t loc = (size_t)ch->Ml * ch->Nl, vv = (size_t)v * v;
    ch->ldp = round_up(ch->Ml, 2) + 2;
    ch->ldb = round_up(ch->Nl, 2) + 2;
#define ALLOC(ptr, n) if ((rc = dmalloc(&(ptr), (n)))) return fail(rc)
    ALLOC(ch->A0, loc); ALLOC(ch->A11, loc);
    ALLOC(ch->PT, (size_t)v * ch->ldp); ALLOC(ch->LT, (size_t)v * ch->ldp); ALLOC(ch->W, (size_t)v * ch->ldp);
    ALLOC(ch->G, 2 * (size_t)Px * v * ch->ldp); ALLOC(ch->Bc, 2 * (size_t)v * ch->ldb);
    ALLOC(ch->D, vv); ALLOC(ch->A00, vv); ALLOC(ch->Uinv, vv); ALLOC(ch->LinvT, vv); ALLOC(ch->acc, 4);
    ALLOC(ch->info, 4);
    if (potrf_tile_blocked(v)) ALLOC(ch->Q, potrf_tile_scratch(v));
#undef ALLOC
    cudaMemsetAsync(ch->PT, 0, (size_t)v * ch->ldp * sizeof(double), c->stream);
    cudaMemsetAsync(ch->LT, 0, (size_t)v * ch->ldp * sizeof(double), c->stream);
    cudaMemsetAsync(ch->W, 0, (size_t)v * ch->ldp * sizeof(double), c->stream);
    cudaMemsetAsync(ch->G, 0, 2 * (size_t)Px * v * ch->ldp * sizeof(double), c->stream);
    cudaMemsetAsync(ch->Bc, 0, 2 * (size_t)v * ch->ldb * sizeof(double), c->stream);
    cudaMemsetAsync(ch->A0, 0, loc * sizeof(double), c->stream);
    cudaMemsetAsync(ch->A00, 0, vv * sizeof(double), c->stream);
    if ((rc = gemm_tn_setup())) return fail(rc);
    {
        const char* e = getenv("CFLX_GEMM");
        if (!(e && !strcmp(e, "dmma")) && ch->nlayr % 128 == 0 && ch->nlayr <= 512) {
            if ((rc = ozaki_workspace_create(&ch->oz, ch->Ml, ch->Nl, ch->nlayr))) return fail(rc);
            ch->use_ozaki = true;
        }
    }
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (cudaStreamCreateWithPriority(&ch->side, cudaStreamNonBlocking, hi) != cudaSuccess) return fail(CFLX_ERR_CUDA);
        for (int i = 0; i < 2; ++i)
            if (cudaEventCreateWithFlags(&ch->ev_col[i], cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&ch->ev_panel[i], cudaEventDisableTiming) != cudaSuccess)
                return fail(CFLX_ERR_CUDA);
    }
    if ((rc = potrf_tile_setup(v))) return fail(rc);
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) return fail(CFLX_ERR_CUDA);
    *out = ch;
    return CFLX_OK;
}

// info_out[16] = {N, v, Kappa, Ml, Nl, nlayr, P, Px, Py, Pz, pi, pj, pk, rank, 0, 0}
int cflx_chol_info(const cflx_chol* ch, int* o) {
    if (!ch || !o) return CFLX_ERR_ARG;
    const int vals[16] = {ch->N, ch->v, ch->Kappa, ch->Ml, ch->Nl, ch->nlayr, ch->P, ch->Px, ch->Py, ch->Pz, ch->pi, ch->pj, ch->pk,
                          ch->rank, 0, 0};
    std::memcpy(o, vals, sizeof(vals));
    return CFLX_OK;
}

int cflx_chol_set_local(cflx_chol* ch, const double* host_local) {
    if (!ch || !host_local) return CFLX_ERR_ARG;
    CFLX_CUDA(cudaSetDevice(ch->comm->device));
    CFLX_CUDA(cudaMemcpyAsync(ch->A0, host_local, (size_t)ch->Ml * ch->Nl * sizeof(double), cudaMemcpyHostToDevice, ch->comm->stream));
    CFLX_CUDA(cudaStreamSynchronize(ch->comm->stream));
    ch->have_input = true;
    ch->factored = false;
    return CFLX_OK;
}

// COLLECTIVE.  parallelCholesky() (Cholesky.cpp:760-921): ms_out = device time of the factorisation loop.
int cflx_chol_factor(cflx_chol* ch, double* ms_out) {
    if (!ch) return CFLX_ERR_ARG;
    if (!ch->have_input) {
        set_last_error("cflx_chol_factor before cflx_chol_set_local");
        return CFLX_ERR_STATE;
    }
    cflx_comm* c = ch->comm;
    cudaStream_t s = c->stream;
    CFLX_CUDA(cudaSetDevice(c->device));
    const int v = ch->v, Py = ch->Py, Ml = ch->Ml, Nl = ch->Nl;
    const int pj = ch->pj;
    CFLX_CUDA(cudaMemcpyAsync(ch->A11, ch->A0, (size_t)Ml * Nl * sizeof(double), cudaMemcpyDeviceToDevice, s));
    CFLX_CUDA(cudaMemsetAsync(ch->info, 0, sizeof(int) * 4, s));
    CFLX_TRY(grid_barrier(c));
    cudaEvent_t e0, e1;
    CFLX_CUDA(cudaEventCreate(&e0));
    CFLX_CUDA(cudaEventCreate(&e1));
    CFLX_CUDA(cudaEventRecord(e0, s));
    // Look-ahead: the panel pipeline of step k+1 (z-reduce, diagonal Cholesky, solve, piece broadcast -- and every NCCL
    // call of the factorisation) runs on the side stream while the main stream applies the rank-v update of step k; the
    // tile column of step k+1 is updated first so that the side stream can start.
    cudaStream_t sp = ch->side;
    CFLX_CUDA(cudaEventRecord(ch->ev_col[0], s));
    CFLX_CUDA(cudaStreamWaitEvent(sp, ch->ev_col[0], 0));
    CFLX_TRY(panel_step(ch, 0, sp));
    CFLX_CUDA(cudaEventRecord(ch->ev_panel[0], sp));
    for (int k = 0; k + 1 < ch->Kappa; ++k) {
        const int b = k & 1, nb1 = (k + 1) & 1;
        CFLX_CUDA(cudaStreamWaitEvent(s, ch->ev_panel[b], 0));             // pieces of step k are in buffer set b
        CFLX_TRY(split_planes(ch, k + 1, k + 1, b, s));                     // (int8 tcgen05 path) digit planes of both operands
        const int ljn = (k + 1) / Py;                                        // local tile of column k+1 on its owners
        const bool own_next = (pj == (k + 1) % Py);
        if (own_next) CFLX_TRY(update_columns(ch, k + 1, k + 1, b, ch->A11, ljn, ljn + 1, s, b));
        CFLX_CUDA(cudaEventRecord(ch->ev_col[nb1], s));
        CFLX_CUDA(cudaStreamWaitEvent(sp, ch->ev_col[nb1], 0));
        CFLX_TRY(panel_step(ch, k + 1, sp));
        CFLX_CUDA(cudaEventRecord(ch->ev_panel[nb1], sp));
        CFLX_TRY(update_columns(ch, k + 1, k + 1, b, ch->A11, own_next ? ljn + 1 : 0, Nl / v, s, b));
    }
    CFLX_CUDA(cudaStreamWaitEvent(s, ch->ev_panel[(ch->Kappa - 1) & 1], 0));
    CFLX_CUDA(cudaEventRecord(e1, s));
    CFLX_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    CFLX_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    CFLX_CUDA(cudaGetLastError());
    // Only the owner of a diagonal tile sees its pivots: the first failing column (the smallest nonzero info) is agreed on
    // by every rank, so that the collective call returns the same answer everywhere.
    int h[4] = {0, 0, 0, 0};
    CFLX_CUDA(cudaMemcpy(h, ch->info, sizeof(h), cudaMemcpyDeviceToHost));
    if (ch->P > 1) {
        const int mine = h[1] != 0 ? h[1] : INT_MAX;
        CFLX_CUDA(cudaMemcpyAsync(ch->info + 2, &mine, sizeof(int), cudaMemcpyHostToDevice, s));
        CFLX_NCCL(ncclAllReduce(ch->info + 2, ch->info + 2, 1, ncclInt32, ncclMin, c->world, s));
        CFLX_CUDA(cudaMemcpyAsync(&h[2], ch->info + 2, sizeof(int), cudaMemcpyDeviceToHost, s));
        CFLX_CUDA(cudaStreamSynchronize(s));
        h[1] = h[2] == INT_MAX ? 0 : h[2];
    }
    if (h[1] != 0) {
        set_last_error("cholesky: the matrix is not positive definite (the leading minor of order %d is not positive: "
                       "column %d, like dpotrf's info)", h[1], h[1]);
        return CFLX_ERR_STATE;
    }
    if (ms_out) *ms_out = ms;
    ch->factored = true;
    return CFLX_OK;
}

// local share of L (Ml x Nl row-major, conflux tile layout; tiles above the diagonal are not meaningful)
int cflx_chol_get_local(cflx_chol* ch, double* L_host) {
    if (!ch || !L_host) return CFLX_ERR_ARG;
    if (!ch->factored) {
        set_last_error("factor requested before cflx_chol_factor");
        return CFLX_ERR_STATE;
    }
    CFLX_CUDA(cudaSetDevice(ch->comm->device));
    CFLX_CUDA(cudaMemcpyAsync(L_host, ch->A11, (size_t)ch->Ml * ch->Nl * sizeof(double), cudaMemcpyDeviceToHost, ch->comm->stream));
    CFLX_CUDA(cudaStreamSynchronize(ch->comm->stream));
    return CFLX_OK;
}

// COLLECTIVE.  ||A - L L^T||_F over the lower triangle (absolute and relative to ||A||_F), on the GPU grid: the update
// sweep is replayed with the stored factor on a copy of the input.  (The reference's checker, examples/cholesky_helper.cpp:
// 183-217, compares against LAPACKE_dpotrf on one node; tests/ do that at small sizes.)
int cflx_chol_validate(cflx_chol* ch, double* abs_out, double* rel_out) {
    if (!ch) return CFLX_ERR_ARG;
    if (!ch->factored) {
        set_last_error("validation requested before cflx_chol_factor");
        return CFLX_ERR_STATE;
    }
    cflx_comm* c = ch->comm;
    cudaStream_t s = c->stream;
    CFLX_CUDA(cudaSetDevice(c->device));
    const int v = ch->v, Px = ch->Px, Py = ch->Py, Ml = ch->Ml, Nl = ch->Nl;
    const size_t loc = (size_t)Ml * Nl;
    double* R = nullptr;
    CFLX_TRY(dmalloc(&R, loc));
    int rc = CFLX_OK;
    // every layer replays with the full contraction on layer 0's factor: only layer 0 holds L, so restrict to pk == 0 by
    // zeroing the other layers' contribution (their A11 holds partial sums, not the factor)
    if (cudaMemcpyAsync(R, ch->A0, loc * sizeof(double), cudaMemcpyDeviceToDevice, s) != cudaSuccess) rc = CFLX_ERR_CUDA;
    const int nlayr_save = ch->nlayr, pk_save = ch->pk;
    for (int t = 0; t < ch->Kappa && !rc; ++t) {
        const int pjt = t % Py;
        const int row0 = first_local_tile(t, ch->pi, Px) * v, n0 = Ml - row0;
        if (ch->pj == pjt && pk_save == 0 && n0 > 0) {
            dim3 grid((n0 + 31) / 32, (v + 31) / 32), block(32, 8);
            extract_l_panel_T_kernel<<<grid, block, 0, s>>>(ch->A11, Nl, row0, (t / Py) * v, n0, v, Px, ch->pi, t, ch->LT,
                                                            piece_ld(ch, t, ch->pi));
        }
        // layer 0 applies the whole contraction, the other layers a zero-length slab (they only take part in the broadcasts)
        ch->nlayr = pk_save == 0 ? v : 0;
        ch->pk = 0;
        if (pk_save == 0) rc = broadcast_and_update(ch, t, t, false, R, s);
        else {
            // participate in the grouped broadcasts only
            ncclGroupStart();
            for (int p = 0; p < Px && !rc; ++p) {
                const int rows = Ml - first_local_tile(t, p, Px) * v;
                if (rows <= 0) continue;
                double* buf = ch->G + (int64_t)p * v * ch->ldp;
                if (ncclBroadcast(buf, buf, (size_t)v * piece_ld(ch, t, p), ncclDouble, (p * Py + pjt) * ch->Pz, c->world, s) != ncclSuccess)
                    rc = CFLX_ERR_NCCL;
            }
            ncclGroupEnd();
        }
        ch->nlayr = nlayr_save;
        ch->pk = pk_save;
    }
    if (!rc && cudaMemsetAsync(ch->acc, 0, 2 * sizeof(double), s) != cudaSuccess) rc = CFLX_ERR_CUDA;
    if (!rc && pk_save == 0) {
        sumsq_lower_kernel<<<1184, 256, 0, s>>>(R, Ml, Nl, v, Px, Py, ch->pi, ch->pj, ch->acc);
        sumsq_lower_kernel<<<1184, 256, 0, s>>>(ch->A0, Ml, Nl, v, Px, Py, ch->pi, ch->pj, ch->acc + 1);
    }
    if (!rc && ch->P > 1 && ncclAllReduce(ch->acc, ch->acc, 2, ncclDouble, ncclSum, c->world, s) != ncclSuccess) rc = CFLX_ERR_NCCL;
    double h[2] = {0, 0};
    if (!rc && cudaMemcpyAsync(h, ch->acc, sizeof(h), cudaMemcpyDeviceToHost, s) != cudaSuccess) rc = CFLX_ERR_CUDA;
    if (cudaStreamSynchronize(s) != cudaSuccess && !rc) {
        set_last_error("cholesky validation: %s", cudaGetErrorString(cudaGetLastError()));
        rc = CFLX_ERR_CUDA;
    }
    cudaFree(R);
    if (rc) return rc;
    if (abs_out) *abs_out = std::sqrt(h[0]);
    if (rel_out) *rel_out = std::sqrt(h[0]) / std::sqrt(h[1]);
    return CFLX_OK;
}

int cflx_chol_launch_count(cflx_chol* ch, int64_t* count_out, int reset) {
    if (!ch || !count_out) return CFLX_ERR_ARG;
    *count_out = ch->launches;
    if (reset) ch->launches = 0;
    return CFLX_OK;
}

void cflx_chol_destroy(cflx_chol* ch) { free_chol(ch); }

// The diagonal-tile Cholesky of cflx_chol_factor alone (the same potrf_tile), on the current device: A v x v row-major (lower
// triangle referenced), L_out = L with zeros above the diagonal, LT_out = L^T, info_out as dpotrf.  L^T starts as NaN, so a
// value the kernels never write shows up.
int cflx_dbg_potrf_tile(int v, int blocked, const double* A, double* L_out, double* LT_out, int* info_out) {
    if (v <= 0 || v % 4 != 0 || v > 512 || (blocked != 0 && blocked != 1) || !A || !L_out || !LT_out || !info_out)
        return CFLX_ERR_ARG;
    if (blocked && !potrf_tile_blocked(v)) {
        set_last_error("blocked tile Cholesky needs v %% 128 == 0 and v >= 256 (v=%d)", v);
        return CFLX_ERR_UNSUPPORTED;
    }
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        cudaGetLastError();
        set_last_error("no CUDA device visible: conflux_b200 has no CPU fallback");
        return CFLX_ERR_NO_DEVICE;
    }
    const size_t vv = (size_t)v * v;
    double *D = nullptr, *UT = nullptr, *Q = nullptr;
    int* info = nullptr;
    int rc = dmalloc(&D, vv);
    if (!rc) rc = dmalloc(&UT, vv);
    if (!rc && blocked) rc = dmalloc(&Q, potrf_tile_scratch(v));
    if (!rc) rc = dmalloc(&info, 1);
    if (!rc) rc = gemm_tn_setup();
    if (!rc) rc = potrf_tile_setup(v);
    if (!rc && (cudaMemcpy(D, A, vv * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess ||
                cudaMemset(UT, 0xff, vv * sizeof(double)) != cudaSuccess || cudaMemset(info, 0, sizeof(int)) != cudaSuccess))
        rc = CFLX_ERR_CUDA;
    int64_t launches = 0;
    if (!rc) rc = potrf_tile(v, D, UT, Q, info, 0, 0, &launches);
    if (!rc && (cudaMemcpy(L_out, D, vv * sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess ||
                cudaMemcpy(LT_out, UT, vv * sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess ||
                cudaMemcpy(info_out, info, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess)) {
        set_last_error("tile Cholesky failed: %s", cudaGetErrorString(cudaGetLastError()));
        rc = CFLX_ERR_CUDA;
    }
    for (void* p : {(void*)D, (void*)UT, (void*)Q, (void*)info}) cudaFree(p);
    return rc;
}

}  // extern "C"
