// conflux_b200/csrc/validate.cu -- the reference's validation flow on the GPU grid (not on the timed path).
//
// Reference (relative to /root/reference):
//   src/conflux/lu/conflux_opt.hpp:1673-1699,1721-1771   factors land in the caller's C in the conflux block-cyclic
//                                                        layout: pivoted row q = k*v + i on rank (k % Px, pj, 0),
//                                                        local row (k / Px)*v + i               -> redistribute_pivoted_rows
//   examples/conflux_miniapp.cpp:349-500                 L = unit-lower(C), U = upper(C), P from pivotIndsBuff,
//                                                        PA - L*U with pdgemm on the Px x Py grid, Frobenius norm
//                                                        reduced over the grid                  -> lu_residual_grid
// The reference goes through COSTA transforms to a ScaLAPACK layout and calls pdgemm; here the conflux block-cyclic
// layout itself is the distribution of a SUMMA sweep: for every tile step t the owner column broadcasts the masked
// L^T block along its grid row, the owner row broadcasts the masked U block along its grid column, and every layer-0
// rank updates its local remainder with the library's own FP64 tensor-core GEMM.
#include <cmath>
#include <cstring>

#include "lu_state.h"

namespace cflx {
namespace {

__global__ void gather_rows_kernel(const double* __restrict__ A, int64_t lda, const int* __restrict__ src_rows, int nrows,
                                   int ncols, double* __restrict__ out) {
    const int i = blockIdx.y;
    if (i >= nrows) return;
    const double2* s = reinterpret_cast<const double2*>(A + (int64_t)src_rows[i] * lda);
    double2* d = reinterpret_cast<double2*>(out + (int64_t)i * ncols);
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < ncols / 2; c += gridDim.x * blockDim.x) d[c] = s[c];
}
__global__ void scatter_rows_kernel(const double* __restrict__ in, int ncols, const int* __restrict__ dst_rows, int nrows,
                                    double* __restrict__ C, int64_t ldc) {
    const int i = blockIdx.y;
    if (i >= nrows) return;
    const double2* s = reinterpret_cast<const double2*>(in + (int64_t)i * ncols);
    double2* d = reinterpret_cast<double2*>(C + (int64_t)dst_rows[i] * ldc);
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < ncols / 2; c += gridDim.x * blockDim.x) d[c] = s[c];
}
__global__ void move_rows_kernel(const double* __restrict__ A, int64_t lda, const int* __restrict__ src_rows,
                                 const int* __restrict__ dst_rows, int nrows, int ncols, double* __restrict__ C, int64_t ldc) {
    const int i = blockIdx.y;
    if (i >= nrows) return;
    const double2* s = reinterpret_cast<const double2*>(A + (int64_t)src_rows[i] * lda);
    double2* d = reinterpret_cast<double2*>(C + (int64_t)dst_rows[i] * ldc);
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < ncols / 2; c += gridDim.x * blockDim.x) d[c] = s[c];
}

// LT[c][r] = L[q(r)][t*v + c] of the packed factors C (conflux layout): multiplier below the diagonal, 1 on it, 0 above
// (discard_upper_half, conflux_miniapp.cpp:352-360).  q(r) = global row of local row r = ((r / v)*Px + pi)*v + r % v.
__global__ void extract_l_block_T_kernel(const double* __restrict__ C, int64_t ldc, int Ml, int v, int Px, int pi, int t,
                                         int lc0, int row_lo, double* __restrict__ LT, int64_t ldp) {
    __shared__ double tile[32][33];
    const int r0 = row_lo + blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int dy = threadIdx.y; dy < 32; dy += blockDim.y) {
        const int r = r0 + dy, c = c0 + threadIdx.x;
        double x = 0.0;
        if (r < Ml && c < v) {
            const int64_t q = ((int64_t)(r / v) * Px + pi) * v + r % v, gc = (int64_t)t * v + c;
            x = q > gc ? C[(int64_t)r * ldc + lc0 + c] : (q == gc ? 1.0 : 0.0);
        }
        tile[dy][threadIdx.x] = x;
    }
    __syncthreads();
    for (int dy = threadIdx.y; dy < 32; dy += blockDim.y) {
        const int c = c0 + dy, r = r0 + threadIdx.x;
        if (r < Ml && c < v) LT[(int64_t)c * ldp + r] = tile[threadIdx.x][dy];
    }
}
// U[r][lc] = upper part of pivoted row t*v + r (discard_lower_half, conflux_miniapp.cpp:363-369)
__global__ void extract_u_block_kernel(const double* __restrict__ C, int64_t ldc, int Nl, int v, int Py, int pj, int t,
                                       int lr0, int col_lo, double* __restrict__ U, int64_t ldu) {
    const int r = blockIdx.y;
    const int64_t q = (int64_t)t * v + r;
    for (int lc = col_lo + blockIdx.x * blockDim.x + threadIdx.x; lc < Nl; lc += gridDim.x * blockDim.x) {
        const int64_t gc = ((int64_t)(lc / v) * Py + pj) * v + lc % v;
        U[(int64_t)r * ldu + lc] = gc >= q ? C[(int64_t)(lr0 + r) * ldc + lc] : 0.0;
    }
}
}  // namespace

// dst (Ml x Nl, conflux layout of the PIVOTED matrix) <- rows of src.  factors: src = A11 (row i of a rank = its i-th
// promoted row);  otherwise src = the pristine input A0 (row of global id g at its original local slot), i.e. dst = P*A.
// Collective over the i-communicator of layer 0 (ranks with pk != 0 must not call).
int redistribute_pivoted_rows(cflx_lu* lu, const std::vector<int>& hist, bool factors, const double* src, double* dst) {
    if (lu->Px > 1 && !lu->xbuf) CFLX_TRY(dmalloc(&lu->xbuf, 2 * (size_t)lu->Ml * lu->Nl));
    return redistribute_pivoted_rows(lu, hist, factors, src, dst, lu->Nl, lu->Nl, lu->xbuf);
}

// The same on rows of `ncols` doubles at leading dimension ld (both even) of src and dst, e.g. the right-hand sides of
// cflx_lu_solve (factors = false: dst = P*B).  stage: 2 * Ml * ncols doubles of staging, needed when Px > 1.
int redistribute_pivoted_rows(cflx_lu* lu, const std::vector<int>& hist, bool factors, const double* src, double* dst,
                              int ncols, int64_t ld, double* stage) {
    cflx_comm* c = lu->comm;
    cudaStream_t s = c->stream;
    const int v = lu->v, Px = lu->Px, Ml = lu->Ml;
    const size_t loc = (size_t)Ml * ncols;
    if (!lu->idx_buf) CFLX_TRY(dmalloc(&lu->idx_buf, 2 * (size_t)Ml));
    std::vector<int> next_local(Px, 0);
    std::vector<std::vector<int>> send_rows(Px), recv_rows(Px);  // send_rows[dst rank] = my source rows; recv_rows[src rank] = my dest rows
    for (int q = 0; q < lu->M; ++q) {
        const int g = hist[q];
        if (g < 0 || g >= lu->M) {
            set_last_error("pivot history entry %d = %d is not a row id", q, g);
            return CFLX_ERR_STATE;
        }
        const int owner = (g / v) % Px;
        const int promoted = next_local[owner]++;
        const int lrow = factors ? promoted : (g / (v * Px)) * v + g % v;
        const int k = q / v, i = q % v;
        const int to = k % Px, drow = (k / Px) * v + i;
        if (owner == lu->pi) send_rows[to].push_back(lrow);
        if (to == lu->pi) recv_rows[owner].push_back(drow);
    }
    std::vector<int> flat_send, flat_recv;
    for (int p = 0; p < Px; ++p) flat_send.insert(flat_send.end(), send_rows[p].begin(), send_rows[p].end());
    for (int p = 0; p < Px; ++p) flat_recv.insert(flat_recv.end(), recv_rows[p].begin(), recv_rows[p].end());
    if ((int)flat_send.size() != Ml || (int)flat_recv.size() != Ml) {
        set_last_error("row redistribution: %zu rows to send, %zu to receive, expected %d", flat_send.size(), flat_recv.size(), Ml);
        return CFLX_ERR_STATE;
    }
    CFLX_CUDA(cudaMemcpyAsync(lu->idx_buf, flat_send.data(), sizeof(int) * Ml, cudaMemcpyHostToDevice, s));
    CFLX_CUDA(cudaMemcpyAsync(lu->idx_buf + Ml, flat_recv.data(), sizeof(int) * Ml, cudaMemcpyHostToDevice, s));
    dim3 grid(std::max(1, std::min(32, ncols / 512)), Ml);
    if (Px == 1) {
        move_rows_kernel<<<grid, 256, 0, s>>>(src, ld, lu->idx_buf, lu->idx_buf + Ml, Ml, ncols, dst, ld);
        CFLX_CUDA(cudaGetLastError());
        CFLX_CUDA(cudaStreamSynchronize(s));  // the index vectors above are stack/heap temporaries
        return CFLX_OK;
    }
    double* sendbuf = stage;
    double* recvbuf = stage + loc;
    gather_rows_kernel<<<grid, 256, 0, s>>>(src, ld, lu->idx_buf, Ml, ncols, sendbuf);
    CFLX_CUDA(cudaGetLastError());
    CFLX_NCCL(ncclGroupStart());
    size_t so = 0, ro = 0;
    for (int p = 0; p < Px; ++p) {
        const size_t ns = send_rows[p].size() * (size_t)ncols, nr = recv_rows[p].size() * (size_t)ncols;
        if (p == lu->pi) {
            CFLX_CUDA(cudaMemcpyAsync(recvbuf + ro, sendbuf + so, ns * sizeof(double), cudaMemcpyDeviceToDevice, s));
        } else {
            if (ns) CFLX_NCCL(ncclSend(sendbuf + so, ns, ncclDouble, p, lu->i_comm.c, s));
            if (nr) CFLX_NCCL(ncclRecv(recvbuf + ro, nr, ncclDouble, p, lu->i_comm.c, s));
        }
        so += ns;
        ro += nr;
    }
    CFLX_NCCL(ncclGroupEnd());
    scatter_rows_kernel<<<grid, 256, 0, s>>>(recvbuf, ncols, lu->idx_buf + Ml, Ml, dst, ld);
    CFLX_CUDA(cudaGetLastError());
    CFLX_CUDA(cudaStreamSynchronize(s));
    return CFLX_OK;
}

// ||P*A - L*U||_F and ||A||_F over the whole grid.  COLLECTIVE over the world communicator (layers pk != 0 take part in
// the broadcasts only).  abs_out / rel_out identical on every rank.
int lu_residual_grid(cflx_lu* lu, const std::vector<int>& hist, double* abs_out, double* rel_out) {
    cflx_comm* c = lu->comm;
    cudaStream_t s = c->stream;
    const int v = lu->v, Px = lu->Px, Py = lu->Py, Pz = lu->Pz, Ml = lu->Ml, Nl = lu->Nl, Nt = lu->Nt;
    const int pi = lu->pi, pj = lu->pj;
    const bool layer0 = lu->pk == 0;
    const size_t loc = (size_t)Ml * Nl;
    double *R = nullptr, *acc = nullptr;
    int rc = CFLX_OK;
    auto cleanup = [&]() {
        cudaFree(R);
        cudaFree(acc);
        cudaFree(lu->xbuf);  // 2 x local matrix of staging: do not keep it alive after validation
        lu->xbuf = nullptr;
    };
    if ((rc = dmalloc(&acc, 2))) return rc;
    if (cudaMemsetAsync(acc, 0, 2 * sizeof(double), s) != cudaSuccess) rc = CFLX_ERR_CUDA;
    if (!rc && layer0) {
        if (!lu->Cbuf) rc = dmalloc(&lu->Cbuf, loc);
        if (!rc) rc = dmalloc(&R, loc);
        if (!rc) rc = redistribute_pivoted_rows(lu, hist, true, lu->A11, lu->Cbuf);   // C   (conflux layout)
        if (!rc) rc = redistribute_pivoted_rows(lu, hist, false, lu->A0, R);          // P*A (conflux layout)
    }
    // every rank must reach the collectives below even after a local failure above would deadlock the others: a
    // failure here is an allocation failure, which the caller treats as fatal for the whole grid anyway
    if (rc) {
        cleanup();
        return rc;
    }
    const int64_t ldp = lu->ldp_max, ldu = Nl;
    for (int t = 0; t < Nt && !rc; ++t) {
        const int ltr = (t - pi + Px - 1) / Px, ltc = (t - pj + Py - 1) / Py;  // first local tile row / col with global tile >= t
        const int row_lo = std::min(Ml, ltr * v), col_lo = std::min(Nl, ltc * v);
        if (layer0 && pj == t % Py && row_lo < Ml) {
            dim3 grid((Ml - row_lo + 31) / 32, (v + 31) / 32), block(32, 8);
            extract_l_block_T_kernel<<<grid, block, 0, s>>>(lu->Cbuf, Nl, Ml, v, Px, pi, t, (t / Py) * v, row_lo, lu->PT, ldp);
        }
        if (Py * Pz > 1) {
            ncclResult_t r = ncclBroadcast(lu->PT, lu->PT, (size_t)v * ldp, ncclDouble, (t % Py) * Pz, lu->jk_comm.c, s);
            if (r != ncclSuccess) {
                set_last_error("residual: ncclBroadcast(L) -> %s", ncclGetErrorString(r));
                rc = CFLX_ERR_NCCL;
                break;
            }
        }
        if (layer0 && pi == t % Px && col_lo < Nl) {
            dim3 grid(std::max(1, std::min(32, (Nl - col_lo) / 256)), v);
            extract_u_block_kernel<<<grid, 256, 0, s>>>(lu->Cbuf, Nl, Nl, v, Py, pj, t, (t / Px) * v, col_lo, lu->U, ldu);
        }
        if (Px * Pz > 1) {
            ncclResult_t r = ncclBroadcast(lu->U, lu->U, (size_t)v * ldu, ncclDouble, (t % Px) * Pz, lu->ik_comm.c, s);
            if (r != ncclSuccess) {
                set_last_error("residual: ncclBroadcast(U) -> %s", ncclGetErrorString(r));
                rc = CFLX_ERR_NCCL;
                break;
            }
        }
        if (layer0 && row_lo < Ml && col_lo < Nl) {
            GemmArgs g{};
            g.M = Ml - row_lo; g.N = Nl - col_lo; g.K = v;
            g.AT = lu->PT + row_lo; g.ldat = ldp;
            g.B = lu->U + col_lo; g.ldb = ldu;
            g.C = R + (int64_t)row_lo * Nl + col_lo; g.ldc = Nl;
            g.D = R + (int64_t)row_lo * Nl + col_lo; g.ldd = Nl;
            g.alpha = -1.0; g.beta = 1.0;
            rc = launch_gemm_tn(g, s);
        }
    }
    if (!rc && cudaGetLastError() != cudaSuccess) rc = CFLX_ERR_CUDA;
    if (!rc && layer0) {
        rc = launch_sumsq(R, (int64_t)loc, acc, s);
        if (!rc) rc = launch_sumsq(lu->A0, (int64_t)loc, acc + 1, s);
    }
    if (!rc && lu->P > 1) {
        ncclResult_t r = ncclAllReduce(acc, acc, 2, ncclDouble, ncclSum, c->world, s);
        if (r != ncclSuccess) {
            set_last_error("residual: ncclAllReduce -> %s", ncclGetErrorString(r));
            rc = CFLX_ERR_NCCL;
        }
    }
    double h[2] = {0, 0};
    if (!rc && cudaMemcpyAsync(h, acc, sizeof(h), cudaMemcpyDeviceToHost, s) != cudaSuccess) rc = CFLX_ERR_CUDA;
    if (cudaStreamSynchronize(s) != cudaSuccess && !rc) {
        set_last_error("residual: %s", cudaGetErrorString(cudaGetLastError()));
        rc = CFLX_ERR_CUDA;
    }
    cleanup();
    // the panels were used as staging: restore the zero padding the factorisation relies on
    if (!rc) {
        cudaMemsetAsync(lu->PT, 0, (size_t)v * ldp * sizeof(double), s);
        cudaMemsetAsync(lu->U, 0, (size_t)v * (Nl + 2) * sizeof(double), s);
        if (cudaStreamSynchronize(s) != cudaSuccess) rc = CFLX_ERR_CUDA;
    }
    if (rc) return rc;
    if (abs_out) *abs_out = std::sqrt(h[0]);
    if (rel_out) *rel_out = std::sqrt(h[0]) / std::sqrt(h[1]);
    return CFLX_OK;
}

}  // namespace cflx
