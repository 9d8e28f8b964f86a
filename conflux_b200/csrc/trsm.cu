// conflux_b200/csrc/trsm.cu -- the two triangular solves of the LU step as blocked GEMMs on the FP64 tensor path.
//
// Replaces, relative to /root/reference/src/conflux/lu/conflux_opt.hpp:
//   :1347-1358  cblas_dtrsm(Right, Upper, NoTrans, NonUnit)  A10 <- A10 * U00^-1     -> trsm_right_upper_T
//   :1539-1550  cblas_dtrsm(Left,  Lower, NoTrans, Unit)     A01 <- L00^-1 * A01     -> trsm_left_lower_unit
// A00 = L00\U00 is v x v (<= 2 MB).  Its nb x nb diagonal blocks (nb = 128 when v allows, like MAGMA's trsm) are inverted
// once per step by a small kernel (substitution in shared memory, one warp per column); the solve is then a right-looking sweep of GEMMs
// (multiply by the inverse block, rank-nb update of the remaining block rows) that all run on gemm.cu's DMMA
// kernel with the panels kept K-major (transposed L panel, row-major U panel).
#include "common.cuh"
#include "kernels.h"

namespace cflx {
namespace {
// grid = (nblk, 2, CS): y == 0 -> Uinv[j] = inv(U_jj) row-major (u_transposed: inv(U_jj)^T, the operand of the left
// upper solve); y == 1 -> LinvT[j] = inv(L_jj)^T row-major; the columns of a block are split over CS = gridDim.z CTAs
// (each stages the whole block in shared memory).
// One WARP per column of the inverse: the column lives in registers spread over the lanes (lane l holds entries l, l + 32,
// ...), every substitution step is a short partial dot product per lane + a warp reduction, so an NB x NB block takes NB
// steps of ~100 cycles per column instead of an NB^2 / 2 serial FMA chain per thread.
template <int NB>
__global__ void __launch_bounds__(1024) diag_inverse_kernel(const double* __restrict__ A00, int v, double* __restrict__ Uinv,
                                                            double* __restrict__ LinvT, int u_transposed) {
    constexpr int EPL = (NB + 31) / 32;  // entries per lane
    extern __shared__ double S[];        // [NB][NB + 1]
    constexpr int LD = NB + 1;
    const int j = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const double* blk = A00 + (size_t)(j * NB) * v + j * NB;
    for (int e = threadIdx.x; e < NB * NB; e += blockDim.x) S[(e / NB) * LD + e % NB] = blk[(size_t)(e / NB) * v + e % NB];
    __syncthreads();
    double* out = (blockIdx.y == 0 ? Uinv : LinvT) + (size_t)j * NB * NB;
    const int cols_per = (NB + gridDim.z - 1) / gridDim.z;
    const int c_lo = blockIdx.z * cols_per, c_hi = min(NB, c_lo + cols_per);
    for (int c = c_lo + warp; c < c_hi; c += nwarps) {
        double x[EPL];
#pragma unroll
        for (int e = 0; e < EPL; ++e) x[e] = 0.0;
        if (blockIdx.y == 0) {  // U X = I: x[c] = 1/U[c][c]; x[r] = -(sum_{t=r+1..c} U[r][t] x[t]) / U[r][r], r < c
            const double xc = 1.0 / S[c * LD + c];
#pragma unroll
            for (int e = 0; e < EPL; ++e)
                if (lane + 32 * e == c) x[e] = xc;
            for (int r = c - 1; r >= 0; --r) {
                double s = 0.0;
#pragma unroll
                for (int e = 0; e < EPL; ++e) {
                    const int t = lane + 32 * e;
                    if (t > r && t <= c) s = fma(S[r * LD + t], x[e], s);
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                const double xr = -s / S[r * LD + r];
#pragma unroll
                for (int e = 0; e < EPL; ++e)
                    if (lane + 32 * e == r) x[e] = xr;
            }
#pragma unroll
            for (int e = 0; e < EPL; ++e) {
                const int t = lane + 32 * e;
                if (t < NB) out[u_transposed ? (size_t)c * NB + t : (size_t)t * NB + c] = x[e];  // Uinv[t][c]
            }
        } else {  // L Y = I (unit diagonal): y[c] = 1; y[r] = -sum_{t=c..r-1} L[r][t] y[t], r > c
#pragma unroll
            for (int e = 0; e < EPL; ++e)
                if (lane + 32 * e == c) x[e] = 1.0;
            for (int r = c + 1; r < NB; ++r) {
                double s = 0.0;
#pragma unroll
                for (int e = 0; e < EPL; ++e) {
                    const int t = lane + 32 * e;
                    if (t >= c && t < r) s = fma(S[r * LD + t], x[e], s);
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
#pragma unroll
                for (int e = 0; e < EPL; ++e)
                    if (lane + 32 * e == r) x[e] = -s;
            }
#pragma unroll
            for (int e = 0; e < EPL; ++e) {
                const int t = lane + 32 * e;
                if (t < NB) out[(size_t)c * NB + t] = x[e];  // LinvT[c][r] = Linv[r][c]
            }
        }
    }
}

template <int NB>
int launch_diag_nb(const double* A00, int v, double* Uinv, double* LinvT, bool u_transposed, cudaStream_t stream) {
    constexpr size_t smem = (size_t)NB * (NB + 1) * sizeof(double);
    constexpr int CS = NB > 64 ? NB / 32 : 1;   // 128-wide blocks: 4 CTAs x 32 columns, one column per warp
    const int warps = NB < 32 ? NB : 32;
    static PerDeviceMax cfg;
    if (cfg.raise(smem))
        CFLX_CUDA(cudaFuncSetAttribute(diag_inverse_kernel<NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    diag_inverse_kernel<NB><<<dim3(v / NB, 2, CS), 32 * warps, smem, stream>>>(A00, v, Uinv, LinvT, u_transposed ? 1 : 0);
    CFLX_CUDA(cudaGetLastError());
    return CFLX_OK;
}
}  // namespace

int launch_diag_inverses(const double* A00, int v, int nb, double* Uinv, double* LinvT, cudaStream_t stream,
                         bool u_transposed) {
    switch (nb) {
        case 128: return launch_diag_nb<128>(A00, v, Uinv, LinvT, u_transposed, stream);
        case 64: return launch_diag_nb<64>(A00, v, Uinv, LinvT, u_transposed, stream);
        case 32: return launch_diag_nb<32>(A00, v, Uinv, LinvT, u_transposed, stream);
        case 16: return launch_diag_nb<16>(A00, v, Uinv, LinvT, u_transposed, stream);
        case 8: return launch_diag_nb<8>(A00, v, Uinv, LinvT, u_transposed, stream);
        case 4: return launch_diag_nb<4>(A00, v, Uinv, LinvT, u_transposed, stream);
        default:
            set_last_error("diag_inverses: unsupported block size %d", nb);
            return CFLX_ERR_UNSUPPORTED;
    }
}

// X * U00 = P  <=>  U00^T X^T = P^T.  PT/LT are the transposed panels [v][ld]; sweep over block rows j:
//   LT_j = inv(U_jj)^T * PT_j ;  PT_i -= U_ji^T * LT_j  (i > j)
int trsm_right_upper_T(const double* A00, const double* Uinv, int v, int nb, double* PT, double* LT, int64_t ld, int n,
                       cudaStream_t stream) {
    if (n <= 0) return CFLX_OK;
    const int nblk = v / nb;
    const int N = (n + 1) & ~1;
    for (int j = 0; j < nblk; ++j) {
        GemmArgs g{};
        g.M = nb; g.N = N; g.K = nb;
        g.AT = Uinv + (size_t)j * nb * nb; g.ldat = nb;              // AT[k][m] = inv(U_jj)[k][m]
        g.B = PT + (int64_t)j * nb * ld; g.ldb = ld;
        g.C = nullptr; g.ldc = ld;
        g.D = LT + (int64_t)j * nb * ld; g.ldd = ld;
        g.alpha = 1.0; g.beta = 0.0;
        CFLX_TRY(launch_gemm_tn(g, stream));
        const int rest = v - (j + 1) * nb;
        if (rest > 0) {
            GemmArgs u{};
            u.M = rest; u.N = N; u.K = nb;
            u.AT = A00 + (size_t)(j * nb) * v + (j + 1) * nb; u.ldat = v;  // AT[k][m] = U[j*nb+k][(j+1)*nb+m]
            u.B = LT + (int64_t)j * nb * ld; u.ldb = ld;
            u.C = PT + (int64_t)(j + 1) * nb * ld; u.ldc = ld;
            u.D = PT + (int64_t)(j + 1) * nb * ld; u.ldd = ld;
            u.alpha = -1.0; u.beta = 1.0;
            CFLX_TRY(launch_gemm_tn(u, stream));
        }
    }
    return CFLX_OK;
}

// L00 * X = R (unit lower).  R/U are [v][ld]:  U_j = inv(L_jj) * R_j ;  R_i -= L_ij * U_j  (i > j)
int trsm_left_lower_unit(const double* A00T, const double* LinvT, int v, int nb, double* R, double* U, int64_t ld, int n,
                         cudaStream_t stream) {
    // (callers solve a column window by offsetting R and U: the columns are independent right-hand sides)
    if (n <= 0) return CFLX_OK;
    const int nblk = v / nb;
    for (int j = 0; j < nblk; ++j) {
        GemmArgs g{};
        g.M = nb; g.N = n; g.K = nb;
        g.AT = LinvT + (size_t)j * nb * nb; g.ldat = nb;             // AT[k][m] = inv(L_jj)[m][k]
        g.B = R + (int64_t)j * nb * ld; g.ldb = ld;
        g.C = nullptr; g.ldc = ld;
        g.D = U + (int64_t)j * nb * ld; g.ldd = ld;
        g.alpha = 1.0; g.beta = 0.0;
        CFLX_TRY(launch_gemm_tn(g, stream));
        const int rest = v - (j + 1) * nb;
        if (rest > 0) {
            GemmArgs u{};
            u.M = rest; u.N = n; u.K = nb;
            u.AT = A00T + (size_t)(j * nb) * v + (j + 1) * nb; u.ldat = v;  // AT[k][m] = L[(j+1)*nb+m][j*nb+k]
            u.B = U + (int64_t)j * nb * ld; u.ldb = ld;
            u.C = R + (int64_t)(j + 1) * nb * ld; u.ldc = ld;
            u.D = R + (int64_t)(j + 1) * nb * ld; u.ldd = ld;
            u.alpha = -1.0; u.beta = 1.0;
            CFLX_TRY(launch_gemm_tn(u, stream));
        }
    }
    return CFLX_OK;
}

// U00 * X = R (non-unit upper), the bottom-up mirror of trsm_left_lower_unit.  R/X are [v][ld]:
//   X_j = inv(U_jj) * R_j ;  R_i -= U_ij * X_j  (i < j, all block rows above j in one GEMM)
// UinvT holds inv(U_jj)^T (launch_diag_inverses with u_transposed), A00T[c][r] = U00[r][c].
int trsm_left_upper(const double* A00T, const double* UinvT, int v, int nb, double* R, double* X, int64_t ld, int n,
                    cudaStream_t stream) {
    if (n <= 0) return CFLX_OK;
    const int nblk = v / nb;
    for (int j = nblk - 1; j >= 0; --j) {
        GemmArgs g{};
        g.M = nb; g.N = n; g.K = nb;
        g.AT = UinvT + (size_t)j * nb * nb; g.ldat = nb;             // AT[k][m] = inv(U_jj)[m][k]
        g.B = R + (int64_t)j * nb * ld; g.ldb = ld;
        g.C = nullptr; g.ldc = ld;
        g.D = X + (int64_t)j * nb * ld; g.ldd = ld;
        g.alpha = 1.0; g.beta = 0.0;
        CFLX_TRY(launch_gemm_tn(g, stream));
        if (j > 0) {
            GemmArgs u{};
            u.M = j * nb; u.N = n; u.K = nb;
            u.AT = A00T + (size_t)(j * nb) * v; u.ldat = v;               // AT[k][m] = U[m][j*nb+k]
            u.B = X + (int64_t)j * nb * ld; u.ldb = ld;
            u.C = R; u.ldc = ld;
            u.D = R; u.ldd = ld;
            u.alpha = -1.0; u.beta = 1.0;
            CFLX_TRY(launch_gemm_tn(u, stream));
        }
    }
    return CFLX_OK;
}

}  // namespace cflx
