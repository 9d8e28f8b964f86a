// conflux_b200/csrc/dbg.cu -- single-device test / micro-benchmark hooks of the C ABI (cflx_dbg_*).
// They drive the SAME kernels the factorisation uses, with host buffers in and out, so that tests/ can check every
// kernel in isolation against numpy / the oracle, and bench.py can time the dominant kernel alone.
#include <vector>

#include "../../include/conflux_b200.h"
#include "common.cuh"
#include "kernels.h"

using namespace cflx;

namespace {
struct DevBuf {
    void* p = nullptr;
    ~DevBuf() { cudaFree(p); }
    int alloc(size_t bytes) {
        CFLX_CUDA(cudaMalloc(&p, bytes + 4096));
        return CFLX_OK;
    }
    template <class T>
    T* as() { return (T*)p; }
};
int check_device() {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        cudaGetLastError();
        set_last_error("no CUDA device visible: conflux_b200 has no CPU fallback");
        return CFLX_ERR_NO_DEVICE;
    }
    return CFLX_OK;
}

// ---- FP64 pipe peak probes ------------------------------------------------------------------------------
__global__ void dmma_peak_kernel(double* out, int iters) {
    double c[16][2];
#pragma unroll
    for (int i = 0; i < 16; ++i) c[i][0] = c[i][1] = 0.0;
    double a = 1.0 + threadIdx.x * 1e-9, b = 1.0 - threadIdx.x * 1e-9;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) dmma884(c[i][0], c[i][1], a, b);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += c[i][0] + c[i][1];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void dfma_peak_kernel(double* out, int iters) {
    double c[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) c[i] = i;
    double a = 1.0 + threadIdx.x * 1e-9, b = 1e-9;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) c[i] = fma(c[i], a, b);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += c[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
}  // namespace

static long long g_panel_cycles[8] = {0};

extern "C" {

int cflx_dbg_last_panel_cycles(long long* out8) {
    for (int i = 0; i < 8; ++i) out8[i] = g_panel_cycles[i];
    return CFLX_OK;
}

// burst = best of a few ~2 ms launches (what a kernel timed alone can reach at the maximum clock); sustained = one
// ~0.5 s launch (what survives the power cap inside a long step)
int cflx_dbg_fp64_peak_ex(int which, double* burst_out, double* sustained_out) {
    CFLX_TRY(check_device());
    int dev = 0, sms = 0;
    CFLX_CUDA(cudaGetDevice(&dev));
    CFLX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int threads = 256, blocks = sms * 4;
    DevBuf out;
    CFLX_TRY(out.alloc(sizeof(double) * threads * blocks));
    cudaEvent_t e0, e1;
    CFLX_CUDA(cudaEventCreate(&e0));
    CFLX_CUDA(cudaEventCreate(&e1));
    auto run = [&](int iters, double* tf) -> int {
        CFLX_CUDA(cudaEventRecord(e0));
        if (which == 0) dmma_peak_kernel<<<blocks, threads>>>(out.as<double>(), iters);
        else dfma_peak_kernel<<<blocks, threads>>>(out.as<double>(), iters);
        CFLX_CUDA(cudaEventRecord(e1));
        CFLX_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        CFLX_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        // DMMA 8x8x4 = 256 FMA = 512 flop per warp instruction; DFMA = 2 flop per lane
        const double flop = which == 0 ? (double)blocks * (threads / 32) * iters * 16 * 512.0
                                       : (double)blocks * threads * iters * 16 * 2.0;
        *tf = flop / (ms * 1e-3) / 1e12;
        return CFLX_OK;
    };
    double burst = 0, tf = 0;
    for (int rep = 0; rep < 4; ++rep) {
        CFLX_TRY(run(1024, &tf));
        if (rep > 0 && tf > burst) burst = tf;
    }
    double sustained = 0;
    CFLX_TRY(run(262144, &sustained));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (burst_out) *burst_out = burst;
    if (sustained_out) *sustained_out = sustained;
    return CFLX_OK;
}
int cflx_dbg_fp64_peak(int which, double* tflops_out) { return cflx_dbg_fp64_peak_ex(which, tflops_out, nullptr); }

int cflx_dbg_gemm_tn(int M, int N, int K, const double* AT, const double* B, const double* C, double alpha, double beta,
                     double* D, int reps, double* ms_out) {
    CFLX_TRY(check_device());
    if (M <= 0 || N <= 0 || K <= 0) return CFLX_ERR_ARG;
    const int64_t ldat = round_up(M, 2), ldb = round_up(N, 2), ldc = ldb;
    DevBuf dA, dB, dC, dD;
    CFLX_TRY(dA.alloc(sizeof(double) * K * ldat));
    CFLX_TRY(dB.alloc(sizeof(double) * K * ldb));
    CFLX_TRY(dC.alloc(sizeof(double) * M * ldc));
    CFLX_TRY(dD.alloc(sizeof(double) * M * ldc));
    CFLX_CUDA(cudaMemset(dA.p, 0, sizeof(double) * K * ldat));
    CFLX_CUDA(cudaMemset(dB.p, 0, sizeof(double) * K * ldb));
    CFLX_CUDA(cudaMemcpy2D(dA.p, ldat * 8, AT, (size_t)M * 8, (size_t)M * 8, K, cudaMemcpyHostToDevice));
    CFLX_CUDA(cudaMemcpy2D(dB.p, ldb * 8, B, (size_t)N * 8, (size_t)N * 8, K, cudaMemcpyHostToDevice));
    if (C) CFLX_CUDA(cudaMemcpy2D(dC.p, ldc * 8, C, (size_t)N * 8, (size_t)N * 8, M, cudaMemcpyHostToDevice));
    else CFLX_CUDA(cudaMemset(dC.p, 0, sizeof(double) * M * ldc));
    GemmArgs g{};
    g.M = M; g.N = (int)ldb; g.K = K;
    g.AT = dA.as<double>(); g.ldat = ldat;
    g.B = dB.as<double>(); g.ldb = ldb;
    g.C = dC.as<double>(); g.ldc = ldc;
    g.D = dD.as<double>(); g.ldd = ldc;
    g.alpha = alpha; g.beta = beta;
    cudaEvent_t e0, e1;
    CFLX_CUDA(cudaEventCreate(&e0));
    CFLX_CUDA(cudaEventCreate(&e1));
    if (reps < 1) reps = 1;
    CFLX_TRY(launch_gemm_tn(g, 0));  // warm-up / the result
    CFLX_CUDA(cudaEventRecord(e0));
    for (int r = 0; r < reps; ++r) CFLX_TRY(launch_gemm_tn(g, 0));
    CFLX_CUDA(cudaEventRecord(e1));
    CFLX_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    CFLX_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    if (ms_out) *ms_out = ms / reps;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (D) CFLX_CUDA(cudaMemcpy2D(D, (size_t)N * 8, dD.p, ldc * 8, (size_t)N * 8, M, cudaMemcpyDeviceToHost));
    CFLX_CUDA(cudaDeviceSynchronize());
    return CFLX_OK;
}

int cflx_dbg_panel(int n, int v, const double* panel, int* perm_out, double* A00_out, double* LU_out, int reps,
                   double* ms_out) {
    CFLX_TRY(check_device());
    if (n < 0 || v <= 0) return CFLX_ERR_ARG;
    const int64_t ld = std::max<int64_t>(2, round_up(n, 2));
    // host transpose into the kernel's K-major layout
    std::vector<double> WT((size_t)v * ld, 0.0);
    for (int r = 0; r < n; ++r)
        for (int c = 0; c < v; ++c) WT[(size_t)c * ld + r] = panel[(size_t)r * v + c];
    DevBuf dW, dW0, dA00, dA00T, dperm;
    CFLX_TRY(dW.alloc(sizeof(double) * v * ld));
    CFLX_TRY(dW0.alloc(sizeof(double) * v * ld));
    CFLX_TRY(dA00.alloc(sizeof(double) * v * v));
    CFLX_TRY(dA00T.alloc(sizeof(double) * v * v));
    CFLX_TRY(dperm.alloc(sizeof(int) * 2 * v));
    CFLX_CUDA(cudaMemcpy(dW0.p, WT.data(), sizeof(double) * v * ld, cudaMemcpyHostToDevice));
    CFLX_CUDA(cudaMemset(dA00.p, 0, sizeof(double) * v * v));
    PanelWorkspace ws{};
    CFLX_TRY(panel_workspace_create(&ws));
    cudaEvent_t e0, e1;
    CFLX_CUDA(cudaEventCreate(&e0));
    CFLX_CUDA(cudaEventCreate(&e1));
    if (reps < 1) reps = 1;
    float total = 0;
    int nb = 0, rc = CFLX_OK;
    for (int r = 0; r < reps + 1 && rc == CFLX_OK; ++r) {
        cudaMemcpyAsync(dW.p, dW0.p, sizeof(double) * v * ld, cudaMemcpyDeviceToDevice, 0);
        cudaEventRecord(e0);
        rc = launch_panel_getrf_a00(dW.as<double>(), ld, n, v, dperm.as<int>(), dA00.as<double>(), &nb, &ws, 0);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) rc = CFLX_ERR_CUDA;
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (r > 0) total += ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (rc == CFLX_OK && n >= v)
        rc = launch_gather_a00(dW.as<double>(), ld, dperm.as<int>(), v, nb, dA00.as<double>(), dA00T.as<double>(), 0);
    cudaMemcpy(g_panel_cycles, ws.dbg, sizeof(g_panel_cycles), cudaMemcpyDeviceToHost);
    panel_workspace_destroy(&ws);
    if (rc != CFLX_OK) {
        if (rc == CFLX_ERR_CUDA) set_last_error("panel kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
        return rc;
    }
    if (ms_out) *ms_out = total / reps;
    if (perm_out) CFLX_CUDA(cudaMemcpy(perm_out, dperm.p, sizeof(int) * v, cudaMemcpyDeviceToHost));
    if (A00_out) CFLX_CUDA(cudaMemcpy(A00_out, dA00.p, sizeof(double) * v * v, cudaMemcpyDeviceToHost));
    if (LU_out) {
        CFLX_CUDA(cudaMemcpy(WT.data(), dW.p, sizeof(double) * v * ld, cudaMemcpyDeviceToHost));
        for (int r = 0; r < n; ++r)
            for (int c = 0; c < v; ++c) LU_out[(size_t)r * v + c] = WT[(size_t)c * ld + r];
    }
    CFLX_CUDA(cudaDeviceSynchronize());
    return CFLX_OK;
}

int cflx_dbg_trsm(int n, int v, const double* A00, const double* B, double* X_out, const double* R, double* Y_out) {
    CFLX_TRY(check_device());
    if (n <= 0 || v <= 0 || v % 4 != 0) return CFLX_ERR_ARG;
    int nb = 0;
    for (int c : {128, 64, 32, 16, 8, 4})
        if (!nb && v % c == 0) nb = c;
    if (nb == 0) return CFLX_ERR_UNSUPPORTED;
    const int64_t ld = round_up(n, 2);
    std::vector<double> A00T((size_t)v * v), BT((size_t)v * ld, 0.0), RT((size_t)v * ld, 0.0);
    for (int i = 0; i < v; ++i)
        for (int j = 0; j < v; ++j) A00T[(size_t)j * v + i] = A00[(size_t)i * v + j];
    DevBuf dA, dAT, dUinv, dLinvT, dP, dL, dR, dU;
    CFLX_TRY(dA.alloc(8 * (size_t)v * v)); CFLX_TRY(dAT.alloc(8 * (size_t)v * v));
    CFLX_TRY(dUinv.alloc(8 * (size_t)v * v)); CFLX_TRY(dLinvT.alloc(8 * (size_t)v * v));
    CFLX_TRY(dP.alloc(8 * (size_t)v * ld)); CFLX_TRY(dL.alloc(8 * (size_t)v * ld));
    CFLX_TRY(dR.alloc(8 * (size_t)v * ld)); CFLX_TRY(dU.alloc(8 * (size_t)v * ld));
    CFLX_CUDA(cudaMemcpy(dA.p, A00, 8 * (size_t)v * v, cudaMemcpyHostToDevice));
    CFLX_CUDA(cudaMemcpy(dAT.p, A00T.data(), 8 * (size_t)v * v, cudaMemcpyHostToDevice));
    CFLX_TRY(launch_diag_inverses(dA.as<double>(), v, nb, dUinv.as<double>(), dLinvT.as<double>(), 0));
    if (B && X_out) {  // X = B * U^-1, B is n x v row-major
        for (int r = 0; r < n; ++r)
            for (int c = 0; c < v; ++c) BT[(size_t)c * ld + r] = B[(size_t)r * v + c];
        CFLX_CUDA(cudaMemcpy(dP.p, BT.data(), 8 * (size_t)v * ld, cudaMemcpyHostToDevice));
        CFLX_CUDA(cudaMemset(dL.p, 0, 8 * (size_t)v * ld));
        CFLX_TRY(trsm_right_upper_T(dA.as<double>(), dUinv.as<double>(), v, nb, dP.as<double>(), dL.as<double>(), ld, n, 0));
        CFLX_CUDA(cudaMemcpy(BT.data(), dL.p, 8 * (size_t)v * ld, cudaMemcpyDeviceToHost));
        for (int r = 0; r < n; ++r)
            for (int c = 0; c < v; ++c) X_out[(size_t)r * v + c] = BT[(size_t)c * ld + r];
    }
    if (R && Y_out) {  // Y = L^-1 * R, R is v x n row-major
        for (int i = 0; i < v; ++i)
            for (int c = 0; c < n; ++c) RT[(size_t)i * ld + c] = R[(size_t)i * n + c];
        CFLX_CUDA(cudaMemcpy(dR.p, RT.data(), 8 * (size_t)v * ld, cudaMemcpyHostToDevice));
        CFLX_CUDA(cudaMemset(dU.p, 0, 8 * (size_t)v * ld));
        CFLX_TRY(trsm_left_lower_unit(dAT.as<double>(), dLinvT.as<double>(), v, nb, dR.as<double>(), dU.as<double>(), ld,
                                      (int)ld, 0));
        CFLX_CUDA(cudaMemcpy(RT.data(), dU.p, 8 * (size_t)v * ld, cudaMemcpyDeviceToHost));
        for (int i = 0; i < v; ++i)
            for (int c = 0; c < n; ++c) Y_out[(size_t)i * n + c] = RT[(size_t)i * ld + c];
    }
    CFLX_CUDA(cudaDeviceSynchronize());
    return CFLX_OK;
}

// the diagonal-tile solve of cflx_lu_solve: X = U^-1 R with the transposed block inverses of diag_inverse_kernel
int cflx_dbg_trsm_left_upper(int v, int n, const double* A00, const double* R, double* X_out) {
    CFLX_TRY(check_device());
    if (n <= 0 || v <= 0 || v % 4 != 0 || !A00 || !R || !X_out) return CFLX_ERR_ARG;
    int nb = 0;
    for (int c : {128, 64, 32, 16, 8, 4})
        if (!nb && v % c == 0) nb = c;
    if (nb == 0) return CFLX_ERR_UNSUPPORTED;
    const int64_t ld = round_up(n, 2);
    std::vector<double> A00T((size_t)v * v), RT((size_t)v * ld, 0.0);
    for (int i = 0; i < v; ++i)
        for (int j = 0; j < v; ++j) A00T[(size_t)j * v + i] = A00[(size_t)i * v + j];
    for (int i = 0; i < v; ++i)
        for (int c = 0; c < n; ++c) RT[(size_t)i * ld + c] = R[(size_t)i * n + c];
    DevBuf dA, dAT, dUinvT, dLinvT, dR, dX;
    CFLX_TRY(dA.alloc(8 * (size_t)v * v)); CFLX_TRY(dAT.alloc(8 * (size_t)v * v));
    CFLX_TRY(dUinvT.alloc(8 * (size_t)v * v)); CFLX_TRY(dLinvT.alloc(8 * (size_t)v * v));
    CFLX_TRY(dR.alloc(8 * (size_t)v * ld)); CFLX_TRY(dX.alloc(8 * (size_t)v * ld));
    CFLX_CUDA(cudaMemcpy(dA.p, A00, 8 * (size_t)v * v, cudaMemcpyHostToDevice));
    CFLX_CUDA(cudaMemcpy(dAT.p, A00T.data(), 8 * (size_t)v * v, cudaMemcpyHostToDevice));
    CFLX_CUDA(cudaMemcpy(dR.p, RT.data(), 8 * (size_t)v * ld, cudaMemcpyHostToDevice));
    CFLX_CUDA(cudaMemset(dX.p, 0, 8 * (size_t)v * ld));
    CFLX_TRY(launch_diag_inverses(dA.as<double>(), v, nb, dUinvT.as<double>(), dLinvT.as<double>(), 0, true));
    CFLX_TRY(trsm_left_upper(dAT.as<double>(), dUinvT.as<double>(), v, nb, dR.as<double>(), dX.as<double>(), ld, (int)ld, 0));
    CFLX_CUDA(cudaMemcpy(RT.data(), dX.p, 8 * (size_t)v * ld, cudaMemcpyDeviceToHost));
    for (int i = 0; i < v; ++i)
        for (int c = 0; c < n; ++c) X_out[(size_t)i * n + c] = RT[(size_t)i * ld + c];
    CFLX_CUDA(cudaDeviceSynchronize());
    return CFLX_OK;
}

// step 2 of the LU loop in isolation on ONE rank (Px = 1): plan_moves (analyze_pivots) + push_phase1..3 (push_pivots_up,
// conflux_opt.hpp:176-218) + the gri/igri bookkeeping, on an n_rows x n_cols row-major matrix (n_cols even).  The npiv
// pivot rows (local indices >= fnpr, tournament order) end up in rows [fnpr, fnpr+npiv) in that order.
// gri_out[n_rows] (optional) = new row -> old row.  a01_out (optional, npiv x n_cols) = the pivot rows phase 1 extracts.
int cflx_dbg_push_pivots(int n_rows, int n_cols, double* A_inout, int npiv, const int* pivot_rows, int fnpr, int* gri_out,
                         double* a01_out) {
    CFLX_TRY(check_device());
    if (n_rows <= 0 || n_cols <= 0 || (n_cols & 1) || npiv < 0 || npiv > n_rows - fnpr || fnpr < 0) return CFLX_ERR_ARG;
    if (npiv == 0) {
        if (gri_out) for (int i = 0; i < n_rows; ++i) gri_out[i] = i;
        return CFLX_OK;
    }
    const int v = npiv;  // every pivot of the "tile" lives on this rank
    DevBuf dA, dtmp, da01, dplan, dgp, dgri, dgrit, digri;
    CFLX_TRY(dA.alloc(8 * (size_t)n_rows * n_cols));
    CFLX_TRY(dtmp.alloc(8 * (size_t)v * n_cols));
    CFLX_TRY(da01.alloc(8 * (size_t)v * n_cols));
    CFLX_TRY(dplan.alloc(sizeof(int) * (6 * (size_t)v + 8 + n_rows)));
    CFLX_TRY(dgp.alloc(sizeof(int) * v));
    CFLX_TRY(dgri.alloc(sizeof(int) * n_rows));
    CFLX_TRY(dgrit.alloc(sizeof(int) * n_rows));
    CFLX_TRY(digri.alloc(sizeof(int) * n_rows));
    CFLX_CUDA(cudaMemcpy(dA.p, A_inout, 8 * (size_t)n_rows * n_cols, cudaMemcpyHostToDevice));
    CFLX_CUDA(cudaMemcpy(dgp.p, pivot_rows, sizeof(int) * v, cudaMemcpyHostToDevice));
    MovePlan plan{};
    int* pm = dplan.as<int>();
    plan.npiv = pm; plan.nel = pm + 4; pm += 8;
    plan.cur_piv = pm; pm += v;
    plan.order = pm; pm += v;
    plan.slot2piv = pm; pm += v;
    plan.early = pm; pm += v;
    plan.late = pm; pm += 2 * v;
    plan.rowsrc = pm;
    // gri = identity with "tile size" n_rows so that global id == local row (Px = 1)
    CFLX_TRY(launch_iota_gri(dgri.as<int>(), digri.as<int>(), n_rows, n_rows, 1, 0, 0));
    // plan_moves maps a global id g to the local slot (g / (v*Px))*v + g % v: with v := n_rows that is g itself
    CFLX_TRY(launch_plan_moves(dgp.as<int>(), v, 1, 0, fnpr, n_rows, digri.as<int>(), plan, 0));
    CFLX_TRY(launch_push_phase1(dA.as<double>(), n_cols, n_cols, 0, plan, v, dtmp.as<double>(), da01.as<double>(), n_cols, 0, 0));
    CFLX_TRY(launch_push_phase2(dA.as<double>(), n_cols, n_cols, 0, plan, v, 0));
    CFLX_TRY(launch_push_phase3(dA.as<double>(), n_cols, n_cols, 0, fnpr, plan, v, dtmp.as<double>(), 0));
    CFLX_TRY(launch_update_gri(dgri.as<int>(), dgrit.as<int>(), digri.as<int>(), plan.rowsrc, fnpr, n_rows, n_rows, 1, 0));
    CFLX_CUDA(cudaMemcpy(A_inout, dA.p, 8 * (size_t)n_rows * n_cols, cudaMemcpyDeviceToHost));
    if (gri_out) CFLX_CUDA(cudaMemcpy(gri_out, dgri.p, sizeof(int) * n_rows, cudaMemcpyDeviceToHost));
    if (a01_out) CFLX_CUDA(cudaMemcpy(a01_out, da01.p, 8 * (size_t)v * n_cols, cudaMemcpyDeviceToHost));
    CFLX_CUDA(cudaDeviceSynchronize());
    return CFLX_OK;
}

// D = C - AT^T * B on the int8 tcgen05 path (ozaki.cu): AT [K x M], B [K x N], C/D [M x N] row-major dense host arrays,
// K a multiple of 128, N even.  Optional outputs for tests: the digit planes [8][M][K] / [8][N][K] (int8) and the
// exponents [M] / [N], exactly as the kernels produced them.  ms_out = mean device time of the GEMM kernel alone.
int cflx_dbg_ozaki_gemm(int M, int N, int K, const double* AT, const double* B, const double* C, double* D,
                        signed char* planesA_out, signed char* planesB_out, int* ea_out, int* eb_out, int reps,
                        double* ms_out, double* split_ms_out) {
    CFLX_TRY(check_device());
    if (M <= 0 || N <= 0 || K <= 0 || (N & 1)) return CFLX_ERR_ARG;
    const int64_t ldat = round_up(M, 2), ldb = N, ldc = N;
    DevBuf dA, dB, dC, dC0;
    CFLX_TRY(dA.alloc(sizeof(double) * K * ldat));
    CFLX_TRY(dB.alloc(sizeof(double) * K * ldb));
    CFLX_TRY(dC.alloc(sizeof(double) * M * ldc));
    CFLX_TRY(dC0.alloc(sizeof(double) * M * ldc));
    CFLX_CUDA(cudaMemset(dA.p, 0, sizeof(double) * K * ldat));
    CFLX_CUDA(cudaMemcpy2D(dA.p, ldat * 8, AT, (size_t)M * 8, (size_t)M * 8, K, cudaMemcpyHostToDevice));
    CFLX_CUDA(cudaMemcpy(dB.p, B, sizeof(double) * K * ldb, cudaMemcpyHostToDevice));
    if (C) CFLX_CUDA(cudaMemcpy(dC0.p, C, sizeof(double) * M * ldc, cudaMemcpyHostToDevice));
    else CFLX_CUDA(cudaMemset(dC0.p, 0, sizeof(double) * M * ldc));
    OzakiWorkspace ws;
    int rc = ozaki_workspace_create(&ws, M, N, K);
    cudaEvent_t e0, e1, e2;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventCreate(&e2);
    if (reps < 1) reps = 1;
    float ms = 0, ms_split = 0;
    for (int r = 0; r < reps + 1 && rc == CFLX_OK; ++r) {
        cudaMemcpyAsync(dC.p, dC0.p, sizeof(double) * M * ldc, cudaMemcpyDeviceToDevice, 0);
        cudaEventRecord(e0);
        rc = ozaki_split_a(&ws, dA.as<double>(), ldat, M, 0);
        if (!rc) rc = ozaki_split_b(&ws, dB.as<double>(), ldb, 0, N, 0);
        cudaEventRecord(e1);
        if (!rc) rc = launch_ozaki_gemm(&ws, M, N, 0, 0, dC.as<double>(), ldc, 0, 0);
        cudaEventRecord(e2);
        if (cudaEventSynchronize(e2) != cudaSuccess) {
            set_last_error("ozaki kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
            rc = CFLX_ERR_CUDA;
        }
        float a = 0, b = 0;
        cudaEventElapsedTime(&a, e0, e1);
        cudaEventElapsedTime(&b, e1, e2);
        if (r > 0) {
            ms_split += a;
            ms += b;
        }
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaEventDestroy(e2);
    if (rc == CFLX_OK) {
        if (D) cudaMemcpy(D, dC.p, sizeof(double) * M * ldc, cudaMemcpyDeviceToHost);
        for (int s = 0; s < 8; ++s) {
            if (planesA_out) cudaMemcpy(planesA_out + (size_t)s * M * K, ws.planesA + (size_t)s * ws.cap_a * K, (size_t)M * K, cudaMemcpyDeviceToHost);
            if (planesB_out) cudaMemcpy(planesB_out + (size_t)s * N * K, ws.planesB + (size_t)s * ws.cap_b * K, (size_t)N * K, cudaMemcpyDeviceToHost);
        }
        if (ea_out) cudaMemcpy(ea_out, ws.ea, sizeof(int) * M, cudaMemcpyDeviceToHost);
        if (eb_out) cudaMemcpy(eb_out, ws.eb, sizeof(int) * N, cudaMemcpyDeviceToHost);
        if (ws.dbg) {
            long long h[16];
            cudaMemcpy(h, ws.dbg, sizeof(h), cudaMemcpyDeviceToHost);
            fprintf(stderr, "[ozaki cycles, CTA 0] producer: wait emptyB %lld emptyA %lld total %lld | mma: wait fullA %lld fullB %lld tempty %lld "
                            "total %lld | epilogue: wait tfull %lld drain %lld rmw %lld total %lld\n",
                    h[0], h[1], h[3], h[4], h[5], h[6], h[7], h[8], h[9], h[10], h[11]);
        }
        if (cudaDeviceSynchronize() != cudaSuccess) rc = CFLX_ERR_CUDA;
    }
    ozaki_workspace_destroy(&ws);
    if (ms_out) *ms_out = ms / reps;
    if (split_ms_out) *split_ms_out = ms_split / reps;
    return rc;
}

// raw tensor-pipe rate of back-to-back tcgen05.mma 128 x n x 32-byte-K instructions (one CTA per SM, operands resident in
// shared memory): which = 0 kind::i8, 1 kind::f16 (bf16).  Returns tera-MACs per second (x2 = TOP/s / TFLOP/s).
int cflx_dbg_umma_peak(int which, int n, double* tmacs_out) {
    CFLX_TRY(check_device());
    if (!tmacs_out) return CFLX_ERR_ARG;
    return umma_peak_probe(n, which, tmacs_out);
}

}  // extern "C"
