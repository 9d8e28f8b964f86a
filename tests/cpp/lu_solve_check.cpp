// tests/cpp/lu_solve_check.cpp -- conflux::LU_solve through the C++ facade on one GPU: factor the seeded N x N matrix,
// solve for 3 right-hand sides, print the normwise backward error ||B - A X||_F / (||A||_F ||X||_F).
//   usage: lu_solve_check [N]        exit 0 when the backward error is <= 1e-12
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <exception>
#include <vector>

#include "conflux/lu/conflux_b200.hpp"

int main(int argc, char** argv) {
    const int N = argc > 1 ? std::atoi(argv[1]) : 256, v = 32, nrhs = 3;
    int ndev = 0;
    cflx_device_count(&ndev);
    if (ndev == 0) {
        std::fprintf(stderr, "no CUDA device visible (no CPU fallback)\n");
        return 2;
    }
    try {
        cflx_comm* comm = nullptr;
        conflux::check(cflx_comm_create(1, 0, nullptr, 0, &comm), "comm");
        double berr = 0;
        {
            conflux::lu_params<double> gv(N, N, v, 1, 1, 1, comm);
            conflux::LU_rep<double>(gv, nullptr, nullptr);
            const int M = gv.M;  // one rank: the local array is the whole (padded) matrix
            std::vector<double> B((size_t)M * nrhs), X((size_t)gv.Nl * nrhs);
            for (size_t i = 0; i < B.size(); ++i) B[i] = std::sin(0.37 * (double)i + 1.0);
            const std::size_t ms = conflux::LU_solve<double>(gv, nrhs, B.data(), X.data());
            double r2 = 0, a2 = 0, x2 = 0;
            for (int i = 0; i < M; ++i)
                for (int c = 0; c < nrhs; ++c) {
                    double s = B[(size_t)i * nrhs + c];
                    for (int k = 0; k < M; ++k) s -= gv.data[(size_t)i * gv.Nl + k] * X[(size_t)k * nrhs + c];
                    r2 += s * s;
                }
            for (double a : gv.data) a2 += a * a;
            for (double x : X) x2 += x * x;
            berr = std::sqrt(r2) / (std::sqrt(a2) * std::sqrt(x2));
            std::printf("lu_solve_check: N=%d v=%d nrhs=%d  %zu ms  backward_error=%.3e\n", M, v, nrhs, ms, berr);
        }
        cflx_comm_destroy(comm);
        return berr <= 1e-12 ? 0 : 1;
    } catch (const std::exception& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 2;
    }
}
