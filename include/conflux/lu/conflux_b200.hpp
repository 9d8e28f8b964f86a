// include/conflux/lu/conflux_b200.hpp -- header-only C++ facade over the C ABI (include/conflux_b200.h) that keeps the
// reference's driver-facing names for the LU path, so that examples/conflux_miniapp.cpp reads like the reference's
// miniapp (examples/conflux_miniapp.cpp:88-167 there).  Reference interfaces mirrored (file:line in eth-cscs/conflux):
//   conflux::lu_params<T>       src/conflux/lu/lu_params.hpp:8-459   (ctors :401-409, public fields :378-397)
//   conflux::LU_rep<T>          src/conflux/lu/conflux_opt.hpp:343-346
//   conflux::conflux_layout<T>  src/conflux/lu/layout.hpp:7-17, layout.cpp:30-135 (both overloads)
// MPI is not part of this image, so the MPI handles become small value types with the same roles:
//   MPI_Comm (world, ctor argument)      -> conflux::comm_t   (a cflx_comm*: one per rank, one GPU per rank)
//   MPI_Comm lu_comm (3-D Cartesian)     -> conflux::cart_t   (handle + dims + coords + rank, what MPI_Cart_get returns)
//   jk_comm / ik_comm / ij_comm / k_comm / i_comm (MPI_Cart_sub)   -> conflux::sub_comm_t (kept dims, size, rank); the
//        NCCL communicators behind them are created by ncclCommSplit inside the plan (cflx_lu_create)
//   costa::grid_layout<T> matrix         -> conflux::grid_layout<T>: the argument list of costa::custom_layout<T>
//        (libs/costa/src/costa/layout.hpp:35-42) held by value + COSTA's initialize/apply/accumulate element visitors;
//        with -DCONFLUX_B200_WITH_COSTA it converts to the real costa::grid_layout<T> (to_costa()).
#pragma once
#include <cctype>
#include <cmath>
#include <cstddef>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../conflux_b200.h"

#ifdef CONFLUX_B200_WITH_COSTA
#include <costa/layout.hpp>
#endif

namespace conflux {

using comm_t = cflx_comm*;

inline void check(int rc, const char* what) {
    if (rc != 0) throw std::runtime_error(std::string(what) + ": " + cflx_last_error());
}

// what MPI_Cart_get / MPI_Comm_rank report for the reference's lu_comm (lu_params.hpp:85-92): dims = {Px, Py, Pz},
// coords = {pi, pj, pk}, rank = (pi*Py + pj)*Pz + pk (row-major, no reordering)
struct cart_t {
    comm_t handle = nullptr;
    int dims[3] = {0, 0, 0};
    int coords[3] = {0, 0, 0};
    int rank = 0;
    bool null() const { return handle == nullptr; }
    int cart_rank(int pi, int pj, int pk) const { return (pi * dims[1] + pj) * dims[2] + pk; }  // MPI_Cart_rank
};
// result of MPI_Cart_sub(lu_comm, keep, &sub): the kept dimensions, the size and this rank's number inside it
struct sub_comm_t {
    int keep[3] = {0, 0, 0};
    int size = 0, rank = 0;
    bool null() const { return size == 0; }
};
inline sub_comm_t cart_sub(const cart_t& c, int k0, int k1, int k2) {
    sub_comm_t s;
    s.keep[0] = k0; s.keep[1] = k1; s.keep[2] = k2;
    s.size = 1; s.rank = 0;
    for (int d = 0; d < 3; ++d)
        if (s.keep[d]) {
            s.rank = s.rank * c.dims[d] + c.coords[d];
            s.size *= c.dims[d];
        }
    return s;
}

// == costa::block_t (libs/costa/src/costa/layout.hpp:14-19)
struct block_t {
    void* data;
    int ld;
    int row;
    int col;
};

// Non-owning description of a distributed matrix: exactly the inputs of costa::custom_layout<T>.
template <typename T>
struct grid_layout {
    int rowblocks = 0, colblocks = 0;
    std::vector<int> rowsplit, colsplit;  // block i covers rows [rowsplit[i], rowsplit[i+1])
    std::vector<int> owners;              // rowblocks x colblocks, row-major: rank owning each block
    std::vector<block_t> localblocks;     // this rank's blocks: pointer, leading dimension, global block coordinates
    char ordering = 'R';                  // storage order inside a local block

    int num_local_blocks() const { return (int)localblocks.size(); }
    T& at(const block_t& b, int li, int lj) const {
        T* p = static_cast<T*>(b.data);
        return ordering == 'R' ? p[(std::size_t)li * b.ld + lj] : p[(std::size_t)lj * b.ld + li];
    }
    // COSTA's element visitors (grid_layout.hpp:68-131): blocks in local order, row by row inside a block;
    // f receives GLOBAL element coordinates
    template <class F>
    void initialize(F f) {
        for (const block_t& b : localblocks)
            for (int li = 0; li < rowsplit[b.row + 1] - rowsplit[b.row]; ++li)
                for (int lj = 0; lj < colsplit[b.col + 1] - colsplit[b.col]; ++lj)
                    at(b, li, lj) = f(rowsplit[b.row] + li, colsplit[b.col] + lj);
    }
    template <class F>
    void apply(F f) {
        for (const block_t& b : localblocks)
            for (int li = 0; li < rowsplit[b.row + 1] - rowsplit[b.row]; ++li)
                for (int lj = 0; lj < colsplit[b.col + 1] - colsplit[b.col]; ++lj)
                    at(b, li, lj) = f(rowsplit[b.row] + li, colsplit[b.col] + lj, at(b, li, lj));
    }
    template <class F>
    T accumulate(F f, T init) const {
        for (const block_t& b : localblocks)
            for (int li = 0; li < rowsplit[b.row + 1] - rowsplit[b.row]; ++li)
                for (int lj = 0; lj < colsplit[b.col + 1] - colsplit[b.col]; ++lj) init = f(init, at(b, li, lj));
        return init;
    }
#ifdef CONFLUX_B200_WITH_COSTA
    costa::grid_layout<T> to_costa() const {
        static_assert(sizeof(costa::block_t) == sizeof(block_t), "block descriptor mismatch");
        return costa::custom_layout<T>(rowblocks, colblocks, rowsplit.data(), colsplit.data(), owners.data(),
                                       (int)localblocks.size(), reinterpret_cast<const costa::block_t*>(localblocks.data()),
                                       ordering);
    }
#endif
};

namespace detail {
inline std::vector<int> line_split(int N, int v) {  // layout.cpp:20-28
    std::vector<int> s;
    s.reserve(N / v + 1);
    for (int i = 0; i < N / v; ++i) s.push_back(i * v);
    s.push_back(N);
    return s;
}
template <typename T>
grid_layout<T> tile_layout(T* data, int M, int N, int v, char ordering, int Px, int Py, int pi, int pj, int rank_stride,
                           int owner_stride_i) {
    ordering = (char)std::toupper((unsigned char)ordering);
    if (ordering != 'R' && ordering != 'C') throw std::invalid_argument("conflux_layout: ordering must be 'R' or 'C'");
    const int Nt = (int)std::ceil((double)N / v), Mt = (int)std::ceil((double)M / v);
    const int tA11x = (int)std::ceil((double)Mt / Px), tA11y = (int)std::ceil((double)Nt / Py);
    const int Ml = tA11x * v, Nl = tA11y * v;
    grid_layout<T> g;
    g.rowblocks = Mt; g.colblocks = Nt; g.ordering = ordering;
    g.rowsplit = line_split(M, v);
    g.colsplit = line_split(N, v);
    g.owners.resize((std::size_t)Mt * Nt);
    for (int i = 0; i < Mt; ++i)
        for (int j = 0; j < Nt; ++j) g.owners[(std::size_t)i * Nt + j] = (i % Px) * owner_stride_i + (j % Py) * rank_stride;
    for (int lti = 0; lti < tA11x; ++lti) {
        const int gti = lti * Px + pi;
        if (gti >= Mt) continue;
        for (int ltj = 0; ltj < tA11y; ++ltj) {
            const int gtj = ltj * Py + pj;
            if (gtj >= Nt) continue;
            block_t b;
            // tile (lti, ltj) of the local Ml x Nl array: row-major storage puts it at lti*v*Nl + ltj*v (layout.cpp:100),
            // column-major storage (the miniapp's "scalapack" buffers) at ltj*v*Ml + lti*v
            b.data = ordering == 'R' ? (void*)(data + (std::size_t)lti * v * Nl + (std::size_t)ltj * v)
                                     : (void*)(data + (std::size_t)ltj * v * Ml + (std::size_t)lti * v);
            b.ld = ordering == 'R' ? Nl : Ml;
            b.row = gti; b.col = gtj;
            g.localblocks.push_back(b);
        }
    }
    return g;
}
}  // namespace detail

// layout.cpp:30-61: 2-D block-cyclic variant, `rank` numbered row-major on the Px x Py grid ('R' grid order)
template <typename T>
grid_layout<T> conflux_layout(T* data, int M, int N, int v, char ordering, int Px, int Py, int rank) {
    return detail::tile_layout(data, M, N, v, ordering, Px, Py, rank / Py, rank % Py, /*rank stride of pj*/ 1,
                               /*rank stride of pi*/ Py);
}
// layout.cpp:63-135: custom layout on the 3-D communicator; tile (i, j) belongs to rank X2p(i % Px, j % Py, 0)
template <typename T>
grid_layout<T> conflux_layout(T* data, int M, int N, int v, char ordering, const cart_t& lu_comm) {
    const int Px = lu_comm.dims[0], Py = lu_comm.dims[1], Pz = lu_comm.dims[2];
    return detail::tile_layout(data, M, N, v, ordering, Px, Py, lu_comm.coords[0], lu_comm.coords[1], Pz, Py * Pz);
}

template <typename T>
class lu_params {
    static_assert(sizeof(T) == sizeof(double), "the B200 path is FP64 only (BASELINE.json)");

   public:
    cart_t lu_comm;
    sub_comm_t jk_comm, ik_comm, ij_comm, k_comm, i_comm;  // lu_params.hpp:94-108
    int rank = 0, pi = 0, pj = 0, pk = 0;
    int M = 0, N = 0, P = 0, Ml = 0, Nl = 0, Px = 0, Py = 0, Pz = 0;
    int v = 0, nlayr = 0, Mt = 0, Nt = 0, t = 0, tA11x = 0, tA11y = 0;
    int seed = 42;
    std::vector<T> data;     // local tiles, row-major Ml x Nl (conflux/COSTA tile layout, layout.cpp:95-109)
    grid_layout<T> matrix;   // non-owning descriptor of `data` (lu_params.hpp:118)
    bool use_collectives = false;
    cflx_lu* plan = nullptr;  // device side of this object (B200 only)

    lu_params() = default;
    lu_params(int inpM, int inpN, int v_, comm_t comm) { initialize(inpM, inpN, v_, -1, -1, -1, comm); }
    lu_params(int inpM, int inpN, int v_, int Px_, int Py_, int Pz_, comm_t comm) {
        initialize(inpM, inpN, v_, Px_, Py_, Pz_, comm);
    }
    lu_params(const lu_params&) = delete;
    lu_params& operator=(const lu_params&) = delete;
    ~lu_params() { free_comms(); }

    void InitMatrix() {  // lu_params.hpp:141-376: zeros, fixed matrices for M = N in {8,9,16,20,27,32}, seeded otherwise
        check(cflx_init_matrix_host(M, N, v, Px, Py, Pz, rank, seed, data.data()), "InitMatrix");
    }
    void free_comms() {  // idempotent like the reference's (lu_params.hpp:434-457)
        if (plan) cflx_lu_destroy(plan);
        plan = nullptr;
        lu_comm = cart_t{};
        jk_comm = ik_comm = ij_comm = k_comm = i_comm = sub_comm_t{};
    }

   private:
    void initialize(int inpM, int inpN, int v_, int Px_, int Py_, int Pz_, comm_t comm) {
        check(cflx_lu_create(comm, inpM, inpN, v_, Px_, Py_, Pz_, &plan), "lu_params");
        int info[16];
        check(cflx_lu_info(plan, info), "lu_info");
        M = info[0]; N = info[1]; Ml = info[2]; Nl = info[3]; Nt = info[4]; nlayr = info[5]; P = info[6];
        Px = info[7]; Py = info[8]; Pz = info[9]; pi = info[10]; pj = info[11]; pk = info[12]; rank = info[13]; v = info[14];
        Mt = M / v; tA11x = Ml / v; tA11y = Nl / v; t = tA11y + 1;
        use_collectives = v > 1024;
        lu_comm.handle = comm;
        lu_comm.dims[0] = Px; lu_comm.dims[1] = Py; lu_comm.dims[2] = Pz;
        lu_comm.coords[0] = pi; lu_comm.coords[1] = pj; lu_comm.coords[2] = pk;
        lu_comm.rank = rank;
        jk_comm = cart_sub(lu_comm, 0, 1, 1);
        ik_comm = cart_sub(lu_comm, 1, 0, 1);
        k_comm = cart_sub(lu_comm, 0, 0, 1);
        i_comm = cart_sub(lu_comm, 1, 0, 0);
        ij_comm = cart_sub(lu_comm, 1, 1, 0);
        data.assign((std::size_t)Ml * Nl, T{0});
        matrix = conflux_layout(data.data(), M, N, v, 'R', lu_comm);
        InitMatrix();
    }
};

// Collective over gv.lu_comm; does not modify gv.data; C (>= Ml*Nl, may be null) and permutation (>= M, may be null)
// are filled as in the reference's validation build; returns the main-loop time in ms (truncated like the reference).
template <class T>
std::size_t LU_rep(lu_params<T>& gv, T* C, int* permutation) {
    double ms = 0;
    check(cflx_lu_set_local(gv.plan, gv.data.data()), "LU_rep: upload");
    check(cflx_lu_factor(gv.plan, &ms), "LU_rep: factor");
    if (C) check(cflx_lu_get_factors(gv.plan, C, permutation), "LU_rep: factors");
    else if (permutation) check(cflx_lu_get_permutation(gv.plan, permutation), "LU_rep: permutation");
    return (std::size_t)ms;
}

// A X = B with the factors of the last LU_rep (no counterpart in the reference).  Collective over gv.lu_comm.
// B: this rank's Ml x nrhs rows of B in A's row distribution (read on ranks with pj == 0 && pk == 0, may be null
// elsewhere); X: Nl x nrhs, filled on every rank with X in A's column distribution (cflx_lu_solve in conflux_b200.h).
// Returns the device time of the solve in ms (truncated like LU_rep).
template <class T>
std::size_t LU_solve(lu_params<T>& gv, int nrhs, const T* B, T* X) {
    double ms = 0;
    check(cflx_lu_solve(gv.plan, nrhs, B, X, &ms), "LU_solve");
    return (std::size_t)ms;
}

// The reference's validation (examples/conflux_miniapp.cpp:349-500) of the last LU_rep, on the GPU grid.  Collective.
// Returns ||P*A - L*U||_F (what the reference prints as "Total Frobenius norm"); *relative = that / ||A||_F.
template <class T>
double validate(lu_params<T>& gv, double* relative = nullptr) {
    double a = 0, r = 0;
    check(cflx_lu_validate(gv.plan, &a, &r), "validate");
    if (relative) *relative = r;
    return a;
}

}  // namespace conflux
