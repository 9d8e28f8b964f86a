// tests/cpp/layout_ref_dump.cpp -- TEST INFRASTRUCTURE, golden generator only (tests/golden/make_golden.py compiles it
// against the reference sources).  Prints the COSTA descriptors produced by the REFERENCE's conflux_layout
// (src/conflux/lu/layout.cpp, both overloads; the 3-D one through lu_params::matrix on the thread-backed MPI stub) in
// the text format of layout_dump.cpp; the output is tests/golden/layouts.txt.
#include <algorithm>
#include <cstdio>
#include <functional>  // lu_params.hpp uses std::bind and <random> without including them
#include <random>
#include <string>
#include <tuple>
#include <vector>

#include <conflux/lu/layout.hpp>
#include <conflux/lu/lu_params.hpp>

static std::string describe(costa::grid_layout<double>& a, const double* base) {
    std::string s = "size " + std::to_string(a.num_rows()) + " " + std::to_string(a.num_cols()) + " " +
                    std::to_string(a.num_blocks_row()) + " " + std::to_string(a.num_blocks_col()) + "\nrows";
    for (int i = 0; i < a.num_blocks_row(); ++i)
        s += " " + std::to_string(a.grid.rows_interval(i).start) + ":" + std::to_string(a.grid.rows_interval(i).end);
    s += "\ncols";
    for (int j = 0; j < a.num_blocks_col(); ++j)
        s += " " + std::to_string(a.grid.cols_interval(j).start) + ":" + std::to_string(a.grid.cols_interval(j).end);
    s += "\nowners";
    for (int i = 0; i < a.num_blocks_row(); ++i)
        for (int j = 0; j < a.num_blocks_col(); ++j) s += " " + std::to_string(a.grid.owner(i, j));
    s += "\n";
    // the order in which a layout enumerates its local blocks is an internal detail (COSTA's ScaLAPACK variant walks
    // them column by column): blocks are listed by global block coordinates
    std::vector<std::tuple<int, int, long, int, int, int>> blocks;
    for (size_t k = 0; k < a.blocks.num_blocks(); ++k) {
        auto& x = a.blocks.get_block(k);
        blocks.emplace_back(x.coordinates.row, x.coordinates.col, (long)(x.data - base), x.stride, x.n_rows(), x.n_cols());
    }
    std::sort(blocks.begin(), blocks.end());
    for (auto& b : blocks)
        s += "block " + std::to_string(std::get<0>(b)) + " " + std::to_string(std::get<1>(b)) + " " +
             std::to_string(std::get<2>(b)) + " " + std::to_string(std::get<3>(b)) + " " + std::to_string(std::get<4>(b)) +
             " " + std::to_string(std::get<5>(b)) + "\n";
    return s;
}

struct Case { int N, v, Px, Py, Pz; std::vector<std::string> out; };
static void rank_main(int, void* p) {
    auto* c = (Case*)p;
    conflux::lu_params<double> params(c->N, c->N, c->v, c->Px, c->Py, c->Pz, MPI_COMM_WORLD);
    char head[160];
    std::snprintf(head, sizeof head, "case cart %d %d %d R %d %d %d %d %d %d\n", params.M, params.N, params.v, params.Px,
                  params.Py, params.Pz, params.pi, params.pj, params.pk);
    c->out[params.rank] = head + describe(params.matrix, params.data.data());
    MPI_Barrier(params.lu_comm);
}

int main() {
    std::vector<double> buf(1 << 16);
    const int cases[][5] = {{16, 16, 4, 1, 1}, {64, 64, 8, 2, 2}, {96, 96, 8, 3, 3}, {48, 48, 4, 2, 2}};
    for (auto& c : cases)
        for (char ord : {'R', 'C'})
            for (int rank = 0; rank < c[3] * c[4]; ++rank) {
                auto ref = conflux::conflux_layout<double>(buf.data(), c[0], c[1], c[2], ord, c[3], c[4], rank);
                std::printf("case bc %d %d %d %c %d %d %d\n%s", c[0], c[1], c[2], ord, c[3], c[4], rank,
                            describe(ref, buf.data()).c_str());
            }
    Case cs[] = {{64, 8, 2, 2, 1}, {64, 8, 2, 2, 2}, {96, 8, 3, 3, 1}, {64, 16, 1, 1, 2}, {100, 16, 2, 2, 1}};
    for (auto& c : cs) {
        c.out.resize(c.Px * c.Py * c.Pz);
        stub_mpi_run(c.Px * c.Py * c.Pz, rank_main, &c);
        for (auto& s : c.out) std::fputs(s.c_str(), stdout);
    }
    return 0;
}
