// tests/cpp/layout_dump.cpp -- TEST INFRASTRUCTURE: this repo's conflux_layout descriptors (both overloads) in a text
// format that tests/test_layout_vs_costa.py compares with the reference's COSTA descriptors (tests/golden/layouts.txt,
// written by layout_ref_dump.cpp).  Reads the "case" lines of that file on stdin and answers each with its descriptor:
//   case bc   M N v ordering Px Py rank           -> conflux_layout(data, M, N, v, ordering, Px, Py, rank)
//   case cart M N v ordering Px Py Pz pi pj pk     -> conflux_layout(data, M, N, v, ordering, lu_comm at (pi, pj, pk))
// Block offsets are counted in elements from the start of the local array.
#include <algorithm>
#include <cstdio>
#include <iostream>
#include <sstream>
#include <string>
#include <tuple>
#include <vector>

#include <conflux/lu/conflux_b200.hpp>

static std::string describe(const conflux::grid_layout<double>& a, const double* base) {
    const int nbr = a.rowblocks, nbc = a.colblocks;
    std::string s = "size " + std::to_string(a.rowsplit[nbr]) + " " + std::to_string(a.colsplit[nbc]) + " " +
                    std::to_string(nbr) + " " + std::to_string(nbc) + "\nrows";
    for (int i = 0; i < nbr; ++i) s += " " + std::to_string(a.rowsplit[i]) + ":" + std::to_string(a.rowsplit[i + 1]);
    s += "\ncols";
    for (int j = 0; j < nbc; ++j) s += " " + std::to_string(a.colsplit[j]) + ":" + std::to_string(a.colsplit[j + 1]);
    s += "\nowners";
    for (int o : a.owners) s += " " + std::to_string(o);
    s += "\n";
    std::vector<std::tuple<int, int, long, int, int, int>> blocks;
    for (const auto& b : a.localblocks)
        blocks.emplace_back(b.row, b.col, (long)(static_cast<const double*>(b.data) - base), b.ld,
                            a.rowsplit[b.row + 1] - a.rowsplit[b.row], a.colsplit[b.col + 1] - a.colsplit[b.col]);
    std::sort(blocks.begin(), blocks.end());
    for (auto& b : blocks)
        s += "block " + std::to_string(std::get<0>(b)) + " " + std::to_string(std::get<1>(b)) + " " +
             std::to_string(std::get<2>(b)) + " " + std::to_string(std::get<3>(b)) + " " + std::to_string(std::get<4>(b)) +
             " " + std::to_string(std::get<5>(b)) + "\n";
    return s;
}

int main() {
    std::vector<double> buf(1 << 16);
    std::string line;
    while (std::getline(std::cin, line)) {
        std::istringstream in(line);
        std::string tag, kind;
        int M, N, v;
        char ord;
        in >> tag >> kind >> M >> N >> v >> ord;
        if (tag != "case") continue;
        if (kind == "bc") {
            int Px, Py, rank;
            in >> Px >> Py >> rank;
            std::cout << line << "\n" << describe(conflux::conflux_layout<double>(buf.data(), M, N, v, ord, Px, Py, rank), buf.data());
        } else {
            conflux::cart_t c;
            in >> c.dims[0] >> c.dims[1] >> c.dims[2] >> c.coords[0] >> c.coords[1] >> c.coords[2];
            c.rank = c.cart_rank(c.coords[0], c.coords[1], c.coords[2]);
            std::cout << line << "\n" << describe(conflux::conflux_layout<double>(buf.data(), M, N, v, ord, c), buf.data());
        }
    }
    return 0;
}
