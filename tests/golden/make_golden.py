"""tests/golden/make_golden.py -- regenerates tests/golden/*.npz by running THE REFERENCE ITSELF
(oracle/_ref/libref_lu.so = /root/reference sources compiled by oracle/build_ref.sh; ranks are threads).
Run in the build container only (needs /root/reference):  python tests/golden/make_golden.py
    [helpers] [lu_cases] [lu_ref_cases] [layouts]   (default: all)

Fixtures:
  helpers.npz  - the reference's building blocks on the inputs of its own unit test
                 (tests/unit/test_utils.cpp:8-84 push_pivots_up 8x8 case) plus seeded random cases:
                 push_pivots_up, inverse_permute_rows, permute_rows, butterfly_pair, g2lnoTile owners, LUP perms.
  lu_cases.npz - full LU_rep outputs (input A, C, permutation) on small grids, incl. the hard-coded
                 matrices of lu_params.hpp:157-363 (N = 16, 27, 32) and multi-rank / multi-layer grids.
  lu_perms.npz - permutation-only known answers for larger seeded inputs (N = 256, 1024, 2048).
  lu_ref_cases.npz - LU_rep on the grids of tests/test_oracle_vs_reference.py: a SHA-256 digest of the generated
                 input, the permutation and a seeded sample of the factors (the full factors would exceed 1 MB).
  layouts.txt  - the reference's conflux_layout / lu_params::matrix COSTA descriptors (tests/cpp/layout_ref_dump.cpp,
                 compiled against the sources under $CONFLUX_REFERENCE), for tests/test_layout_vs_costa.py.
"""
import ctypes
import hashlib
import os
import subprocess
import sys
import sysconfig
import tempfile
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref, layout  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
L = ref.lib()
dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
ip = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_int))


def helpers():
    out = {}
    rng = np.random.default_rng(7)
    # the reference's own unit-test input (tests/unit/test_utils.cpp:10-19), pivots {2,1,5}, fnpr 0
    ut = np.array([9, 1, 1, 9, 5, 5, 3, 3, 7, 3, 4, 5, 2, 4, 5, 2, 5, 5, 1, 3, 3, 9, 1, 9, 9, 2, 3, 9, 5, 2, 2, 9,
                   7, 6, 5, 7, 8, 1, 4, 4, 2, 2, 4, 6, 5, 2, 6, 5, 3, 7, 4, 4, 4, 7, 1, 7, 3, 8, 1, 6, 4, 8, 7, 8],
                  dtype=np.float64).reshape(8, 8)
    cases = [(ut, np.array([3, 2, 1, 5], dtype=np.int32), 0)]
    for (n, c, fnpr, npiv) in [(12, 5, 3, 4), (16, 3, 0, 8), (9, 4, 5, 2), (20, 7, 6, 0), (10, 2, 2, 8), (6, 6, 0, 6)]:
        m = rng.integers(0, 100, size=(n, c)).astype(np.float64)
        piv = rng.permutation(np.arange(fnpr, n))[:npiv].astype(np.int32)
        cases.append((m, np.concatenate([[npiv], piv]).astype(np.int32), fnpr))
    out["push_n"] = np.array(len(cases))
    for i, (m, cp, fnpr) in enumerate(cases):
        res = np.ascontiguousarray(m.copy())
        L.ref_push_pivots_up(dp(res), m.shape[0], m.shape[1], ip(np.ascontiguousarray(cp)), int(fnpr))
        out[f"push{i}_in"], out[f"push{i}_piv"], out[f"push{i}_fnpr"], out[f"push{i}_out"] = m, cp, np.array(fnpr), res
    # inverse_permute_rows / permute_rows (utils.hpp:49-138): strided + column-offset shapes
    pcases = [(4, 3, 4, 3), (4, 5, 4, 3), (6, 4, 3, 4), (8, 5, 4, 2), (1, 1, 1, 1)]
    out["perm_n"] = np.array(len(pcases))
    for i, (nr, nc, onr, onc) in enumerate(pcases):
        m = rng.standard_normal((nr, nc))
        p = rng.permutation(nr).astype(np.int32)
        inv = np.zeros((onr, onc))
        L.ref_inverse_permute_rows(dp(m), dp(inv), nr, nc, onr, onc, ip(p), nr)
        out[f"perm{i}_in"], out[f"perm{i}_p"], out[f"perm{i}_inv"] = m, p, inv
        if onr == nr:
            fw = np.zeros((onr, onc))
            L.ref_permute_rows(dp(m), dp(fw), nr, nc, onr, onc, ip(p), nr)
            out[f"perm{i}_fwd"] = fw
    # butterfly_pair table (conflux_opt.cpp:59-72)
    bp = np.full((9, 4, 9), -1, dtype=np.int32)
    for Px in range(1, 9):
        for r in range(4):
            for pi in range(Px):
                bp[Px, r, pi] = L.ref_butterfly_pair(pi, r, Px)
    out["butterfly"] = bp
    # g2lnoTile owners (conflux_opt.cpp:74-98)
    g = rng.integers(0, 96, size=24).astype(np.int32)
    own = np.zeros(24, dtype=np.int32)
    L.ref_g2l_owner(ip(g), 24, 3, 8, ip(own))
    out["g2l_rows"], out["g2l_owner"] = g, own
    # LUP (conflux_opt.hpp:143-166): perm of seeded panels, incl. n < v and integer ties
    lcases = [(rng.standard_normal((24, 9)), 24, 8), (rng.standard_normal((16, 9)), 16, 8),
              (rng.integers(0, 4, size=(16, 5)).astype(np.float64), 16, 4),
              (rng.standard_normal((3, 9)), 3, 8), (rng.standard_normal((64, 17)), 64, 16)]
    out["lup_n"] = np.array(len(lcases))
    for i, (c, n, v) in enumerate(lcases):
        m = max(2 * v, n)
        perm = np.zeros(m, dtype=np.int32)
        pb = np.zeros((max(n, 1), v))
        L.ref_lup(n, v, dp(np.ascontiguousarray(c)), ip(perm), dp(pb))
        out[f"lup{i}_cand"], out[f"lup{i}_perm"], out[f"lup{i}_lu"] = c, perm, pb
    np.savez_compressed(os.path.join(HERE, "helpers.npz"), **out)


def lu_cases():
    out = {}
    cases = [(16, 4, 1, 1, 1), (16, 4, 2, 2, 1), (27, 3, 3, 3, 1), (32, 4, 2, 2, 2), (64, 8, 1, 1, 1),
             (64, 8, 2, 2, 1), (64, 8, 2, 2, 2), (64, 16, 1, 1, 2), (96, 8, 3, 3, 1), (128, 16, 2, 2, 2)]
    out["cases"] = np.array(cases, dtype=np.int32)
    for i, (N, v, Px, Py, Pz) in enumerate(cases):
        r = ref.lu_run(N, v, Px, Py, Pz)
        out[f"c{i}_A"] = np.stack(r["A"])
        out[f"c{i}_C"] = np.stack(r["C"])
        out[f"c{i}_perm"] = r["perm"]
        A = layout.assemble(r["A"], N, v, Px, Py, Pz)
        LU = layout.assemble(r["C"], N, v, Px, Py, Pz)
        out[f"c{i}_res"] = np.array(layout.residual(A, LU, r["perm"]))
    np.savez_compressed(os.path.join(HERE, "lu_cases.npz"), **out)
    perms = {}
    pc = [(256, 32, 1, 1, 1), (256, 16, 2, 2, 1), (512, 32, 2, 2, 2), (1024, 64, 1, 1, 1), (1024, 64, 2, 2, 2),
          (1024, 128, 1, 1, 2), (2048, 128, 1, 1, 1)]
    perms["cases"] = np.array(pc, dtype=np.int32)
    for i, c in enumerate(pc):
        perms[f"p{i}"] = ref.lu_run(*c, want_factors=False, blas_threads=4)["perm"]
    np.savez_compressed(os.path.join(HERE, "lu_perms.npz"), **perms)


REF_CASES = [(48, 4, 1, 1, 1), (128, 16, 2, 2, 1), (128, 8, 2, 2, 2), (96, 16, 1, 1, 2), (72, 4, 3, 3, 2), (256, 32, 4, 4, 1)]
REF_SAMPLE = 1024        # factor entries kept per case


def lu_ref_cases():
    out = {"cases": np.array(REF_CASES, dtype=np.int32)}
    for i, (N, v, Px, Py, Pz) in enumerate(REF_CASES):
        r = ref.lu_run(N, v, Px, Py, Pz)
        out[f"c{i}_A_sha256"] = np.array(hashlib.sha256(np.ascontiguousarray(np.stack(r["A"])).tobytes()).hexdigest())
        out[f"c{i}_perm"] = r["perm"]
        C = np.stack(r["C"]).reshape(-1)
        idx = np.sort(np.random.default_rng(i).choice(C.size, size=min(REF_SAMPLE, C.size), replace=False))
        out[f"c{i}_C_idx"] = idx.astype(np.int32)
        out[f"c{i}_C_val"] = C[idx]
    np.savez_compressed(os.path.join(HERE, "lu_ref_cases.npz"), **out)


def layouts():
    src = os.environ.get("CONFLUX_REFERENCE")
    if not src or not os.path.isdir(os.path.join(src, "libs", "costa", "src")):
        sys.exit("layouts: set CONFLUX_REFERENCE to the reference checkout (eth-cscs/conflux with libs/costa)")
    costa = os.path.join(src, "libs", "costa", "src")
    sp = sysconfig.get_paths()["purelib"]
    libs = os.path.join(sp, "opencv_python_headless.libs")
    blas = os.path.join(libs, sorted(f for f in os.listdir(libs) if f.startswith("libopenblasp"))[0])
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "layout_ref_dump")
        srcs = [f"{src}/src/conflux/lu/layout.cpp", f"{costa}/costa/layout.cpp", f"{ROOT}/oracle/mpi_stub/mpi_threads.cpp"] + \
               [f"{costa}/costa/grid2grid/{f}.cpp" for f in ("block", "grid2D", "interval", "scalapack_layout", "ranks_reordering")]
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fopenmp", "-w", "-DNDEBUG", f"-I{ROOT}/oracle/mpi_stub", f"-I{costa}",
                               f"-I{src}/src", f"{ROOT}/tests/cpp/layout_ref_dump.cpp"] + srcs +
                              [blas, f"-Wl,-rpath,{libs}", f"-Wl,-rpath,{sp}/scipy.libs", "-lpthread", "-o", exe])
        txt = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    with open(os.path.join(HERE, "layouts.txt"), "w") as f:
        f.write(txt)


if __name__ == "__main__":
    if not ref.available():
        sys.exit("oracle/_ref/libref_lu.so missing: run oracle/build_ref.sh in the build container first")
    steps = {"helpers": helpers, "lu_cases": lu_cases, "lu_ref_cases": lu_ref_cases, "layouts": layouts}
    for name in [a for a in sys.argv[1:] if a in steps] or list(steps):
        steps[name]()
    print("golden fixtures written to", HERE)
