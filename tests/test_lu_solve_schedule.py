"""CPU: the fan-in tile schedule of cflx_lu_solve (oracle/solve_ref.py) solves A X = B on every grid shape, the
right-hand-side / solution layouts round-trip, the C ABI refuses bad arguments without a device, and the C++ facade's
LU_solve compiles."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import scipy.linalg

import conflux_b200 as cb
from conflux_b200 import _lib
from oracle import layout, restate, solve_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("N,v,Px,Py,Pz", [(64, 8, 1, 1, 1), (100, 16, 1, 1, 1), (64, 8, 2, 2, 1), (100, 8, 2, 2, 1),
                                          (64, 8, 2, 2, 2), (72, 8, 3, 3, 1), (100, 4, 3, 3, 1), (72, 8, 3, 3, 2)])
@pytest.mark.parametrize("nrhs", [1, 5])
def test_schedule_solves_the_system(N, v, Px, Py, Pz, nrhs):
    A_locals = restate.init_matrix(N, v, Px, Py, Pz)
    o = restate.lu(A_locals, N, v, Px, Py, Pz)
    A = layout.assemble(A_locals, N, v, Px, Py, Pz)
    B = np.random.default_rng(N + nrhs).standard_normal((A.shape[0], nrhs))
    X_locals = solve_ref.solve(o["C"], o["perm"], solve_ref.scatter_rows(B, N, v, Px, Py, Pz), N, v, Px, Py, Pz)
    X = solve_ref.gather_cols(X_locals, N, v, Px, Py, Pz)            # also: replicas bitwise equal
    want = scipy.linalg.lu_solve(scipy.linalg.lu_factor(A), B)
    assert np.abs(X - want).max() <= 1e-11 * np.abs(want).max()


def test_layout_helpers_round_trip():
    for (N, v, Px, Py, Pz) in [(64, 8, 1, 1, 1), (100, 16, 2, 2, 1), (72, 8, 3, 3, 2)]:
        d = layout.dims(N, v, Px, Py, Pz)
        B = np.arange(d["M"] * 3, dtype=np.float64).reshape(d["M"], 3)
        parts = solve_ref.scatter_rows(B, N, v, Px, Py, Pz)
        assert all(p.shape == (d["Ml"], 3) for p in parts)
        assert np.array_equal(solve_ref.gather_rows(parts, N, v, Px, Py, Pz), B)
        cols = solve_ref.scatter_cols(B, N, v, Px, Py, Pz)
        assert all(c.shape == (d["Nl"], 3) for c in cols)
        assert np.array_equal(solve_ref.gather_cols(cols, N, v, Px, Py, Pz), B)
        if d["P"] > 1:
            cols[-1] = cols[-1].copy()
            cols[-1][0, 0] += 1.0
            with pytest.raises(AssertionError):
                solve_ref.gather_cols(cols, N, v, Px, Py, Pz)


def test_solve_refuses_bad_arguments_without_a_handle():
    X = np.zeros(4)
    B = np.zeros(4)
    assert _lib.lib().cflx_lu_solve(None, 1, B.ctypes.data, X.ctypes.data, None) == -1   # CFLX_ERR_ARG
    assert _lib.lib().cflx_lu_solve(None, 0, B.ctypes.data, X.ctypes.data, None) == -1


def test_facade_lu_solve_compiles(tmp_path):
    lib = os.path.join(ROOT, "conflux_b200")
    if not os.path.exists(os.path.join(lib, "libconflux_b200.so")):
        pytest.skip("library not built")
    exe = tmp_path / "lu_solve_check"
    subprocess.check_call(["g++", "-std=c++17", "-O1", f"-I{ROOT}/include", f"{ROOT}/tests/cpp/lu_solve_check.cpp", "-o",
                           str(exe), f"-L{lib}", "-lconflux_b200", f"-Wl,-rpath,{lib}", "-lpthread"])
    n = ctypes.c_int()
    ctypes.CDLL(os.path.join(lib, "libconflux_b200.so")).cflx_device_count(ctypes.byref(n))
    if n.value == 0:
        out = subprocess.run([str(exe), "256"], capture_output=True, text=True)
        assert out.returncode != 0 and "no CPU fallback" in out.stderr
