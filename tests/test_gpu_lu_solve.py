"""GPU: LU_solve / cflx_lu_solve -- A X = B with the factors of the last LU_rep, on 1-8 GPUs, against the host
(normwise backward error), the numpy restatement of the tile schedule (oracle/solve_ref.py) on the GPU's own factors,
and its own state rules."""
import os
import subprocess

import numpy as np
import pytest
import scipy.linalg

import conflux_b200 as cb
from oracle import layout, solve_ref
from tests._harness import n_gpus, run_ranks
from tests.test_gpu_lu import GRIDS

pytestmark = pytest.mark.gpu
RESIDUAL_TOL = 1e-12      # BASELINE.json's bar, here on ||B - A X||_F / (||A||_F ||X||_F)
SCHEDULE_TOL = 1e-11      # X against solve_ref on the same factors, relative max-norm
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rhs(M, nrhs, seed=7):
    return np.random.default_rng(seed).standard_normal((M, nrhs))


def gpu_solve(N, v, Px, Py, Pz, nrhs_list):
    """Factor the seeded matrix on the grid and solve for each nrhs in turn.  Returns dict(A, C, perm, X={nrhs: [per
    rank X_local]}, ms={nrhs: max ms}, dims)."""
    d = layout.dims(N, v, Px, Py, Pz)
    Bs = {n: solve_ref.scatter_rows(_rhs(d["M"], n), N, v, Px, Py, Pz) for n in nrhs_list}

    def body(comm):
        gv = cb.lu_params(N, N, v, Px, Py, Pz, comm)
        C = np.zeros((gv.Ml, gv.Nl))
        perm = np.zeros(gv.M, dtype=np.int32)
        cb.LU_rep(gv, C, perm)
        out = dict(A=gv.data.copy(), C=C, perm=perm, X={}, ms={})
        for n in nrhs_list:
            out["X"][n], out["ms"][n] = cb.LU_solve(gv, Bs[n][gv.rank])
        gv.free_comms()
        return out

    rs = run_ranks(d["P"], body)
    return dict(A=[r["A"] for r in rs], C=[r["C"] for r in rs], perm=rs[0]["perm"], dims=d,
                X={n: [r["X"][n] for r in rs] for n in nrhs_list}, ms={n: max(r["ms"][n] for r in rs) for n in nrhs_list})


def backward_error(A, X, B):
    return float(np.linalg.norm(B - A @ X) / (np.linalg.norm(A) * np.linalg.norm(X)))


def _check(N, v, Px, Py, Pz, nrhs_list):
    if n_gpus() < Px * Py * Pz:
        pytest.skip(f"needs {Px * Py * Pz} GPUs")
    g = gpu_solve(N, v, Px, Py, Pz, nrhs_list)
    A = layout.assemble(g["A"], N, v, Px, Py, Pz)
    for n in nrhs_list:
        X = solve_ref.gather_cols(g["X"][n], N, v, Px, Py, Pz)    # every replica (all pi, all pk) bitwise equal
        B = _rhs(A.shape[0], n)
        assert backward_error(A, X, B) <= RESIDUAL_TOL, (N, v, n)
        ref = solve_ref.gather_cols(solve_ref.solve(g["C"], g["perm"], solve_ref.scatter_rows(B, N, v, Px, Py, Pz), N, v,
                                                     Px, Py, Pz), N, v, Px, Py, Pz)
        assert np.abs(X - ref).max() <= SCHEDULE_TOL * np.abs(ref).max(), (N, v, n)
    return g


@pytest.mark.parametrize("N,v", [(64, 8), (256, 32), (1024, 128), (768, 256), (100, 16)])
def test_single_gpu_solves(N, v):
    _check(N, v, 1, 1, 1, [1, 3, 64, 300])


@pytest.mark.parametrize("N,v,Px,Py,Pz", GRIDS)
def test_multi_gpu_solves(N, v, Px, Py, Pz):
    _check(N, v, Px, Py, Pz, [1, 3, 64])


def test_skinny_and_wide_updates_agree():
    """nrhs = 1 runs the bandwidth-bound update kernel, nrhs = 64 the DMMA GEMM: the same column agrees."""
    g = gpu_solve(1024, 128, 1, 1, 1, [64])
    B = _rhs(1024, 64)
    comm = cb.Comm(1, 0, None, 0)
    gv = cb.lu_params(1024, 1024, 128, 1, 1, 1, comm)
    cb.LU_rep(gv)
    x1, _ = cb.LU_solve(gv, np.ascontiguousarray(B[:, :1]))
    gv.free_comms()
    comm.close()
    wide = g["X"][64][0][:, 0]
    assert np.abs(x1[:, 0] - wide).max() <= 1e-13 * np.abs(wide).max()


def test_solve_state_rules():
    comm = cb.Comm(1, 0, None, 0)
    gv = cb.lu_params(512, 512, 64, 1, 1, 1, comm)
    B = _rhs(gv.M, 4)
    with pytest.raises(cb.ConfluxError):
        cb.LU_solve(gv, B)                                        # before any factorisation
    C0, p0 = np.zeros((gv.Ml, gv.Nl)), np.zeros(gv.M, dtype=np.int32)
    cb.LU_rep(gv, C0, p0)
    v0 = cb.validate(gv)
    x1, _ = cb.LU_solve(gv, B)
    x2, _ = cb.LU_solve(gv, B)
    assert np.array_equal(x1, x2)                                 # a second solve is bitwise the first
    C1, p1 = np.zeros((gv.Ml, gv.Nl)), np.zeros(gv.M, dtype=np.int32)
    cb._lib.check(cb._lib.lib().cflx_lu_get_factors(gv._h, C1.ctypes.data, p1.ctypes.data), "get_factors")
    assert np.array_equal(C0, C1) and np.array_equal(p0, p1)      # the solve left the factors as they were
    v1 = cb.validate(gv)                                          # (its norms are summed with atomics: last-bit noise)
    assert abs(v1[1] - v0[1]) <= 1e-6 * v0[1] and v1[1] <= RESIDUAL_TOL
    assert backward_error(gv.data, x1, B) <= RESIDUAL_TOL
    a = np.ascontiguousarray(gv.data)
    cb._lib.check(cb._lib.lib().cflx_lu_set_local(gv._h, a.ctypes.data), "set_local")
    with pytest.raises(cb.ConfluxError):
        cb.LU_solve(gv, B)                                        # re-uploaded input, not factored yet
    with pytest.raises(AssertionError):
        cb.LU_solve(gv, np.asfortranarray(B))                     # layout checked like LU_rep
    gv.free_comms()
    comm.close()


def test_streamed_factorisation_solves_the_factored_matrix():
    comm = cb.Comm(1, 0, None, 0)
    gv = cb.lu_params(1024, 1024, 128, 1, 1, 1, comm)
    rng = np.random.default_rng(3)
    first, nxt = gv.data.copy(), cb.pinned_empty((gv.Ml, gv.Nl))
    nxt[...] = rng.standard_normal((gv.Ml, gv.Nl))
    B = _rhs(gv.M, 2)
    cb.LU_rep(gv, next_data=nxt)                                  # factors `first`, uploads `nxt` behind it
    x, _ = cb.LU_solve(gv, B)
    assert backward_error(first, x, B) <= RESIDUAL_TOL
    assert np.abs(x - np.linalg.solve(first, B)).max() <= 1e-9 * np.abs(x).max()
    cb.LU_rep(gv, upload=False)                                   # now the queued matrix
    y, _ = cb.LU_solve(gv, B)
    assert backward_error(np.asarray(nxt), y, B) <= RESIDUAL_TOL
    cb.pinned_free(nxt)
    gv.free_comms()
    comm.close()


def test_larger_solve_on_the_tcgen05_factors():
    comm = cb.Comm(1, 0, None, 0)
    gv = cb.lu_params(4096, 4096, 256, 1, 1, 1, comm)
    assert cb._lib.lib().cflx_lu_uses_tcgen05(gv._h) == 1
    cb.LU_rep(gv)
    B = _rhs(gv.M, 16)
    x, ms = cb.LU_solve(gv, B)
    assert backward_error(gv.data, x, B) <= RESIDUAL_TOL and ms > 0
    gv.free_comms()
    comm.close()


@pytest.mark.parametrize("v", [64, 256, 512])
def test_trsm_left_upper_kernel(v):
    rng = np.random.default_rng(v)
    A00 = rng.standard_normal((v, v)) + v * np.eye(v)
    R = rng.standard_normal((v, 37))
    X = cb.dbg.trsm_left_upper(A00, R)
    want = scipy.linalg.solve_triangular(np.triu(A00), R, lower=False)
    assert np.abs(X - want).max() <= 1e-12 * np.abs(want).max()


def test_cpp_facade_lu_solve(tmp_path):
    lib = os.path.join(ROOT, "conflux_b200")
    exe = tmp_path / "lu_solve_check"
    subprocess.check_call(["g++", "-std=c++17", "-O1", f"-I{ROOT}/include", f"{ROOT}/tests/cpp/lu_solve_check.cpp", "-o",
                           str(exe), f"-L{lib}", "-lconflux_b200", f"-Wl,-rpath,{lib}", "-lpthread"])
    out = subprocess.run([str(exe), "256"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    berr = float(out.stdout.split("backward_error=")[1].split()[0])
    assert berr <= RESIDUAL_TOL
