"""GPU: the CONFCHOX path (conflux_b200/csrc/chol.cu) through the reference-facing interface against the oracle the
reference's own checker uses (LAPACK dpotrf on the assembled matrix, examples/cholesky_helper.cpp:183-217), on the
reference's generated input, on single- and multi-rank grids; plus the grid-wide device residual."""
import numpy as np
import pytest

import conflux_b200 as cb
from oracle import chol_ref
from tests._harness import n_gpus, run_ranks

pytestmark = pytest.mark.gpu


def _run(N, v, grid, A_global=None, twice=False, catch=False):
    """Factor A_global (default: the reference's generator) on the grid.  Returns (A, L, per-rank results).
    twice: factor a second time without uploading again, L of that run in r["L2"] (assembled: r["L2g"] of rank 0).
    catch: a ConfluxError of parallelCholesky() is returned as r["error"] on each rank (A and L are then None)."""
    P = grid[0] * grid[1] * grid[2]
    if n_gpus() < P:
        pytest.skip(f"needs {P} GPUs")

    def body(comm):
        ch = cb.cholesky.initialize(N, v, grid, comm)
        if A_global is not None and ch.pz == 0:
            for lti in range(ch.Ml // v):
                for ltj in range(ch.Nl // v):
                    gi, gj = lti * ch.PX + ch.px, ltj * ch.PY + ch.py
                    if gi < ch.Kappa and gj < ch.Kappa:
                        ch.data[lti * v:(lti + 1) * v, ltj * v:(ltj + 1) * v] = A_global[gi * v:(gi + 1) * v, gj * v:(gj + 1) * v]
        try:
            ms = ch.parallelCholesky()
        except cb.ConfluxError as e:
            if not catch:
                raise
            ch.finalize()
            return dict(error=str(e), rank=ch.rank)
        res = dict(A=ch.data.copy(), L=ch.local_factor() if ch.pz == 0 else None, resid=ch.validate(), ms=ms, rank=ch.rank)
        if twice:
            ch.parallelCholesky(upload=False)
            res["L2"] = ch.local_factor() if ch.pz == 0 else None
        ch.finalize()
        return res

    rs = run_ranks(P, body)
    if any("error" in r for r in rs):
        return None, None, rs
    A = chol_ref.assemble([r["A"] for r in rs], N, v, *grid)
    L = np.tril(chol_ref.assemble([r["L"] for r in rs], N, v, *grid))
    if twice:
        rs[0]["L2g"] = np.tril(chol_ref.assemble([r["L2"] for r in rs], N, v, *grid))
    return A, L, rs


@pytest.mark.parametrize("N,v,grid", [(64, 16, (1, 1, 1)), (256, 32, (1, 1, 1)), (512, 128, (1, 1, 1)), (1024, 256, (1, 1, 1)),
                                      (2048, 512, (1, 1, 1)), (100, 16, (1, 1, 1))])
def test_cholesky_single_gpu_matches_lapack(N, v, grid):
    A, L, rs = _run(N, v, grid)
    S = chol_ref.lower_sym(A)
    Lref = np.linalg.cholesky(S)
    assert np.abs(L - Lref).max() <= 1e-12 * np.abs(Lref).max() * 8
    assert np.linalg.norm(S - L @ L.T) / np.linalg.norm(S) <= 1e-14
    assert rs[0]["resid"][1] <= 1e-14


def test_cholesky_generator_is_the_references():
    N, v = 96, 16
    comm = cb.Comm(1, 0, None, 0)
    ch = cb.cholesky.initialize(N, v, (1, 1, 1), comm)
    A, T, mx = chol_ref.init_matrix(N, v)
    assert np.allclose(np.tril(ch.data), A, rtol=1e-15, atol=1e-15)       # dsyrk summation order may differ in the last bit
    assert np.array_equal(np.diag(ch.data), np.diag(A)) or np.allclose(np.diag(ch.data), np.diag(A), rtol=1e-15)
    ch.finalize()
    comm.close()


def test_cholesky_random_spd_input():
    rng = np.random.default_rng(3)
    N, v = 384, 64
    M = rng.standard_normal((N, N))
    S = M @ M.T + N * np.eye(N)
    A, L, rs = _run(N, v, (1, 1, 1), A_global=S)
    Lref = np.linalg.cholesky(S)
    assert np.abs(L - Lref).max() <= 1e-11 * np.abs(Lref).max()


def test_cholesky_not_positive_definite_is_reported():
    comm = cb.Comm(1, 0, None, 0)
    ch = cb.cholesky.initialize(64, 16, (1, 1, 1), comm)
    ch.data[...] = -np.eye(64)
    with pytest.raises(cb.ConfluxError, match="positive definite"):
        ch.parallelCholesky()
    ch.finalize()
    comm.close()


@pytest.mark.parametrize("N,v,grid", [(256, 32, (2, 1, 1)), (256, 32, (1, 1, 2)), (512, 64, (2, 2, 1)), (512, 64, (2, 2, 2)),
                                      (1024, 128, (4, 2, 1)), (768, 64, (2, 1, 2))])
def test_cholesky_multi_gpu_matches_lapack(N, v, grid):
    A, L, rs = _run(N, v, grid)
    S = chol_ref.lower_sym(A)
    Lref = np.linalg.cholesky(S)
    assert np.abs(L - Lref).max() <= 1e-12 * np.abs(Lref).max() * 8
    assert all(r["resid"] == rs[0]["resid"] for r in rs) and rs[0]["resid"][1] <= 1e-14
