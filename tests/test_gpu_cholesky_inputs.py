"""GPU: the Cholesky path (conflux_b200/csrc/chol.cu) on general SPD inputs, not just the reference's generator.

Inputs (oracle/chol_ref.py): spd_random (cond ~ 80, every tile different: the precision check), spd_exact (an exact
integer factor: wiring and indexing), grade (D S D with D = diag(2^e): the factor must be D L(S) bit for bit, which checks
the per-row / per-column exponents of the tcgen05 digit planes) and not_pd (a known first failing column).

Bars: backward error ||S - L L^T||_F / ||S||_F <= 2e-15 and <= 8x LAPACK's; forward error against LAPACK <= 4e-15.  A
numpy model whose update keeps 44 bits fails both (tests/test_cholesky_acceptance.py).  Run with -s to see the measured
errors (lines starting with "chol-errors")."""
import re

import numpy as np
import pytest

import conflux_b200 as cb
from oracle import chol_ref as C
from tests.test_gpu_cholesky import _run

pytestmark = pytest.mark.gpu

ONE_CTA_V = [4, 8, 12, 20, 32, 36, 60, 64, 100, 128, 160, 252, 256, 384, 448, 512]
BLOCKED_V = [256, 384, 512]
TILE_PATHS = [pytest.param(v, False, id=f"onecta-{v}") for v in ONE_CTA_V] + \
             [pytest.param(v, True, id=f"blocked-{v}") for v in BLOCKED_V]


def _report(what, **m):
    print("chol-errors " + what + " " + " ".join(f"{k}={v:.3g}" for k, v in m.items()))


def _assert_bars(S, L, what):
    ok, m = C.acceptance(S, L)
    _report(what, **m)
    assert ok, (what, m)


def _nan_upper(S):
    X = np.tril(S)
    X[np.triu_indices(len(S), 1)] = np.nan
    return X


# ------------------------------------------------------------------------------------------ the diagonal-tile kernels
@pytest.mark.parametrize("v,blocked", TILE_PATHS)
def test_potrf_tile_exact_factor_and_triangles(v, blocked):
    S, L0 = C.spd_exact(v, seed=v)
    L, LT, info = cb.dbg.potrf_tile(S, blocked)
    assert info == 0
    assert np.abs(L - L0).max() <= 1e-14 * np.abs(L0).max()
    assert not np.triu(L, 1).any()                       # exactly zero above the diagonal
    assert np.array_equal(LT, L.T)                       # L^T written everywhere (it starts as NaN)


@pytest.mark.parametrize("v,blocked", TILE_PATHS)
def test_potrf_tile_random_spd(v, blocked):
    S = C.spd_random(v, 100 + v)
    L, LT, info = cb.dbg.potrf_tile(S, blocked)
    assert info == 0 and np.array_equal(LT, L.T) and not np.triu(L, 1).any()
    _assert_bars(S, L, f"tile {'blocked' if blocked else 'onecta'} v={v}")
    # graded input: every operation scales exactly by powers of two
    e = C.grade_exponents(v, v)
    Lg, LTg, info = cb.dbg.potrf_tile(C.grade(S, e), blocked)
    assert info == 0 and C.equivariant(Lg, L, e)
    # the strict upper triangle is never read
    Ln, LTn, info = cb.dbg.potrf_tile(_nan_upper(S), blocked)
    assert info == 0 and np.array_equal(Ln, L) and np.array_equal(LTn, LT)


@pytest.mark.parametrize("v", BLOCKED_V)
def test_potrf_tile_paths_agree(v):
    S = C.spd_random(v, 7 * v)
    L0, _, _ = cb.dbg.potrf_tile(S, False)
    L1, _, _ = cb.dbg.potrf_tile(S, True)
    assert np.linalg.norm(L0 - L1) / np.linalg.norm(L0) <= C.BACKWARD_BAR


@pytest.mark.parametrize("v,blocked", TILE_PATHS)
def test_potrf_tile_reports_first_failing_column(v, blocked):
    S, L0 = C.spd_exact(v, seed=v + 1)
    for c in [c for c in (0, 1, 31, 32, 33, 127, 128, 129, 255, 300, v - 1) if c < v]:
        _, _, info = cb.dbg.potrf_tile(C.not_pd(S, L0, c), blocked)
        assert info == c + 1, (v, blocked, c, info)


def test_potrf_tile_refuses_unsupported_shapes():
    with pytest.raises(cb.ConfluxError, match="status"):
        cb.dbg.potrf_tile(np.eye(128), True)             # blocked needs v >= 256
    with pytest.raises(cb.ConfluxError, match="status"):
        cb.dbg.potrf_tile(np.eye(6), False)              # v % 4 != 0
    with pytest.raises(cb.ConfluxError, match="status"):
        cb.dbg.potrf_tile(np.eye(516), False)            # v > 512


# ------------------------------------------------------------------------------------------ the factorisation
SINGLE = [(480, 48), (400, 100), (512, 128), (1024, 256), (1536, 384), (2048, 512), (4096, 512)]


def _path(v, Pz, dmma):
    tile = "blocked" if v % 128 == 0 and v >= 256 else "onecta"
    upd = "tcgen05" if not dmma and (v // Pz) % 128 == 0 else "dmma"
    return f"{tile}/{upd}"


def _check_random_graded_determinism(N, v, grid, dmma, check_validate):
    what = f"N={N} v={v} grid={'x'.join(map(str, grid))} {_path(v, grid[2], dmma)}"
    S = C.spd_random(N, N + v)
    _, L, rs = _run(N, v, grid, A_global=np.tril(S), twice=True)
    _assert_bars(S, L, what)
    assert np.array_equal(rs[0]["L2g"], L), "two factorisations of the same input differ"
    if check_validate:
        host = np.linalg.norm(np.tril(S - L @ L.T)) / np.linalg.norm(np.tril(S))
        assert 0.1 * host <= rs[0]["resid"][1] <= 10 * host, (rs[0]["resid"], host)
    assert all(r["resid"] == rs[0]["resid"] for r in rs)
    e = C.grade_exponents(N, N - v)
    _, Lg, _ = _run(N, v, grid, A_global=np.tril(C.grade(S, e)))
    assert C.equivariant(Lg, L, e), f"{what}: L(DSD) != D L(S), first mismatch in row " \
        f"{int(np.argwhere(Lg != np.ldexp(L, e[:, None]))[0][0])}"
    return S, L


@pytest.mark.parametrize("dmma", [False, True], ids=["default", "dmma"])
@pytest.mark.parametrize("N,v", SINGLE)
def test_single_gpu_general_inputs(N, v, dmma, monkeypatch):
    if dmma:
        monkeypatch.setenv("CFLX_GEMM", "dmma")          # read in cflx_chol_create
    S, L = _check_random_graded_determinism(N, v, (1, 1, 1), dmma, check_validate=True)
    # the strict upper triangle is never read: NaN there, or the full symmetric matrix, give the same factor
    _, Ln, _ = _run(N, v, (1, 1, 1), A_global=_nan_upper(S))
    assert np.array_equal(Ln, L)
    _, Ls, _ = _run(N, v, (1, 1, 1), A_global=S)
    assert np.array_equal(Ls, L)
    # exact truth
    Se, L0 = C.spd_exact(N, seed=v)
    _, Le, _ = _run(N, v, (1, 1, 1), A_global=np.tril(Se))
    assert np.abs(Le - L0).max() <= 1e-14 * np.abs(L0).max()


MULTI = [(256, 32, (2, 1, 1)), (256, 32, (1, 1, 2)), (512, 64, (2, 2, 1)), (512, 64, (2, 2, 2)), (1024, 128, (4, 2, 1)),
         (768, 64, (2, 1, 2)), (2048, 256, (2, 1, 1)), (2048, 512, (2, 2, 1)), (2048, 256, (2, 2, 2)), (2048, 512, (2, 1, 2)),
         (4096, 512, (4, 2, 1))]


@pytest.mark.parametrize("N,v,grid", MULTI)
def test_multi_gpu_general_inputs(N, v, grid):
    _check_random_graded_determinism(N, v, grid, False, check_validate=False)


# ------------------------------------------------------------------------------------------ not positive definite
def _column_in(msg):
    m = re.search(r"column (\d+)\b", msg)
    return int(m.group(1)) if m else None


@pytest.mark.parametrize("c", [5, 300, 700])
def test_not_positive_definite_names_the_first_failing_column(c):
    N, v = 1024, 256
    S, L0 = C.spd_exact(N, seed=c)
    _, _, rs = _run(N, v, (1, 1, 1), A_global=np.tril(C.not_pd(S, L0, c)), catch=True)
    msg = rs[0].get("error", "")
    assert "positive definite" in msg and _column_in(msg) == c + 1, msg


@pytest.mark.parametrize("grid", [(2, 1, 1), (2, 2, 1)])
def test_not_positive_definite_is_reported_on_every_rank(grid):
    N, v = 1024, 256
    for c in (300, 700):
        S, L0 = C.spd_exact(N, seed=c)
        _, _, rs = _run(N, v, grid, A_global=np.tril(C.not_pd(S, L0, c)), catch=True)
        msgs = [r.get("error", "") for r in rs]
        assert all("positive definite" in m for m in msgs), msgs
        assert [_column_in(m) for m in msgs] == [c + 1] * len(rs), msgs
