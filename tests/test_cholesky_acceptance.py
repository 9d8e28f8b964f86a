"""CPU: the acceptance bars of the Cholesky tests (oracle/chol_ref.py) can tell a correct factorisation from a subtly wrong
one.  They are applied to a numpy model of the tiled right-looking Cholesky of chol.cu (N=1024, v=256): exact, and with
the rank-v update rounded to 48 or 44 significant bits, or with the update's operand rows scaled by the exponent of the
neighbouring row.  Also checks the input builders the GPU tests rely on."""
import numpy as np
import pytest
import scipy.linalg.lapack

from oracle import chol_ref as C

N, V = 1024, 256


@pytest.fixture(scope="module")
def S():
    return C.spd_random(N, 1)


def test_exact_model_is_accepted(S):
    ok, m = C.acceptance(S, C.tiled_model(S, V))
    assert ok, m


def test_48_bit_update_is_accepted(S):
    ok, m = C.acceptance(S, C.tiled_model(S, V, bits=48))
    assert ok, m


def test_44_bit_update_is_rejected_on_both_bars(S):
    _, m = C.acceptance(S, C.tiled_model(S, V, bits=44))
    assert m["backward"] > 2 * C.BACKWARD_BAR and m["forward"] > 2 * C.FORWARD_BAR, m


def test_reference_generator_cannot_tell_a_44_bit_update():
    """why the general inputs exist: on the generator's matrix a 44-bit update stays under the old elementwise bar"""
    A, _, _ = C.init_matrix(N, V)
    S = C.lower_sym(A)
    L = C.tiled_model(S, V, bits=44)
    Lref = np.linalg.cholesky(S)
    assert np.abs(L - Lref).max() <= 8e-12 * np.abs(Lref).max()


def test_misindexed_row_exponent_fails_equivariance_only(S):
    e = C.grade_exponents(N, 2)
    L = C.tiled_model(S, V)
    assert C.equivariant(C.tiled_model(C.grade(S, e), V), L, e)
    Lbad = C.tiled_model(S, V, exp_from_neighbour=True)
    assert C.acceptance(S, Lbad)[0]                        # the precision bars do not see it ...
    assert not C.equivariant(C.tiled_model(C.grade(S, e), V, exp_from_neighbour=True), Lbad, e)   # ... this does


def test_48_bit_update_is_still_equivariant(S):
    """rounding to significant bits scales with the input: equivariance tests indexing, not precision"""
    e = C.grade_exponents(N, 3)
    assert C.equivariant(C.tiled_model(C.grade(S, e), V, bits=48), C.tiled_model(S, V, bits=48), e)


def test_spd_random_conditioning():
    w = np.linalg.eigvalsh(C.spd_random(512, 4))
    assert 40 < w[-1] / w[0] < 120
    S = C.spd_random(256, 5)
    assert np.array_equal(S, S.T)
    assert not np.array_equal(S[:64, :64], S[64:128, 64:128])          # tiles differ


@pytest.mark.parametrize("n", [4, 100, 512, 4096])
def test_spd_exact_factor_is_exact(n):
    S, L0 = C.spd_exact(n, seed=n)
    assert np.abs(S).max() < 2.0 ** 53 and np.array_equal(S, S.T)
    assert np.array_equal(np.tril(L0 @ L0.T), np.tril(S))
    if n <= 512:
        L, info = scipy.linalg.lapack.dpotrf(S, lower=1)
        assert info == 0 and np.array_equal(np.tril(L), L0)
        assert np.linalg.cond(S) <= 30


def test_grade_scales_the_factor_exactly():
    S, L0 = C.spd_exact(256, seed=1)
    e = C.grade_exponents(256, 1)
    assert e.min() >= -20 and e.max() <= 20 and len(set(e.tolist())) > 20
    G = C.grade(S, e)
    L, info = scipy.linalg.lapack.dpotrf(G, lower=1)
    assert info == 0 and C.equivariant(L, L0, e)


@pytest.mark.parametrize("c", [0, 1, 31, 128, 300, 1023])
def test_not_pd_first_failing_column(c):
    S, L0 = C.spd_exact(1024, seed=7)
    _, info = scipy.linalg.lapack.dpotrf(C.not_pd(S, L0, c), lower=1)
    assert info == c + 1
