"""oracle/chol_ref.py -- TEST INFRASTRUCTURE: CPU oracle of the CONFCHOX path.
  * assemble(): local conflux-layout shares -> the global matrix (same tile map as the LU path, oracle/layout.py);
  * reference factor = numpy.linalg.cholesky (LAPACK dpotrf, lower) of the assembled input, which is exactly what the
    reference's own checker compares against (examples/cholesky_helper.cpp:183-217: LAPACKE_dpotrf(ROW_MAJOR, 'L'));
  * init_matrix(): restatement of CholeskyIO::generateInputMatrixDistributed (CholeskyIO.cpp:100-172) with glibc's rand()
    through ctypes (srand(1)), for checking the library's generator."""
import ctypes

import numpy as np


def dims(N, v, Px, Py, Pz):
    K = -(-N // v)
    return dict(N=K * v, Kappa=K, Ml=-(-K // Px) * v, Nl=-(-K // Py) * v, P=Px * Py * Pz)


def assemble(locals_, N, v, Px, Py, Pz):
    d = dims(N, v, Px, Py, Pz)
    A = np.zeros((d["N"], d["N"]))
    for r, loc in enumerate(locals_):
        if r % Pz or loc is None:
            continue
        pi, pj = r // (Py * Pz), (r // Pz) % Py
        loc = np.asarray(loc).reshape(d["Ml"], d["Nl"])
        for lti in range(d["Ml"] // v):
            for ltj in range(d["Nl"] // v):
                gi, gj = lti * Px + pi, ltj * Py + pj
                if gi < d["Kappa"] and gj < d["Kappa"]:
                    A[gi * v:(gi + 1) * v, gj * v:(gj + 1) * v] = loc[lti * v:(lti + 1) * v, ltj * v:(ltj + 1) * v]
    return A


def lower_sym(A):
    """the symmetric matrix whose lower triangle is the lower triangle of A"""
    L = np.tril(A)
    return L + np.tril(A, -1).T


def init_matrix(N, v):
    """global lower triangle as the reference generates it (every tile = lower(R^T R), strengthened diagonal)"""
    libc = ctypes.CDLL(None)
    libc.srand(1)
    libc.rand.restype = ctypes.c_int
    RAND_MAX = 2147483647
    R = np.array([libc.rand() / RAND_MAX * 2 - 1 for _ in range(v * v)]).reshape(v, v)
    T = np.tril(R.T @ R)
    K = -(-N // v)
    mx = np.abs(T).sum(axis=1).max() * K * 2
    A = np.zeros((K * v, K * v))
    for i in range(K):
        for j in range(i + 1):
            A[i * v:(i + 1) * v, j * v:(j + 1) * v] = T
        A[i * v:(i + 1) * v, i * v:(i + 1) * v][np.diag_indices(v)] = mx
    return A, T, mx


# ---------------------------------------------------------------------------------------------------------------------
# General SPD inputs and the acceptance bars of the Cholesky path.  The generator above makes every tile the same and the
# diagonal dominant, so L is nearly diagonal and the rank-v update carries little of the answer; these inputs do not.

BACKWARD_BAR = 2e-15      # ||S - L L^T||_F / ||S||_F
LAPACK_FACTOR = 8.0       # ... and at most this many times LAPACK's on the same S
FORWARD_BAR = 4e-15       # ||L - L_lapack||_F / ||L_lapack||_F on spd_random (cond ~ 80)


def spd_random(N, seed):
    """M M^T / N + 0.05 I with M standard normal: cond ~ 80, every tile different."""
    M = np.random.default_rng(seed).standard_normal((N, N))
    S = M @ M.T / N + 0.05 * np.eye(N)
    return (S + S.T) / 2                                     # exactly symmetric


def spd_exact(N, d=64, seed=0):
    """(S, L0): S = L0 L0^T with L0 = d I plus strictly-lower integers in {-1, 0, 1}.  Every entry of S is an integer
    below 2^53 (N <= 4096 at d = 64), so S is exact in FP64, and L0 is its exact Cholesky factor (cond(S) <= 30).  An
    exact truth for wiring and indexing; it cannot show lost precision (the update is exact in few bits)."""
    rng = np.random.default_rng(seed)
    L0 = np.tril(rng.integers(-1, 2, size=(N, N)), -1).astype(np.float64) + d * np.eye(N)
    return L0 @ L0.T, L0


def grade_exponents(N, seed):
    return np.random.default_rng(seed).integers(-20, 21, size=N)


def grade(S, e):
    """D S D with D = diag(2^e_i): its Cholesky factor is exactly D L(S), row i scaled by 2^e_i."""
    e = np.asarray(e)
    return np.ldexp(np.ldexp(S, e[:, None]), e[None, :])


def not_pd(S, L0, c):
    """S with the pivot of column c made -L0[c,c]^2: the leading minors of order <= c are unchanged, so the first failing
    column (dpotrf's info) is exactly c + 1."""
    S = S.copy()
    S[c, c] -= 2 * L0[c, c] ** 2
    return S


def backward_error(S, L):
    L = np.tril(L)
    return float(np.linalg.norm(S - L @ L.T) / np.linalg.norm(S))


def forward_error(L, Lref):
    return float(np.linalg.norm(np.tril(L) - Lref) / np.linalg.norm(Lref))


def acceptance(S, L, check_forward=True):
    """(ok, measured) of a factor L of S against the bars: backward error <= BACKWARD_BAR and <= LAPACK_FACTOR times
    LAPACK's, forward error against LAPACK <= FORWARD_BAR (on well-conditioned inputs such as spd_random)."""
    Lref = np.linalg.cholesky(S)
    m = dict(backward=backward_error(S, L), lapack_backward=backward_error(S, Lref), forward=forward_error(L, Lref))
    ok = m["backward"] <= BACKWARD_BAR and m["backward"] <= LAPACK_FACTOR * max(m["lapack_backward"], 1e-17)
    if check_forward:
        ok = ok and m["forward"] <= FORWARD_BAR
    return ok, m


def equivariant(L_graded, L, e):
    """L(D S D) == D L(S) bit for bit (every operation of a correct factorisation scales exactly by powers of two)."""
    return np.array_equal(np.tril(L_graded), np.ldexp(np.tril(L), np.asarray(e)[:, None]))


def _round_significant(X, bits):
    """every entry of X to `bits` significant bits"""
    m, E = np.frexp(X)
    return np.ldexp(np.round(np.ldexp(m, bits)), E - bits)


def _round_rows_to_neighbour_exponent(X, bits=52):
    """rows of X to `bits` bits below a power of two per row, the exponent of the largest entry of the NEXT row: digit
    planes whose per-row exponent is read one row off"""
    _, E = np.frexp(np.abs(X).max(axis=1))
    E = np.concatenate([E[1:], E[-1:]])
    step = np.ldexp(1.0, E - bits)[:, None]
    return np.round(X / step) * step


def tiled_model(S, v, bits=None, exp_from_neighbour=False):
    """numpy model of the tiled right-looking Cholesky of chol.cu: LAPACK on the diagonal tile, triangular solve of the
    tile column, rank-v update of the trailing matrix.  bits: the update is rounded to that many significant bits before
    it is subtracted (None = exact FP64); exp_from_neighbour: the update's operand rows are kept to 52 bits below the
    exponent of the neighbouring row instead of their own."""
    import scipy.linalg
    A = np.tril(S).copy()
    N = A.shape[0]
    for k in range(0, N, v):
        e = min(k + v, N)
        A[k:e, k:e] = np.linalg.cholesky(lower_sym(A[k:e, k:e]))
        if e == N:
            break
        A[e:, k:e] = scipy.linalg.solve_triangular(A[k:e, k:e], A[e:, k:e].T, lower=True).T
        X = A[e:, k:e]
        if exp_from_neighbour:
            X = _round_rows_to_neighbour_exponent(X)
        upd = np.tril(X @ X.T)
        if bits is not None:
            upd = _round_significant(upd, bits)
        A[e:, e:] -= upd
    return np.tril(A)
