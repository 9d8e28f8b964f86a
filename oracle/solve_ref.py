"""oracle/solve_ref.py -- TEST INFRASTRUCTURE (never imported by the product).

numpy restatement of the SCHEDULE of cflx_lu_solve (conflux_b200/csrc/solve.cu): the fan-in tile sweeps over the
Px x Py x Pz grid, rank by rank.  Every rank's work buffer W is simulated; the reductions over a grid row, the zeroing
of the non-root slots and the broadcasts over a grid column happen exactly where the CUDA path issues them, so the
per-rank X_local lists can be compared replica by replica.  Also the row / column layouts of right-hand sides and
solutions (next to oracle/layout.py's assemble / scatter of the matrix itself).
"""
import numpy as np
from scipy.linalg import solve_triangular

from . import layout


def scatter_rows(B, N, v, Px, Py, Pz):
    """Global B (M x nrhs, or M) -> per-rank B_local list in A's ROW distribution: global row g on grid row (g // v) % Px
    at local row (g // (v*Px))*v + g % v.  Every rank of a grid row gets its rows (they are read on pj == 0, pk == 0)."""
    d = layout.dims(N, v, Px, Py, Pz)
    B = np.asarray(B, dtype=np.float64)
    assert B.shape[0] == d["M"]
    out = []
    for r in range(d["P"]):
        pi = r // (Py * Pz)
        rows = [g for g in range(d["M"]) if (g // v) % Px == pi]
        loc = np.zeros((d["Ml"],) + B.shape[1:])
        loc[[(g // (v * Px)) * v + g % v for g in rows]] = B[rows]
        out.append(loc)
    return out


def gather_rows(B_locals, N, v, Px, Py, Pz):
    """Inverse of scatter_rows (reads the ranks pj == 0, pk == 0)."""
    d = layout.dims(N, v, Px, Py, Pz)
    first = np.asarray(B_locals[0])
    B = np.zeros((d["M"],) + first.shape[1:])
    for g in range(d["M"]):
        B[g] = B_locals[layout.rank_of((g // v) % Px, 0, 0, Px, Py, Pz)][(g // (v * Px)) * v + g % v]
    return B


def gather_cols(X_locals, N, v, Px, Py, Pz):
    """Per-rank X_local list (Nl x nrhs) in A's COLUMN distribution -> global X (M x nrhs).  Global row g lives on every
    rank with pj == (g // v) % Py (all pi, all pk) at local row (g // (v*Py))*v + g % v; the replicas must be bitwise
    equal (AssertionError otherwise)."""
    d = layout.dims(N, v, Px, Py, Pz)
    first = np.asarray(X_locals[0])
    X = np.zeros((d["N"],) + first.shape[1:])
    for pj in range(Py):
        ranks = [layout.rank_of(pi, pj, pk, Px, Py, Pz) for pi in range(Px) for pk in range(Pz)]
        ref = np.asarray(X_locals[ranks[0]])
        for r in ranks[1:]:
            assert np.array_equal(np.asarray(X_locals[r]), ref), f"replica on rank {r} differs from rank {ranks[0]}"
        for g in range(d["N"]):
            if (g // v) % Py == pj:
                X[g] = ref[(g // (v * Py)) * v + g % v]
    return X


def scatter_cols(X, N, v, Px, Py, Pz):
    """Global X (M x nrhs) -> the per-rank X_local list of the column distribution (every replica)."""
    d = layout.dims(N, v, Px, Py, Pz)
    X = np.asarray(X, dtype=np.float64)
    out = []
    for r in range(d["P"]):
        pj = (r // Pz) % Py
        loc = np.zeros((d["Nl"],) + X.shape[1:])
        for g in range(d["N"]):
            if (g // v) % Py == pj:
                loc[(g // (v * Py)) * v + g % v] = X[g]
        out.append(loc)
    return out


def solve(C_locals, perm, B_locals, N, v, Px=1, Py=1, Pz=1):
    """C_locals: per-rank factors in the conflux pivoted layout (cflx_lu_get_factors / restate.lu), perm: pivot history
    (pivoted row q = original row perm[q]), B_locals: per-rank B_local (Ml x nrhs, read on pj == 0, pk == 0).
    Returns the per-rank X_local list (Nl x nrhs)."""
    d = layout.dims(N, v, Px, Py, Pz)
    P, M, Ml, Nl, Nt = d["P"], d["M"], d["Ml"], d["Nl"], d["Nt"]
    ranks = [(r // (Py * Pz), (r // Pz) % Py, r % Pz) for r in range(P)]
    nrhs = np.asarray(B_locals[layout.rank_of(0, 0, 0, Px, Py, Pz)]).reshape(Ml, -1).shape[1]
    C = [np.asarray(c).reshape(Ml, Nl) if c is not None else None for c in C_locals]
    W = [np.zeros((Ml, nrhs)) for _ in range(P)]
    X = [np.zeros((Nl, nrhs)) for _ in range(P)]
    # P B inside grid column 0: pivoted row q = k*v + i to grid row k % Px, local row (k // Px)*v + i
    for q in range(M):
        g, k = int(perm[q]), q // v
        src = np.asarray(B_locals[layout.rank_of((g // v) % Px, 0, 0, Px, Py, Pz)]).reshape(Ml, nrhs)
        W[layout.rank_of(k % Px, 0, 0, Px, Py, Pz)][(k // Px) * v + q % v] = src[(g // (v * Px)) * v + g % v]

    def sweep(forward):
        for t in (range(Nt) if forward else range(Nt - 1, -1, -1)):
            pr, pc = t % Px, t % Py
            lr, lc = (t // Px) * v, (t // Py) * v
            root = layout.rank_of(pr, pc, 0, Px, Py, Pz)
            row = [r for r in range(P) if ranks[r][0] == pr]
            red = W[row[0]][lr:lr + v].copy()               # reduce over the grid row (jk_comm) to (pr, pc, 0)
            for r in row[1:]:
                red += W[r][lr:lr + v]
            D = C[root][lr:lr + v, lc:lc + v]
            if forward:
                tile = solve_triangular(D, red, lower=True, unit_diagonal=True)
                for r in row:
                    W[r][lr:lr + v] = tile if r == root else 0.0
            else:
                tile = solve_triangular(D, red, lower=False)
            for r in range(P):                              # broadcast over the grid column (ik_comm), every layer
                if ranks[r][1] == pc:
                    X[r][lc:lc + v] = tile
                    if ranks[r][2] != 0:
                        continue
                    pi = ranks[r][0]
                    if forward:                             # local rows of the tiles below t: W -= L[., t] Y_t
                        lo = min(Ml, (t + 1 - pi + Px - 1) // Px * v)
                        W[r][lo:] -= C[r][lo:, lc:lc + v] @ tile
                    else:                                   # local rows of the tiles above t: W -= U[., t] X_t
                        hi = min(Ml, (t - pi + Px - 1) // Px * v)
                        W[r][:hi] -= C[r][:hi, lc:lc + v] @ tile

    sweep(True)
    sweep(False)
    return X
