"""CPU: the restatement oracle against what the reference's own LU_rep produced (oracle/_ref/libref_lu.so built by
oracle/build_ref.sh, ranks = threads) on the same grids, stored in tests/golden/lu_ref_cases.npz by
tests/golden/make_golden.py: a digest of the generated input, the permutation and a seeded sample of the factors."""
import hashlib
import os

import numpy as np
import pytest

from oracle import layout, restate

CASES = [(48, 4, 1, 1, 1), (128, 16, 2, 2, 1), (128, 8, 2, 2, 2), (96, 16, 1, 1, 2), (72, 4, 3, 3, 2), (256, 32, 4, 4, 1)]


@pytest.fixture(scope="module")
def G(golden_dir):
    return np.load(os.path.join(golden_dir, "lu_ref_cases.npz"))


@pytest.mark.parametrize("case", CASES)
def test_matches_live_reference(case, G):
    i = [tuple(int(x) for x in c) for c in G["cases"]].index(case)
    N, v, Px, Py, Pz = case
    A0 = restate.init_matrix(N, v, Px, Py, Pz)
    # generator is bit-identical to lu_params::InitMatrix
    assert hashlib.sha256(np.ascontiguousarray(np.stack(A0)).tobytes()).hexdigest() == str(G[f"c{i}_A_sha256"])
    o = restate.lu(A0, N, v, Px, Py, Pz)
    assert np.array_equal(o["perm"], G[f"c{i}_perm"])
    C = np.stack(o["C"]).reshape(-1)
    assert np.abs(C[G[f"c{i}_C_idx"]] - G[f"c{i}_C_val"]).max() <= 1e-10 * 6.0
    A = layout.assemble(A0, N, v, Px, Py, Pz)
    assert layout.residual(A, layout.assemble(o["C"], N, v, Px, Py, Pz), o["perm"]) <= 1e-12
