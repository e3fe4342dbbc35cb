"""CPU checks of the references the 34- and 36-site sector tests compare against: the Bethe-ansatz ground-state energy of
the periodic Heisenberg chain (tests/bethe_chain.py) and the per-row restatement of the sector convention for halves of
more than 16 bits (tests/repr_rows_wide.py)."""
import numpy as np
import pytest

import bethe_chain as B
import repr_builders as R
import repr_rows_wide as W


def test_bethe_ansatz_reproduces_the_reference_chain_energies():
    assert abs(B.ground_state_energy(16) - (-7.142296361)) < 1e-9              # main_test.cc
    assert abs(B.ground_state_energy(20) - (-8.9043865298764)) < 1e-12         # config 1 on the compiled reference


@pytest.mark.parametrize("L", [8, 10, 12])
def test_bethe_ansatz_equals_exact_diagonalisation(L):
    import scipy.sparse as sp
    import scipy.sparse.linalg as sla
    from itertools import combinations
    states = np.array(sorted(sum(1 << s for s in c) for c in combinations(range(L), L // 2)), dtype=np.int64)
    index = {int(s): i for i, s in enumerate(states)}
    rows, cols, vals = [], [], []
    for i, s in enumerate(states.tolist()):
        d = 0.0
        for x in range(L):
            y = (x + 1) % L
            if ((s >> x) & 1) == ((s >> y) & 1):
                d += 0.25
            else:
                d -= 0.25
                rows.append(i); cols.append(index[s ^ ((1 << x) | (1 << y))]); vals.append(0.5)
        rows.append(i); cols.append(i); vals.append(d)
    H = sp.csr_matrix((vals, (rows, cols)), shape=(states.size, states.size))
    E0 = sla.eigsh(H, k=1, which="SA", tol=1e-14)[0][0]
    assert abs(B.ground_state_energy(L) - E0) < 1e-10


def test_bethe_ansatz_values_at_34_and_36_sites():
    assert abs(B.ground_state_energy(34) - (-15.091296465658)) < 1e-11
    assert abs(B.ground_state_energy(36) - (-15.976235822064)) < 1e-11
    assert B.ground_state_momentum(34) == 17 and B.ground_state_momentum(36) == 0


@pytest.mark.parametrize("L,ndown,k,bonds", [([16], 8, [3], "chain"), ([12], 6, [0], "chain"), ([4, 4], 8, [1, 2], "tri"),
                                             ([6, 2], 6, [3, 1], "tri"), ([14], 6, [2], "chain")])
def test_per_row_restatement_equals_the_enumerating_builder(L, ndown, k, bonds):
    """The per-row restatement (no enumeration: representative test, norm, and H x row by row) against repr_builders on
    sectors it can enumerate -- the stored matrix times a random vector."""
    bl = R.chain_bonds(L[0]) if bonds == "chain" else R.triangular_bonds(*L)
    S, ia, ja, val = R.heisenberg_sector_upper_csr(L, ndown, k, bl)
    T = W.SectorTables(L, k)
    canon, nu = T.representative_and_norm(S.states)
    assert np.all(canon) and np.array_equal(nu, S.nu)
    # a state that is not its own representative is recognised
    a, b = S.unzip(S.states)
    moved = S.zip(*S._move(S.fwd[1], a, b))
    c2, _ = T.representative_and_norm(moved)
    assert not np.all(c2[moved != S.states])
    n = S.n
    rng = np.random.default_rng(3)
    x = rng.normal(size=n) + 1j * rng.normal(size=n)
    full = np.zeros((n, n), dtype=np.complex128)
    for r in range(n):
        for e in range(ia[r], ia[r + 1]):
            full[r, ja[e]] = val[e]
            if ja[e] != r:
                full[ja[e], r] = np.conj(val[e])
    rows = np.arange(0, n, 3)
    y = T.rows_times(S.states, nu, bl, rows, x)
    ref = full[rows] @ x
    assert np.abs(y - ref).max() <= 1e-12 * np.abs(ref).max()
