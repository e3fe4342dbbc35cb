"""Bethe-ansatz ground-state energy of the periodic spin-1/2 Heisenberg chain H = sum_x S_x . S_{x+1} (even L).

TEST INFRASTRUCTURE ONLY.  The ground state has M = L/2 magnons with rapidities lambda_j solving
    L * 2 atan(2 lambda_j) = 2 pi I_j + sum_k 2 atan(lambda_j - lambda_k),
I_j = -(M-1)/2, ..., (M-1)/2 (integers for odd M, half-integers for even M), and energy
    E = L/4 - sum_j 2 / (4 lambda_j^2 + 1).
Its momentum is 0 for even M and pi for odd M (Marshall's sign rule), so the level lies in the sector k = 0 or k = L/2.
"""
import numpy as np


def ground_state_energy(L):
    if L % 2:
        raise ValueError("even L only")
    M = L // 2
    I = np.arange(M) - (M - 1) / 2.0
    lam = 0.5 * np.tan(np.pi * I / L)                      # the equations without the scattering phases
    for _ in range(100):
        d = lam[:, None] - lam[None, :]
        F = 2.0 * L * np.arctan(2.0 * lam) - 2.0 * np.pi * I - 2.0 * np.arctan(d).sum(axis=1)
        g = 2.0 / (1.0 + d * d)                             # d/dx 2 atan(x)
        Jm = g.copy()                                       # dF_j / dlam_k = +2/(1 + d_jk^2) for k != j
        np.fill_diagonal(Jm, 0.0)
        Jm[np.diag_indices(M)] = 4.0 * L / (1.0 + 4.0 * lam * lam) - (g.sum(axis=1) - 2.0)
        step = np.linalg.solve(Jm, F)
        lam = lam - step
        if np.abs(step).max() < 1e-15 * max(1.0, np.abs(lam).max()):
            break
    return L / 4.0 - float((2.0 / (4.0 * lam * lam + 1.0)).sum())


def ground_state_momentum(L):
    """k in units of 2 pi / L: 0 for even L/2, L/2 for odd L/2."""
    return 0 if (L // 2) % 2 == 0 else L // 2
