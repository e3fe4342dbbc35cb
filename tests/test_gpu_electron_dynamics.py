"""GPU tests of the one-site electron operators between Hubbard momentum sectors (qbgpu_sector_apply_density / _spin_flip /
_fermion: model::moprXvec_repr, src/model.cc:1716-1846) and of measure_repr_dynamic_electron on top of them: every device entry
against the restatement in tests/repr_ops_fermion.py (itself pinned in tests/test_electron_ops_cpu.py), run-to-run
bit-identity, and the dynamic flows from the device's own ground state against the compiled reference's goldens, SU(2) and an
independent full-basis computation."""
import json
import os

import numpy as np
import pytest

import lin_builders as B
import repr_builders_fermion as F
import repr_ops_fermion as O
import quantum_basis_b200 as qb

pytestmark = pytest.mark.gpu


def rel_l2(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def _random(S, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(size=S.n) + 1j * rng.normal(size=S.n)
    x[S.nu == 0] = 0.0
    x[rng.random(S.n) < 0.05] = 1e-13                                  # below lanczos_precision: must not contribute
    return x


# (lattice, (N_up, N_dn), K): 4x2 at half filling (no zero-norm rows at (0,0)), 4x3 (6,6,(2,1)) with zero-norm rows on both ends
CASES = [([4, 2], (4, 4), (0, 0), (1, 1)), ([4, 2], (4, 4), (2, 1), (3, 0)), ([4, 3], (6, 6), (2, 1), (0, 2))]


@pytest.mark.parametrize("L,nn,K,q", CASES)
def test_device_electron_operators_match_the_restatement(L, nn, K, q):
    """Density, spin flip both ways, c and c+ for both spins: device against the reference's scatter (restated) to 1e-13, and
    a second call bit-identical to the first.  Coefficients e^{+i q.r} (times a complex constant), target momentum K + q."""
    N = int(np.prod(L))
    nup, ndn = nn
    S0r = F.ElectronSector(L, nup, ndn, list(K))
    S0 = qb.ElectronSector(L, nup, ndn, list(K))
    assert np.array_equal(S0.states().astype(np.uint64), S0r.states) and np.array_equal(S0.norms(), S0r.nu)
    kt = [(K[d] + q[d]) % L[d] for d in range(len(L))]
    c = O.plane_wave(L, q) * (0.4 - 0.9j) / np.sqrt(N)
    x = _random(S0r, 3)
    xd = qb.DeviceVector.from_numpy(x)
    ops = [("density", (nup, ndn), None), ("flip", (nup - 1, ndn + 1), dict(lower=True)), ("flip", (nup + 1, ndn - 1), dict(lower=False))]
    ops += [("fermion", (nup + (d if s == 0 else 0), ndn + (d if s == 1 else 0)), dict(create=d > 0, spin=s)) for d in (-1, 1) for s in (0, 1)]
    for kind, tgt, kw in ops:
        S1r = F.ElectronSector(L, tgt[0], tgt[1], kt)
        S1 = qb.ElectronSector(L, tgt[0], tgt[1], kt)
        if kind == "density":
            cu, cd = c, c[::-1].copy() * 0.5
            want = O.apply_density(S0r, S1r, cu, cd, x)
            run = lambda: S0.apply_density(S1, cu, cd, xd).to_numpy()          # noqa: E731
        elif kind == "flip":
            want = O.apply_scatter(S0r, S1r, kind, c, x, **kw)
            run = lambda: S0.apply_spin_flip(S1, c, xd, **kw).to_numpy()       # noqa: E731
        else:
            want = O.apply_scatter(S0r, S1r, kind, c, x, **kw)
            run = lambda: S0.apply_fermion(S1, c, xd, **kw).to_numpy()         # noqa: E731
        y1, y2 = run(), run()
        assert np.linalg.norm(want) > 0.1 * np.linalg.norm(x) * np.abs(c).max(), (kind, kw)
        assert rel_l2(y1, want) < 1e-13, (kind, kw, rel_l2(y1, want))
        assert np.array_equal(y1.view(np.float64), y2.view(np.float64)), (kind, kw)
        S1.free()
    xd.free()
    S0.free()


def test_electron_operators_refuse_wrong_sectors():
    S0 = qb.ElectronSector([4, 2], 4, 4, [0, 0])
    x = np.zeros(S0.dim, dtype=np.complex128)
    c = np.ones(8, dtype=np.complex128)
    same = qb.ElectronSector([4, 2], 4, 4, [1, 0])
    fewer_up = qb.ElectronSector([4, 2], 3, 4, [1, 0])
    flipped = qb.ElectronSector([4, 2], 3, 5, [1, 0])
    other_lattice = qb.ElectronSector([2, 4], 3, 4, [1, 0])
    spins = qb.Sector([8], 4, [0])
    with pytest.raises(qb.QbgpuError):
        S0.apply_density(fewer_up, c, c, x)                              # particle numbers
    with pytest.raises(qb.QbgpuError):
        S0.apply_spin_flip(same, c, x)
    with pytest.raises(qb.QbgpuError):
        S0.apply_spin_flip(flipped, c, x, lower=False)                  # S^+ raises N_up
    with pytest.raises(qb.QbgpuError):
        S0.apply_fermion(flipped, c, x)
    with pytest.raises(qb.QbgpuError):
        S0.apply_fermion(fewer_up, c, x, spin=1)                         # c_dn keeps N_up
    with pytest.raises(qb.QbgpuError):
        S0.apply_fermion(fewer_up, c, x, create=True)
    with pytest.raises(qb.QbgpuError):
        S0.apply_fermion(other_lattice, c, x)                            # another lattice
    with pytest.raises(qb.QbgpuError, match="electron sectors only"):
        S0.apply_fermion(spins, c, x)                                    # a spin sector
    xs, ys = qb.DeviceVector(spins.dim), qb.DeviceVector(S0.dim)
    with pytest.raises(qb.QbgpuError, match="electron sectors only"):                # a spin sector as the source, through the C entry
        qb._lib.check(qb.lib().qbgpu_sector_apply_density(spins._h, S0._h, c.ctypes.data, c.ctypes.data, xs.ptr, ys.ptr))
    S0.apply_fermion(fewer_up, c, x)                                    # the right target works


# ------------------------------------------------------------------ dynamic flows from the device's ground state
_state = {}


def _ground():
    """E0 and phi0 of the half-filled 4x2 cluster (t = 1, U = 1.1) in k = (0,0) by the device's Lanczos + CG."""
    if not _state:
        S0 = qb.ElectronSector([4, 2], 4, 4, [0, 0])
        H0 = S0.hubbard(F.square_hops(4, 2), 1.0, 1.1)
        res = qb.locate_E0_lanczos(H0, nev=1, ncv=1, device_vectors=True)
        _state.update(S0=S0, H0=H0, E0=res["eigenvals"][0], phi0=res["eigenvecs_device"][0])
    return _state


def _dyn(op, coefs, tgt, kt, maxit):
    g = _ground()
    S1 = qb.ElectronSector([4, 2], tgt[0], tgt[1], list(kt))
    H1 = S1.hubbard(F.square_hops(4, 2), 1.0, 1.1)
    hess = np.zeros(2 * maxit)
    m, norm = qb.measure_repr_dynamic_electron(op, coefs, g["S0"], S1, H1, g["phi0"], maxit, hess)
    H1.destroy()
    S1.free()
    return m, norm, hess[maxit:maxit + m], hess[:m]


@pytest.mark.parametrize("name", ["hubbard4x2_szq10", "hubbard4x2_szq21"])
def test_szq_flow_in_the_momentum_basis_matches_the_reference(name):
    """S^z_q of the Hubbard model between momentum sectors (density rule, cd = -cu) from the device's phi0: the norm and dnmcs
    coefficients of the compiled reference's full-basis flow (golden).  Coefficients from step 5 on differ by round-off
    amplification (tests/test_gpu_dynamics.py), so they are compared through the continued fraction."""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    meta = json.loads(str(z["meta"]))
    assert abs(_ground()["E0"] - meta["E0"]) < 1e-10
    c = B.square_szq_coefficients(4, 2, meta["qm"], meta["qn"])
    m, norm, a, b = _dyn("density", (c, -c), (4, 4), (meta["qm"], meta["qn"]), meta["maxit"])
    assert m >= 8
    assert abs(norm - meta["dyn_norm"]) < 1e-11
    assert np.abs(a[:5] - z["dyn_a"][:5]).max() < 1e-9
    assert np.abs(b[1:5] - z["dyn_b"][1:5]).max() < 1e-9
    w = np.linspace(-14.0, 8.0, 221) + 0.1j
    mr = min(m, len(z["dyn_a"]))
    g, g_ref = qb.continued_fraction(a[:mr], b[:mr], w), qb.continued_fraction(z["dyn_a"][:mr], z["dyn_b"][:mr], w)
    assert np.abs(g - g_ref).max() <= 1e-3 * np.abs(g_ref).max()


@pytest.mark.parametrize("q", [(1, 0), (2, 1), (1, 1)])
def test_spin_flip_flow_obeys_su2(q):
    """|S^-_q phi0|^2 = 2 |S^z_q phi0|^2 and equal dnmcs coefficients: the ground state is a singlet."""
    c = O.plane_wave([4, 2], q) / np.sqrt(8)
    mz, nz, az, bz = _dyn("density", (0.5 * c, -0.5 * c), (4, 4), q, 40)
    mm, nm, am, bm = _dyn("s-", c, (3, 5), q, 40)
    assert abs((nm / nz) ** 2 - 2.0) < 1e-10
    assert np.abs(az[:6] - am[:6]).max() < 1e-9 and np.abs(bz[:6] - bm[:6]).max() < 1e-9
    mp, npl, ap, bp = _dyn("s+", c, (5, 3), q, 40)
    assert abs((npl / nz) ** 2 - 2.0) < 1e-10


def test_szq_at_q_zero_gives_nothing():
    """S^z_total phi0 = 0 for the singlet ground state: norm below lanczos_precision, m = 0, no Lanczos run."""
    c = np.full(8, 0.5 / np.sqrt(8), dtype=np.complex128)
    m, norm, a, b = _dyn("density", (c, -c), (4, 4), (0, 0), 40)
    assert m == 0 and norm < qb.lanczos_precision


_full = {}


def _full_block(nup, ndn):
    if (nup, ndn) not in _full:
        Fb = O.FullBasis([4, 2], nup, ndn)
        w, v = np.linalg.eigh(Fb.hamiltonian())
        _full[(nup, ndn)] = (Fb, w, v)
    return _full[(nup, ndn)]


@pytest.mark.parametrize("create", [False, True])
def test_spectral_function_matches_the_full_basis(create):
    """A(k, omega) for spin up: photoemission (c_k phi0, sector K = -k) and inverse photoemission (c+_k phi0, K = +k) from the
    device's phi0 through measure_repr_dynamic_electron and the continued fraction, against an independent full-basis
    computation (plain occupation numbers, dense diagonalisation): weights to 1e-11, <H> to 1e-9, the spectrum at eta = 0.1
    to 1e-3 of its maximum; the sum rules hold on the device's weights."""
    F0, w0, v0 = _full_block(4, 4)
    phi_full = v0[:, 0]
    d = 1 if create else -1
    Fn, w, v = _full_block(4 + d, 4)
    z = np.linspace(-16.0, 8.0, 241) + 0.1j
    total = 0.0
    for k in [(m, n) for m in range(4) for n in range(2)]:
        c = O.plane_wave([4, 2], k, d) / np.sqrt(8)
        m, norm, a, b = _dyn("cdag_up" if create else "c_up", c, (4 + d, 4), tuple(d * x for x in k), 150)
        yf = F0.apply_fermion(Fn, F0.plane_wave(k, d) / np.sqrt(8), phi_full, create, 0)
        wt = np.abs(v.T @ yf) ** 2
        assert abs(norm ** 2 - wt.sum()) < 1e-11, k
        total += norm ** 2
        if wt.sum() < 1e-20:
            continue
        assert abs(a[0] - (wt * w).sum() / wt.sum()) < 1e-9, k
        Af = -(wt[None, :] / (z[:, None] - w[None, :])).sum(1).imag
        Ad = -(norm ** 2 * qb.continued_fraction(a, b, z)).imag
        assert np.abs(Ad - Af).max() <= 1e-3 * Af.max(), k
    assert abs(total - 4.0) < 1e-10                  # sum_k |c_k phi0|^2 = N_up = 4 ; sum_k |c+_k phi0|^2 = N - N_up = 4
