"""One-site electron operators between Hubbard momentum sectors (model::moprXvec_repr, src/model.cc:1716-1846), restated in
tests/repr_ops_fermion.py, against what pins them without a GPU:
  * S^z_q through the density rule against the compiled reference's full-basis dynamic flow (tests/golden/hubbard4x2_szq*);
  * S^-_q through the spin-flip rule against S^z_q (SU(2): the 4x2 ground state is a singlet);
  * c_k, c+_k against an independent full-basis computation (own Jordan-Wigner order, dense diagonalisation);
  * the adjoint identities, and the row-by-row (gather) form the device computes against the reference's scatter.
Everything on the half-filled 4x2 cluster, t = 1, U = 1.1, whose ground state is unique at k = (0,0)."""
import json
import os

import numpy as np
import pytest

import lin_builders as B
import repr_ops_fermion as O
import quantum_basis_b200 as qb

L = [4, 2]
N = 8
E0_4X2 = -14.076058658879


def lanczos(H, y, m):
    """The dnmcs recursion (no re-orthogonalisation) from y/|y|: (a[0..m), b[0..m)), b[0] = 0."""
    v = y / np.linalg.norm(y)
    vp = np.zeros_like(v)
    a, b = np.zeros(m), np.zeros(m + 1)
    for j in range(m):
        w = H @ v - b[j] * vp
        a[j] = np.vdot(v, w).real
        w = w - a[j] * v
        b[j + 1] = np.linalg.norm(w)
        vp, v = v, w / b[j + 1]
    return a, b[:m]


_cache = {}


def sector(nup, ndn, k):
    key = (nup, ndn, tuple(int(x) % l for x, l in zip(k, L)))
    if key not in _cache:
        _cache[key] = O.dense_sector(L, nup, ndn, list(key[2]))
    return _cache[key]


def ground():
    if "phi0" not in _cache:
        S0, H0 = sector(4, 4, (0, 0))
        w, v = np.linalg.eigh(H0)
        _cache["phi0"] = (w[0], v[:, 0])
    return _cache["phi0"]


def test_ground_state_of_the_4x2_cluster():
    E0, phi0 = ground()
    assert abs(E0 - E0_4X2) < 1e-11


@pytest.mark.parametrize("name", ["hubbard4x2_szq10", "hubbard4x2_szq21"])
def test_density_rule_reproduces_the_reference_szq_flow(name):
    """S^z_q = sum_r c_r (n_up,r - n_dn,r), c_r = e^{+i q.r}/(2 sqrt N), maps k = (0,0) to q: its norm and dnmcs coefficients
    are those of the compiled reference's full-basis flow (examples/trans_absent/latt_square/square_Fermi_Hubbard.cc)."""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    meta = json.loads(str(z["meta"]))
    E0, phi0 = ground()
    S0, _ = sector(4, 4, (0, 0))
    q = (meta["qm"], meta["qn"])
    c = B.square_szq_coefficients(4, 2, *q)
    assert np.abs(c - 0.5 / np.sqrt(N) * O.plane_wave(L, q)).max() < 1e-15
    S1, H1 = sector(4, 4, q)
    y = O.apply_density(S0, S1, c, -c, phi0)
    assert abs(np.linalg.norm(y) - meta["dyn_norm"]) < 1e-11
    m = len(z["dyn_a"])
    a, b = lanczos(H1, y, m)
    assert np.abs(a[:5] - z["dyn_a"][:5]).max() < 1e-9
    assert np.abs(b[1:5] - z["dyn_b"][1:5]).max() < 1e-9
    w = np.linspace(-14.0, 8.0, 221) + 0.1j
    g, g_ref = qb.continued_fraction(a, b, w), qb.continued_fraction(z["dyn_a"], z["dyn_b"], w)
    assert np.abs(g - g_ref).max() <= 1e-3 * np.abs(g_ref).max()


@pytest.mark.parametrize("q", [(1, 0), (2, 1), (1, 1)])
def test_spin_flip_rule_obeys_su2(q):
    """S^-_q = sum_r e^{+i q.r}/sqrt N c+_{r,dn} c_{r,up}: for a singlet, S^-_q phi0 is a rotated copy of S^z_q phi0, so
    |S^-_q phi0|^2 = 2 |S^z_q phi0|^2 and both dnmcs runs give the same coefficients (targets (4,4,q) and (3,5,q))."""
    E0, phi0 = ground()
    S0, _ = sector(4, 4, (0, 0))
    c = O.plane_wave(L, q) / np.sqrt(N)
    Sz, Hz = sector(4, 4, q)
    Sm, Hm = sector(3, 5, q)
    yz = O.apply_density(S0, Sz, 0.5 * c, -0.5 * c, phi0)
    ym = O.apply_scatter(S0, Sm, "flip", c, phi0, lower=True)
    assert abs((np.linalg.norm(ym) / np.linalg.norm(yz)) ** 2 - 2.0) < 1e-12
    az, bz = lanczos(Hz, yz, 6)
    am, bm = lanczos(Hm, ym, 6)
    assert np.abs(az - am).max() < 1e-10 and np.abs(bz - bm).max() < 1e-10
    yg = O.apply_gather(S0, Sm, "flip", c, phi0, lower=True)
    assert np.abs(yg - ym).max() < 1e-15


# ------------------------------------------------------------------ single-electron operators against the full basis
def _full():
    if "full" not in _cache:
        F0 = O.FullBasis(L, 4, 4)
        w, v = np.linalg.eigh(F0.hamiltonian())
        _cache["full"] = (F0, w[0], v[:, 0])
    return _cache["full"]


def _full_block(nup, ndn):
    key = ("full", nup, ndn)
    if key not in _cache:
        F = O.FullBasis(L, nup, ndn)
        w, v = np.linalg.eigh(F.hamiltonian())
        _cache[key] = (F, w, v)
    return _cache[key]


def _cases():
    return [(k, create, spin) for k in [(m, n) for m in range(4) for n in range(2)] for create in (False, True) for spin in (0, 1)]


def _sector_vector(k, create, spin):
    """c_{k,s} phi0 (N^{-1/2} sum_r e^{-i k.r} c_{r,s}, lands in K = -k) or c+_{k,s} phi0 (e^{+i k.r}, lands in K = +k)."""
    E0, phi0 = ground()
    S0, _ = sector(4, 4, (0, 0))
    d = 1 if create else -1
    c = O.plane_wave(L, k, d) / np.sqrt(N)
    kt = tuple(d * x for x in k)
    Sn, Hn = sector(4 + d * (spin == 0), 4 + d * (spin == 1), kt)
    return S0, Sn, Hn, c, O.apply_scatter(S0, Sn, "fermion", c, phi0, create=create, spin=spin)


def _full_vector(k, create, spin):
    F0, E0, phi0 = _full()
    d = 1 if create else -1
    Fn, w, v = _full_block(4 + d * (spin == 0), 4 + d * (spin == 1))
    c = F0.plane_wave(k, d) / np.sqrt(N)
    return Fn, w, v, F0.apply_fermion(Fn, c, phi0, create, spin)


@pytest.mark.parametrize("k,create,spin", _cases())
def test_single_electron_operators_match_the_full_basis(k, create, spin):
    """|c_ks phi0|^2, |c+_ks phi0|^2, the first Lanczos coefficient <H> and the spectral function at eta = 0.1 from the sector
    restatement against plain occupation numbers (its own Jordan-Wigner order) and dense diagonalisation of the N -+ 1 blocks."""
    S0, Sn, Hn, c, y = _sector_vector(k, create, spin)
    Fn, w, v, yf = _full_vector(k, create, spin)
    n2, n2f = np.vdot(y, y).real, np.vdot(yf, yf).real
    assert abs(n2 - n2f) < 1e-12
    if n2 < 1e-20:
        return
    assert abs(np.vdot(y, Hn @ y).real / n2 - np.sum(np.abs(v.T @ yf) ** 2 * w) / n2f) < 1e-10
    z = np.linspace(-16.0, 8.0, 241) + 0.1j
    ws, vs = np.linalg.eigh(Hn)
    g = (np.abs(vs.conj().T @ y) ** 2)[None, :] / (z[:, None] - ws[None, :])
    gf = (np.abs(v.T @ yf) ** 2)[None, :] / (z[:, None] - w[None, :])
    A, Af = -g.sum(1).imag, -gf.sum(1).imag
    assert np.abs(A - Af).max() <= 1e-3 * Af.max()
    a, b = lanczos(Hn, y, min(150, int((Sn.nu > 0).sum()) - 1))
    Ac = -(n2 * qb.continued_fraction(a, b, z)).imag
    assert np.abs(Ac - Af).max() <= 1e-3 * Af.max()
    assert np.abs(O.apply_gather(S0, Sn, "fermion", c, ground()[1], create=create, spin=spin) - y).max() < 1e-15


@pytest.mark.parametrize("spin", [0, 1])
def test_single_electron_sum_rules(spin):
    """sum_k |c_ks phi0|^2 = N_s and |c_ks phi0|^2 + |c+_ks phi0|^2 = 1 for every k."""
    tot = 0.0
    for k in [(m, n) for m in range(4) for n in range(2)]:
        nc = np.linalg.norm(_sector_vector(k, False, spin)[4]) ** 2
        nd = np.linalg.norm(_sector_vector(k, True, spin)[4]) ** 2
        assert abs(nc + nd - 1.0) < 1e-12
        tot += nc
    assert abs(tot - 4.0) < 1e-11


def test_adjoint_identities():
    """<w, A v> = <A^+ w, v> for the three operator families, with random v, w (zero on zero-norm rows), through the
    reference's scatter and the device's gather, between sectors whose norms differ ((2,1) has zero-norm rows)."""
    rng = np.random.default_rng(5)

    def rnd(S):
        x = rng.normal(size=S.n) + 1j * rng.normal(size=S.n)
        x[S.nu == 0] = 0.0
        return x

    S0, _ = sector(4, 4, (2, 1))
    q = (1, 1)
    cu, cd = rng.normal(size=N) + 1j * rng.normal(size=N), rng.normal(size=N) + 1j * rng.normal(size=N)
    S1, _ = sector(4, 4, (3, 0))
    v, w = rnd(S0), rnd(S1)
    lhs = np.vdot(w, O.apply_density(S0, S1, cu, cd, v))
    assert abs(lhs - np.vdot(O.apply_density(S1, S0, np.conj(cu), np.conj(cd), w), v)) < 1e-12 * abs(lhs)
    c = O.plane_wave(L, q) * (0.3 + 0.7j)
    for kind, kw, tgt, back in (("flip", dict(lower=True), (3, 5), dict(lower=False)),
                                ("flip", dict(lower=False), (5, 3), dict(lower=True)),
                                ("fermion", dict(create=False, spin=0), (3, 4), dict(create=True, spin=0)),
                                ("fermion", dict(create=False, spin=1), (4, 3), dict(create=True, spin=1))):
        kt = (2 + q[0], 1 + q[1])
        S1, _ = sector(*tgt, kt)
        v, w = rnd(S0), rnd(S1)
        for f in (O.apply_scatter, O.apply_gather):
            Av = f(S0, S1, kind, c, v, **kw)
            Aw = f(S1, S0, kind, np.conj(c), w, **back)
            lhs = np.vdot(w, Av)
            assert abs(lhs) > 1e-3 and abs(lhs - np.vdot(Aw, v)) < 1e-12 * abs(lhs), (kind, kw, f.__name__)
        assert np.abs(O.apply_gather(S0, S1, kind, c, v, **kw) - O.apply_scatter(S0, S1, kind, c, v, **kw)).max() < 1e-13


def test_continued_fraction_is_the_resolvent_of_the_tridiagonal_matrix():
    rng = np.random.default_rng(1)
    a, b = rng.normal(size=7), np.concatenate([[0.0], rng.uniform(0.5, 1.5, size=6)])
    T = np.diag(a) + np.diag(b[1:], 1) + np.diag(b[1:], -1)
    z = np.array([0.3 + 0.1j, -1.0 + 0.05j])
    want = [np.linalg.inv(zz * np.eye(7) - T)[0, 0] for zz in z]
    assert np.abs(qb.continued_fraction(a, b, z) - want).max() < 1e-12


def test_cpp_adaptor_electron_operators_compile_and_link(tmp_path):
    """qbgpu::electron_sector::apply_density / apply_spin_flip / apply_fermion: every entry they use exists in libqbgpu.so, and
    without a device the sector constructor throws instead of falling back."""
    import shutil
    import subprocess
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "electron_ops.cc"
    src.write_text('''
#include <cstdio>
#include "qbgpu_csr_mat.hpp"
int main(int argc, char **) {
    try {
        qbgpu::electron_sector s({4, 2}, 4, 4, {0, 0}), t({4, 2}, 3, 4, {1, 0});
        std::vector<std::complex<double>> c(8, 1.0);
        std::complex<double> *x = nullptr, *y = nullptr;
        if (argc == 1000) { s.apply_density(s, c, c, x, y); s.apply_spin_flip(t, true, c, x, y); s.apply_fermion(t, false, 0, c, x, y); }
    } catch (const std::runtime_error &e) { std::printf("electron_sector: %s\\n", e.what()); return 1; }
    return 0;
}
''')
    exe = tmp_path / "electron_ops"
    libdir = os.path.join(root, "quantum_basis_b200")
    subprocess.run([gxx, "-std=c++17", "-O1", "-I", os.path.join(root, "include"), str(src), "-o", str(exe), "-L", libdir, "-lqbgpu",
                    "-Wl,-rpath," + libdir], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 1 and "electron_sector:" in r.stdout, r.stdout + r.stderr
