"""The numpy Lin-order builders (tests/lin_builders.py) pinned against CSR matrices assembled by the reference."""
import numpy as np
import pytest

import lin_builders as B


def test_hubbard4x2_is_bit_identical_to_reference(oracle):
    A, meta, ex = oracle.load_golden("hubbard4x2")
    n, ia, ja, val = B.hubbard_upper_csr(8, 4, 4, B.square_bonds(4, 2), t=1.0, U=1.1)
    assert n == A.dim and np.array_equal(ia, A.ia) and np.array_equal(ja, A.ja)
    assert np.array_equal(val, A.val)


@pytest.mark.parametrize("args,mk", [
    (["heis_chain", 12, "sz", 0], lambda: B.heisenberg_upper_csr(12, 6, B.chain_bonds(12))),
    (["heis_chain", 15, "sz", 0.5], lambda: B.heisenberg_upper_csr(15, 7, B.chain_bonds(15))),
    (["hubbard", 3, 3, 4, 5, 1, 2.3], lambda: B.hubbard_upper_csr(9, 4, 5, B.square_bonds(3, 3), U=2.3)),
])
def test_against_live_reference(oracle, args, mk, tmp_path):
    if not oracle.have_qb_ref():
        pytest.skip("oracle/_ref/qb_ref not built (needs the reference's sources at build time)")
    f = str(tmp_path / "H.qbcsr")
    oracle.run_qb_ref(args + ["--dump", f], workdir=str(tmp_path))
    A = oracle.read_qbcsr(f)
    n, ia, ja, val = mk()
    assert n == A.dim and np.array_equal(ia, A.ia) and np.array_equal(ja, A.ja) and np.array_equal(val, A.val)


# ------------------------------------------------------------------ translation-symmetric sectors (repr_builders.py)
def _repr_cases():
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "repr_hashes.json")) as f:
        return json.load(f)


def _build_repr(args):
    import repr_builders as R
    if args[0] == "hubbard_k":
        import repr_builders_fermion as F
        _, Lx, Ly, nup, ndn, t, U, m, n = args
        return F.hubbard_sector_upper_csr([Lx, Ly], nup, ndn, [m, n], F.square_hops(Lx, Ly), t, U)
    if args[0] == "heis_chain_k":
        _, L, sz, k = args
        return R.heisenberg_sector_upper_csr([L], L // 2 - sz, [k], R.chain_bonds(L))
    _, Lx, Ly, sz, m, n = args
    return R.heisenberg_sector_upper_csr([Lx, Ly], Lx * Ly // 2 - sz, [m, n], R.triangular_bonds(Lx, Ly))


@pytest.mark.parametrize("case", _repr_cases(), ids=lambda c: "-".join(str(a) for a in c["qb_ref_args"]))
def test_sector_builder_reproduces_reference_hashes(case):
    """dim, ia, ja and every matrix element of generate_Ham_sparse_repr (src/model.cc:688-836), bit for bit: the
    SHA-256 digests were taken from matrices assembled by the compiled reference (oracle/make_repr_hashes.py)."""
    import hashlib
    S, ia, ja, val = _build_repr(case["qb_ref_args"])
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()   # noqa: E731
    assert S.n == case["dim"] and ja.size == case["nnz"]
    assert sha(ia.astype(np.int64)) == case["ia"] and sha(ja.astype(np.int64)) == case["ja"]
    val = val.astype(np.complex128)
    val = (val.real + 0.0) + 1j * (val.imag + 0.0)          # -0.0 -> +0.0, as in oracle/make_repr_hashes.py
    assert sha(val) == case["val"]


@pytest.mark.parametrize("name,L,k,tri", [("heis16_k3", [16], [3], False), ("tri4x4_k01", [4, 4], [0, 1], True),
                                          ("tri4x4_k12", [4, 4], [1, 2], True)])
def test_sector_builder_against_golden_matrices(oracle, name, L, k, tri):
    import repr_builders as R
    A, meta, ex = oracle.load_golden(name)
    bonds = R.triangular_bonds(*L) if tri else R.chain_bonds(L[0])
    S, ia, ja, val = R.heisenberg_sector_upper_csr(L, 8, k, bonds)
    assert S.n == A.dim and np.array_equal(ia, A.ia) and np.array_equal(ja, A.ja) and np.array_equal(val, A.val)
    # zero-norm representatives carry only the artificial diagonal fake_pos + i/dim (src/model.cc:737-740)
    dead = np.nonzero(S.nu == 0)[0]
    for i in dead[:5]:
        assert ia[i + 1] - ia[i] == 1 and val[ia[i]] == 100.0 + i / S.n


@pytest.mark.parametrize("name", ["heis16_szq3", "heis16_szq8", "heis12_szq1"])
def test_sector_sz_operator_matches_reference_moprXvec(name):
    """A = sum_x exp(-i 2 pi q x/L)/sqrt(L) S^z_x applied between momentum sectors: the restatement of
    model::moprXvec_repr against the vector the compiled reference produced from its own phi0 (golden)."""
    import json
    import os
    import repr_builders as R
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    meta = json.loads(str(z["meta"]))
    L, q, k0 = meta["L"], meta["q"], meta["k0"]
    S0 = R.Sector([L], L // 2, [k0])
    S1 = R.Sector([L], L // 2, [k0 - q])
    y = R.apply_sz(S0, S1, R.szq_coefficients(L, q), z["phi0"])
    assert np.abs(y - z["Aphi0"]).max() < 1e-15
    assert abs(np.linalg.norm(y) - meta["dyn_norm"]) < 1e-14


# ------------------------------------------------------------------ arbitrary translation groups (orbit_builders.py, config 4)
def _dense_from_upper(n, ia, ja, val):
    D = np.zeros((n, n), dtype=np.complex128)
    for i in range(n):
        for p in range(ia[i], ia[i + 1]):
            D[i, ja[p]] = val[p]
            if ja[p] != i:
                D[ja[p], i] = np.conj(val[p])
    return D


def test_cluster_translation_groups_are_groups_with_homomorphic_characters():
    from quantum_basis_b200.clusters import Cluster
    for A in (((2, 1), (-1, 3)), ((3, 1), (-1, 4)), ((3, 1), (-1, 3)), ((5, 1), (-1, 6)), ((4, 0), (0, 3))):
        c = Cluster(*A)
        P = c.translations()
        assert all(sorted(p) == list(range(c.det)) for p in P.tolist()) and P[0].tolist() == list(range(c.det))
        index = {tuple(p): i for i, p in enumerate(P.tolist())}
        mom = c.distinct_momenta()
        assert len(mom) == c.det
        chi = c.characters(mom[min(1, len(mom) - 1)])
        for a in range(c.det):
            for b in range(c.det):
                ab = index[tuple(P[a][P[b]].tolist())]           # closure
                assert abs(chi[ab] - chi[a] * chi[b]) < 1e-12     # chi is a character
        assert len(c.triangular_bonds()) == 3 * c.det


@pytest.mark.parametrize("A0,A1,ndown", [((2, 1), (-1, 3), 3), ((3, 1), (-1, 3), 5), ((3, 1), (-1, 4), 6), ((4, 0), (0, 3), 6)])
def test_orbit_convention_partitions_the_full_spectrum(A0, A1, ndown):
    """The convention the device assembler for tilted clusters follows (no reference exists for config 4, SURVEY F5): all
    momentum sectors together have exactly the spectrum of the full Sz sector, whose matrix is the reference-pinned
    full-basis restatement."""
    import orbit_builders as OB
    from quantum_basis_b200.clusters import Cluster
    cl = Cluster(A0, A1)
    bonds = cl.triangular_bonds()
    n, ia, ja, val = B.heisenberg_upper_csr(cl.det, ndown, bonds)
    full = np.linalg.eigvalsh(_dense_from_upper(n, ia, ja, val))
    ev = []
    for m in cl.distinct_momenta():
        reps, stab, sia, sja, sval = OB.heisenberg_orbit_upper_csr(cl.det, ndown, cl.translations(), cl.characters(m), bonds)
        ev.append(np.linalg.eigvalsh(_dense_from_upper(reps.size, sia, sja, sval)))
    ev = np.sort(np.concatenate(ev))
    assert ev.size == full.size and np.abs(ev - full).max() < 1e-10


# published ground-state energies of the momentum sectors (the reference's own example asserts)
CHAIN16_E0 = [-7.142296361, -6.523407057, -5.990986863, -5.615175598, -5.451965668, -5.525353087, -5.823231143, -6.298652725,
              -6.872106678, -6.298652725, -5.823231143, -5.525353087, -5.451965668, -5.615175598, -5.990986863, -6.523407057]
TRI4X4_E0 = {(0, 0): -8.555514918, (0, 1): -8.002263841, (0, 2): -7.944709784, (0, 3): -8.002263841, (1, 2): -7.588987242}


def _oracle_E0(oracle, S, ia, ja, val):
    from oracle_lib import Csr
    A = Csr(S.n, ia, ja, val, True)
    x = oracle.vec_randomize(S.n, 1)
    m, a, b, _ = oracle.lanczos(A, x, 1000, "sr_val0")
    hess = np.zeros(2000)
    hess[:m + 1] = b
    hess[1000:1000 + m] = a
    return oracle.hess_eigen(hess, 1000, m, vectors=False)[0][0]


@pytest.mark.parametrize("k", range(16))
def test_chain16_sector_energies_match_the_published_list(oracle, k):
    """examples/trans_symmetric/latt_chain/chain_Heisenberg_spin_half.cc:102-117: E0 of every momentum sector of the
    L = 16 chain, from the restated assembler + the restated Lanczos (start vector and stop rule of the reference)."""
    import repr_builders as R
    S, ia, ja, val = R.heisenberg_sector_upper_csr([16], 8, [k], R.chain_bonds(16))
    assert abs(_oracle_E0(oracle, S, ia, ja, val) - CHAIN16_E0[k]) < 1e-8


@pytest.mark.parametrize("mn", sorted(TRI4X4_E0))
def test_triangular4x4_sector_energies_match_the_published_list(oracle, mn):
    """examples/trans_symmetric/latt_triangular/triangular_Heisenberg_spin_half.cc:135-139 (E0_list index = 4 m + n)."""
    import repr_builders as R
    S, ia, ja, val = R.heisenberg_sector_upper_csr([4, 4], 8, list(mn), R.triangular_bonds(4, 4))
    assert abs(_oracle_E0(oracle, S, ia, ja, val) - TRI4X4_E0[mn]) < 1e-8


HUBBARD4X2_E0 = [-14.07605866, -10.50470669, -12.16861094, -12.19847764, -10.54300366, -14.03137587, -12.16861094, -12.19847764]


@pytest.mark.parametrize("idx", range(8))
def test_hubbard4x2_sector_energies_match_the_published_list(oracle, idx):
    """examples/trans_symmetric/latt_square/square_Fermi_Hubbard.cc:112-119 (E0_list index = Ly m + n = 2 m + n): the
    fermionic restatement (translation signs in norms and matrix elements) + the restated Lanczos."""
    import repr_builders_fermion as F
    m, n = idx // 2, idx % 2
    S, ia, ja, val = F.hubbard_sector_upper_csr([4, 2], 4, 4, [m, n], F.square_hops(4, 2), 1.0, 1.1)
    assert abs(_oracle_E0(oracle, S, ia, ja, val) - HUBBARD4X2_E0[idx]) < 1e-8


@pytest.mark.parametrize("name", ["heis16_smq3", "heis12_smq5"])
def test_sector_sminus_operator_matches_reference_moprXvec(name):
    """The off-diagonal branch of model::moprXvec_repr (src/model.cc:1762-1834): S^-_q phi0 lands in the sector with one
    more down spin and momentum k0 - q; restatement against the vector the compiled reference produced (golden)."""
    import json
    import os
    import repr_builders as R
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    meta = json.loads(str(z["meta"]))
    L, q, k0 = meta["L"], meta["q"], meta["k0"]
    S0 = R.Sector([L], L // 2, [k0])
    S1 = R.Sector([L], L // 2 + 1, [k0 - q])
    y = R.apply_sminus(S0, S1, R.szq_coefficients(L, q), z["phi0"])
    assert y.size == z["Aphi0"].size and np.abs(y - z["Aphi0"]).max() < 1e-14
    assert abs(np.linalg.norm(y) - meta["dyn_norm"]) < 1e-13
    # S^+ with conjugated coefficients is the adjoint map between the two sectors: <w, A v> = <A^+ w, v>
    rng = np.random.default_rng(2)
    w = rng.normal(size=S1.n) + 1j * rng.normal(size=S1.n)
    w[S1.nu == 0] = 0.0
    up = R.apply_splus(S1, S0, np.conj(R.szq_coefficients(L, q)), w)
    assert abs(np.vdot(w, y) - np.vdot(up, z["phi0"])) < 1e-13


@pytest.mark.parametrize("name", ["hubbard4x2_szq10", "hubbard4x2_szq21"])
def test_full_basis_szq_matches_reference_moprXvec_full(name):
    """model::moprXvec_full (src/model.cc:1468-1538) for S^z_q of the Hubbard model in the full basis: the numpy restatement
    and the library's row function (run on the host through qbgpu_debug_full_apply_diag_host) against the vector the
    compiled reference produced in the flow of examples/trans_absent/latt_square/square_Fermi_Hubbard.cc (golden)."""
    import ctypes as C
    import json
    import os
    import lin_builders as LB
    from quantum_basis_b200 import _lib
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    meta = json.loads(str(z["meta"]))
    Lx, Ly, nup, ndn = meta["Lx"], meta["Ly"], meta["nup"], meta["ndn"]
    c = LB.square_szq_coefficients(Lx, Ly, meta["qm"], meta["qn"])
    y = LB.apply_onsite_diag(Lx * Ly, 2, (nup, ndn), c, -c, z["phi0"])
    assert np.abs(y - z["Aphi0"]).max() < 1e-15
    assert abs(np.linalg.norm(y) - meta["dyn_norm"]) < 1e-14
    yl = np.zeros_like(y)
    c0, c1, x = np.ascontiguousarray(c), np.ascontiguousarray(-c), np.ascontiguousarray(z["phi0"])
    p = lambda a: C.c_void_p(a.ctypes.data)   # noqa: E731
    _lib.check(_lib.lib().qbgpu_debug_full_apply_diag_host(1, Lx * Ly, nup, ndn, p(c0), p(c1), p(x), p(yl)))
    assert np.abs(yl - z["Aphi0"]).max() < 1e-15
    # spins through the same entry point: S^z_total on any Sz-sector vector is Sz times the vector
    n = 924
    xs = (np.random.default_rng(1).standard_normal(n) + 0j)
    ys = np.zeros(n, dtype=np.complex128)
    ones = np.ones(12, dtype=np.complex128)
    _lib.check(_lib.lib().qbgpu_debug_full_apply_diag_host(0, 12, 6, 0, p(ones), p(ones), p(xs), p(ys)))
    assert np.abs(ys).max() < 1e-15                                   # Sz_total = 0 at half filling
    _lib.check(_lib.lib().qbgpu_debug_full_apply_diag_host(0, 12, 5, 0, p(ones), p(ones), p(np.ascontiguousarray(xs[:792])), p(ys)))
    assert np.abs(ys[:792] - 1.0 * xs[:792]).max() < 1e-15            # 7 up, 5 down: Sz_total = +1
    assert np.array_equal(LB.apply_onsite_diag(12, 1, (5,), ones, None, xs[:792]), ys[:792])


@pytest.mark.parametrize("name", ["hubbard4x2"])
def test_host_row_function_against_the_reference_assembled_matrix(oracle, name):
    """qbgpu_debug_rows_host (the sampled-row parity check bench.py runs on the BASELINE-size matrices: rows regenerated on the
    host from the Lin tables by the generators' own row function, accumulated in long double) against the long-double product
    on the matrix the compiled reference assembled."""
    import ctypes as C
    import quantum_basis_b200 as qb
    L = qb.lib()
    A, meta, ex = oracle.load_golden(name)
    n = A.dim
    x = oracle.vec_randomize(n, 1) + 1j * oracle.vec_randomize(n, 2).real
    want = oracle.spmv_ld(A, x)
    rows = np.arange(n, dtype=np.int64)
    y = np.zeros(2 * n)
    bonds = np.array(B.square_bonds(4, 2), dtype=np.int32).ravel()
    rc = L.qbgpu_debug_rows_host(1, 8, 4, 4, len(bonds) // 2, bonds.ctypes.data, 0.0, 1.0, 1.1, n, rows.ctypes.data, x.ctypes.data, 1, y.ctypes.data)
    assert rc == 0
    assert np.linalg.norm(y.view(np.complex128) - want) <= 1e-15 * np.linalg.norm(want)
    with pytest.raises(Exception):
        bad = np.array([n], dtype=np.int64)
        from quantum_basis_b200 import _lib
        _lib.check(L.qbgpu_debug_rows_host(1, 8, 4, 4, len(bonds) // 2, bonds.ctypes.data, 0.0, 1.0, 1.1, 1, bad.ctypes.data, x.ctypes.data, 1, y.ctypes.data))
