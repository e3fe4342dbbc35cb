"""Spin-1/2 momentum sectors with 64-bit states (34 and 36 sites): enumeration, matrix-free product, stored build and
the S^z / S^+- operators of the wide path -- against the narrow path on the same sectors (qbgpu_debug_sector_words(64)),
against tests/repr_builders.py and its per-row restatement (tests/repr_rows_wide.py), and against the Bethe ansatz
(tests/bethe_chain.py) and the published 6x6 square-lattice energy."""
import ctypes as C
from math import comb

import numpy as np
import pytest

import bethe_chain as BA
import quantum_basis_b200 as qb
import repr_builders as R
import repr_rows_wide as W

pytestmark = pytest.mark.gpu

TOL_MV = 1e-12
ERR_ARG, ERR_STATE = 1, 4

# the ten sectors of tests/test_gpu_parity.py (_SECTOR_CASES): zero-norm rows, Lin and integer row order
SECTOR_CASES = [
    ("chain16_k3", [16], 8, [3]), ("chain12_k5", [12], 6, [5]), ("chain14_sz1_k2", [14], 6, [2]),
    ("chain20_k7", [20], 10, [7]), ("chain22_sz1_k5", [22], 10, [5]), ("chain24_k0", [24], 12, [0]),
    ("tri4x4_k12", [4, 4], 8, [1, 2]), ("tri3x4_k23", [3, 4], 6, [2, 3]), ("tri6x3_k12", [6, 3], 9, [1, 2]),
    ("tri4x5_k32", [4, 5], 10, [3, 2]),
]
# the sectors of test_matrix_free_sector_product_equals_the_stored_sector_matrix
MATFREE_CASES = [([16], 8, [3]), ([12], 6, [0]), ([4, 4], 8, [1, 2]), ([4, 4], 8, [2, 2]), ([6, 2], 6, [3, 1])]


def _bonds(L):
    return R.chain_bonds(L[0]) if len(L) == 1 else R.triangular_bonds(*L)


def rel_l2(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


@pytest.fixture
def wide():
    L = qb.lib()
    assert L.qbgpu_debug_sector_words(64) == 0
    try:
        yield L
    finally:
        assert L.qbgpu_debug_sector_words(0) == 0


def _pair(L, ndown, k):
    """The same sector on both paths: (narrow, wide)."""
    lib = qb.lib()
    sn = qb.Sector(L, ndown, k)
    assert lib.qbgpu_debug_sector_words(64) == 0
    try:
        sw = qb.Sector(L, ndown, k)
    finally:
        assert lib.qbgpu_debug_sector_words(0) == 0
    assert sn.state_bits == 32 and sw.state_bits == 64
    return sn, sw


# ------------------------------------------------------------------------------------------ forced wide at <= 32 sites
@pytest.mark.parametrize("name,L,ndown,k", SECTOR_CASES, ids=[c[0] for c in SECTOR_CASES])
def test_forced_wide_sector_is_the_reference_convention(oracle, wide, name, L, ndown, k):
    from oracle_lib import Csr
    bonds = _bonds(L)
    S, ia, ja, val = R.heisenberg_sector_upper_csr(L, ndown, k, bonds)
    sec = qb.Sector(L, ndown, k)
    assert sec.state_bits == 64 and sec.dim == S.n and sec.lin_order == S.lin_order and sec.zero_norm == int((S.nu == 0).sum())
    st = sec.states()
    assert st.dtype == np.uint64 and np.array_equal(st, S.states)
    assert np.array_equal(sec.norms(), S.nu)
    M = sec.heisenberg(bonds, flags=1)
    rowptr, col, v = M.download_expanded()
    eia, eja, ev = oracle.expand_upper(Csr(S.n, ia, ja, val, True))
    assert M.dim == S.n and M.info.nnz_input == ja.size
    assert np.array_equal(rowptr, eia) and np.array_equal(col.astype(np.int64), eja) and np.array_equal(v, ev)
    del M
    sec.free()


@pytest.mark.parametrize("name,L,ndown,k", SECTOR_CASES, ids=[c[0] for c in SECTOR_CASES])
def test_wide_operators_equal_the_narrow_ones(name, L, ndown, k):
    """apply_sz bit for bit, apply_ladder (fp64 atomics) to 1e-13, between sectors of both widths."""
    N = int(np.prod(L))
    lat = R.Lattice(L)
    k2 = [k[0] - 1] + list(k[1:])
    coef = np.array([np.exp(-2j * np.pi * lat.coor[s][0] / L[0]) / np.sqrt(N) for s in range(N)])
    a_n, a_w = _pair(L, ndown, k)
    b_n, b_w = _pair(L, ndown, k2)
    x = qb.vec_randomize(a_n.dim, 1)
    yn = a_n.apply_sz(b_n, coef, x).to_numpy()
    yw = a_w.apply_sz(b_w, coef, x).to_numpy()
    assert np.array_equal(yn, yw)
    if ndown + 1 <= N:
        c_n, c_w = _pair(L, ndown + 1, k)
        ln = a_n.apply_ladder(c_n, coef, x, lower=True).to_numpy()
        lw = a_w.apply_ladder(c_w, coef, x, lower=True).to_numpy()
        assert np.abs(ln - lw).max() <= 1e-13 * max(1.0, np.abs(ln).max())
        un = c_n.apply_ladder(a_n, coef, ln, lower=False).to_numpy()
        uw = c_w.apply_ladder(a_w, coef, ln, lower=False).to_numpy()
        assert np.abs(un - uw).max() <= 1e-13 * max(1.0, np.abs(un).max())


@pytest.mark.parametrize("L,ndown,k", MATFREE_CASES)
def test_wide_matrix_free_product_is_bit_identical_to_the_narrow_one(L, ndown, k):
    """The same rows, the same arithmetic in the same order: MultMv, MultMv2 and the fused Lanczos loop (dots in the
    kernel epilogue) agree bit for bit between the widths, and with the stored matrix to TOL_MV."""
    bl = _bonds(L)
    sn, sw = _pair(L, ndown, k)
    assert np.array_equal(sn.states().astype(np.uint64), sw.states())
    Hn, Hw, Hs = sn.heisenberg_matrix_free(bl), sw.heisenberg_matrix_free(bl), sw.heisenberg(bl, flags=1)
    n = sn.dim
    rng = np.random.default_rng(5)
    x = rng.normal(size=n) + 1j * rng.normal(size=n)
    yn, yw, ys = (np.zeros(n, dtype=np.complex128) for _ in range(3))
    Hn.MultMv(x, yn); Hw.MultMv(x, yw); Hs.MultMv(x, ys)
    assert np.array_equal(yn, yw) and rel_l2(yw, ys) < TOL_MV
    y0 = rng.normal(size=n) + 1j * rng.normal(size=n)
    y2n, y2w = y0.copy(), y0.copy()
    Hn.MultMv2(x, y2n); Hw.MultMv2(x, y2w)
    assert np.array_equal(y2n, y2w)
    if n > 40:
        rn = qb.locate_E0_lanczos(Hn, nev=1, ncv=0)
        rw = qb.locate_E0_lanczos(Hw, nev=1, ncv=0)
        assert rn["eigenvals"][0] == rw["eigenvals"][0] and rn["lanczos_steps"] == rw["lanczos_steps"]
    del Hn, Hw, Hs


def test_narrow_sectors_are_unaffected_after_a_reset_to_size_selection():
    lib = qb.lib()
    assert lib.qbgpu_debug_sector_words(64) == 0
    assert lib.qbgpu_debug_sector_words(0) == 0
    S, _, _, _ = R.heisenberg_sector_upper_csr([16], 8, [3], R.chain_bonds(16))
    sec = qb.Sector([16], 8, [3])
    assert sec.state_bits == 32
    st = sec.states()
    assert st.dtype == np.uint32 and np.array_equal(st.astype(np.uint64), S.states)
    assert np.array_equal(sec.states64(), S.states)


def test_errors_of_the_wide_interface():
    lib = qb.lib()
    h = C.c_void_p()
    Ls, k = np.array([38], dtype=np.int32), np.array([0], dtype=np.int32)
    assert lib.qbgpu_sector_create(C.byref(h), 1, C.c_void_p(Ls.ctypes.data), 19, C.c_void_p(k.ctypes.data)) == ERR_ARG
    Le, ke = np.array([6, 3], dtype=np.int32), np.array([0, 0], dtype=np.int32)
    assert lib.qbgpu_sector_create_electron(C.byref(h), 2, C.c_void_p(Le.ctypes.data), 9, 9, C.c_void_p(ke.ctypes.data)) == ERR_ARG
    for bits in (1, 16, 32, 63, 128, -1):
        assert lib.qbgpu_debug_sector_words(bits) == ERR_ARG
    assert lib.qbgpu_debug_sector_words(64) == 0
    try:
        sec = qb.Sector([12], 6, [1])
    finally:
        assert lib.qbgpu_debug_sector_words(0) == 0
    out = np.empty(sec.dim, dtype=np.uint32)
    assert lib.qbgpu_sector_states(sec._h, C.c_void_p(out.ctypes.data)) == ERR_STATE
    assert b"qbgpu_sector_states64" in lib.qbgpu_last_error()
    assert lib.qbgpu_sector_states64(sec._h, None) == ERR_ARG


# ------------------------------------------------------------------------------------------ 34 and 36 sites
def test_chain34_all_momenta_partition_the_sz0_states():
    """sum_k (dim - zero_norm) = C(34, 17); every sector's states are distinct representatives."""
    live = 0
    for k in range(34):
        sec = qb.Sector([34], 17, [k])
        assert sec.state_bits == 64
        live += sec.dim - sec.zero_norm
        st = sec.states()
        st.sort()
        assert np.all(st[1:] != st[:-1]), k
        del st
        sec.free()
    assert live == comb(34, 17) == 2333606220


def test_chain34_stored_sector_matrix_equals_the_matrix_free_product():
    sec = qb.Sector([34], 17, [1])
    bl = R.chain_bonds(34)
    Hf = sec.heisenberg_matrix_free(bl)
    x = qb.vec_randomize(sec.dim, 1, device=True)
    yf = qb.DeviceVector(sec.dim)
    Hf.MultMv(x, yf)
    yf = yf.to_numpy()
    del Hf
    Hs = sec.heisenberg(bl)
    ys = qb.DeviceVector(sec.dim)
    Hs.MultMv(x, ys)
    assert rel_l2(yf, ys.to_numpy()) < TOL_MV
    del Hs


@pytest.mark.parametrize("L", [36, 34])
def test_chain_E0_of_the_matrix_free_sector_equals_the_bethe_ansatz(L):
    """The ground state sits at k = 0 for even L/2 and k = L/2 for odd L/2 (Marshall's sign rule)."""
    sec = qb.Sector([L], L // 2, [BA.ground_state_momentum(L)])
    H = sec.heisenberg_matrix_free(R.chain_bonds(L))
    E = qb.locate_E0_lanczos(H, nev=1, ncv=0)["eigenvals"][0]
    Eb = BA.ground_state_energy(L)
    assert abs(E - Eb) <= 1e-10 * abs(Eb), (E, Eb)


@pytest.mark.parametrize("case", ["chain36_k0", "square6x6_k00"])
def test_sampled_rows_at_36_sites_follow_the_restated_convention(case):
    L, bl = ([36], R.chain_bonds(36)) if case == "chain36_k0" else ([6, 6], R.square_bonds(6, 6))
    k = [0] * len(L)
    sec = qb.Sector(L, 18, k)
    assert sec.state_bits == 64
    H = sec.heisenberg_matrix_free(bl)
    x = qb.vec_randomize(sec.dim, 1, device=True)
    y = qb.DeviceVector(sec.dim)
    H.MultMv(x, y)
    y = y.to_numpy()
    xh = x.to_numpy()
    del H
    states, nu = sec.states(), sec.norms()
    rows = np.sort(np.random.default_rng(7).choice(sec.dim, size=10000, replace=False))
    T = W.SectorTables(L, k)
    is_rep, nu_r = T.representative_and_norm(states[rows])
    assert np.all(is_rep) and np.array_equal(nu_r, nu[rows])
    ref = T.rows_times(states, nu, bl, rows, xh)
    assert np.abs(y[rows] - ref).max() <= 1e-12 * np.abs(ref).max()


def test_square6x6_ground_state_energy_and_singlet_structure_factor():
    """E0/N = -0.678872 (Schulz, Ziman & Poilblanc, J. Phys. I France 6, 675 (1996)); the ground state is a singlet, so
    |S^-_q phi0|^2 = 2 |S^z_q phi0|^2 at q = (pi, pi) -- the wide apply_sz and apply_ladder between 2.5e8-row sectors."""
    L, bl = [6, 6], R.square_bonds(6, 6)
    s0 = qb.Sector(L, 18, [0, 0])
    H = s0.heisenberg_matrix_free(bl)
    res = qb.locate_E0_lanczos(H, nev=1, ncv=1, device_vectors=True)
    E0 = res["eigenvals"][0]
    assert abs(E0 / 36 - (-0.678872)) < 5e-7, E0
    phi0 = res["eigenvecs_device"][0]
    del H
    lat = R.Lattice(L)
    coef = np.array([(-1.0) ** int(lat.coor[s].sum()) / 6.0 for s in range(36)], dtype=np.complex128)
    sq = qb.Sector(L, 18, [3, 3])
    yz = s0.apply_sz(sq, coef, phi0).to_numpy()
    sm = qb.Sector(L, 19, [3, 3])
    ym = s0.apply_ladder(sm, coef, phi0, lower=True).to_numpy()
    nz, nm = np.vdot(yz, yz).real, np.vdot(ym, ym).real
    assert nz > 0.1 and abs(nm - 2.0 * nz) <= 1e-10 * nm, (nz, nm)
