"""GPU tests of the slice-granular product of packed cross parts (quantum_basis_b200/csrc/sjds_bulk.cu,
sjds_cross_slices_kernel): the closing pass of a stored species-order handle built without a row range, with real values
and fp64 vectors.

Every 32-row slice of a cross part that stays inside one up configuration is uniform (all rows have the up-hop count of
that configuration); the others -- slices that straddle two blocks of D_dn rows, the last partial slice, slices with empty
rows -- take the ragged path of the same kernel.  The shapes below special-case: mostly uniform slices (D_dn >= 32; D_dn is
never a multiple of 32 on the at most 24 sites a species-order handle takes: 32 divides no C(n, k) with n < 32), many
straddling slices (D_dn < 32), D_dn = 1, n < 32, an empty cross part (it is not packed and takes the bulk-streamed kernel),
and rows longer than one trip of diagonals.  Each product is held row by row to the long-double bound of
tests/kernel_routes.py; the matrix the bound is computed from is the ordinary handle's, whose rows are checked first
against qbgpu_debug_rows_host (long double, on the host).
"""
import ctypes as C

import numpy as np
import pytest

import kernel_routes as K
import lin_builders as B
import quantum_basis_b200 as qb
from quantum_basis_b200 import _lib

pytestmark = pytest.mark.gpu

SPECIES = _lib.SPECIES_ORDER
# name: (Lx, Ly, N_up, N_dn)
SHAPES = {
    "4x4_2_3": (4, 4, 2, 3),       # D_dn = 560: mostly uniform slices, one straddler per block of 17.5 slices
    "4x3_3_1": (4, 3, 3, 1),       # D_dn = 12: every slice straddles blocks
    "4x3_5_0": (4, 3, 5, 0),       # D_dn = 1
    "2x2_1_2": (2, 2, 1, 2),       # n = 24 < 32: one partial slice
    "4x3_0_4": (4, 3, 0, 4),       # no up electron: empty cross part
    "4x4_6_2": (4, 4, 6, 2),       # D_dn = 120: uniform and straddling slices, rows of up to 24 entries (two trips)
}
ALPHA, GAMMA, BETA = 0.7, 0.2, -0.6
STATE = (0.8, 1.3, 0.45)                                      # sx, sz, b_prev of qbgpu_lanczos_step_a
REL = 1e-13


def cd(z):
    z = complex(z)
    return (C.c_double * 2)(z.real, z.imag)


def vp(v):
    return C.c_void_p(v.ptr) if v is not None else None


def fused(M, x, z, y, alpha=1.0, gamma=0.0, beta=0.0, dots=None):
    _lib.check(qb.lib().qbgpu_spmv_fused(M.handle, vp(x), vp(z), vp(y), cd(alpha), cd(gamma), cd(beta), vp(dots)))


def build(name, **kw):
    Lx, Ly, nu, nd = SHAPES[name]
    return qb.hubbard(Lx * Ly, nu, nd, B.square_bonds(Lx, Ly), 1.0, 1.1, **kw)


_REFS = {}


def reference(name):
    """(expanded CSR of H in the reference's order, its cross part, the ordinary handle), the rows of H pinned against
    qbgpu_debug_rows_host."""
    if name in _REFS:
        return _REFS[name]
    Lx, Ly, nu, nd = SHAPES[name]
    ns, bonds = Lx * Ly, B.square_bonds(Lx, Ly)
    P = build(name, is_complex=True, flags=K.NO_AUTOTUNE | K.FORMAT_CSR)
    rp, col, v = P.download_expanded()
    n = P.dim
    rng = np.random.default_rng(23)
    rows = np.arange(n, dtype=np.int64) if n <= 100_000 else np.sort(rng.choice(n, 3_000, replace=False)).astype(np.int64)
    x = rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)
    yh = np.zeros(2 * rows.size)
    b = np.ascontiguousarray(np.asarray(bonds, dtype=np.int32).ravel())
    _lib.check(qb.lib().qbgpu_debug_rows_host(1, ns, nu, nd, len(bonds), b.ctypes.data, 0.0, 1.0, 1.1, rows.size,
                                              rows.ctypes.data, x.ctypes.data, 1, yh.ctypes.data))
    K.assert_rows(yh[0::2] + 1j * yh[1::2], K.RowRef(rp, col, v, x, rows), x, what=f"{name}: generator vs host rows")
    _REFS[name] = (rp, col, v, P)
    return _REFS[name]


def cross_of(rp, col, v, perm, Dd):
    """The entries of H between different up configurations (the cross part), reference order."""
    return K.csr_rows_of(rp, col, v, lambda r, c: perm[r] // Dd != perm[c] // Dd)


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_cross_part_products(name):
    """The fused product on the cross part alone (fp64 vectors, internal order): y = H_c x; alpha, gamma, beta with
    z != y and the running dots; z = y with beta = 1 (rows without entries keep y) and with other scalars; the Lanczos
    step a (scal_mode 1)."""
    rp, col, v, _ = reference(name)
    M = build(name, is_complex=False, flags=SPECIES)
    n, perm = M.dim, M.native_perm()
    Lx, Ly, nu, nd = SHAPES[name]
    _, Dd = K.species_dims(Lx, Ly, nu, nd)
    crp, ccol, cv = cross_of(rp, col, v.real, perm, Dd)
    _, cross = M.species_parts()
    rng = np.random.default_rng(41)
    x, z, y0 = rng.uniform(-1, 1, n), rng.uniform(-1, 1, n), rng.uniform(-1, 1, n)   # reference order
    ref = K.RowRef(crp, ccol, cv, x)

    def dev(a):                                                # reference order -> internal order, on the device
        out = np.empty_like(a)
        out[perm] = a
        return qb.DeviceVector.from_numpy(out)

    def back(d):
        return d.to_numpy()[perm]

    xd, zd = dev(x), dev(z)
    yd = dev(y0)
    fused(cross, xd, None, yd)
    K.assert_rows(back(yd), ref, x, cplx=False, what=f"{name} y=Hc x")
    dots = qb.DeviceVector.from_numpy(np.zeros(4))
    yd = dev(y0)
    fused(cross, xd, zd, yd, ALPHA, GAMMA, BETA, dots)
    y = back(yd)
    K.assert_rows(y, ref, x, z, ALPHA, GAMMA, BETA, cplx=False, what=f"{name} epilogue")
    K.assert_dots(dots.to_numpy(), x, y, cplx=False, what=f"{name} dots")
    yd = dev(y0)
    fused(cross, xd, yd, yd, 1.0, 0.0, 1.0)
    y = back(yd)
    K.assert_rows(y, ref, x, y0, 1.0, 0.0, 1.0, cplx=False, what=f"{name} y+=Hc x")
    assert np.array_equal(y[ref.L == 0], y0[ref.L == 0]), f"{name}: a row without entries did not keep y"
    yd = dev(y0)
    fused(cross, xd, yd, yd, ALPHA, 0.0, BETA)
    K.assert_rows(back(yd), ref, x, y0, ALPHA, 0.0, BETA, cplx=False, what=f"{name} y=aHc x+by")
    sx, sz, bp = STATE
    st = qb.DeviceVector.from_numpy(np.array([sx, sz, bp, 0, 0, 0, 0, 0], dtype=np.float64))
    uz = dev(y0)
    _lib.check(qb.lib().qbgpu_lanczos_step_a(cross.handle, vp(xd), vp(uz), vp(st)))
    w = back(uz)
    K.assert_rows(w, ref, x, y0, sx, 0.0, -bp * sz, cplx=False, what=f"{name} lanczos_step_a w")
    dot = np.sum(sx * x.astype(K.LD) * w.astype(K.LD))
    assert abs(st.to_numpy()[3] - float(dot)) <= 4 * K.U_RND * n * sx * float(np.sum(np.abs(x) * np.abs(w))), f"{name}: state[3]"


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_handle_products(name):
    """Through the whole handle: MultMv in the reference's order with real-content vectors (the closing pass writes the
    reference's order itself) against the long-double rows and the ordinary handle (relative 1e-13), and the Lanczos step
    a, whose closing pass runs with scal_mode 2 and the running dots."""
    rp, col, v, P = reference(name)
    Mc = build(name, is_complex=True, flags=SPECIES)
    n = Mc.dim
    rng = np.random.default_rng(43)
    x = rng.uniform(-1, 1, n)
    ref_all = K.RowRef(rp, col, v.real, x)
    xd, yd = qb.DeviceVector.from_numpy(x.astype(np.complex128)), qb.DeviceVector(n)
    Mc.MultMv(xd, yd)
    y = yd.to_numpy()
    K.assert_rows(y, ref_all, x, cplx=False, what=f"{name} MultMv")
    want = np.zeros(n, dtype=np.complex128)
    P.MultMv(x.astype(np.complex128), want)
    nrm = np.linalg.norm(want)
    assert np.linalg.norm(y - want) <= REL * max(nrm, 1e-300) or nrm == 0.0, f"{name}: MultMv vs the ordinary handle"
    assert np.linalg.norm(y - ref_all.hx) <= REL * max(np.linalg.norm(ref_all.hx), 1e-300) or nrm == 0.0
    # Lanczos step a on the real handle (internal order): w = sx H ux - b_prev sz uz
    M = build(name, is_complex=False, flags=SPECIES)
    perm = M.native_perm()
    y0 = rng.uniform(-1, 1, n)
    xi, yi = np.empty(n), np.empty(n)
    xi[perm], yi[perm] = x, y0
    sx, sz, bp = STATE
    st = qb.DeviceVector.from_numpy(np.array([sx, sz, bp, 0, 0, 0, 0, 0], dtype=np.float64))
    xid, uz = qb.DeviceVector.from_numpy(xi), qb.DeviceVector.from_numpy(yi)
    _lib.check(qb.lib().qbgpu_lanczos_step_a(M.handle, vp(xid), vp(uz), vp(st)))
    w = uz.to_numpy()[perm]
    K.assert_rows(w, ref_all, x, y0, sx, 0.0, -bp * sz, cplx=False, what=f"{name} handle lanczos_step_a w")
    dot = np.sum(sx * x.astype(K.LD) * w.astype(K.LD))
    assert abs(st.to_numpy()[3] - float(dot)) <= 4 * K.U_RND * n * sx * float(np.sum(np.abs(x) * np.abs(w))), f"{name}: state[3]"


def test_shapes_cover_the_special_cases():
    """The table above holds what its comments say (host only: dimensions and hop counts)."""
    dims = {k: K.species_dims(*s) for k, s in SHAPES.items()}
    assert dims["4x4_2_3"][1] > 32
    assert dims["4x3_3_1"][1] < 32 and 32 % dims["4x3_3_1"][1] != 0
    assert dims["4x3_5_0"][1] == 1
    assert dims["2x2_1_2"][0] * dims["2x2_1_2"][1] < 32
    assert SHAPES["4x3_0_4"][2] == 0
    Lx, Ly, nu, _ = SHAPES["4x4_6_2"]
    bonds = B.square_bonds(Lx, Ly)
    assert dims["4x4_6_2"][1] % 32 != 0
    # the longest cross row: 6 electrons on the 4x4 torus, each bond with one occupied end is one hop
    occ = np.zeros(Lx * Ly, dtype=bool)
    occ[[0, 2, 5, 7, 8, 10]] = True
    hops = sum(1 for (a, b) in bonds if occ[a] != occ[b])
    assert hops > 16
