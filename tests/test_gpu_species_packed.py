"""GPU tests of the packed entry words of stored species-order handles (quantum_basis_b200/csrc/species.cu, sjds.cu,
sjds_bulk.cu).

A stored handle built without a row range, with real values, keeps each entry as one 32-bit word (column | value code): 4 bytes per entry instead
of 12.  Row shards (also one covering all rows) and QBGPU_KEEP_COMPLEX handles keep separate values.  The products of every kernel that reads a packed
part -- the block-local pass 1, the plain sliced-jagged pass 1 (blocks of x too large for shared memory), the bulk-streamed
pass 2 with and without the running dots and with the fused way out -- are compared with the ordinary handle.  The host
rules of the packing are checked in tests/test_species_packed_cpu.py.
"""
import ctypes as C

import numpy as np
import pytest

import lin_builders as B
import quantum_basis_b200 as qb
from quantum_basis_b200 import _lib
from gpu_species_common import SPECIES, rel_l2

pytestmark = pytest.mark.gpu

# Lx, Ly, nup, ndn: 4x3 -- both passes block-local / bulk-streamed; 4x4 with D_dn = 8008 -- the complex block of x (125 KB)
# exceeds the block-local limit, so pass 1 with complex vectors takes the plain kernel; 6x3 with D_dn = 48620 -- the fp64
# block too
CASES = {"hub4x3_66": (4, 3, 6, 6), "hub4x4_16": (4, 4, 1, 6), "hub6x3_19": (6, 3, 1, 9)}
ONE, ZERO = (C.c_double * 2)(1.0, 0.0), (C.c_double * 2)(0.0, 0.0)


def _make(name, **kw):
    Lx, Ly, nu, nd = CASES[name]
    return qb.hubbard(Lx * Ly, nu, nd, B.square_bonds(Lx, Ly), 1.0, 1.1, **kw)


@pytest.mark.parametrize("name", sorted(CASES))
def test_packed_layout_info(name):
    M = _make(name, flags=SPECIES)
    K = _make(name, flags=SPECIES | _lib.KEEP_COMPLEX)
    inf, kinf = M.info, K.info
    assert inf.val_is_real and inf.value_dict > 0
    assert kinf.value_dict == 0 and not kinf.val_is_real
    assert inf.nnz_stored == kinf.nnz_stored
    # same tables and row metadata: the difference is 4 bytes per packed entry against 4 + 16 per complex one
    assert kinf.device_bytes - inf.device_bytes == 16 * inf.nnz_stored


def test_row_shards_keep_fp64_values():
    Lx, Ly, nu, nd = CASES["hub4x3_66"]
    Dd = 924
    n = Dd * Dd
    S = qb.hubbard(Lx * Ly, nu, nd, B.square_bonds(Lx, Ly), 1.0, 1.1, flags=SPECIES, rows=(0, 300 * Dd))
    SK = qb.hubbard(Lx * Ly, nu, nd, B.square_bonds(Lx, Ly), 1.0, 1.1, flags=SPECIES | _lib.KEEP_COMPLEX, rows=(0, 300 * Dd))
    assert S.info.n == n and S.info.value_dict == 0 and S.info.val_is_real
    assert SK.info.device_bytes - S.info.device_bytes == 8 * S.info.nnz_stored      # 12 bytes per entry against 20
    # a one-rank shard (row range = all rows) keeps fp64 values too: its cross part can be split by columns
    S1 = qb.hubbard(Lx * Ly, nu, nd, B.square_bonds(Lx, Ly), 1.0, 1.1, flags=SPECIES, rows=(0, n))
    assert S1.info.value_dict == 0 and S1.info.val_is_real
    hs1 = (C.c_void_p * 2)()
    b1 = np.array([0, 462 * Dd, n], dtype=np.int64)
    _lib.check(qb.lib().qbgpu_species_split_cross(S1.handle, 2, b1.ctypes.data, hs1))
    for h1 in hs1:
        _lib.check(qb.lib().qbgpu_destroy(C.c_void_p(h1)))
    M = _make("hub4x3_66", flags=SPECIES)
    loc, cross = M.species_parts()
    h = C.c_void_p()
    assert qb.lib().qbgpu_row_view(cross.handle, 0, 32 * Dd, Dd, 64, C.byref(h)) != 0          # packed parts cannot be cut
    assert "packed" in qb.lib().qbgpu_last_error().decode()
    b = np.array([0, n // 2 // Dd * Dd, n], dtype=np.int64)
    hs = (C.c_void_p * 2)()
    assert qb.lib().qbgpu_species_split_cross(M.handle, 2, b.ctypes.data, hs) != 0
    assert "packed" in qb.lib().qbgpu_last_error().decode()


@pytest.mark.parametrize("name", sorted(CASES))
def test_packed_products_match_the_ordinary_handle(name):
    M, P = _make(name, flags=SPECIES), _make(name, flags=0)
    n = M.dim
    perm = M.native_perm()
    rng = np.random.default_rng(7)
    xr = rng.normal(size=n)
    xc = rng.normal(size=n) + 1j * rng.normal(size=n)
    want_r, want_c = np.zeros(n, dtype=np.complex128), np.zeros(n, dtype=np.complex128)
    P.MultMv(xr.astype(np.complex128), want_r)
    P.MultMv(xc, want_c)
    # MultMv, reference order: real content (fp64 passes, closing pass writes the reference's order) and genuinely complex
    for x, want in ((xr.astype(np.complex128), want_r), (xc, want_c)):
        xd, yd = qb.DeviceVector.from_numpy(x), qb.DeviceVector(n)
        M.MultMv(xd, yd)
        assert rel_l2(yd.to_numpy(), want) <= 1e-12
    # fused product in the internal order: fp64 vectors through the real view, complex vectors through the handle
    L = qb.lib()
    Mr = M.real_view()
    x_int = np.empty(n); x_int[perm] = xr
    xn, yn = qb.DeviceVector.from_numpy(x_int), qb.DeviceVector(n, np.float64)
    _lib.check(L.qbgpu_spmv_fused(Mr.handle, C.c_void_p(xn.ptr), None, C.c_void_p(yn.ptr), ONE, ZERO, ZERO, None))
    assert rel_l2(yn.to_numpy()[perm], want_r.real) <= 1e-12
    xc_int = np.empty_like(xc); xc_int[perm] = xc
    xn, yn = qb.DeviceVector.from_numpy(xc_int), qb.DeviceVector(n)
    dots = qb.DeviceVector(4, np.float64)
    _lib.check(L.qbgpu_spmv_fused(M.handle, C.c_void_p(xn.ptr), None, C.c_void_p(yn.ptr), ONE, ZERO, ZERO, C.c_void_p(dots.ptr)))
    assert rel_l2(yn.to_numpy()[perm], want_c) <= 1e-12
    d = dots.to_numpy()
    assert abs(d[2] - np.vdot(want_c, want_c).real) <= 1e-12 * np.vdot(want_c, want_c).real


@pytest.mark.parametrize("name", ["hub4x3_66", "hub6x3_19"])
def test_packed_lanczos_matches_the_ordinary_handle(name):
    M, P = _make(name, flags=SPECIES), _make(name, flags=0)
    n = M.dim
    hs, hp = np.zeros(200), np.zeros(200)
    vs, vp = np.zeros(2 * n, dtype=np.complex128), np.zeros(2 * n, dtype=np.complex128)
    v0 = np.random.default_rng(3).normal(size=n)
    vs[:n] = v0 / np.linalg.norm(v0); vp[:n] = vs[:n]                        # real start vector: the fp64 loop
    ms = qb.lanczos(0, 40, 100, n, M, vs, hs, "dnmcs")
    mp = qb.lanczos(0, 40, 100, n, P, vp, hp, "dnmcs")
    assert ms == mp == 40
    for k in (slice(100, 140), slice(1, 40)):                                # the alphas and betas of the recursion
        assert np.all(np.abs(hs[k] - hp[k]) <= 1e-10 * np.maximum(1.0, np.abs(hp[k])))
