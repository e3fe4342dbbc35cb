"""Every H*v kernel route and fused epilogue against a long-double reference, at the shapes each route special-cases.

Each device product is held, row by row, to the error bound of tests/kernel_routes.py (long-double reference, bound
c*u*(L_i+4)*(|alpha| sum|h||x| + |gamma||x_i| + |beta||z_i|)); where the code promises identical bits, the test asserts
identical bits.  The route each case takes is predicted by kernel_routes.predict_* (a restatement of the launchers'
rules) and confirmed through the handle's info where the handle can show it.  The CPU side of the helpers is checked in
tests/test_kernel_routes_cpu.py.
"""
import ctypes as C
import time

import numpy as np
import pytest

import kernel_routes as K
import lin_builders as B
import quantum_basis_b200 as qb
from quantum_basis_b200 import _lib

pytestmark = pytest.mark.gpu

SPECIES = _lib.SPECIES_ORDER
ALPHA, GAMMA, BETA = 0.7 - 0.3j, 0.2 + 0.45j, -0.6 + 0.25j
STATE = (0.8, 1.3, 0.45)                                      # sx, sz, b_prev of qbgpu_lanczos_step_a


def cd(z):
    z = complex(z)
    return (C.c_double * 2)(z.real, z.imag)


def vp(v):
    return C.c_void_p(v.ptr) if v is not None else None


def L():
    return qb.lib()


def fused(M, x, z, y, alpha=1.0, gamma=0.0, beta=0.0, dots=None):
    _lib.check(L().qbgpu_spmv_fused(M.handle, vp(x), vp(z), vp(y), cd(alpha), cd(gamma), cd(beta), vp(dots)))


def rnd(rng, n, cplx):
    return rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n) if cplx else rng.uniform(-1, 1, n)


def scal(s, cplx):
    return complex(s) if cplx else complex(s).real


# ---------------------------------------------------------------------------------------------- ordinary handles
def make_ordinary(up, kind, flags, sym=True):
    n, ia, ja, val = up
    if not sym:
        ia, ja, val = K.lower_too(n, ia, ja, val)
    if kind == "d":
        return qb.csr_mat(n, ia, ja, np.ascontiguousarray(val.real), sym, flags=flags)
    if kind == "z_real":
        return qb.csr_mat(n, ia, ja, val.real.astype(np.complex128), sym, flags=flags)
    return qb.csr_mat(n, ia, ja, val.astype(np.complex128), sym, flags=flags | _lib.KEEP_COMPLEX)


def kind_values(up, kind):
    n, ia, ja, val = up
    return (n, ia, ja, val.real if kind != "z_cplx" else val.astype(np.complex128))


def run_epilogues(M, up, kind, seed, what):
    """Every epilogue of the fused product, the Lanczos step and the reference-shaped products on handle M."""
    n, ia, ja, val = kind_values(up, kind)
    rp, col, v = K.expand(n, ia, ja, val)
    cplx = kind != "d"
    ar = kind == "z_cplx"                                       # complex arithmetic in the matrix entries too
    rng = np.random.default_rng(seed)
    x, z, y0 = rnd(rng, n, cplx), rnd(rng, n, cplx), rnd(rng, n, cplx)
    ref = K.RowRef(rp, col, v, x)
    dt = np.complex128 if cplx else np.float64
    xd = qb.DeviceVector.from_numpy(x)
    c8 = cplx or ar
    # plain y = H x
    yd = qb.DeviceVector.from_numpy(y0)
    fused(M, xd, None, yd)
    y_plain = yd.to_numpy()
    K.assert_rows(y_plain, ref, x, cplx=c8, what=f"{what} y=Hx")
    # alpha, gamma, beta (complex on complex vectors), z != y, running dots
    a, g, b = scal(ALPHA, cplx), scal(GAMMA, cplx), scal(BETA, cplx)
    zd, dots = qb.DeviceVector.from_numpy(z), qb.DeviceVector(4, np.float64)
    fused(M, xd, zd, yd, a, g, b, dots)
    y = yd.to_numpy()
    K.assert_rows(y, ref, x, z, a, g, b, cplx=c8, what=f"{what} epilogue")
    K.assert_dots(dots.to_numpy(), x, y, cplx=c8, what=f"{what} dots")
    # z aliasing y with beta = 1 (the KEEP instantiations: rows without entries keep y), from a non-zero y
    yd = qb.DeviceVector.from_numpy(y0)
    fused(M, xd, yd, yd, 1.0, 0.0, 1.0)
    y = yd.to_numpy()
    K.assert_rows(y, ref, x, y0, 1.0, 0.0, 1.0, cplx=c8, what=f"{what} y+=Hx")
    empty = ref.L == 0
    assert np.array_equal(y[empty], y0[empty]), f"{what}: a row without entries did not keep y"
    # z aliasing y with complex scalars (not KEEP)
    yd = qb.DeviceVector.from_numpy(y0)
    fused(M, xd, yd, yd, a, 0.0, b)
    K.assert_rows(yd.to_numpy(), ref, x, y0, a, 0.0, b, cplx=c8, what=f"{what} y=aHx+by")
    # Lanczos step a with a state set here: w = sx H ux - b_prev sz uz ; state[3] = sum Re conj(sx ux_i) w_i
    sx, sz, bp = STATE
    st = qb.DeviceVector.from_numpy(np.array([sx, sz, bp, 0, 0, 0, 0, 0], dtype=np.float64))
    uz = qb.DeviceVector.from_numpy(y0)
    _lib.check(L().qbgpu_lanczos_step_a(M.handle, vp(xd), vp(uz), vp(st)))
    w = uz.to_numpy()
    K.assert_rows(w, ref, x, y0, sx, 0.0, -bp * sz, cplx=c8, what=f"{what} lanczos_step_a w")
    s3 = st.to_numpy()[3]
    dot = np.sum((np.conj(sx * x.astype(K.CLD)) * w.astype(K.CLD)).real)
    assert abs(s3 - float(dot)) <= 8 * K.U_RND * n * sx * float(np.sum(np.abs(x) * np.abs(w))), f"{what}: state[3]"
    # the reference-shaped products: MultMv (host and device vectors), y = alpha H x + beta y through qbgpu_zmv / qbgpu_dmv
    yh = np.full(n, 3.0, dtype=dt)
    M.MultMv(x.astype(dt), yh)
    K.assert_rows(yh, ref, x, cplx=c8, what=f"{what} MultMv host")
    assert np.array_equal(yh, y_plain), f"{what}: MultMv and the fused product differ"
    yh = y0.astype(dt).copy()
    M._mv(a, x.astype(dt), b, yh)
    K.assert_rows(yh, ref, x, y0, a, 0.0, b, cplx=c8, what=f"{what} mv host")
    yd = qb.DeviceVector.from_numpy(y0)
    M._mv(a, xd, b, yd)
    assert np.array_equal(yd.to_numpy(), yh), f"{what}: host and device vectors differ"
    yh2 = y0.astype(dt).copy()
    M.MultMv2(x.astype(dt), yh2)
    K.assert_rows(yh2, ref, x, y0, 1.0, 0.0, 1.0, cplx=c8, what=f"{what} MultMv2")
    return ref


FMTS = {"csr": K.NO_AUTOTUNE | K.FORMAT_CSR, "sell": K.NO_AUTOTUNE | K.FORMAT_SELL}


@pytest.mark.parametrize("sym", [True, False], ids=["upper", "full"])
@pytest.mark.parametrize("fmt", sorted(FMTS))
@pytest.mark.parametrize("kind", K.VALUE_KINDS)
@pytest.mark.parametrize("lanes", K.LANES)
def test_lane_counts_and_row_structures(lanes, kind, fmt, sym):
    """Rows of exactly 1, LANES, 2*LANES-1, 2*LANES and 2*LANES+1 entries and empty rows, at a mean row length that makes
    the untimed choice take LANES: the paired loop and the tail of the CSR-vector kernel, and the same rows in the
    sliced-jagged kernel (full trips, ragged trips, slices with empty rows, whole slices without entries)."""
    up = K.lane_case(lanes, kind="complex" if kind == "z_cplx" else "real")
    M = make_ordinary(up, kind, FMTS[fmt], sym)
    n, ia, ja, val = up
    rp, _, _ = K.expand(n, ia, ja, val)
    p = K.predict_ordinary(int(rp[-1]), n, FMTS[fmt], kind != "z_cplx")
    inf = M.info
    assert inf.lanes == p["lanes"] == lanes and inf.format == p["format"] and inf.value_dict == 0
    assert bool(inf.val_is_real) == (kind != "z_cplx") and inf.nnz_stored == rp[-1]
    assert K.empty_slices(rp).size >= 1
    run_epilogues(M, up, kind, 11 + lanes, f"lanes={lanes} {kind} {fmt}")


@pytest.mark.parametrize("fmt", ["csr", "sell", "default"])
@pytest.mark.parametrize("kind", K.VALUE_KINDS)
@pytest.mark.parametrize("n", [1, 31, 33, 40_007])
def test_small_and_odd_dimensions(n, kind, fmt):
    rng = np.random.default_rng(n)
    up = K.band_upper(n, 3, rng, "complex" if kind == "z_cplx" else "real")
    flags = {"csr": FMTS["csr"], "sell": FMTS["sell"], "default": 0}[fmt]
    M = make_ordinary(up, kind, flags)
    run_epilogues(M, up, kind, 5, f"n={n} {kind} {fmt}")


@pytest.mark.parametrize("fmt", ["csr", "sell", "default"])
@pytest.mark.parametrize("kind", ["d", "z_cplx"])
def test_hub_row_longer_than_65536(kind, fmt):
    """A star: row 0 holds 70,000 entries, every other row one (the Hermitian image) and a diagonal on every third."""
    n = 70_001
    rng = np.random.default_rng(3)
    r = np.concatenate([np.zeros(n, np.int64), np.arange(3, n, 3)])
    c = np.concatenate([np.arange(n), np.arange(3, n, 3)])
    up = K._upper_csr(n, r, c, rng, "complex" if kind == "z_cplx" else "real")
    flags = {"csr": FMTS["csr"], "sell": FMTS["sell"], "default": 0}[fmt]
    M = make_ordinary(up, kind, flags)
    ref = run_epilogues(M, up, kind, 9, f"hub {kind} {fmt}")
    assert ref.L[0] > 65_536


def _dict_matrix(nvals, seed=2):
    rng = np.random.default_rng(seed)
    n, ia, ja, _ = K.band_upper(3001, 4, rng, "real")
    table = np.concatenate([[0.0, -0.0], np.unique(rng.uniform(-2, 2, nvals + 50))[:nvals - 2]])
    assert table.size == nvals
    val = table[np.arange(ja.size) % nvals]
    return n, ia, ja, val


@pytest.mark.parametrize("kind", ["d", "z_real"])
def test_value_dictionary_with_256_and_257_values(kind):
    """Exactly 256 distinct values (+0.0 and -0.0 among them: code 255 is used): 1-byte codes, products bit-identical to the
    fp64 sliced-jagged handle and inside the bound; 257 values: the handle keeps fp64 values."""
    up = _dict_matrix(256)
    D = make_ordinary(up, kind, K.NO_AUTOTUNE | K.VALUE_DICT)
    J = make_ordinary(up, kind, FMTS["sell"])
    n, ia, ja, val = up
    rp, _, v = K.expand(n, ia, ja, val)
    assert len({x.tobytes() for x in np.asarray(v, dtype=np.float64)}) == 256        # -0.0 and +0.0 are two codes
    p = K.predict_ordinary(int(rp[-1]), n, K.NO_AUTOTUNE | K.VALUE_DICT, True, 256)
    assert D.info.value_dict == p["value_dict"] == 256 and D.info.format == p["format"] == K.FORMAT_SELL
    assert D.info.device_bytes < J.info.device_bytes
    ref = run_epilogues(D, up, kind, 21, f"dict256 {kind}")
    rng = np.random.default_rng(4)
    cplx = kind != "d"
    x, z = rnd(rng, n, cplx), rnd(rng, n, cplx)
    outs = []
    for M in (D, J):
        yd = qb.DeviceVector.from_numpy(z)
        fused(M, qb.DeviceVector.from_numpy(x), yd, yd, scal(ALPHA, cplx), 0.0, 1.0)
        outs.append(yd.to_numpy())
    assert np.array_equal(outs[0], outs[1])                                             # the table holds the identical doubles
    assert ref.rows.size == n
    up2 = _dict_matrix(257)
    D2 = make_ordinary(up2, kind, K.NO_AUTOTUNE | K.VALUE_DICT)
    assert D2.info.value_dict == 0 and K.predict_ordinary(1, 1, K.NO_AUTOTUNE | K.VALUE_DICT, True, 257)["value_dict"] == 0
    run_epilogues(D2, up2, kind, 22, f"dict257 {kind}")


@pytest.mark.parametrize("kind", ["d", "z_real", "z_cplx"])
def test_host_vector_product_in_eight_chunks(kind):
    """where = QBGPU_HOST with n >= 2^20: the product runs in 8 row chunks cut on 32-row boundaries while the results are
    copied back.  beta != 0, n not a multiple of 256: bit-identical to the device product and inside the bound."""
    n0 = (1 << 20) + 4133
    rng = np.random.default_rng(8)
    up = K.band_upper(n0, 2, rng, "complex" if kind == "z_cplx" else "real")
    n = up[0]
    assert n >= 1 << 20 and n % 256
    M = make_ordinary(up, kind, 0)
    cplx = kind != "d"
    dt = np.complex128 if cplx else np.float64
    x, y0 = rnd(rng, n, cplx).astype(dt), rnd(rng, n, cplx).astype(dt)
    a, b = scal(ALPHA, cplx), scal(BETA, cplx)
    yh = y0.copy()
    M._mv(a, x, b, yh)
    yd = qb.DeviceVector.from_numpy(y0)
    M._mv(a, qb.DeviceVector.from_numpy(x), b, yd)
    assert np.array_equal(yh, yd.to_numpy())
    nn, ia, ja, val = kind_values(up, kind)
    rp, col, v = K.expand(nn, ia, ja, val)
    rows = np.unique(np.concatenate([np.random.default_rng(1).integers(0, n, 20_000), np.arange(0, n, n // 8), [n - 1]]))
    ref = K.RowRef(rp, col, v, x, rows)
    K.assert_rows(yh[rows], ref, x, y0, a, 0.0, b, cplx=cplx, what="host chunks")


def test_row_of_2_pow_24_entries_keeps_csr_vector():
    """One row of 2^24 entries: the sliced-jagged layout cannot hold it (24-bit length field).  Default create keeps the
    CSR-vector kernel and the arrays intact; QBGPU_FORMAT_SELL refuses."""
    n = (1 << 24) + 40
    h = 1 << 24
    rng = np.random.default_rng(12)
    val0 = rng.uniform(-1, 1, h)
    ia = np.zeros(n + 1, dtype=np.int64)
    ia[1:] = h
    ja = np.arange(h, dtype=np.int64)
    with pytest.raises(qb.QbgpuError, match="longer than 2\\^24-1"):
        qb.csr_mat(n, ia, ja, val0, True, flags=K.FORMAT_SELL)
    M = qb.csr_mat(n, ia, ja, val0, True)
    assert M.info.format == K.FORMAT_CSR and M.info.nnz_stored == 2 * h - 1
    # expanded: row 0 = (0..h-1, val0); rows 1..h-1 = (0, val0[j]); rows >= h empty
    rp = np.concatenate([[0, h], h + np.arange(1, h), np.full(n - h, 2 * h - 1)]).astype(np.int64)
    col = np.concatenate([np.arange(h), np.zeros(h - 1, np.int64)])
    v = np.concatenate([val0, val0[1:]])
    x = rng.uniform(-1, 1, n)
    y = np.zeros(n)
    M.MultMv(x, y)
    rows = np.concatenate([[0, 1, 2, h - 1, h, n - 1], rng.integers(0, n, 5000)])
    K.assert_rows(y[rows], K.RowRef(rp, col, v, x, rows), x, cplx=False, what="2^24 row")


# ---------------------------------------------------------------------------------------------- species order
SHAPES = {s[0]: s[1:] for s in K.species_shapes()}
SAMPLED = {"5x3_3_7": 20_000, "6x3_1_9": 40_000}                  # rows checked (all rows for the other shapes)
_REFS = {}


def species_reference(name):
    """(expanded CSR in the reference's order, rows to check).  Sectors of <= 8 sites: the numpy restatement of the
    reference's assembly (it enumerates all 4^sites occupation patterns, which takes tens of seconds per sector at 12 sites
    and is out of reach at 15 or more).  Larger ones: the matrix of the ordinary device generator, whose entries are pinned
    first by the host row function qbgpu_debug_rows_host (long double, no device): H x for a random complex x on every row
    of sectors up to 200,000 states, on 2,000 sampled rows of the larger ones."""
    if name in _REFS:
        return _REFS[name]
    Lx, Ly, nu, nd = SHAPES[name]
    ns, bonds = Lx * Ly, B.square_bonds(Lx, Ly)
    if ns <= 8:
        n, ia, ja, val = B.hubbard_upper_csr(ns, nu, nd, bonds, 1.0, 1.1, dtype=np.float64)
        rp, col, v = K.expand(n, ia, ja, val)
    else:
        P = qb.hubbard(ns, nu, nd, bonds, 1.0, 1.1, is_complex=False, flags=K.NO_AUTOTUNE | K.FORMAT_CSR)
        rp, col, v = P.download_expanded()
        n = P.dim
        P.destroy()
        rng = np.random.default_rng(17)
        rows = np.arange(n, dtype=np.int64) if n <= 200_000 else np.sort(rng.choice(n, 2_000, replace=False)).astype(np.int64)
        x = rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)
        yh = np.zeros(2 * rows.size)
        b = np.ascontiguousarray(np.asarray(bonds, dtype=np.int32).ravel())
        _lib.check(L().qbgpu_debug_rows_host(1, ns, nu, nd, len(bonds), b.ctypes.data, 0.0, 1.0, 1.1, rows.size, rows.ctypes.data,
                                              x.ctypes.data, 1, yh.ctypes.data))
        K.assert_rows(yh[0::2] + 1j * yh[1::2], K.RowRef(rp, col, v, x, rows), x, what=f"{name}: generator vs host rows")
    rows = None
    if name in SAMPLED:
        rows = np.sort(np.random.default_rng(5).choice(rp.size - 1, SAMPLED[name], replace=False)).astype(np.int64)
    _REFS[name] = (rp, col, v, rows)
    return _REFS[name]


def build_species(name, how, cplx=True):
    Lx, Ly, nu, nd = SHAPES[name]
    ns, bonds = Lx * Ly, B.square_bonds(Lx, Ly)
    n = qb.lib().qbgpu_dim_hubbard(ns, nu, nd)
    if how == "packed":
        return qb.hubbard(ns, nu, nd, bonds, 1.0, 1.1, is_complex=cplx, flags=SPECIES)
    if how == "keep_complex":
        return qb.hubbard(ns, nu, nd, bonds, 1.0, 1.1, is_complex=True, flags=SPECIES | _lib.KEEP_COMPLEX)
    if how == "rows_all":
        return qb.hubbard(ns, nu, nd, bonds, 1.0, 1.1, is_complex=cplx, flags=SPECIES, rows=(0, n))
    return qb.hubbard(ns, nu, nd, bonds, 1.0, 1.1, is_complex=cplx, flags=SPECIES, matrix_free=True)


def internal(perm, a):
    out = np.empty_like(a)
    out[perm] = a
    return out


def species_perm(name, M):
    if M.has_internal_order():
        return M.native_perm()
    # a handle built with a row range keeps no permutation of its own, but its internal order is the one of the handle
    # built without one: take the permutation from such a handle
    return build_species(name, "packed").native_perm()


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_species_packing_matches_the_prediction(name):
    """Packed parts against the handle: the local part always packs (value_dict > 0); the cross part packs unless it is
    empty (no up electron can hop: its values stay fp64, 0 entries).  Against the KEEP_COMPLEX handle a packed entry saves 16
    bytes (4 against 4 + 16), an unpacked fp64 one 8."""
    Lx, Ly, nu, nd = SHAPES[name]
    Du, Dd = K.species_dims(Lx, Ly, nu, nd)
    M, Kc = build_species(name, "packed"), build_species(name, "keep_complex")
    rp, col, v, _ = species_reference(name)
    perm = M.native_perm()
    r = np.repeat(np.arange(rp.size - 1), np.diff(rp))
    nnz_l = int(np.count_nonzero(perm[r] // Dd == perm[np.asarray(col, dtype=np.int64)] // Dd))
    nnz_c = int(rp[-1]) - nnz_l
    assert M.info.n == Du * Dd and M.info.nnz_stored == rp[-1] and Kc.info.value_dict == 0
    routes = K.species_route_table()[name]["fp64"]
    assert M.info.value_dict > 0
    assert ("empty_cross" in routes) == (nnz_c == 0)
    assert Kc.info.device_bytes - M.info.device_bytes == 16 * nnz_l + 16 * nnz_c


@pytest.mark.parametrize("how", ["packed", "keep_complex", "rows_all", "matrix_free"])
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_species_products(name, how):
    """MultMv / MultMv2 in the reference's order (host and device vectors), the fused product in the internal order
    (complex alpha, gamma, beta; z != y; z == y; dots), the two stored parts, and the Lanczos step, on each shape."""
    rp, col, v, rows = species_reference(name)
    M = build_species(name, how)
    n = M.dim
    perm = species_perm(name, M)
    Lx, Ly, nu, nd = SHAPES[name]
    Du, Dd = K.species_dims(Lx, Ly, nu, nd)
    rng = np.random.default_rng(31)
    x = rnd(rng, n, True)
    xr = rnd(rng, n, False)
    z, y0 = rnd(rng, n, True), rnd(rng, n, True)
    ref = K.RowRef(rp, col, v, x, rows)
    refr = K.RowRef(rp, col, v, xr, rows)
    sel = ref.rows
    if M.has_internal_order():
        # reference order: complex x, real-content x, host and device vectors, MultMv2
        for xx, rr, tag in ((x, ref, "complex"), (xr.astype(np.complex128), refr, "real content")):
            yh = np.full(n, 2.0 - 1.0j)
            M.MultMv(xx, yh)
            K.assert_rows(yh[sel], rr, xx, what=f"{name} {how} MultMv host {tag}")
            yd = qb.DeviceVector(n)
            M.MultMv(qb.DeviceVector.from_numpy(xx), yd)
            assert np.array_equal(yd.to_numpy(), yh), f"{name} {how}: host and device vectors differ ({tag})"
            y2 = y0.copy()
            M.MultMv2(xx, y2)
            K.assert_rows(y2[sel], rr, xx, y0, 1.0, 0.0, 1.0, what=f"{name} {how} MultMv2 {tag}")
            yd2 = qb.DeviceVector.from_numpy(y0)
            M.MultMv2(qb.DeviceVector.from_numpy(xx), yd2)
            assert np.array_equal(yd2.to_numpy(), y2), f"{name} {how}: MultMv2 with host and device vectors differ ({tag})"
            y3 = y0.copy()
            M._mv(ALPHA, xx, BETA, y3)
            K.assert_rows(y3[sel], rr, xx, y0, ALPHA, 0.0, BETA, what=f"{name} {how} zmv {tag}")
        # a complex-API handle routes real-content x through its fp64 passes: the same bits as the fp64 (d API) handle
        if how != "keep_complex":
            ya, yb = np.zeros(n, dtype=np.complex128), np.zeros(n, dtype=np.complex128)
            M.MultMv(xr.astype(np.complex128), ya)
            Mr = build_species(name, how, cplx=False)
            yr = np.zeros(n)
            Mr.MultMv(xr, yr)
            assert np.array_equal(ya.real, yr) and not ya.imag.any()
            K.assert_rows(yr[sel], refr, xr, cplx=False, what=f"{name} {how} fp64 handle")
    # internal order: fused product with complex scalars, z != y, dots
    xi, zi, y0i = internal(perm, x), internal(perm, z), internal(perm, y0)
    pos = perm[sel]                                                 # internal positions of the checked rows
    xd = qb.DeviceVector.from_numpy(xi)
    yd, zd, dots = qb.DeviceVector(n), qb.DeviceVector.from_numpy(zi), qb.DeviceVector(4, np.float64)
    fused(M, xd, zd, yd, ALPHA, GAMMA, BETA, dots)
    y = yd.to_numpy()
    K.assert_rows(y[pos], ref, x, z, ALPHA, GAMMA, BETA, what=f"{name} {how} fused")
    if rows is None:
        K.assert_dots(dots.to_numpy(), xi, y, what=f"{name} {how} fused dots")
    yd = qb.DeviceVector.from_numpy(y0i)
    fused(M, xd, yd, yd, ALPHA, 0.0, BETA)
    K.assert_rows(yd.to_numpy()[pos], ref, x, y0, ALPHA, 0.0, BETA, what=f"{name} {how} fused z == y")
    yd = qb.DeviceVector.from_numpy(y0i)
    fused(M, xd, yd, yd, 1.0, 0.0, 1.0)
    K.assert_rows(yd.to_numpy()[pos], ref, x, y0, 1.0, 0.0, 1.0, what=f"{name} {how} fused y += Hx")
    # fp64 vectors in the internal order (real view / fp64 handle), with an x that is only 8-byte aligned
    if how != "keep_complex":
        Mr = M.real_view() if how != "matrix_free" else build_species(name, how, cplx=False)
        xri = internal(perm, xr)
        buf = qb.DeviceVector(n + 1, np.float64)
        _lib.check(L().qbgpu_memcpy_h2d(C.c_void_p(buf.ptr + 8), C.c_void_p(xri.ctypes.data), 8 * n))
        for xv, tag in ((qb.DeviceVector.from_numpy(xri), "aligned"), (buf.view(1, n), "8-byte aligned")):
            yd, dots = qb.DeviceVector(n, np.float64), qb.DeviceVector(4, np.float64)
            fused(Mr, xv, None, yd, 0.9, 0.0, 0.0, dots)
            yr = yd.to_numpy()
            K.assert_rows(yr[pos], refr, xr, alpha=0.9, cplx=False, what=f"{name} {how} fp64 fused {tag}")
            if rows is None:
                K.assert_dots(dots.to_numpy(), xri, yr, cplx=False, what=f"{name} {how} fp64 dots")
            if tag == "aligned":
                y_al = yr
            else:
                assert np.array_equal(yr, y_al)
        # real parts of a complex x with zero imaginary parts: the same bits as the fp64 vectors
        if how == "packed":
            yc = qb.DeviceVector(n)
            fused(M, qb.DeviceVector.from_numpy(xri.astype(np.complex128)), None, yc, 0.9, 0.0, 0.0)
            ycn = yc.to_numpy()
            K.assert_rows(ycn[pos], refr, xr, alpha=0.9, what=f"{name} {how} complex zero-imag")
            assert np.array_equal(ycn.real, y_al) and not ycn.imag.any(), f"{name}: complex zero-imag and fp64 vectors differ"
    # Lanczos step a, complex vectors (dots fused into the closing pass, scaled by sx)
    sx, sz, bp = STATE
    st = qb.DeviceVector.from_numpy(np.array([sx, sz, bp, 0, 0, 0, 0, 0], dtype=np.float64))
    uz = qb.DeviceVector.from_numpy(y0i)
    _lib.check(L().qbgpu_lanczos_step_a(M.handle, vp(xd), vp(uz), vp(st)))
    w = uz.to_numpy()
    K.assert_rows(w[pos], ref, x, y0, sx, 0.0, -bp * sz, what=f"{name} {how} lanczos_step_a")
    dot = np.sum((np.conj(sx * xi.astype(K.CLD)) * w.astype(K.CLD)).real)
    assert abs(st.to_numpy()[3] - float(dot)) <= 8 * K.U_RND * n * sx * float(np.sum(np.abs(xi) * np.abs(w))), f"{name} {how} state[3]"
    # the two stored parts: local part y = alpha*H_loc x + gamma x + beta z, then cross part y += alpha*H_cross x
    if how in ("packed", "keep_complex", "rows_all"):
        loc, cross = M.species_parts()
        perm_inv = np.empty_like(perm); perm_inv[perm] = np.arange(n, dtype=perm.dtype)
        same_block = lambda r, c: perm[r] // Dd == perm[c] // Dd            # noqa: E731 (reference-order rows and columns)
        rpl, cl, vl = K.csr_rows_of(rp, col, v, same_block)
        refl = K.RowRef(rpl, cl, vl, x, rows)
        yd, zd = qb.DeviceVector(n), qb.DeviceVector.from_numpy(zi)
        fused(loc, xd, zd, yd, ALPHA, GAMMA, BETA)
        K.assert_rows(yd.to_numpy()[pos], refl, x, z, ALPHA, GAMMA, BETA, what=f"{name} {how} local part")
        fused(cross, xd, yd, yd, ALPHA, 0.0, 1.0)
        K.assert_rows(yd.to_numpy()[pos], ref, x, z, ALPHA, GAMMA, BETA, what=f"{name} {how} local + cross parts")


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_species_stored_kinds_give_identical_bits(name):
    """The stored kinds accumulate every row in the same order, so their products are the same bits: packed entry words,
    fp64 values (a handle built with a row range covering all rows) and complex values (QBGPU_KEEP_COMPLEX), with complex
    vectors; packed and fp64 values with fp64 vectors; and a complex x with zero imaginary parts gives, in its real parts,
    the bits of the fp64 vectors.  Between these the routes differ: block-local against plain pass 1 (4x4_1_7: fp64 blocks
    fit the shared memory, complex ones do not), thread-copied against bulk-copied x (5x3_3_7), packed against separate
    values in both passes."""
    rp, col, v, rows = species_reference(name)
    P, R, Kc = build_species(name, "packed"), build_species(name, "rows_all"), build_species(name, "keep_complex")
    n = P.dim
    perm = P.native_perm()
    rng = np.random.default_rng(77)
    xi, zi = rnd(rng, n, True), rnd(rng, n, True)
    xri = rnd(rng, n, False)
    ys = []
    for M in (P, R, Kc):
        yd = qb.DeviceVector(n)
        fused(M, qb.DeviceVector.from_numpy(xi), qb.DeviceVector.from_numpy(zi), yd, ALPHA, GAMMA, BETA)
        ys.append(yd.to_numpy())
    assert np.array_equal(ys[0], ys[1]), f"{name}: packed and fp64-valued parts differ (complex vectors)"
    assert np.array_equal(ys[0], ys[2]), f"{name}: packed and complex-valued parts differ (complex vectors)"
    x, z = xi[perm], zi[perm]                                       # the reference's order, for the bound
    ref = K.RowRef(rp, col, v, x, rows)
    K.assert_rows(ys[0][perm[ref.rows]], ref, x, z, ALPHA, GAMMA, BETA, what=f"{name} stored kinds")
    y64 = []
    for M in (P.real_view(), R.real_view()):
        yd = qb.DeviceVector(n, np.float64)
        fused(M, qb.DeviceVector.from_numpy(xri), None, yd, 0.9, 0.0, 0.0)
        y64.append(yd.to_numpy())
    assert np.array_equal(y64[0], y64[1]), f"{name}: packed and fp64-valued parts differ (fp64 vectors)"
    for M in (P, R, Kc):
        yd = qb.DeviceVector(n)
        fused(M, qb.DeviceVector.from_numpy(xri.astype(np.complex128)), None, yd, 0.9, 0.0, 0.0)
        yc = yd.to_numpy()
        assert np.array_equal(yc.real, y64[0]) and not yc.imag.any(), f"{name}: complex zero-imag x and fp64 x differ"


@pytest.mark.parametrize("name", ["4x3_2_4", "4x4_1_7"])
@pytest.mark.parametrize("how", ["packed", "matrix_free"])
def test_species_tile_widths(name, how, monkeypatch):
    """QBGPU_SPECIES_TILE (read at create) at 32 and at 96 (which divides neither D_dn): same bits as the default tile for the
    stored kind (the tile orders the slices, not the sums), inside the bound for both."""
    rp, col, v, rows = species_reference(name)
    base = build_species(name, how)
    n = base.dim
    x = rnd(np.random.default_rng(2), n, True)
    ref = K.RowRef(rp, col, v, x, rows)
    y_base = np.zeros(n, dtype=np.complex128)
    base.MultMv(x, y_base)
    for tile in ("32", "96"):
        monkeypatch.setenv("QBGPU_SPECIES_TILE", tile)
        M = build_species(name, how)
        monkeypatch.delenv("QBGPU_SPECIES_TILE")
        y = np.zeros(n, dtype=np.complex128)
        M.MultMv(x, y)
        K.assert_rows(y[ref.rows], ref, x, what=f"{name} {how} tile {tile}")
        if how == "packed":
            assert np.array_equal(y, y_base)


@pytest.mark.parametrize("how", ["packed", "matrix_free"])
@pytest.mark.parametrize("name", ["4x3_1_4", "4x4_1_7"])
def test_species_stateful_sequence(name, how):
    """mv_species remembers whether the last x had imaginary parts: real, complex, complex, real with beta = 0, the same with
    beta != 0, host and device vectors interleaved -- every result against the reference."""
    rp, col, v, rows = species_reference(name)
    M = build_species(name, how)
    n = M.dim
    rng = np.random.default_rng(44)
    seq = []
    for beta in (0.0, BETA):
        for cx in (False, True, True, False):
            seq.append((cx, beta))
    for k, (cx, beta) in enumerate(seq):
        x = rnd(rng, n, True) if cx else rnd(rng, n, False).astype(np.complex128)
        y0 = rnd(rng, n, True)
        ref = K.RowRef(rp, col, v, x, rows)
        dev = k % 2 == 1
        if dev:
            yd = qb.DeviceVector.from_numpy(y0)
            M._mv(ALPHA, qb.DeviceVector.from_numpy(x), beta, yd)
            y = yd.to_numpy()
        else:
            y = y0.copy()
            M._mv(ALPHA, x, beta, y)
        K.assert_rows(y[ref.rows], ref, x, y0, ALPHA, 0.0, beta, what=f"{name} {how} step {k} complex={cx} beta={beta} device={dev}")


def test_baseline_size_complex_route():
    """Hubbard 4x4, 8 + 8 electrons (n = 165,636,900): the packed handle with a genuinely complex x and complex alpha (plain
    pass 1, the packed complex ring of pass 2, 4 code bits), 10^5 seeded rows against the host row function in long double;
    then the fp64 fused product in the internal order with dots.  Needs ~29 GB for the handle and ~16 GB of vectors."""
    torch = pytest.importorskip("torch")
    free = torch.cuda.mem_get_info()[0] if torch.cuda.is_available() else 0
    if free < 64 * 2 ** 30:
        pytest.skip(f"needs ~64 GB of free device memory, {free / 2 ** 30:.1f} GB free")
    t0 = time.time()
    ns, nu, nd = 16, 8, 8
    bonds = B.square_bonds(4, 4)
    barr = np.ascontiguousarray(np.asarray(bonds, dtype=np.int32).ravel())
    M = qb.hubbard(ns, nu, nd, bonds, 1.0, 1.1, flags=SPECIES)
    n = M.dim
    assert n == 165_636_900 and M.info.value_dict > 0 and K.packed_col_bits(n) == 28
    rng = np.random.default_rng(2024)
    x = (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex128)
    xd, yd = qb.DeviceVector.from_numpy(x), qb.DeviceVector(n)
    M._mv(ALPHA, xd, 0.0, yd)
    y = yd.to_numpy()
    del yd
    rows = np.sort(rng.choice(n, 100_000, replace=False)).astype(np.int64)

    def host_rows(xh, cplx, t=1.0, U=1.1):
        out = np.zeros(2 * rows.size)
        _lib.check(L().qbgpu_debug_rows_host(1, ns, nu, nd, len(bonds), barr.ctypes.data, 0.0, t, U, rows.size, rows.ctypes.data,
                                              xh.ctypes.data, int(cplx), out.ctypes.data))
        return out[0::2] + 1j * out[1::2]

    # the bound with sum_j |h_ij||x_j| <= |H_ii x_i| + t * (off-diagonal entries <= 2 * bonds) * max|x|
    def check(yv, xh, cplx, alpha, what):
        want = alpha * host_rows(xh, cplx)
        diag = np.abs(host_rows(xh, cplx, t=0.0))
        m = abs(alpha) * (diag + 1.0 * 2 * len(bonds) * np.max(np.abs(xh)))
        bnd = 8 * K.U_RND * (2 * len(bonds) + 1 + 4) * m + 4 * K.U_RND * np.abs(want)
        bad = np.nonzero(np.abs(yv - want) > bnd)[0]
        assert bad.size == 0, f"{what}: {bad.size} rows break the bound, first row {rows[bad[0]]}: {yv[bad[0]]} vs {want[bad[0]]}"

    check(y[rows], x, True, ALPHA, "config 3 complex")
    del y
    # fp64 vectors, internal order, fused product with dots
    Mr = M.real_view()
    xr = rng.uniform(-1, 1, n)
    xrd = qb.DeviceVector.from_numpy(xr)
    xn = Mr.to_native(xrd)
    yn, dots = qb.DeviceVector(n, np.float64), qb.DeviceVector(4, np.float64)
    fused(Mr, xn, None, yn, 1.0, 0.0, 0.0, dots)
    yr = Mr.from_native(yn).to_numpy()
    check(yr[rows].astype(np.complex128), xr, False, 1.0, "config 3 fp64 fused")
    d = dots.to_numpy()
    ynh, xnh = yn.to_numpy(), xn.to_numpy()
    dot, nrm, mag = K.LD(0), K.LD(0), 0.0
    for s in range(0, n, 1 << 24):
        a, b = xnh[s:s + (1 << 24)].astype(K.LD), ynh[s:s + (1 << 24)].astype(K.LD)
        dot += np.sum(a * b); nrm += np.sum(b * b); mag += float(np.sum(np.abs(a * b)))
    assert abs(d[0] - float(dot)) <= 4 * K.U_RND * n * mag and abs(d[2] - float(nrm)) <= 4 * K.U_RND * n * float(nrm)
    print(f"baseline-size test: {time.time() - t0:.1f} s")
