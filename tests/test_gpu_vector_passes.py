"""The vector passes of the Krylov drivers (csrc/vecops.cu, csrc/trlan.cu and the reduction of csrc/common.cuh) against
long-double references, at the lengths where their loops take batch tails and more than one grid-stride trip
(tests/vector_passes.py: grids, length table, references and bounds; their calibration: tests/test_vector_passes_cpu.py).

  - the BLAS-1 C entries on windows of sentinel-filled buffers (nothing outside the window may change), n = 0, repeated
    calls (identical bits) and an interleaving of one-block and capped-grid reductions (the self-resetting ticket);
  - Lanczos steps b and c and the CG step entries, one call at a time, fed and checked with the device's own scalars;
  - the whole Lanczos loop (sr_val0, sr_val1, dnmcs) and the sharded sr_val1 loop on one rank, coefficient by coefficient;
  - thick-restart Lanczos at every multi_dot chunk remainder and the largest basis, eigenpairs known from small blocks.
"""
import ctypes as C

import numpy as np
import pytest

import kernel_routes as K
import quantum_basis_b200 as qb
import vector_passes as V
from kernel_routes import CLD, LD, U_RND
from quantum_basis_b200 import dist as qd
from quantum_basis_b200._lib import check as ok

pytestmark = pytest.mark.gpu

SENTINEL = 0x7FF4_0BAD_C0DE_0BAD         # a NaN payload no pass writes
PAD = 32                                  # guard words (8 bytes each) before and after every window


@pytest.fixture(scope="module")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def L():
    return qb.lib()


class Window:
    """A vector placed inside a larger device buffer filled with SENTINEL; shift: extra 8-byte words before the window (an
    fp64 vector 8 bytes off a 16-byte boundary).  Complex windows stay 16-byte aligned, as the library requires."""

    def __init__(self, data, shift=0):
        data = np.ascontiguousarray(data)
        self.dtype, self.n = data.dtype, data.size
        self.words = data.nbytes // 8
        self.off = PAD + shift
        host = np.full(self.off + self.words + PAD, SENTINEL, dtype=np.uint64)
        host[self.off:self.off + self.words] = data.view(np.uint64)
        self.buf = qb.DeviceVector.from_numpy(host.view(np.float64))
        self.ptr = C.c_void_p(self.buf.ptr + 8 * self.off)

    def read(self):
        """(the window's contents, whether every guard word still holds SENTINEL)"""
        h = self.buf.to_numpy().view(np.uint64)
        guards = np.concatenate([h[:self.off], h[self.off + self.words:]])
        return h[self.off:self.off + self.words].view(self.dtype).copy(), bool(np.all(guards == SENTINEL))

    def free(self):
        self.buf.free()


def same_bits(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


def dev_scalars(vals):
    return qb.DeviceVector.from_numpy(np.asarray(vals, dtype=np.float64))


# ================================================================================================= BLAS-1 C entries
def _dot(L, cplx, n, x, y):
    if cplx:
        out = (C.c_double * 2)(7.0, 7.0)
        ok(L.qbgpu_zdotc(n, x.ptr, y.ptr, out))
        return complex(out[0], out[1])
    out = C.c_double(7.0)
    ok(L.qbgpu_ddot(n, x.ptr, y.ptr, C.byref(out)))
    return out.value


def _nrm2(L, cplx, n, x):
    out = C.c_double(7.0)
    ok((L.qbgpu_dznrm2 if cplx else L.qbgpu_dnrm2)(n, x.ptr, C.byref(out)))
    return out.value


def _check_dot(got, x, y, n, num_sms, cplx, what):
    ref, mag = V.dot_ref(x, y)
    b = V.reduce_bound(n, V.vec_grid(n, num_sms), mag, cplx)
    d = complex(got) - complex(ref)
    assert abs(d.real) <= b and abs(d.imag) <= b, f"{what}: n={n} dot {got!r} vs {complex(ref)!r} (bound {b:.3g})"


def _check_nrm2(got, x, n, num_sms, cplx, what):
    ref, mag = V.nrm2sq_ref(x)
    b = V.sqrt_bound(n, V.vec_grid(n, num_sms), mag, cplx)
    assert abs(got - float(np.sqrt(ref))) <= b, f"{what}: n={n} nrm2 {got!r} vs {float(np.sqrt(ref))!r} (bound {b:.3g})"


@pytest.mark.parametrize("cplx", [False, True], ids=["d", "z"])
def test_blas1_reductions_at_every_length(L, num_sms, cplx):
    S = V.trip_vec(num_sms)
    rng = np.random.default_rng(100 + cplx)
    for n in [0] + V.lengths(S, large=True):
        x, y = V.unit_entries(n, rng, cplx), V.unit_entries(n, rng, cplx)
        wx, wy = Window(x), Window(y)
        d1 = _dot(L, cplx, n, wx, wy)
        d2 = _dot(L, cplx, n, wx, wy)
        r1 = _nrm2(L, cplx, n, wx)
        r2 = _nrm2(L, cplx, n, wx)
        assert same_bits(d1, d2) and same_bits(r1, r2), f"n={n}: a repeated reduction changed its bits"
        if n == 0:
            assert d1 == 0 and r1 == 0.0
        _check_dot(d1, x, y, n, num_sms, cplx, "dot")
        _check_nrm2(r1, x, n, num_sms, cplx, "nrm2")
        for w, want in ((wx, x), (wy, y)):                            # inputs are read only; nothing around them written
            got, guards = w.read()
            assert guards and same_bits(got, want), f"n={n}: a reduction wrote to its input or past the window"
            w.free()


@pytest.mark.parametrize("cplx", [False, True], ids=["d", "z"])
def test_blas1_updates_at_every_length(L, num_sms, cplx):
    S = V.trip_vec(num_sms)
    rng = np.random.default_rng(200 + cplx)
    a = complex(0.8, -0.55) if cplx else -0.7
    ca = (C.c_double * 2)(a.real, a.imag) if cplx else None
    for n in [0] + V.lengths(S):
        x, y = V.unit_entries(n, rng, cplx), V.unit_entries(n, rng, cplx)
        wx, wy = Window(x), Window(y)
        ok(L.qbgpu_zaxpy(n, ca, wx.ptr, wy.ptr) if cplx else L.qbgpu_daxpy(n, a, wx.ptr, wy.ptr))
        got, guards = wy.read()
        xs, xguards = wx.read()
        assert guards and xguards and same_bits(xs, x), f"n={n}: axpy wrote past its window or to x"
        want, mag = V.axpy_ref(a, x, y)
        bad = V.elementwise_bad(got, want, mag, cplx)
        assert bad.size == 0, f"n={n}: axpy breaks the bound at {bad[:8]} of {n}"
        ok(L.qbgpu_zscal(n, ca, wx.ptr) if cplx else L.qbgpu_dscal(n, a, wx.ptr))
        got, guards = wx.read()
        want, mag = V.scal_ref(a, x)
        bad = V.elementwise_bad(got, want, mag, cplx)
        assert guards and bad.size == 0, f"n={n}: scal breaks the bound at {bad[:8]} of {n} (guards intact: {guards})"
        wx.free(); wy.free()


def test_fp64_windows_8_bytes_off_a_16_byte_boundary(L, num_sms):
    S = V.trip_vec(num_sms)
    rng = np.random.default_rng(300)
    n = 4 * S + 3
    x, y = V.unit_entries(n, rng, False), V.unit_entries(n, rng, False)
    wx, wy = Window(x, shift=1), Window(y, shift=1)
    assert wx.ptr.value % 16 == 8
    _check_dot(_dot(L, False, n, wx, wy), x, y, n, num_sms, False, "ddot, shifted")
    _check_nrm2(_nrm2(L, False, n, wx), x, n, num_sms, False, "dnrm2, shifted")
    ok(L.qbgpu_daxpy(n, 0.3, wx.ptr, wy.ptr))
    ok(L.qbgpu_dscal(n, -1.1, wx.ptr))
    gy, gy_ok = wy.read()
    gx, gx_ok = wx.read()
    assert gy_ok and gx_ok
    assert V.elementwise_bad(gy, *V.axpy_ref(0.3, x, y), False).size == 0
    assert V.elementwise_bad(gx, *V.scal_ref(-1.1, x), False).size == 0
    wx.free(); wy.free()


@pytest.mark.parametrize("cplx", [False, True], ids=["d", "z"])
def test_interleaved_one_block_and_capped_reductions(L, num_sms, cplx):
    """Every reduction leaves the shared ticket at 0 for the next: a one-block reduction, then a capped grid, then two blocks,
    then a capped grid again, each on fresh data, each within its bound."""
    S = V.trip_vec(num_sms)
    rng = np.random.default_rng(400 + cplx)
    for n in (1, 4 * S + 3, 257, 5 * S + 7, 1):
        x, y = V.unit_entries(n, rng, cplx), V.unit_entries(n, rng, cplx)
        wx, wy = Window(x), Window(y)
        _check_dot(_dot(L, cplx, n, wx, wy), x, y, n, num_sms, cplx, "interleaved dot")
        _check_nrm2(_nrm2(L, cplx, n, wy), y, n, num_sms, cplx, "interleaved nrm2")
        wx.free(); wy.free()


# ================================================================================================= Lanczos steps b and c
def diag_handle(n, cplx):
    """A diagonal matrix of size n: qbgpu_lanczos_step_b takes only n and the vector type from its handle."""
    return qb.csr_mat(n, np.arange(n + 1), np.arange(n), np.ones(n, dtype=np.complex128 if cplx else np.float64), True)


@pytest.mark.parametrize("cplx", [False, True], ids=["d", "z"])
def test_lanczos_step_b_and_c(L, num_sms, cplx):
    S = V.trip_vec(num_sms)
    rng = np.random.default_rng(500 + cplx)
    m = 3
    for n in V.lengths(S):
        M = diag_handle(n, cplx)
        ux, w = V.unit_entries(n, rng, cplx), V.unit_entries(n, rng, cplx)
        wux, wuz = Window(ux), Window(w)
        state0 = np.array([0.61, 0.87, 1.3, 1.7, 5.0, 6.0, -1.0, 8.0])
        st = dev_scalars(state0)
        ab_host = np.full(8, 9.5)
        ab = Window(ab_host)                                          # b at [0, 4), a at [4, 8); sentinel around both
        ok(L.qbgpu_lanczos_step_b(M.handle, wux.ptr, wuz.ptr, C.c_void_p(st.ptr)))
        uz, g1 = wuz.read()
        uxs, g2 = wux.read()
        s1 = st.to_numpy()
        assert g1 and g2 and same_bits(uxs, ux), f"n={n}: step b wrote past its windows or to ux"
        want, mag = V.lanczos_b_ref(state0, ux, w)
        bad = V.elementwise_bad(uz, want, mag, cplx)
        assert bad.size == 0, f"n={n}: step b breaks the bound at {bad[:8]}"
        ref6, mag6 = V.nrm2sq_ref(uz)                                 # |w'|^2 of the device's own w'
        b6 = V.reduce_bound(n, V.vec_grid(n, num_sms), mag6, cplx)
        assert abs(s1[6] - float(ref6)) <= b6, f"n={n}: state[6] {s1[6]!r} vs {float(ref6)!r}"
        assert same_bits(np.delete(s1, 6), np.delete(state0, 6)), f"n={n}: step b changed a state entry other than [6]"
        b_ptr = ab.ptr
        a_ptr = C.c_void_p(ab.ptr.value + 8 * 4)
        ok(L.qbgpu_lanczos_step_c(C.c_void_p(st.ptr), a_ptr, b_ptr, m))
        s2 = st.to_numpy()
        abv, g3 = ab.read()
        bm = np.sqrt(s1[6])                                           # IEEE sqrt and division: bit-exact on both sides
        want_ab = ab_host.copy()
        want_ab[m], want_ab[4 + m - 1] = bm, s1[3]
        assert g3 and same_bits(abv, want_ab), f"n={n}: step c wrote {abv} (want {want_ab})"
        want_s = s1.copy()
        want_s[0], want_s[1], want_s[2] = 1.0 / bm, s1[0], bm
        assert same_bits(s2, want_s), f"n={n}: step c state {s2} (want {want_s})"
        wux.free(); wuz.free(); ab.free(); st.free(); M.destroy()


# ================================================================================================= CG step entries
def row_bad(y, want_ld, H, x, gamma, cplx):
    """Rows of y = alpha H x + gamma x (alpha = +-1) that break kernel_routes' row bound (band rows: at most 5 entries)."""
    c = 8.0 if cplx else 4.0
    bnd = c * U_RND * (5 + 4) * (H.mul_abs(x) + abs(gamma) * np.abs(x))
    return np.nonzero(~(np.abs(np.asarray(y).astype(CLD) - want_ld).astype(np.float64) <= bnd))[0]


@pytest.mark.parametrize("kind", ["real", "complex"])
def test_cg_step_entries_pass_by_pass(L, num_sms, kind):
    """qbgpu_cg_restart, then qbgpu_cg_step three times, at 4 S_v + 3 rows: every batch tail of cg_vr (2 strides) and cg_p (4)
    runs.  Each call is checked against the long-double restatement fed with the device's previous vectors and sc."""
    cplx = kind == "complex"
    S = V.trip_vec(num_sms)
    n = 4 * S + 3
    rng = np.random.default_rng(600 + cplx)
    up = K.band_upper(n, 2, rng, kind)
    H = V.Band(*up, 2)
    M = qb.csr_mat(*up, True)                                         # fp64 values: a csr_mat<double>, fp64 vectors
    dt = np.complex128 if cplx else np.float64
    E0 = complex(-6.0, 0.4) if cplx else -6.0                         # below the band's spectrum (|rows| <= 5)
    e = (C.c_double * 2)(complex(E0).real, complex(E0).imag)
    v = qb.DeviceVector.from_numpy(V.unit_entries(n, rng, cplx).astype(dt))
    r, p, pp = (qb.DeviceVector(n, dt) for _ in range(3))
    for w in (r, p, pp):
        w.zero()
    sc = qb.DeviceVector(8, np.float64)
    sc.zero()
    grid = V.vec_grid(n, num_sms)
    ldt = CLD if cplx else LD
    vn, accu = C.c_double(), C.c_double()
    # restart: v /= |v| ; r = (E0 - H) v ; p = r ; accu = |r|
    v0 = v.to_numpy()
    ok(L.qbgpu_cg_restart(M.handle, e, C.c_void_p(sc.ptr), C.c_void_p(v.ptr), C.c_void_p(r.ptr), C.c_void_p(p.ptr), C.byref(vn), C.byref(accu)))
    _check_nrm2(vn.value, v0, n, num_sms, cplx, "cg_restart |v|")
    v1, r1, p1, s1 = v.to_numpy(), r.to_numpy(), p.to_numpy(), sc.to_numpy()
    assert V.elementwise_bad(v1, *V.scal_ref(1.0 / vn.value, v0), cplx).size == 0
    bad = row_bad(r1, ldt(E0) * V.ld(v1) - H.mul(v1, ldt), H, v1, E0, cplx)
    assert bad.size == 0, f"restart: r breaks the row bound at {bad[:8]}"
    assert same_bits(p1, r1) and same_bits(s1[0], accu.value) and same_bits(accu.value, np.sqrt(s1[3]))
    for step in range(3):
        v0, r0, p0, s0 = v1, r1, p1, s1
        ok(L.qbgpu_cg_step(M.handle, e, C.c_void_p(sc.ptr), C.c_void_p(v.ptr), C.c_void_p(r.ptr), C.c_void_p(p.ptr), C.c_void_p(pp.ptr), C.byref(accu)))
        v1, r1, p1, pp1, s1 = v.to_numpy(), r.to_numpy(), p.to_numpy(), pp.to_numpy(), sc.to_numpy()
        gam = complex(2.0 ** -52 - complex(E0).real, -complex(E0).imag) if cplx else 2.0 ** -52 - E0
        bad = row_bad(pp1, H.mul(p0, ldt) + ldt(gam) * V.ld(p0), H, p0, gam, cplx)
        assert bad.size == 0, f"step {step}: pp breaks the row bound at {bad[:8]}"
        # cg_vr: alpha from gamma = the previous sc[0] and delta = the product's <p, pp> (sc[1], sc[2])
        v_ld, v_mag, r_ld, r_mag, _ = V.cg_vr_ref([s0[0], s1[1], s1[2]], v0, r0, p0, pp1, cplx)
        for name, got, want, mag in (("v", v1, v_ld, v_mag), ("r", r1, r_ld, r_mag)):
            bad = V.elementwise_bad(got, want, mag, cplx)
            assert bad.size == 0, f"step {step}: {name} breaks the bound at {bad[:8]}"
        ref4, mag4 = V.nrm2sq_ref(r1)
        assert abs(s1[4] - float(ref4)) <= V.reduce_bound(n, grid, mag4, cplx), f"step {step}: sc[4]"
        # cg_p: p = r + beta^2 p, sc[5] = gamma * beta
        p_ld, p_mag, sc5 = V.cg_p_ref(s0[0], s1[4], r1, p0)
        bad = V.elementwise_bad(p1, p_ld, p_mag, cplx)
        assert bad.size == 0, f"step {step}: p breaks the bound at {bad[:8]}"
        assert abs(s1[5] - float(sc5)) <= 4 * U_RND * float(sc5), f"step {step}: sc[5] {s1[5]!r} vs {float(sc5)!r}"
        assert same_bits(s1[0], s1[5]) and same_bits(accu.value, s1[5])
    for w in (v, r, p, pp, sc):
        w.free()
    M.destroy()


# ================================================================================================= whole Lanczos loops
_REFS = {}


def lanczos_ref(kind, S, val1):
    """(case, long-double (a, b) of the first 20 steps) -- computed once per module."""
    key = (kind, S, val1)
    if key not in _REFS:
        case = V.lanczos_case(kind, S)
        H, up, x0, phi = case
        ldt = CLD if kind == "complex" else LD
        a, b, _, _ = V.lanczos_restated(H, x0, V.LANCZOS_STEPS, ldt, phi=phi if val1 else None)
        _REFS[key] = (case, a, b)
    return _REFS[key]


MAXIT = 40


@pytest.mark.parametrize("purpose", ["sr_val0", "sr_val1", "dnmcs"])
@pytest.mark.parametrize("kind", ["real", "complex"])
def test_lanczos_loop_coefficients(num_sms, kind, purpose):
    """qb.lanczos at 4 S_v + 3 rows for 20 steps: real values on a complex handle (the loop runs in real mode, fp64 vectors) and
    complex values; (a_m, b_m) against the long-double restatement of the same loop."""
    S = V.trip_vec(num_sms)
    val1 = purpose == "sr_val1"
    (H, up, x0, phi), a_ref, b_ref = lanczos_ref(kind, S, val1)
    n = H.n
    n_, ia, ja, val = up
    M = qb.csr_mat(n, ia, ja, val.astype(np.complex128), True)
    v = np.zeros((3 if val1 else 2) * n, dtype=np.complex128)
    v[:n] = x0
    if val1:
        v[2 * n:] = phi
    hess = np.zeros(2 * MAXIT)
    m = qb.lanczos(0, V.LANCZOS_STEPS, MAXIT, n, M, v, hess, purpose)
    assert m == V.LANCZOS_STEPS
    dev = V.ab_deviation(hess[MAXIT:MAXIT + m], hess[1:m + 1], a_ref, b_ref)
    assert dev <= V.TOL_AB, f"{kind} {purpose}: (a_m, b_m) deviate by {dev:.3g} from the long-double loop"
    if val1:
        for s in range(2):
            ov = abs(np.vdot(phi, v[s * n:(s + 1) * n]))
            assert ov <= 1e-12, f"returned vector {s}: <phi0, v> = {ov:.3g}"
    M.destroy()


@pytest.mark.parametrize("kind", ["real", "complex"])
def test_sharded_sr_val1_on_one_rank(num_sms, kind):
    """qbgpu_dist_lanczos_val1 on a one-rank NativeDist: the only caller of lanczos_b_phi (B = 4 real, 2 complex strides),
    lanczos_c_phi and lanczos_project, held to the same restatement."""
    S = V.trip_vec(num_sms)
    cplx = kind == "complex"
    (H, up, x0, phi), a_ref, b_ref = lanczos_ref(kind, S, True)
    n = H.n
    dt = np.complex128 if cplx else np.float64
    part = qb.csr_mat(*up, True, rows=(0, n))                          # fp64 values: fp64 vectors; complex: complex
    D = qd.NativeDist(qb, n, [0, n], 0, 1, cplx, lambda b: [b])
    ph = qb.DeviceVector.from_numpy(phi.astype(dt))
    try:
        D.upload_own(0, x0.astype(dt))
        D.barrier()
        m, hess = D.lanczos_val1(None, part, ph.ptr, V.LANCZOS_STEPS, MAXIT)
        assert m == V.LANCZOS_STEPS
        dev = V.ab_deviation(hess[MAXIT:MAXIT + m], hess[1:m + 1], a_ref, b_ref)
        assert dev <= V.TOL_AB, f"{kind}: (a_m, b_m) deviate by {dev:.3g} from the long-double loop"
        for b in range(2):
            ov = abs(np.vdot(phi, D.download_own(b)))
            assert ov <= 1e-12, f"returned vector {b}: <phi0, v> = {ov:.3g}"
    finally:
        D.destroy()
        ph.free()
        part.destroy()


# ================================================================================================= thick-restart Lanczos
N_LO, N_HI = 40, 24


def _dense_block(w, rng, cplx):
    """A dense Hermitian block with eigenvalues w, as an upper CSR, and the block itself."""
    m = len(w)
    Z = rng.normal(size=(m, m)) + (1j * rng.normal(size=(m, m)) if cplx else 0.0)
    Q, _ = np.linalg.qr(Z)
    A = (Q * np.asarray(w)) @ Q.conj().T
    A = 0.5 * (A + A.conj().T)
    ia = np.concatenate([[0], np.cumsum(np.arange(m, 0, -1))]).astype(np.int64)
    ja = np.concatenate([np.arange(r, m) for r in range(m)]).astype(np.int64)
    val = np.concatenate([A[r, r:] for r in range(m)])
    return (m, ia, ja, val if cplx else val.real.copy()), (A if cplx else A.real.copy())


_TRLAN = {}


def trlan_case(kind, St):
    """block_diag(dense 40 x 40 with the lowest levels, band of half-width 2, dense 24 x 24 with the highest levels), n = 4 S_t + 5."""
    key = (kind, St)
    if key not in _TRLAN:
        cplx = kind == "complex"
        rng = np.random.default_rng(700 + cplx)
        w_lo = np.concatenate([[-40.0, -35.0, -31.0, -28.0], np.linspace(-26.0, -12.0, N_LO - 4)])
        w_hi = np.concatenate([[40.0, 35.0, 31.0, 28.0], np.linspace(26.0, 12.0, N_HI - 4)])
        lo, A_lo = _dense_block(w_lo, rng, cplx)
        hi, A_hi = _dense_block(w_hi, rng, cplx)
        n = 4 * St + 5
        band = K.band_upper(n - N_LO - N_HI, 2, rng, kind)           # rows of at most 5 entries of |.| <= 1: spectrum in [-5, 5]
        _TRLAN[key] = (K.block_diag_upper(lo, band, hi), A_lo, V.Band(*band, 2), A_hi)
    return _TRLAN[key]


def trlan_residual_rows(A_lo, B, A_hi, U, theta):
    """|H u - theta u| per row, in long double, for each column u of U."""
    out = []
    for j in range(U.shape[1]):
        u = U[:, j]
        ldt = CLD if np.iscomplexobj(u) else LD
        ul = u.astype(ldt)
        r_lo = A_lo.astype(ldt) @ ul[:N_LO]
        r_mid = B.mul(u[N_LO:B.n + N_LO], ldt)
        r_hi = A_hi.astype(ldt) @ ul[N_LO + B.n:]
        r = np.concatenate([r_lo, r_mid, r_hi]) - ldt(theta[j]) * ul
        out.append(np.abs(r).astype(np.float64))
    return np.stack(out, axis=1)


# On a B200 (1000 W): eigenvalue errors up to 1.8e-13, max |V^H V - I| up to 5.6e-15, row residuals up to 7.2e-14 in the small
# block and 3.5e-14 outside it (|H| <= 40).  One wrong row of a returned vector leaves a residual of about 0.06 there.
TOL_EIG = 1e-11
TOL_ORTH = 1e-12
TOL_ROW = 1e-12


@pytest.mark.parametrize("largest", [False, True], ids=["lowest", "largest"])
@pytest.mark.parametrize("ncv,nev", [(9, 2), (16, 3), (17, 4), (48, 4)])
@pytest.mark.parametrize("kind", ["real", "complex"])
def test_trlan_eigenpairs_per_row(num_sms, kind, ncv, nev, largest):
    """qb.trlan at n = 4 S_t + 5: multi_dot / multi_axpy in chunks of 8 with every remainder (ncv = 9, 16, 17: 1, 0 and 1 column
    in the last chunk, and all remainders on the way up) and basis_rotate at m = 48.  The extreme levels are those of the small
    dense blocks; every row of every returned vector is checked through its residual."""
    St = V.trip_trlan(num_sms)
    (n, ia, ja, val), A_lo, B, A_hi = trlan_case(kind, St)
    M = qb.csr_mat(n, ia, ja, val, True)
    nconv, ev, U, nprod = qb.trlan(M, nev, ncv, largest=largest)
    M.destroy()
    assert nconv == nev
    want = np.sort(np.linalg.eigvalsh(A_hi))[::-1][:nev] if largest else np.linalg.eigvalsh(A_lo)[:nev]
    assert np.abs(ev - want).max() <= TOL_EIG, f"eigenvalues {ev} vs {want}"
    G = U.conj().T @ U
    assert np.abs(G - np.eye(nev)).max() <= TOL_ORTH, f"max |V^H V - I| = {np.abs(G - np.eye(nev)).max():.3g}"
    R = trlan_residual_rows(A_lo, B, A_hi, U, ev)
    blk = slice(N_LO + B.n, n) if largest else slice(0, N_LO)
    outside = np.ones(n, dtype=bool)
    outside[blk] = False
    worst_in, worst_out = R[blk].max(), R[outside].max()
    bad = np.nonzero(R.max(axis=1) > TOL_ROW)[0]
    assert bad.size == 0, f"{bad.size} rows break the residual tolerance; first {bad[:8]} (worst in the block {worst_in:.3g}, outside {worst_out:.3g})"
