"""CPU checks of the vector-pass test helpers (tests/vector_passes.py): the grid and length tables, and that every bound and
the Lanczos tolerance accept correct fp64 results (the long-double reference itself, numpy's fp64 in another summation order)
and reject a result with one element dropped or doubled at each batch tail of the length table."""
import numpy as np
import pytest

import vector_passes as V
from kernel_routes import LD

S_V, S_T = V.trip_vec(V.CPU_NUM_SMS), V.trip_trlan(V.CPU_NUM_SMS)


def test_grids_and_length_tables():
    assert (S_V, S_T) == (303104, 151552)                       # 148 SMs: 1184 and 592 blocks of 256
    for f, cap in ((V.vec_grid, 1184), (V.tgrid, 592)):
        assert [f(n, 148) for n in (0, 1, 256, 257, 256 * cap, 256 * cap + 1, V.LARGE)] == [1, 1, 1, 2, cap, cap, cap]
    assert V.vec_grid(1 << 40, 400) == V.MAX_PARTIAL_BLOCKS     # the partial buffer caps any grid
    for S in (S_V, S_T):
        L = V.lengths(S, large=True)
        assert L[-1] == V.LARGE and len(set(L)) == len(L) == 14
        assert {4 * S - 1, 4 * S, 4 * S + 1, 4 * S + 3, 5 * S + 7} <= set(L)
    # every batch tail of a 4-stride loop below 5S+7: k = 1, 2, 3 of the first batch and the second trip's start
    ti = V.tail_indices(S_V, 5 * S_V + 7)
    assert {S_V, 2 * S_V, 3 * S_V, 4 * S_V - 1, 4 * S_V, 4 * S_V + 2, 5 * S_V + 6} <= set(ti)


def _complex_err(got, want):
    d = complex(got) - complex(want)
    return max(abs(d.real), abs(d.imag))


@pytest.mark.parametrize("cplx", [False, True], ids=["real", "complex"])
def test_reduction_bounds_accept_fp64_and_reject_one_term(cplx):
    rng = np.random.default_rng(11 + cplx)
    for n in V.lengths(S_V, large=True):
        x, y = V.unit_entries(n, rng, cplx), V.unit_entries(n, rng, cplx)
        g = V.vec_grid(n, V.CPU_NUM_SMS)
        # dot: sum conj(x) y
        ref, mag = V.dot_ref(x, y)
        b = V.reduce_bound(n, g, mag, cplx)
        terms = np.conj(x) * y
        s64 = np.sum(terms)                                        # pairwise: another order than the device's tree
        assert _complex_err(complex(ref), ref) == 0.0 and _complex_err(s64, ref) <= b, n
        for j in V.tail_indices(S_V, n):
            for wrong in (s64 - terms[j], s64 + terms[j]):
                assert _complex_err(wrong, ref) > 100 * b, (n, j)
        # nrm2: sum |x|^2, and its square root
        ref2, mag2 = V.nrm2sq_ref(x)
        b2, bs = V.reduce_bound(n, g, mag2, cplx), V.sqrt_bound(n, g, mag2, cplx)
        sq = np.abs(x) ** 2
        s2 = np.sum(sq)
        assert abs(LD(s2) - ref2) <= b2 and abs(np.sqrt(s2) - np.sqrt(ref2)) <= bs
        for j in V.tail_indices(S_V, n):
            for wrong in (s2 - sq[j], s2 + sq[j]):
                assert abs(LD(wrong) - ref2) > 100 * b2 and abs(np.sqrt(wrong) - np.sqrt(ref2)) > 100 * bs, (n, j)


@pytest.mark.parametrize("cplx", [False, True], ids=["real", "complex"])
def test_elementwise_bounds_accept_fp64_and_reject_one_element(cplx):
    rng = np.random.default_rng(21 + cplx)
    a = complex(0.8, -0.55) if cplx else -0.7
    for n in [0] + V.lengths(S_V):
        x, y, z, w = (V.unit_entries(n, rng, cplx) for _ in range(4))
        state = np.array([0.61, 0.9, 1.3, 1.7, 0, 0, 0, 0])
        sc = np.array([0.8, 1.9, -0.4 if cplx else 0.0, 0, 2.3, 0, 0, 0])
        vr = V.cg_vr_ref(sc, x, y, z, w, cplx)
        al = complex(vr[4]) if cplx else float(vr[4])
        pp = V.cg_p_ref(sc[0], sc[4], y, z)
        b2 = float(np.sqrt(sc[4]) / sc[0]) ** 2
        cases = {   # name: (fp64 result, its single-element update, long-double reference, magnitudes)
            "axpy": (y + a * x, a * x) + V.axpy_ref(a, x, y),
            "scal": (a * x, (a - 1) * x) + V.scal_ref(a, x),
            "lanczos_b": (w + (-state[3] * state[0]) * x, (-state[3] * state[0]) * x) + V.lanczos_b_ref(state, x, w),
            "cg_v": (x + al * z, al * z, vr[0], vr[1]),
            "cg_r": (y - al * w, -al * w, vr[2], vr[3]),
            "cg_p": (y + b2 * z, y + (b2 - 1) * z, pp[0], pp[1]),
        }
        for name, (got, upd, want, mag) in cases.items():
            assert V.elementwise_bad(got, want, mag, cplx).size == 0, (name, n)
            for j in V.tail_indices(S_V, n):                              # (every other element passes: checked above)
                for wrong_j in (got[j] - upd[j], got[j] + upd[j]):        # dropped, applied twice
                    assert V.elementwise_bad(np.array([wrong_j]), want[j:j + 1], mag[j:j + 1], cplx).size == 1, (name, n, j)


@pytest.fixture(scope="module", params=["real", "complex"])
def lanczos_case(request):
    return request.param, V.lanczos_case(request.param, S_V)


@pytest.mark.parametrize("val1", [False, True], ids=["sr_val0", "sr_val1"])
def test_lanczos_tolerance_is_calibrated(lanczos_case, val1):
    kind, (H, up, x0, phi) = lanczos_case
    n = H.n
    cplx = kind == "complex"
    ldt, f64 = (np.clongdouble, np.complex128) if cplx else (np.longdouble, np.float64)
    ph = phi if val1 else None
    a0, b0, vm, vm1 = V.lanczos_restated(H, x0, V.LANCZOS_STEPS, ldt, phi=ph)
    a1, b1, _, _ = V.lanczos_restated(H, x0, V.LANCZOS_STEPS, f64, phi=ph)
    assert 100 * V.ab_deviation(a1, b1, a0, b0) <= V.TOL_AB
    for j in (S_V, 4 * S_V, 4 * S_V + 2, n - 1):                   # batch tails of the 4-stride update pass, the last element
        a2, b2, _, _ = V.lanczos_restated(H, x0, V.LANCZOS_STEPS, f64, phi=ph, skip=j)
        assert V.ab_deviation(a2, b2, a0, b0) >= 100 * V.TOL_AB, j
    if val1:                                                        # the restatement projects: the vectors are orthogonal to phi0
        assert abs(complex(np.sum(np.conj(phi) * vm.astype(f64)))) < 1e-14
        assert abs(complex(np.sum(np.conj(phi) * vm1.astype(f64)))) < 1e-14
