"""Shared helpers of the vector-pass tests (TEST INFRASTRUCTURE; importable without a GPU).

The Krylov drivers run BLAS-1-like passes around every product (quantum_basis_b200/csrc/vecops.cu: dot, nrm2, axpy, scal,
Lanczos steps b and c, the sr_val1 projection passes, the CG passes; csrc/trlan.cu: multi_dot, multi_axpy, basis_rotate).
This module restates what those passes compute, in long double, and bounds how far an fp64 result may lie from it:

  - the launch grid of the passes, as a function of the device's SM count (vecops.cu vec_grid, trlan.cu tgrid), and the
    table of lengths at which every loop of the passes takes its batch tails and more than one trip;
  - long-double references of each pass, fed with the device's own scalar inputs;
  - the error bounds below;
  - a long-double restatement of the single-GPU Lanczos loop (krylov.cu lanczos_impl) on a banded Hermitian matrix.

Elementwise passes.  y_i = p_i + s * q_i (axpy, Lanczos step b, the CG updates) or y_i = s * q_i (scal) rounds at most twice
per real component (product, then sum; once with fma) and, for a complex s, three times (two products and their sum, then the
add).  So per component

    |y_i - yhat_i| <= c * u * (|p_i| + |s| |q_i|),      c = 2 (real vectors), 4 (complex vectors), u = 2^-53,

with yhat the exact value from the same fp64 inputs.  Every element is checked.  A pass that drops element i leaves
|s q_i| >= 0.5 |s| there, a pass that applies it twice adds as much: both are more than 10^14 times the bound.

Reductions.  Every reducing pass sums in a fixed tree (common.cuh block_reduce_finalize): a thread adds the terms of its
grid-stride loop one after the other (at most T = ceil(n / (256 grid)) terms), the block adds its 32 lanes by 5 shuffles and
its 8 warps one after the other (7 adds), the last block to finish adds ceil(grid / 256) per-block partials per thread and
then the same 5 shuffles and 7 adds.  A term therefore passes through at most

    depth = T + 5 + 7 + ceil(grid / 256) + 5 + 7 + 2

roundings (the +2: the product that forms the term, and the complex term's own sum), and for every order of summation

    |s - shat| <= c * u * depth * sum_i |t_i|,           c = 2 (real terms), 4 (complex terms).

This bound tracks the depth of the tree instead of n: at n = 2^24 it is about 10^-14 * sum |t_i|, where the bound
c * u * n * sum |t_i| of kernel_routes.assert_dots allows 4 * 10^-9 * sum |t_i| and so cannot see a dropped element.  The
test inputs have |x_i| in [0.5, 1] (random sign or phase), so each |t_i| >= sum |t_i| / (4n): one dropped or doubled term
moves the sum by at least sum |t_i| / (4n), which is more than 100 times the bound at every length of the table.

The bound is not a bit-exact restatement of the tree: the library is compiled with fma contraction on, so the host and the
device may round a multiply-add differently.  Bit identity is asserted only where the operation is IEEE-rounded on both
sides (sqrt, a division, a copy) or between two device calls.
"""
import math

import numpy as np

from kernel_routes import CLD, LD, U_RND

BLOCK = 256
MAX_PARTIAL_BLOCKS = 148 * 16      # common.cuh kMaxPartialBlocks
CPU_NUM_SMS = 148                  # a B200; the GPU tests read the device's own count
LARGE = 2 ** 24 + 13               # the one length past the table, for the reductions only
LANCZOS_PRECISION = 2e-12          # krylov.cu kLanczosPrecision: the sr_val1 projection threshold


# ------------------------------------------------------------------------------------------------ grids and lengths
def _grid(n, num_sms, per_sm):
    want = max(1, -(-int(n) // BLOCK))
    return min(want, min(num_sms * per_sm, MAX_PARTIAL_BLOCKS))


def vec_grid(n, num_sms):
    """vecops.cu vec_grid: blocks of 256, at most num_sms * 8 of them (and never more than the partial buffer holds)."""
    return _grid(n, num_sms, 8)


def tgrid(n, num_sms):
    """trlan.cu tgrid: blocks of 256, at most num_sms * 4."""
    return _grid(n, num_sms, 4)


def trip_vec(num_sms):
    """S_v: elements covered by one grid-stride trip of a vecops.cu pass at its capped grid."""
    return BLOCK * vec_grid(1 << 62, num_sms)


def trip_trlan(num_sms):
    """S_t: the same for the trlan.cu passes."""
    return BLOCK * tgrid(1 << 62, num_sms)


def lengths(S, large=False):
    """The length table for one trip size S: lengths that fit one block, one trip, a trip and a bit, a whole batch of 4 strides
    and the partial batches around it."""
    out = [1, 255, 256, 257, S - 1, S, S + 1, 2 * S + 1, 4 * S - 1, 4 * S, 4 * S + 1, 4 * S + 3, 5 * S + 7]
    if large:
        out.append(LARGE)
    return out


def tail_indices(S, n):
    """Indices at which a batched loop over 2 or 4 grid strides of S elements runs a batch tail (k >= 1 of its batch) or starts
    another trip, plus the first and the last index: where a dropped or doubled element must be seen."""
    cand = {0, n - 1, S - 1, S, S + 1, 2 * S - 1, 2 * S, 2 * S + 1, 3 * S, 4 * S - 1, 4 * S, 4 * S + 1, 4 * S + 2, 5 * S, 5 * S + 6}
    return sorted(i for i in cand if 0 <= i < n)


# ------------------------------------------------------------------------------------------------ inputs
def unit_entries(n, rng, cplx):
    """Entries with |x_i| in [0.5, 1] and a random sign (real) or phase (complex)."""
    r = rng.uniform(0.5, 1.0, size=n)
    if cplx:
        return r * np.exp(2j * np.pi * rng.uniform(0.0, 1.0, size=n))
    return r * rng.choice((-1.0, 1.0), size=n)


# ------------------------------------------------------------------------------------------------ bounds
def reduce_depth(n, grid):
    T = -(-int(n) // (BLOCK * grid))
    return T + 5 + 7 + -(-grid // BLOCK) + 5 + 7 + 2


def reduce_bound(n, grid, mag, cplx):
    """Bound on |s - shat| of a reduction of n terms with sum |t_i| = mag on `grid` blocks."""
    return (4.0 if cplx else 2.0) * U_RND * reduce_depth(n, grid) * float(mag)


def sqrt_bound(n, grid, mag, cplx):
    """Bound on |sqrt(s) - sqrt(shat)| for a reduced sum of squares s (nrm2: the host takes the square root, IEEE-rounded)."""
    rel = reduce_bound(n, grid, mag, cplx) / max(float(mag), 1e-300)
    return (0.5 * rel + U_RND) * math.sqrt(float(mag)) * 1.01


def elementwise_bound(mag, cplx):
    """Per-component bound of an elementwise pass, mag_i = |p_i| + |s| |q_i| (or |s| |q_i| for scal)."""
    return (4.0 if cplx else 2.0) * U_RND * np.asarray(mag, dtype=np.float64)


def elementwise_bad(got, want_ld, mag, cplx):
    """Indices where the device's result breaks the elementwise bound (each component checked on its own)."""
    got = np.asarray(got)
    bnd = elementwise_bound(mag, cplx)
    if cplx:
        d = got.astype(CLD) - want_ld
        err = np.maximum(np.abs(d.real), np.abs(d.imag)).astype(np.float64)
    else:
        err = np.abs(got.astype(LD) - want_ld).astype(np.float64)
    return np.nonzero(~(err <= bnd))[0]


# ------------------------------------------------------------------------------------------------ references
def ld(a):
    a = np.asarray(a)
    return a.astype(CLD) if np.iscomplexobj(a) else a.astype(LD)


def dot_ref(x, y):
    """(sum conj(x_i) y_i in long double, sum |x_i| |y_i|)"""
    xl, yl = ld(x), ld(y)
    s = np.sum(np.conj(xl) * yl) if np.iscomplexobj(xl) else np.sum(xl * yl)
    return s, float(np.sum(np.abs(x) * np.abs(y)))


def nrm2sq_ref(x):
    """(sum |x_i|^2 in long double, the same: its own magnitude)"""
    xl = ld(x)
    s = np.sum(xl.real * xl.real + xl.imag * xl.imag) if np.iscomplexobj(xl) else np.sum(xl * xl)
    return s, float(s)


def axpy_ref(a, x, y):
    """(y + a x in long double, |y| + |a| |x|)"""
    return ld(y) + ld(a) * ld(x), np.abs(y) + abs(a) * np.abs(x)


def scal_ref(a, x):
    return ld(a) * ld(x), abs(a) * np.abs(x)


def lanczos_b_ref(state, ux, w):
    """Lanczos step b (vecops.cu lanczos_b_kernel) from the device's state: f = -state[3] * state[0] (one fp64 product, the
    same on both sides), uz = w + f ux.  Returns (uz in long double, its magnitudes)."""
    f = -state[3] * state[0]
    return axpy_ref(f, ux, w)


def cg_alpha(sc, cplx):
    """alpha = gamma^2 / delta of vecops.cu cg_vr_kernel, in long double, from the device's sc[0..2]."""
    g2 = LD(sc[0]) * LD(sc[0])
    if not cplx:
        return g2 / LD(sc[1])
    return g2 / CLD(complex(sc[1], sc[2]))


# The CG passes derive their scalar on the device (alpha = sc[0]^2 / delta: up to 6 roundings for a complex delta; beta^2 =
# (sqrt(sc[4]) / sc[0])^2: 5), so the scalar term of their magnitudes is counted CG_SCALAR times: c * u * CG_SCALAR >= c * u + 8 u.
CG_SCALAR = 5.0


def cg_vr_ref(sc, v, r, p, pp, cplx):
    """cg_vr: v + alpha p, r - alpha pp (alpha from sc[0..2]).  Returns (v_ld, v_mag, r_ld, r_mag, alpha)."""
    al = cg_alpha(sc, cplx)
    aa = CG_SCALAR * float(abs(al))
    return (ld(v) + al * ld(p), np.abs(v) + aa * np.abs(p), ld(r) - al * ld(pp), np.abs(r) + aa * np.abs(pp), al)


def cg_p_ref(sc0, sc4, r, p):
    """cg_p: beta = sqrt(sc[4]) / sc[0], p = r + beta^2 p, sc[5] = sc[0] beta.  Returns (p_ld, p_mag, sc5_ld)."""
    beta = np.sqrt(LD(sc4)) / LD(sc0)
    b2 = beta * beta
    return ld(r) + b2 * ld(p), np.abs(r) + CG_SCALAR * float(b2) * np.abs(p), LD(sc0) * beta


# ------------------------------------------------------------------------------------------------ banded Hermitian matrices
class Band:
    """A Hermitian band matrix given by kernel_routes.band_upper(n, m, ...) (diagonal and m upper diagonals, every entry
    stored), kept as its diagonals: diag[k][r] = H[r, r + k].  The product is written with slices."""

    def __init__(self, n, ia, ja, val, m):
        ia = np.asarray(ia, dtype=np.int64)
        self.n, self.m = int(n), int(m)
        self.diag = []
        for k in range(min(m, n - 1) + 1):
            idx = ia[:n - k] + k
            assert np.array_equal(np.asarray(ja)[idx], np.arange(k, n)), "not a full band"
            self.diag.append(np.asarray(val)[idx])

    def mul(self, x, dtype):
        """H x in the scalar type `dtype` (long double or fp64, real or complex)."""
        x = np.asarray(x).astype(dtype)
        n = self.n
        y = self.diag[0].astype(dtype) * x
        for k in range(1, len(self.diag)):
            d = self.diag[k].astype(dtype)
            y[:n - k] += d * x[k:]
            y[k:] += np.conj(d) * x[:n - k]
        return y

    def mul_abs(self, x):
        """|H| |x| in fp64 (the magnitudes of a row bound)."""
        x = np.abs(np.asarray(x))
        n = self.n
        y = np.abs(self.diag[0]) * x
        for k in range(1, len(self.diag)):
            d = np.abs(self.diag[k])
            y[:n - k] += d * x[k:]
            y[k:] += d * x[:n - k]
        return y


# ------------------------------------------------------------------------------------------------ the Lanczos loop
def lanczos_restated(H, x0, steps, dtype, phi=None, skip=None):
    """krylov.cu lanczos_impl for `steps` steps (no stop rule: the callers stop far before it could act), in the scalar type
    `dtype`.  State as on the device: U buffers unnormalised with scales sx (the newest) and sz, b_prev.
      step a: w = sx H ux - b_prev sz uz ; alpha = Re sum conj(sx ux_i) w_i
      step b: w' = w - alpha sx ux ; |w'|^2            (skip = i: element i keeps w_i, the defect the tests must see)
      step c: b_m = sqrt(|w'|^2) ; (sx, sz, b_prev) <- (1/b_m, sx, b_m)
      sr_val1 (phi given), m > 1: h = <phi, w'> ; if |h sx| > 2e-12: w' -= h phi, sx = 1/|w'|
    Returns (a[0..steps), b[1..steps]) as float64 arrays and the last two vectors, normalised."""
    one = dtype(1)
    U = [np.asarray(x0).astype(dtype), np.zeros(np.asarray(x0).size, dtype=dtype)]
    ph = None if phi is None else np.asarray(phi).astype(dtype)
    sx, sz, bprev = one, dtype(0), dtype(0)
    a, b = [], []
    for m in range(1, steps + 1):
        ux, uz = U[(m - 1) % 2], U[m % 2]
        w = sx * H.mul(ux, dtype) - (bprev * sz) * uz
        alpha = np.sum(np.conj(sx * ux) * w).real
        upd = w + (-alpha * sx) * ux
        if skip is not None:
            upd[skip] = w[skip]
        nn = np.sum((np.conj(upd) * upd).real)
        bm = np.sqrt(nn)
        a.append(alpha); b.append(bm)
        sz, sx, bprev = sx, one / bm, bm
        U[m % 2] = upd
        if ph is not None and m > 1:
            h = np.sum(np.conj(ph) * upd)
            if abs(h * sx) > LANCZOS_PRECISION:
                upd = upd - h * ph
                U[m % 2] = upd
                sx = one / np.sqrt(np.sum((np.conj(upd) * upd).real))
    vm, vm1 = U[steps % 2] * sx, U[(steps - 1) % 2] * sz
    return np.array(a, dtype=np.float64), np.array(b, dtype=np.float64), vm, vm1


def ab_deviation(a, b, a_ref, b_ref):
    """max |a - a_ref|, |b - b_ref| over the steps compared"""
    return float(max(np.abs(np.asarray(a) - a_ref).max(), np.abs(np.asarray(b) - b_ref).max()))


def lanczos_case(kind, S):
    """The Lanczos test problem at n = 4 S + 3 rows: a band of half-width 2 with |H_ij| <= 1 ("real" or "complex" values), a
    normalised start vector and a normalised phi0 (entries as unit_entries).  Returns (Band, (n, ia, ja, val), x0, phi0)."""
    from kernel_routes import band_upper
    n = 4 * S + 3
    rng = np.random.default_rng(5 if kind == "real" else 6)
    up = band_upper(n, 2, rng, kind)
    cplx = kind == "complex"
    x0 = unit_entries(n, rng, cplx)
    phi = unit_entries(n, rng, cplx)
    return Band(*up, 2), up, x0 / np.linalg.norm(x0), phi / np.linalg.norm(phi)


LANCZOS_STEPS = 20
# Tolerance on (a_m, b_m), m <= 20, of a Lanczos run of lanczos_case() against its long-double restatement.  Calibrated in
# tests/test_vector_passes_cpu.py on those matrices: an fp64 run of the same loop (another rounding of every pass) deviates by
# about 4e-16, a run whose update pass skips one element at a trip boundary by 1.7e-7 or more; the test asserts a margin of
# at least 100 on both sides.
TOL_AB = 1e-11
