"""Shared helpers of the kernel-route tests (TEST INFRASTRUCTURE; importable without a GPU).

  - reference products in long double, row by row, with the magnitudes the error bound needs;
  - the per-row error bound every device product is held to;
  - matrix generators with the row structures the H*v kernels special-case;
  - a route predictor that restates the launchers' documented rules (quantum_basis_b200/csrc/spmv.cu, sjds.cu,
    sjds_bulk.cu, species.cu) and the case tables the GPU tests run, each case naming the routes it takes.

The error bound.  For one row i of y = alpha*H*x + gamma*x + beta*z, computed in fp64 by any summation order,

    |y_i - yhat_i| <= c * u * (L_i + 4) * ( |alpha| * sum_j |h_ij| |x_j|  +  |gamma| |x_i|  +  |beta| |z_i| )

with yhat the exact (long double) value, L_i the number of stored entries of the row, u = 2^-53 and c = 4 for real
arithmetic, 8 for complex (a complex multiply-add rounds up to twice per component; the epilogue adds at most four more
roundings).  The bound holds for every order of summation, so it tells a correct kernel from a wrong one without
depending on which kernel ran, and it is per row: one wrong entry in one row of 10^6 fails it.  A row whose bound is 0
(no entries, no gamma or beta term) must be exactly 0 -- or exactly z_i for a product that keeps it.

The running dots (d0 + i d1 = sum conj(x_i) y_i, d2 = sum |y_i|^2 over the device's y) are held to
|d - dhat| <= c * u * n * sum |x_i| |y_i|  and  c * u * n * sum |y_i|^2, with dhat computed in long double from the same y.
"""
import math

import numpy as np

U_RND = 2.0 ** -53
LD, CLD = np.longdouble, np.clongdouble

# ------------------------------------------------------------------------------------------------ references
class RowRef:
    """H x for the rows `rows` of an expanded CSR (every entry stored; rows in CSR order), in long double.
    hx: complex128 (rounded once from long double); habs: sum_j |h_ij||x_j|; L: stored entries per row."""

    def __init__(self, rowptr, col, val, x, rows=None):
        rowptr = np.asarray(rowptr, dtype=np.int64)
        nrows = rowptr.size - 1
        rows = np.arange(nrows, dtype=np.int64) if rows is None else np.asarray(rows, dtype=np.int64)
        s, e = rowptr[rows], rowptr[rows + 1]
        L = e - s
        idx = np.repeat(s - np.concatenate(([0], np.cumsum(L)[:-1])), L) + np.arange(int(L.sum()), dtype=np.int64)
        c = np.asarray(col)[idx].astype(np.int64)
        v = np.asarray(val)[idx]
        xv = np.asarray(x)[c]
        prod = v.astype(CLD) * xv.astype(CLD)
        mag = np.abs(v).astype(LD) * np.abs(xv).astype(LD)
        seg = np.repeat(np.arange(rows.size), L)
        hx = np.zeros(rows.size, dtype=CLD)
        ha = np.zeros(rows.size, dtype=LD)
        np.add.at(hx, seg, prod)
        np.add.at(ha, seg, mag)
        self.rows, self.L = rows, L
        self.hx_ld, self.habs = hx, ha.astype(np.float64)
        self.hx = hx.astype(np.complex128)


def csr_rows_of(rowptr, col, val, keep):
    """The entries of an expanded CSR for which keep(row, col) holds (same rows): a split of H into two parts."""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    r = np.repeat(np.arange(rowptr.size - 1), np.diff(rowptr))
    k = keep(r, np.asarray(col, dtype=np.int64))
    rp = np.zeros_like(rowptr)
    np.add.at(rp, r[k] + 1, 1)
    return np.cumsum(rp), np.asarray(col)[k], np.asarray(val)[k]


def expected(ref, x, z=None, alpha=1.0, gamma=0.0, beta=0.0):
    """alpha*H x + gamma*x_i + beta*z_i on ref.rows, in long double."""
    rows = ref.rows
    want = CLD(complex(alpha)) * ref.hx_ld
    if gamma != 0:
        want = want + CLD(complex(gamma)) * np.asarray(x)[rows].astype(CLD)
    if beta != 0:
        want = want + CLD(complex(beta)) * np.asarray(z)[rows].astype(CLD)
    return want


def row_bound(ref, x, z=None, alpha=1.0, gamma=0.0, beta=0.0, cplx=True):
    c = 8.0 if cplx else 4.0
    m = abs(complex(alpha)) * ref.habs
    if gamma != 0:
        m = m + abs(complex(gamma)) * np.abs(np.asarray(x)[ref.rows])
    if beta != 0:
        m = m + abs(complex(beta)) * np.abs(np.asarray(z)[ref.rows])
    return c * U_RND * (ref.L + 4) * m


def row_errors(y_rows, ref, x, z=None, alpha=1.0, gamma=0.0, beta=0.0, cplx=True):
    """(rows that break the bound, the largest error / bound): y_rows are the device's values at ref.rows."""
    want = expected(ref, x, z, alpha, gamma, beta)
    err = np.abs(np.asarray(y_rows).astype(CLD) - want).astype(np.float64)
    bnd = row_bound(ref, x, z, alpha, gamma, beta, cplx)
    bad = np.nonzero(err > bnd)[0]
    with np.errstate(divide="ignore", invalid="ignore"):
        worst = float(np.max(np.where(bnd > 0, err / np.where(bnd > 0, bnd, 1), np.where(err > 0, np.inf, 0.0)), initial=0.0))
    return bad, worst


def assert_rows(y_rows, ref, x, z=None, alpha=1.0, gamma=0.0, beta=0.0, cplx=True, what=""):
    bad, worst = row_errors(y_rows, ref, x, z, alpha, gamma, beta, cplx)
    if bad.size:
        i = bad[0]
        want = expected(ref, x, z, alpha, gamma, beta)[i]
        raise AssertionError(f"{what}: {bad.size} of {ref.rows.size} rows break the error bound; first: row {ref.rows[i]} "
                             f"(length {ref.L[i]}) got {np.asarray(y_rows)[i]!r}, want {complex(want)!r}")
    return worst


def assert_dots(d, x_rows, y, cplx=True, what=""):
    """d[0..2] from the device against sum conj(x_i) y_i and sum |y_i|^2 of the device's own y, in long double."""
    c = 8.0 if cplx else 4.0
    xl, yl = np.asarray(x_rows).astype(CLD), np.asarray(y).astype(CLD)
    n = max(1, y.size)
    dot = np.sum(np.conj(xl) * yl)
    nrm = np.sum((np.abs(yl) ** 2).astype(LD))
    b01 = c * U_RND * n * float(np.sum(np.abs(xl) * np.abs(yl)))
    b2 = c * U_RND * n * float(nrm)
    assert abs(d[0] - float(dot.real)) <= b01 and abs(d[1] - float(dot.imag)) <= b01, f"{what}: dots {d[:2]} vs {complex(dot)}"
    assert abs(d[2] - float(nrm)) <= b2, f"{what}: |y|^2 {d[2]} vs {float(nrm)}"


# ------------------------------------------------------------------------------------------------ matrices
def band_upper(n, m, rng, kind, diag=True):
    """Hermitian band matrix of half-width m as an upper-triangle CSR (strictly ascending columns).  kind: "real" or
    "complex" values (complex: non-zero imaginary parts off the diagonal, real diagonal)."""
    rows, cols = [], []
    if diag:
        rows.append(np.arange(n)); cols.append(np.arange(n))
    for k in range(1, min(m, n - 1) + 1):
        rows.append(np.arange(n - k)); cols.append(np.arange(k, n))
    return _upper_csr(n, np.concatenate(rows) if rows else np.zeros(0, np.int64),
                      np.concatenate(cols) if cols else np.zeros(0, np.int64), rng, kind)


def designed_upper(lengths, rng, kind, diag_rows=()):
    """Rows 0..R-1 with exactly lengths[r] off-diagonal entries each (a row of length 0 without a diagonal is empty in the
    expanded matrix too), pointing at filler rows that carry one entry each (the Hermitian image).  n = R + sum(lengths)."""
    R = len(lengths)
    tot = int(sum(lengths))
    n = R + tot
    r = np.repeat(np.arange(R), lengths)
    c = R + np.arange(tot)
    d = np.asarray(sorted(diag_rows), dtype=np.int64)
    return _upper_csr(n, np.concatenate([r, d]), np.concatenate([c, d]), rng, kind)


def _upper_csr(n, r, c, rng, kind):
    r, c = np.asarray(r, dtype=np.int64), np.asarray(c, dtype=np.int64)
    o = np.lexsort((c, r))
    r, c = r[o], c[o]
    ia = np.zeros(n + 1, dtype=np.int64)
    np.add.at(ia, r + 1, 1)
    ia = np.cumsum(ia)
    v = rng.uniform(-1.0, 1.0, size=r.size)
    if kind == "complex":
        v = v + 1j * np.where(r == c, 0.0, rng.uniform(-1.0, 1.0, size=r.size))
    return n, ia, c, v


def block_diag_upper(*parts):
    """Upper CSRs (n, ia, ja, val) placed on the diagonal of one matrix."""
    n = sum(p[0] for p in parts)
    ia, ja, val, off, base = [np.zeros(1, np.int64)], [], [], 0, 0
    for (m, a, j, v) in parts:
        ia.append(a[1:] + base); ja.append(j + off); val.append(v)
        off += m; base += a[-1]
    return n, np.concatenate(ia), np.concatenate(ja), np.concatenate(val)


def expand(n, ia, ja, val):
    """Upper triangle -> every entry stored (row-sorted), the layout the device keeps (v at (i,j) and conj(v) at (j,i))."""
    r = np.repeat(np.arange(n), np.diff(ia))
    off = ja != r
    R = np.concatenate([r, ja[off]])
    Cc = np.concatenate([ja, r[off]])
    V = np.concatenate([val, np.conj(val[off])])
    o = np.lexsort((Cc, R))
    rp = np.zeros(n + 1, dtype=np.int64)
    np.add.at(rp, R + 1, 1)
    return np.cumsum(rp), Cc[o], V[o]


def lower_too(n, ia, ja, val):
    """The same Hermitian matrix given as the full (non-symmetric-storage) CSR: sym_upper = 0 input."""
    return expand(n, ia, ja, val)


# ------------------------------------------------------------------------------------------------ route predictor
NO_AUTOTUNE, FORMAT_CSR, FORMAT_SELL, VALUE_DICT, KEEP_COMPLEX = 2, 4, 8, 16, 1
BLOCK_LOCAL_MAX_BYTES = 112 * 1024


def lanes_for(nnz, nrows):
    """spmv.cu autotune: about 4 entries per lane, the count used under QBGPU_NO_AUTOTUNE."""
    mean = nnz / nrows if nrows else 0.0
    lanes = 2
    while lanes < 32 and mean > 4.0 * lanes:
        lanes *= 2
    return lanes


def predict_ordinary(nnz, nrows, flags, val_real, ndistinct=None):
    """Route of an ordinary handle created with `flags` and QBGPU_NO_AUTOTUNE (the untimed choice)."""
    out = {"lanes": lanes_for(nnz, nrows), "format": FORMAT_CSR, "value_dict": 0}
    if flags & VALUE_DICT and val_real and nnz > 0 and ndistinct is not None and ndistinct <= 256:
        out["value_dict"], out["format"] = ndistinct, FORMAT_SELL
    elif flags & FORMAT_SELL:
        out["format"] = FORMAT_SELL
    route = "sjds_dict" if out["value_dict"] else ("sjds" if out["format"] == FORMAT_SELL else f"csr_vector_{out['lanes']}")
    out["route"] = route
    return out


def packed_col_bits(n):
    return max(1, int(n - 1).bit_length())


def predict_species(Du, Dd, cplx_vec, packed_local=None, cross_nnz=1, x_aligned16=True):
    """Routes of the stored two-pass product (species.cu launch_spmv_species) for vectors of 16 (complex) or 8 bytes."""
    vb = 16 if cplx_vec else 8
    routes = []
    if Dd * vb <= BLOCK_LOCAL_MAX_BYTES:
        bulk = (Dd * vb) % 16 == 0 and Dd * vb < (1 << 20) and x_aligned16
        routes.append("pass1_block_bulk_x" if bulk else "pass1_block_thread_x")
    else:
        routes.append("pass1_plain")
    g = math.gcd(32, Dd)
    routes.append("periodic_meta" if Du >= 2 * (32 // g) else "no_periodic_meta")
    if packed_local is not None:
        routes.append("packed" if packed_local else "unpacked")
    if cross_nnz == 0:
        routes.append("empty_cross")
    if Dd == 1:
        routes.append("dn_dim_1")
    if Du * Dd < 32:
        routes.append("n_below_32")
    routes.append("pass2_bulk")
    return routes


# ------------------------------------------------------------------------------------------------ case tables
LANES = (2, 4, 8, 16, 32)
VALUE_KINDS = ("d", "z_real", "z_cplx")     # fp64 values + fp64 vectors; fp64 values + complex vectors; complex values


def lane_case(lanes, seed=0, kind="real"):
    """A matrix whose mean expanded row length makes QBGPU_NO_AUTOTUNE pick `lanes`, with rows of exactly 1, LANES,
    2*LANES-1, 2*LANES and 2*LANES+1 entries, single empty rows and a run of 70 empty rows (it holds at least one whole
    32-row slice without entries: the slice the KEEP kernel skips).  Returns the upper CSR."""
    rng = np.random.default_rng(1000 + 7 * lanes + seed)
    # designed rows: lengths (the row's own off-diagonal entries; its diagonal is added for half of them)
    L = lanes
    lengths = [1, L, 2 * L - 1, 2 * L, 2 * L + 1, 0, 0, 1, L - 1 if L > 1 else 1, 0]
    # rows 0 and 8 also get a diagonal: expanded lengths 2, L, 2L-1, 2L, 2L+1, 0, 0, 1, L, 0; the filler rows have 1
    des = designed_upper(lengths, rng, kind, diag_rows=(0, 8))
    # a band block that brings the mean expanded length to about 3 * LANES
    m = max(1, int(round((3 * L - 1) / 2)))
    band = band_upper(40 * L + 37, m, rng, kind)
    empty = (70, np.zeros(71, dtype=np.int64), np.zeros(0, dtype=np.int64), np.zeros(0))
    return block_diag_upper(des, empty, band)


def empty_slices(rowptr):
    """Indices of the 32-row slices whose rows hold no entry at all (the last, partial slice counts if its rows are empty)."""
    lens = np.diff(np.asarray(rowptr, dtype=np.int64))
    pad = np.concatenate([lens, np.zeros((-lens.size) % 32, dtype=np.int64)])
    return np.nonzero(pad.reshape(-1, 32).sum(axis=1) == 0)[0]


def species_shapes():
    """(name, Lx, Ly, N_up, N_dn): the shapes of the species-order tests (square lattice, periodic bonds)."""
    return [("2x2_1_2", 2, 2, 1, 2), ("4x3_0_0", 4, 3, 0, 0), ("4x3_5_0", 4, 3, 5, 0), ("4x3_0_4", 4, 3, 0, 4),
            ("4x3_1_4", 4, 3, 1, 4), ("4x3_2_4", 4, 3, 2, 4), ("4x4_2_1", 4, 4, 2, 1), ("4x4_1_7", 4, 4, 1, 7),
            ("5x3_3_7", 5, 3, 3, 7), ("6x3_1_9", 6, 3, 1, 9)]


def species_dims(Lx, Ly, nup, ndn):
    ns = Lx * Ly
    return math.comb(ns, nup), math.comb(ns, ndn)


def species_route_table(packed_lookup=None):
    """{shape name: {vector kind: routes}}; packed_lookup(name) -> local part packed (None: not asked)."""
    out = {}
    for (name, Lx, Ly, nu, nd) in species_shapes():
        Du, Dd = species_dims(Lx, Ly, nu, nd)
        cross_nnz = 0 if nu in (0, Lx * Ly) else 1
        pk = packed_lookup(name) if packed_lookup else None
        out[name] = {"fp64": predict_species(Du, Dd, False, pk, cross_nnz), "complex": predict_species(Du, Dd, True, pk, cross_nnz)}
    return out


def ordinary_route_table():
    """{(case, value kind, flags): predicted routes} for the lane cases of the ordinary-handle tests."""
    out = {}
    for L in LANES:
        n, ia, ja, val = lane_case(L)
        rp, _, V = expand(n, ia, ja, val)
        nnz = int(rp[-1])
        for kind in VALUE_KINDS:
            vr = kind != "z_cplx"
            for fl in (NO_AUTOTUNE | FORMAT_CSR, NO_AUTOTUNE | FORMAT_SELL, NO_AUTOTUNE | VALUE_DICT):
                p = predict_ordinary(nnz, n, fl, vr, len(np.unique(V.real)) if vr else None)
                out[(f"lanes{L}", kind, fl)] = p
    return out
