"""GPU parity tests: the CUDA path, called through the C ABI (libqbgpu.so via quantum_basis_b200), against the oracle,
the committed reference outputs (tests/golden) and the reference's published golden values.

Tolerances (BASELINE.json north_star): per-product relative l2 <= 1e-12; E0 relative <= 1e-10; KPM moments <= 1e-9.
Integer/index work (expanded layout, generator output, vec_randomize sequence) is compared exactly.
"""
import os

import numpy as np
import pytest

import lin_builders as B
import quantum_basis_b200 as qb

pytestmark = pytest.mark.gpu

ALL = ["heis12_full", "heis16_full", "heis16_k3", "tri4x4_k00", "tri4x4_k01", "tri4x4_k12", "hubbard4x2",
       "honeycomb3x2_general", "tj12"]
SMALL = [c for c in ALL if c not in ("heis16_full", "tj12")]
TOL_MV = 1e-12
TOL_E0 = 1e-10
TOL_KPM = 1e-9


def rel_l2(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def make(A, **kw):
    return qb.csr_mat(A.dim, A.ia, A.ja, A.val, A.sym, **kw)


# ------------------------------------------------------------------------------------------------ layout
@pytest.mark.parametrize("name", ALL)
def test_expanded_layout_is_exact(oracle, name):
    A, meta, ex = oracle.load_golden(name)
    M = make(A)
    rowptr, col, val = M.download_expanded()
    inf = M.info
    if A.sym:
        ia, ja, v = oracle.expand_upper(A)
    else:
        ia, ja, v = A.ia, A.ja, A.val
    assert np.array_equal(rowptr, ia)
    assert np.array_equal(col.astype(np.int64), ja)
    all_real = np.abs(A.val.imag).max() == 0.0
    assert bool(inf.val_is_real) == all_real                 # fp64 storage iff every imaginary part is exactly 0
    assert np.array_equal(val, v.real if all_real else v)    # bit-exact values (conjugated lower half)
    assert inf.nnz_stored == ia[-1] and inf.nnz_input == A.nnz and inf.n == A.dim
    K = make(A, flags=1)                                     # QBGPU_KEEP_COMPLEX
    assert not K.info.val_is_real
    assert np.array_equal(K.download_expanded()[2], v)


def test_to_dense_matches_reference_semantics(oracle):
    A, meta, ex = oracle.load_golden("honeycomb3x2_general")
    D = make(A).to_dense()
    assert np.array_equal(D, A.to_scipy_full().toarray())
    A, meta, ex = oracle.load_golden("tri4x4_k01")
    D = make(A).to_dense()
    assert np.array_equal(D, A.to_scipy_full().toarray())
    assert np.abs(D - D.conj().T).max() == 0.0


def test_create_rejects_bad_input(oracle):
    A, meta, ex = oracle.load_golden("hubbard4x2")
    ja = A.ja.copy(); ja[5] = A.dim + 3
    with pytest.raises(qb.QbgpuError):
        qb.csr_mat(A.dim, A.ia, ja, A.val, True)
    with pytest.raises(qb.QbgpuError):
        qb.csr_mat(A.dim, A.ia[:-1], A.ja, A.val, True)
    # columns of a row out of order (two referenced entries swapped): refused, not silently mis-split later
    r = int(np.argmax(np.diff(A.ia) >= 3))
    ja2, val2 = A.ja.copy(), A.val.copy()
    p = A.ia[r]
    ja2[p + 1], ja2[p + 2] = A.ja[p + 2], A.ja[p + 1]
    val2[p + 1], val2[p + 2] = A.val[p + 2], A.val[p + 1]
    with pytest.raises(qb.QbgpuError, match="ascending"):
        qb.csr_mat(A.dim, A.ia, ja2, val2, True)


# ---------------------------------------------------------------------------------------------- products
@pytest.mark.parametrize("name", ALL)
def test_multmv_matches_reference_product(oracle, name):
    A, meta, ex = oracle.load_golden(name)
    M = make(A)
    x = oracle.vec_randomize(A.dim, 1)
    y = np.full(A.dim, 7.0 + 1.0j)                           # MultMv must overwrite, not accumulate
    M.MultMv(x, y)
    assert rel_l2(y, ex["y1"]) <= TOL_MV                     # vs the compiled reference's csr_mat::MultMv
    assert rel_l2(y, oracle.spmv_ld(A, x)) <= TOL_MV         # vs the long-double arbiter
    y2 = y.copy()
    M.MultMv2(x, y2)                                         # y += H x
    assert rel_l2(y2, 2 * ex["y1"]) <= TOL_MV
    # device-resident vectors
    dx = qb.DeviceVector.from_numpy(x); dy = qb.DeviceVector(A.dim)
    M.MultMv(dx, dy)
    assert np.array_equal(dy.to_numpy(), y)                  # same kernel, same order: bit-identical
    # the untimed choice: QBGPU_NO_AUTOTUNE keeps the lane count of the mean row length (every lane count is pinned
    # against the long-double reference in test_gpu_kernel_routes.py)
    for flags in (2,):
        y3 = np.zeros(A.dim, dtype=np.complex128)
        make(A, flags=flags).MultMv(x, y3)
        assert rel_l2(y3, ex["y1"]) <= TOL_MV
    # complex values kept complex
    y4 = np.zeros(A.dim, dtype=np.complex128)
    make(A, flags=1).MultMv(x, y4)
    assert rel_l2(y4, ex["y1"]) <= TOL_MV


@pytest.mark.parametrize("name", ALL)
def test_sliced_jagged_layout_gives_the_same_product(oracle, name):
    """QBGPU_FORMAT_SELL (8): in-place re-ordering of every 32-row slice; QBGPU_FORMAT_CSR (4): forced CSR-vector."""
    A, meta, ex = oracle.load_golden(name)
    x = oracle.vec_randomize(A.dim, 1)
    J = make(A, flags=8)
    assert J.info.format == 8
    C4 = make(A, flags=4 | 2)
    assert C4.info.format == 4
    yj = np.zeros(A.dim, dtype=np.complex128); yc = np.zeros_like(yj)
    J.MultMv(x, yj); C4.MultMv(x, yc)
    assert rel_l2(yj, ex["y1"]) <= TOL_MV and rel_l2(yc, ex["y1"]) <= TOL_MV
    # the conversion is a pure permutation: converting back returns the exact CSR arrays
    rp, cj, vj = J.download_expanded()
    rp2, cc, vc = C4.download_expanded()
    assert np.array_equal(rp, rp2) and np.array_equal(cj, cc) and np.array_equal(vj, vc)
    assert J.info.format == 8                                   # and the resident layout is restored afterwards
    y2 = np.zeros_like(yj)
    J.MultMv(x, y2)
    assert np.array_equal(y2, yj)
    # fused Lanczos on the jagged layout
    v = np.zeros(2 * A.dim, dtype=np.complex128); v[:A.dim] = x
    hess = np.zeros(2000)
    m = qb.lanczos(0, 999, 1000, A.dim, J, v, hess, "sr_val0")
    ritz, _ = qb.hess_eigen(hess, 1000, m)
    assert abs(ritz[0] - meta["lanczos_E0"]) <= TOL_E0 * abs(meta["lanczos_E0"])


@pytest.mark.parametrize("name", ALL)
def test_value_dictionary_is_lossless(oracle, name):
    """QBGPU_VALUE_DICT (16): fp64 values replaced by 1-byte codes when there are <= 256 distinct ones."""
    A, meta, ex = oracle.load_golden(name)
    x = oracle.vec_randomize(A.dim, 1)
    D = make(A, flags=16 | 2)
    J = make(A, flags=8 | 2)
    all_real = np.abs(A.val.imag).max() == 0.0
    ndistinct = len(np.unique(oracle.expand_upper(A)[2].real)) if (all_real and A.sym) else None
    inf = D.info
    if all_real and ndistinct is not None and ndistinct <= 256:
        assert inf.value_dict == ndistinct and inf.format == 8
        assert inf.device_bytes < J.info.device_bytes
    if not all_real:
        assert inf.value_dict == 0                           # complex values are left alone
    yd = np.zeros(A.dim, dtype=np.complex128); yj = np.zeros_like(yd)
    D.MultMv(x, yd); J.MultMv(x, yj)
    if inf.value_dict:
        assert np.array_equal(yd, yj)                        # decoded values are the identical doubles, same kernel order
    else:
        assert rel_l2(yd, yj) <= 1e-14
    assert rel_l2(yd, ex["y1"]) <= TOL_MV
    rp, c1, v1 = D.download_expanded()
    rp2, c2, v2 = J.download_expanded()
    assert np.array_equal(rp, rp2) and np.array_equal(c1, c2) and np.array_equal(v1, v2)
    v = np.zeros(2 * A.dim, dtype=np.complex128); v[:A.dim] = x
    hess = np.zeros(2000)
    m = qb.lanczos(0, 999, 1000, A.dim, D, v, hess, "sr_val0")
    ritz, _ = qb.hess_eigen(hess, 1000, m)
    assert abs(ritz[0] - meta["lanczos_E0"]) <= TOL_E0 * abs(meta["lanczos_E0"])


@pytest.mark.parametrize("name", ["heis12_full", "hubbard4x2", "tri4x4_k00", "tj12"])
def test_double_precision_real_matrix_path(oracle, name):
    """csr_mat<double> (reachable in the reference only by constructing it directly, SURVEY F3)."""
    A, meta, ex = oracle.load_golden(name)
    assert np.abs(A.val.imag).max() == 0.0
    Ad = A.astype(np.float64)
    M = make(Ad)
    assert not M.is_complex
    x = oracle.vec_randomize(A.dim, 1, dtype=np.float64)
    y = np.zeros(A.dim)
    M.MultMv(x, y)
    assert rel_l2(y, ex["y1"].real) <= TOL_MV
    assert rel_l2(y, oracle.spmv(Ad, x)) <= TOL_MV
    hess = np.zeros(2000)
    v = np.zeros(2 * A.dim); v[:A.dim] = x
    m = qb.lanczos(0, 999, 1000, A.dim, M, v, hess, "sr_val0")
    ritz, _ = qb.hess_eigen(hess, 1000, m)
    assert abs(ritz[0] - meta["lanczos_E0"]) <= TOL_E0 * abs(meta["lanczos_E0"])


def test_complex_x_with_nonzero_imag(oracle):
    A, meta, ex = oracle.load_golden("tri4x4_k12")
    rng = np.random.default_rng(5)
    x = rng.normal(size=A.dim) + 1j * rng.normal(size=A.dim)
    for flags in (0, 1):
        y = np.zeros(A.dim, dtype=np.complex128)
        make(A, flags=flags).MultMv(x, y)
        assert rel_l2(y, oracle.spmv_ld(A, x)) <= TOL_MV
    A, meta, ex = oracle.load_golden("hubbard4x2")           # real values, complex vector
    x = rng.normal(size=A.dim) + 1j * rng.normal(size=A.dim)
    y = np.zeros(A.dim, dtype=np.complex128)
    make(A).MultMv(x, y)
    assert rel_l2(y, oracle.spmv_ld(A, x)) <= TOL_MV


def test_row_shards_reproduce_the_full_product(oracle):
    A, meta, ex = oracle.load_golden("tj12")
    x = oracle.vec_randomize(A.dim, 1)
    L = qb.lib()
    for parts in (2, 3):
        b = np.zeros(parts + 1, dtype=np.int64)
        assert L.qbgpu_partition_rows(A.dim, A.ia.ctypes.data, A.ia.ctypes.data + 8, A.ja.ctypes.data, 1, parts, b.ctypes.data) == 0
        ys = []
        for p in range(parts):
            S = qb.csr_mat(A.dim, A.ia, A.ja, A.val, True, rows=(b[p], b[p + 1]))
            y = np.zeros(b[p + 1] - b[p], dtype=np.complex128)
            S.MultMv(x, y)
            ys.append(y)
        assert rel_l2(np.concatenate(ys), ex["y1"]) <= TOL_MV


@pytest.mark.parametrize("name,nparts,shard", [("tj12", 8, None), ("heis16_full", 8, None), ("heis16_full", 3, None), ("tri4x4_k12", 5, None),
                                               ("tj12", 8, (0.375, 0.5)), ("heis16_full", 8, (0.125, 0.25)), ("heis16_full", 8, (0.875, 1.0))])
def test_column_blocks_reproduce_the_fused_step(oracle, name, nparts, shard):
    """qbgpu_split_columns + qbgpu_lanczos_step_a_part (what every rank does in the overlapped multi-GPU exchange) on ONE
    GPU: the per-owner column blocks, multiplied one after the other with the accumulate flags, must give the same w and
    the same alpha as the unsplit fused step -- for complex and for fp64 (real-view) vectors."""
    import ctypes as C
    A, meta, ex = oracle.load_golden(name)
    L = qb.lib()
    n = A.dim
    lo, hi = (0, n) if shard is None else (int(shard[0] * n), int(shard[1] * n))     # a rank's row block (row_lo != 0)
    M = make(A) if shard is None else make(A, rows=(lo, hi))
    nl = hi - lo
    chunk = (n + nparts - 1) // nparts
    bounds = np.array([min(n, p * chunk) for p in range(nparts)] + [n], dtype=np.int64)
    real_ok = bool(M.info.val_is_real)
    for part_flags, real in [(f, r) for f in (0, 4 | 2, 8 | 2) for r in ([False, True] if real_ok else [False])]:
        # part layouts: autotuned, forced CSR-vector, forced sliced-jagged
        hs = (C.c_void_p * nparts)()
        assert L.qbgpu_split_columns(M.handle, nparts, bounds.ctypes.data, hs, part_flags) == 0, L.qbgpu_last_error()
        parts = [qb.csr_mat._adopt(C.c_void_p(hs[p]), True) for p in range(nparts)]
        assert sum(p.info.nnz_stored for p in parts) == M.info.nnz_stored
        dt = np.float64 if real else np.complex128
        H = M.real_view() if real else M
        P = [p.real_view() for p in parts] if real else parts
        rng = np.random.default_rng(3)
        ux = rng.normal(size=n) if real else rng.normal(size=n) + 1j * rng.normal(size=n)
        uz0 = rng.normal(size=nl) if real else rng.normal(size=nl) + 1j * rng.normal(size=nl)
        state0 = np.array([0.7, 1.3, 0.9, 0, 0, 0, 0, 0], dtype=np.float64)       # sx, sz, b_prev
        dux = qb.DeviceVector.from_numpy(ux.astype(dt))
        # unsplit
        duz = qb.DeviceVector.from_numpy(uz0.astype(dt)); st = qb.DeviceVector.from_numpy(state0)
        assert L.qbgpu_lanczos_step_a(H.handle, C.c_void_p(dux.ptr), C.c_void_p(duz.ptr), C.c_void_p(st.ptr)) == 0
        w_ref, a_ref = duz.to_numpy(), st.to_numpy()[3]
        w_exact = 0.7 * oracle.spmv_ld(A, ux)[lo:hi] - 0.9 * 1.3 * uz0
        assert rel_l2(w_ref, w_exact if not real else w_exact.real) <= TOL_MV
        assert abs(a_ref - np.real(np.vdot(0.7 * ux[lo:hi], w_ref))) <= 1e-12 * abs(a_ref)
        # per-owner blocks, own block first (rank r = 2 of nparts), the others in ring order
        order = [2 % nparts] + [(2 + d) % nparts for d in range(1, nparts)]
        duz2 = qb.DeviceVector.from_numpy(uz0.astype(dt)); st2 = qb.DeviceVector.from_numpy(state0)
        for idx, p in enumerate(order):
            rc = L.qbgpu_lanczos_step_a_part(P[p].handle, C.c_void_p(dux.ptr), C.c_void_p(duz2.ptr), C.c_void_p(st2.ptr),
                                             int(idx == 0), int(idx == nparts - 1))
            assert rc == 0, L.qbgpu_last_error()
        w_blk, a_blk = duz2.to_numpy(), st2.to_numpy()[3]
        assert rel_l2(w_blk, w_ref) <= 1e-14
        assert abs(a_blk - a_ref) <= 1e-12 * abs(a_ref)
        # and the plain accumulate form (y = sum_p H_p x)
        y = qb.DeviceVector(nl, dt)
        for idx, p in enumerate(order):
            P[p]._mv(complex(1.0), dux, complex(1.0 if idx else 0.0), y)
        assert rel_l2(y.to_numpy(), oracle.spmv_ld(A, ux)[lo:hi] if not real else oracle.spmv_ld(A, ux)[lo:hi].real) <= TOL_MV


# ---------------------------------------------------------------------------------------- vec_randomize
def test_vec_randomize_is_the_reference_sequence(oracle):
    # 4 S_v + 3 (S_v = 303104: one trip of the vector passes on 148 SMs) and 2^24 + 13: the last drawing thread draws 3 and 13
    # of its 64 values, and the normalising nrm2 runs several trips
    for n, seed in ((10, 1), (65536, 1), (100003, 8), (7, 0), (4 * 303104 + 3, 5), (2 ** 24 + 13, 3)):
        g = qb.vec_randomize(n, seed)
        o = oracle.vec_randomize(n, seed)
        assert np.abs(g.imag).max() == 0.0
        # the raw Lehmer values are identical; the common 1/nrm2 factor differs by summation order only
        assert np.abs(g.real - o.real).max() <= 1e-13 * np.abs(o.real).max()
        ratio = g.real[np.abs(o.real) > 1e-6] / o.real[np.abs(o.real) > 1e-6]
        assert ratio.max() - ratio.min() < 1e-12              # one common factor
        assert abs(np.linalg.norm(g) - 1.0) < 1e-14
    gd = qb.vec_randomize(1000, 1, dtype=np.float64)
    assert np.abs(gd - oracle.vec_randomize(1000, 1, dtype=np.float64)).max() <= 1e-14


# ------------------------------------------------------------------------------------------------ Lanczos
@pytest.mark.parametrize("name", ALL)
def test_lanczos_E0_matches_reference_and_published_golden(oracle, name):
    A, meta, ex = oracle.load_golden(name)
    M = make(A)
    n = A.dim
    v = np.zeros(2 * n, dtype=np.complex128)
    v[:n] = oracle.vec_randomize(n, 1)
    hess = np.zeros(2000)
    m = qb.lanczos(0, 999, 1000, n, M, v, hess, "sr_val0")
    ritz, s = qb.hess_eigen(hess, 1000, m)
    assert abs(m - meta["lanczos_steps"]) <= 2                                   # stop rule parity (SURVEY 7)
    assert abs(ritz[0] - meta["lanczos_E0"]) <= TOL_E0 * abs(meta["lanczos_E0"])
    if meta["golden_E0"] is not None:
        assert abs(ritz[0] - meta["golden_E0"]) < 1e-8                           # the reference's own assert
    k = min(20, m - 1)
    assert np.abs(hess[1000:1000 + k] - ex["lanczos_a"][:k]).max() < 1e-11
    assert np.abs(hess[:k] - ex["lanczos_b"][:k]).max() < 1e-11
    assert hess[0] == 0.0 and np.all(hess[m + 1:1000] == 0.0)
    # the two live vectors come back normalised and mutually orthogonal like the reference's v[]
    assert abs(np.linalg.norm(v[:n]) - 1.0) < 1e-10 and abs(np.linalg.norm(v[n:]) - 1.0) < 1e-10
    assert abs(np.vdot(v[:n], v[n:])) < 1e-6


@pytest.mark.parametrize("name", SMALL)
def test_dnmcs_coefficients(oracle, name):
    A, meta, ex = oracle.load_golden(name)
    M = make(A)
    n = A.dim
    dv = qb.DeviceVector(2 * n)
    dv.zero()
    x = qb.DeviceVector.from_numpy(oracle.vec_randomize(n, 1))
    v = np.zeros(2 * n, dtype=np.complex128); v[:n] = x.to_numpy()
    hess = np.zeros(120)
    m = qb.lanczos(0, 59, 60, n, M, v, hess, "dnmcs")
    assert m == meta["dn_steps"] == 59                       # no stop rule in dnmcs mode (src/lanczos.cc:228)
    assert np.abs(hess[60:80] - ex["dn_a"][:20]).max() < 1e-11
    assert np.abs(hess[:20] - ex["dn_b"][:20]).max() < 1e-11


def test_lanczos_complex_start_vector_on_real_matrix(oracle):
    """Real stored values + a genuinely complex start vector: the complex-vector kernels (no real-mode shortcut)."""
    A, meta, ex = oracle.load_golden("hubbard4x2")
    n = A.dim
    rng = np.random.default_rng(11)
    x = rng.normal(size=n) + 1j * rng.normal(size=n)
    x /= np.linalg.norm(x)
    mo, ao, bo, _ = oracle.lanczos(A, x, 1000, "sr_val0")
    v = np.zeros(2 * n, dtype=np.complex128); v[:n] = x
    hess = np.zeros(2000)
    m = qb.lanczos(0, 999, 1000, n, make(A), v, hess, "sr_val0")
    assert abs(m - mo) <= 2
    assert np.abs(hess[1000:1020] - ao[:20]).max() < 1e-11 and np.abs(hess[:20] - bo[:20]).max() < 1e-11
    ritz, _ = qb.hess_eigen(hess, 1000, m)
    assert abs(ritz[0] - meta["lanczos_E0"]) <= TOL_E0 * abs(meta["lanczos_E0"])
    # and the real-mode run of the same matrix from a real start agrees with the forced-complex run to round-off
    # (row sums are the same fma sequence; only the grouping of the block-level dot reductions differs)
    import os
    xr = oracle.vec_randomize(n, 1)
    h1 = np.zeros(2000); h2 = np.zeros(2000)
    v1 = np.zeros(2 * n, dtype=np.complex128); v1[:n] = xr
    m1 = qb.lanczos(0, 999, 1000, n, make(A), v1, h1, "sr_val0")
    os.environ["QBGPU_NO_REAL_MODE"] = "1"
    try:
        v2 = np.zeros(2 * n, dtype=np.complex128); v2[:n] = xr
        m2 = qb.lanczos(0, 999, 1000, n, make(A), v2, h2, "sr_val0")
    finally:
        del os.environ["QBGPU_NO_REAL_MODE"]
    assert abs(m1 - m2) <= 1 and np.abs(h1[:20] - h2[:20]).max() < 1e-13 and np.abs(h1[1000:1020] - h2[1000:1020]).max() < 1e-13
    assert np.abs(v1.imag).max() == 0.0


def test_lanczos_argument_checks(oracle):
    A, meta, ex = oracle.load_golden("hubbard4x2")
    M = make(A)
    v = np.zeros(2 * A.dim, dtype=np.complex128); v[:A.dim] = oracle.vec_randomize(A.dim, 1)
    hess = np.zeros(20)
    with pytest.raises(qb.QbgpuError):
        qb.lanczos(0, 10, 10, A.dim, M, v, hess, "sr_val0")  # the reference asserts k+np < maxit (src/lanczos.cc:147)
    with pytest.raises(qb.QbgpuError):
        qb.lanczos(0, 5, 10, A.dim, M, v, hess, "bogus")
    assert qb.lanczos(0, 0, 10, A.dim, M, v, hess, "sr_val0") == 0   # np == 0 returns immediately (:150)


# ---------------------------------------------------------------------------------------------------- CG
@pytest.mark.parametrize("name", SMALL)
def test_eigenvec_cg(oracle, name):
    A, meta, ex = oracle.load_golden(name)
    M = make(A)
    n = A.dim
    v = oracle.vec_randomize(n, 1)
    r = np.zeros(n, dtype=np.complex128); p = np.zeros_like(r); pp = np.zeros_like(r)
    m, accu = qb.eigenvec_CG(n, 1000, 0, M, meta["lanczos_E0"], v, r, p, pp)
    assert accu < 2e-12
    assert abs(m - meta["cg_steps"]) <= 5
    res = oracle.spmv(A, v) - meta["lanczos_E0"] * v
    assert np.linalg.norm(res) < 1e-9
    assert abs(np.linalg.norm(v) - 1.0) < 1e-9
    ov = abs(np.vdot(ex["cg_vec"], v))
    if name not in ("tri4x4_k01", "tri4x4_k12", "heis16_k3"):        # non-degenerate ground states
        assert ov > 1 - 1e-8


def test_locate_E0_lanczos_heisenberg16_golden(oracle):
    """src/main_test.cc:18-111: E0 and the three ground-state correlators."""
    A, meta, ex = oracle.load_golden("heis16_full")
    out = qb.locate_E0_lanczos(make(A), nev=1, ncv=1)
    assert abs(out["eigenvals"][0] + 7.142296361) < 1e-8
    v = out["eigenvecs"][0]
    st = B.basis_states(16, 1, (None,))
    sz = lambda s: 0.5 - ((st >> s) & 1)                     # noqa: E731
    w = np.abs(v) ** 2
    assert abs((w * sz(0) * sz(1)).sum() + 0.1487978408) < 1e-8
    assert abs((w * sz(0) * sz(2)).sum() - 0.0617414604) < 1e-8
    # <S+_0 S-_1>: flips (down at 0, up at 1) -> (up at 0, down at 1)
    byval = np.argsort(st); sv = st[byval]
    act = np.nonzero((((st >> 0) & 1) == 0) & (((st >> 1) & 1) == 1))[0]     # result states: site0 up(0), site1 down(1)
    src = byval[np.searchsorted(sv, st[act] ^ 0b11)]
    assert abs(np.vdot(v[act], v[src]).real + 0.2975956817) < 1e-8


def test_locate_E0_lanczos_gap_and_excited_vector(oracle):
    A, meta, ex = oracle.load_golden("hubbard4x2")
    out = qb.locate_E0_lanczos(make(A), nev=2, ncv=2)
    F = A.to_scipy_full().toarray()
    w = np.linalg.eigvalsh(F)
    assert abs(out["eigenvals"][0] - w[0]) < 1e-9
    assert abs(out["eigenvals"][0] + 14.07605866) < 1e-8     # examples/trans_absent/latt_square/square_Fermi_Hubbard.cc:113
    e1 = w[np.nonzero(w - w[0] > 1e-9)[0][0]] if out["gap"] > 1e-9 else w[1]
    assert abs(out["eigenvals"][1] - e1) < 1e-8
    for E, vec in zip(out["eigenvals"], out["eigenvecs"]):
        assert np.linalg.norm(F @ vec - E * vec) < 1e-7


# ------------------------------------------------------------------------------------------- ARPACK seam
def test_arpack_callback_seam_tJ_golden(oracle):
    """src/main_test.cc:113-211: t-J chain L=12, locate_E0_iram(full, 4, 8) -> E0 = E1 = -9.762087307.  ARPACK (scipy's
    bundled copy, complex znaupd like the reference's call_arpack) runs on the host and calls MultMv on its own host work
    vectors: the reverse-communication seam of src/lanczos.cc:476."""
    A, meta, ex = oracle.load_golden("tj12")
    out = qb.locate_E0_iram(make(A), nev=4, ncv=8)
    assert out["nconv"] == 4
    assert abs(out["eigenvals"][0] + 9.762087307) < 1e-8
    assert abs(out["eigenvals"][1] + 9.762087307) < 1e-8
    for E, v in zip(out["eigenvals"], out["eigenvecs"]):
        assert np.linalg.norm(oracle.spmv(A, v) - E * v) < 1e-7
    assert qb.iram.last_products > 8


def test_device_resident_thick_restart_lanczos(oracle):
    """qbgpu_trlan: the locate_E0_iram contract with the Krylov basis kept in HBM.  Eigenvalue parity with the reference's
    ARPACK golden (t-J chain, nev=4, ncv=8: E0 = E1 = -9.762087307, src/main_test.cc:207-208) and with dense
    diagonalisation; eigenvectors checked through their residuals and orthonormality."""
    A, meta, ex = oracle.load_golden("tj12")
    out = qb.locate_E0_iram(make(A), nev=4, ncv=8, device_resident=True)
    assert out["nconv"] == 4
    assert abs(out["eigenvals"][0] + 9.762087307) < 1e-8 and abs(out["eigenvals"][1] + 9.762087307) < 1e-8
    U = np.stack(out["eigenvecs"], axis=1)
    for j, E in enumerate(out["eigenvals"]):
        assert np.linalg.norm(oracle.spmv(A, U[:, j]) - E * U[:, j]) < 1e-7
    assert np.abs(U.conj().T @ U - np.eye(4)).max() < 1e-9
    host = qb.locate_E0_iram(make(A), nev=4, ncv=8)                            # ARPACK on the host through the MultMv seam
    assert np.abs(np.array(out["eigenvals"]) - np.array(host["eigenvals"])).max() < 1e-9
    for name, nev, ncv in (("hubbard4x2", 3, 10), ("tri4x4_k12", 2, 12), ("honeycomb3x2_general", 2, 8)):
        A, meta, ex = oracle.load_golden(name)
        w = np.linalg.eigvalsh(A.to_scipy_full().toarray())
        nconv, ev, U, nprod = qb.trlan(make(A), nev, ncv)
        assert nconv == nev and np.abs(ev - w[:nev]).max() < 1e-9
        assert abs(ev[0] - meta["lanczos_E0"]) <= 1e-9 * abs(meta["lanczos_E0"])
    A, meta, ex = oracle.load_golden("hubbard4x2")                             # csr_mat<double> handle
    nconv, ev, U, nprod = qb.trlan(make(A.astype(np.float64)), 2, 8)
    assert nconv == 2 and abs(ev[0] + 14.07605866) < 1e-8 and U.dtype == np.float64
    with pytest.raises(qb.QbgpuError):
        qb.trlan(make(A), 4, 5)                                                # the reference asserts ncv > nev + 1


def test_iram_small_matrix_uses_dense_fallback(oracle):
    """dim <= 30: mat.to_dense() + dense eigensolver (src/lanczos.cc:508-542)."""
    import scipy.sparse as sp
    from oracle_lib import Csr
    rng = np.random.default_rng(2)
    n = 24
    Mx = rng.normal(size=(n, n)) + 1j * rng.normal(size=(n, n))
    Hd = np.triu(Mx + Mx.conj().T)
    S = sp.csr_matrix(Hd)
    S.sort_indices()
    A = Csr(n, S.indptr, S.indices, S.data.astype(np.complex128), True)
    nconv, w, U = qb.iram(n, make(A), np.ones(n, dtype=np.complex128), 3, 8, 100, "sr")
    full = Hd + np.triu(Hd, 1).conj().T
    assert np.abs(w - np.linalg.eigvalsh(full)[:3]).max() < 1e-12


# ------------------------------------------------------------------------------------- energy_scale / KPM
@pytest.mark.parametrize("name", ["heis12_full", "tri4x4_k01", "hubbard4x2"])
def test_energy_scale_matches_reference(oracle, name):
    A, meta, ex = oracle.load_golden(name)
    v = np.zeros(2 * A.dim, dtype=np.complex128)
    lo, hi = qb.energy_scale(A.dim, make(A), v, 0.1, 40)
    assert abs(lo - meta["escale_lo"]) < 1e-8 * abs(meta["escale_lo"])
    assert abs(hi - meta["escale_hi"]) < 1e-8 * abs(meta["escale_hi"])


@pytest.mark.parametrize("name", ["tri4x4_k01", "hubbard4x2", "heis16_k3"])
def test_kpm_moments(oracle, name):
    A, meta, ex = oracle.load_golden(name)
    phi = oracle.vec_randomize(A.dim, 3)
    lo, hi = meta["escale_lo"], meta["escale_hi"]
    for nmom in (1, 2, 7, 64, 129):
        mu = qb.kpm_moments(make(A), phi, lo, hi, nmom)
        ref = oracle.kpm_moments(A, phi, lo, hi, nmom)
        assert np.abs(mu - ref).max() <= TOL_KPM


# --------------------------------------------------------------------------------------------- generators
def _expanded(n, ia, ja, val, oracle):
    from oracle_lib import Csr
    return oracle.expand_upper(Csr(n, ia, ja, val, True))


@pytest.mark.parametrize("case", ["heis12", "heis15", "hub4x2", "hub3x3"])
def test_device_generators_match_the_reference_matrix(oracle, case):
    L = qb.lib()
    import ctypes as C
    if case == "heis12":
        bonds, args = B.chain_bonds(12), (12, 6)
        n, ia, ja, val = B.heisenberg_upper_csr(12, 6, bonds)
    elif case == "heis15":
        bonds, args = B.chain_bonds(15), (15, 7)
        n, ia, ja, val = B.heisenberg_upper_csr(15, 7, bonds)
    elif case == "hub4x2":
        bonds, args = B.square_bonds(4, 2), (8, 4, 4)
        n, ia, ja, val = B.hubbard_upper_csr(8, 4, 4, bonds, 1.0, 1.1)
    else:
        bonds, args = B.square_bonds(3, 3), (9, 4, 5)
        n, ia, ja, val = B.hubbard_upper_csr(9, 4, 5, bonds, 1.0, 2.3)
    barr = np.array(bonds, dtype=np.int32).ravel()
    h = C.c_void_p()
    if case.startswith("heis"):
        rc = L.qbgpu_build_heisenberg(C.byref(h), args[0], args[1], len(bonds), barr.ctypes.data, 1.0, 1, 0, 0, -1)
    else:
        U = 1.1 if case == "hub4x2" else 2.3
        rc = L.qbgpu_build_hubbard(C.byref(h), args[0], args[1], args[2], len(bonds), barr.ctypes.data, 1.0, U, 1, 0, 0, -1)
    assert rc == 0, L.qbgpu_last_error()
    M = qb.csr_mat._adopt(h, True)
    rowptr, col, v = M.download_expanded()
    eia, eja, ev = _expanded(n, ia, ja, val, oracle)
    assert M.dim == n
    assert np.array_equal(rowptr, eia) and np.array_equal(col.astype(np.int64), eja)
    assert np.array_equal(v, ev.real)                        # bit-identical values, fp64 storage
    if case == "hub4x2":
        A, meta, ex = oracle.load_golden("hubbard4x2")       # and therefore equal to the reference-assembled matrix
        rp2, c2, v2 = make(A).download_expanded()
        assert np.array_equal(rowptr, rp2) and np.array_equal(col, c2) and np.array_equal(v, v2)


@pytest.mark.parametrize("case", ["heis12", "heis15", "hub4x2", "hub3x3"])
def test_matrix_free_product_equals_the_stored_matrix(oracle, case):
    """The device counterpart of model::MultMv2 with matrix_free == true (src/model.cc:942-1109): no stored H."""
    from oracle_lib import Csr
    if case == "heis12":
        bonds = B.chain_bonds(12); n, ia, ja, val = B.heisenberg_upper_csr(12, 6, bonds)
        mk = lambda mf, cx=True: qb.heisenberg(12, 6, bonds, 1.0, is_complex=cx, matrix_free=mf)      # noqa: E731
    elif case == "heis15":
        bonds = B.chain_bonds(15); n, ia, ja, val = B.heisenberg_upper_csr(15, 7, bonds)
        mk = lambda mf, cx=True: qb.heisenberg(15, 7, bonds, 1.0, is_complex=cx, matrix_free=mf)      # noqa: E731
    elif case == "hub4x2":
        bonds = B.square_bonds(4, 2); n, ia, ja, val = B.hubbard_upper_csr(8, 4, 4, bonds, 1.0, 1.1)
        mk = lambda mf, cx=True: qb.hubbard(8, 4, 4, bonds, 1.0, 1.1, is_complex=cx, matrix_free=mf)  # noqa: E731
    else:
        bonds = B.square_bonds(3, 3); n, ia, ja, val = B.hubbard_upper_csr(9, 4, 5, bonds, 1.0, 2.3)
        mk = lambda mf, cx=True: qb.hubbard(9, 4, 5, bonds, 1.0, 2.3, is_complex=cx, matrix_free=mf)  # noqa: E731
    A = Csr(n, ia, ja, val, True)
    F = mk(True)
    assert F.info.format == 32 and F.info.nnz_stored == 0 and F.dim == n
    rng = np.random.default_rng(9)
    x = rng.normal(size=n) + 1j * rng.normal(size=n)
    y = np.zeros(n, dtype=np.complex128)
    F.MultMv(x, y)
    assert rel_l2(y, oracle.spmv_ld(A, x)) <= TOL_MV                 # vs the reference-identical matrix on the CPU
    ys = np.zeros(n, dtype=np.complex128)
    mk(False).MultMv(x, ys)
    assert rel_l2(y, ys) <= 1e-14                                    # vs the stored device matrix
    y2 = y.copy()
    F.MultMv2(x, y2)
    assert rel_l2(y2, 2 * y) <= 1e-14
    # fp64 handle and the fused loops on the matrix-free handle
    Fd = mk(True, False)
    xr = rng.normal(size=n); yr = np.zeros(n)
    Fd.MultMv(xr, yr)
    assert rel_l2(yr, oracle.spmv_ld(A, xr).real) <= TOL_MV
    out_f = qb.locate_E0_lanczos(F, nev=1, ncv=1)
    out_s = qb.locate_E0_lanczos(mk(False), nev=1, ncv=1)
    assert abs(out_f["eigenvals"][0] - out_s["eigenvals"][0]) <= TOL_E0 * abs(out_s["eigenvals"][0])
    v = out_f["eigenvecs"][0]
    assert np.linalg.norm(oracle.spmv(A, v) - out_f["eigenvals"][0] * v) < 1e-8
    with pytest.raises(qb.QbgpuError):
        F.download_expanded()


def test_matrix_free_config1_and_a_sector_too_large_to_store(oracle):
    """BASELINE config 1 through the matrix-free handle (E0 = -8.9043865298764 from the compiled reference), and the uniform
    vector check (H 1 = L/4 * 1 in any Sz sector) on the Heisenberg chain L = 30, Sz = 0: 155,117,520 states whose stored
    matrix would take 57 GB; the matrix-free handle keeps 1.2 GB."""
    F = qb.heisenberg(20, 10, B.chain_bonds(20), 1.0, matrix_free=True)
    out = qb.locate_E0_lanczos(F, nev=1, ncv=0)
    assert abs(out["eigenvals"][0] + 8.9043865298764) <= TOL_E0 * 8.9043865298764
    L30 = qb.heisenberg(30, 15, B.chain_bonds(30), 1.0, is_complex=False, matrix_free=True)
    n = L30.dim
    assert n == 155117520 and L30.info.device_bytes < 1.5e9
    ones = qb.DeviceVector.from_numpy(np.ones(n)); y = qb.DeviceVector(n, np.float64)
    L30.MultMv(ones, y)
    assert np.abs(y.to_numpy() - 7.5).max() < 1e-12


def test_config1_heisenberg_L20_E0(oracle):
    """BASELINE config 1: Heisenberg chain L=20, Sz=0 (dim 184,756); E0 from the compiled reference = -8.9043865298764
    in 77 steps (SURVEY.md section 6 / BASELINE.md section 3)."""
    L = qb.lib()
    import ctypes as C
    bonds = np.array(B.chain_bonds(20), dtype=np.int32).ravel()
    h = C.c_void_p()
    assert L.qbgpu_build_heisenberg(C.byref(h), 20, 10, 20, bonds.ctypes.data, 1.0, 1, 0, 0, -1) == 0, L.qbgpu_last_error()
    M = qb.csr_mat._adopt(h, True)
    inf = M.info
    assert inf.n == 184756 and inf.nnz_stored == 2129556 and inf.val_is_real == 1
    out = qb.locate_E0_lanczos(M, nev=1, ncv=0)
    assert abs(out["eigenvals"][0] + 8.9043865298764) <= TOL_E0 * 8.9043865298764
    assert abs(out["lanczos_steps"] - 77) <= 2


def test_large_generated_matrix_properties(oracle):
    """Size-independent properties at a size the oracle would not finish quickly: Heisenberg chain L=26, Sz=0
    (dim 10,400,600): Hermiticity <x,Hy> = conj<y,Hx>, linearity, and agreement between row shards and the whole."""
    L = qb.lib()
    import ctypes as C
    nsites = 26
    bonds = np.array(B.chain_bonds(nsites), dtype=np.int32).ravel()
    h = C.c_void_p()
    assert L.qbgpu_build_heisenberg(C.byref(h), nsites, nsites // 2, nsites, bonds.ctypes.data, 1.0, 1, 0, 0, -1) == 0, L.qbgpu_last_error()
    M = qb.csr_mat._adopt(h, True)
    n = M.dim
    assert n == 10400600
    x = qb.vec_randomize(n, 1, device=True); y = qb.vec_randomize(n, 8, device=True)
    hx = qb.DeviceVector(n); hy = qb.DeviceVector(n)
    M.MultMv(x, hx); M.MultMv(y, hy)
    d1 = (C.c_double * 2)(); d2 = (C.c_double * 2)()
    L.qbgpu_zdotc(n, C.c_void_p(x.ptr), C.c_void_p(hy.ptr), d1)
    L.qbgpu_zdotc(n, C.c_void_p(y.ptr), C.c_void_p(hx.ptr), d2)
    assert abs(complex(d1[0], d1[1]) - complex(d2[0], -d2[1])) < 1e-12
    # a shard of the same generator gives the same rows
    lo, hi = n // 3, n // 3 + 100000
    h2 = C.c_void_p()
    assert L.qbgpu_build_heisenberg(C.byref(h2), nsites, nsites // 2, nsites, bonds.ctypes.data, 1.0, 1, 0, lo, hi) == 0
    S = qb.csr_mat._adopt(h2, True)
    ys = qb.DeviceVector(hi - lo)
    S.MultMv(x, ys)
    assert rel_l2(ys.to_numpy(), hx.to_numpy()[lo:hi]) < 1e-14        # (the shard may have picked another kernel variant)
    # sum of each row of H for the Heisenberg chain in the Sz=0 sector: H applied to the uniform vector is an
    # eigenvector-free check of the generator: (H 1)_i = diag_i + 0.5 * (#antiparallel bonds) = L/4 for every i
    ones = qb.DeviceVector.from_numpy(np.ones(n, dtype=np.complex128))
    M.MultMv(ones, hx)
    assert np.abs(hx.to_numpy() - nsites * 0.25).max() < 1e-12


# ------------------------------------------------------------------ translation-symmetric sectors built on the device
_SECTOR_CASES = [
    ("chain16_k3", [16], 8, [3]), ("chain12_k5", [12], 6, [5]), ("chain14_sz1_k2", [14], 6, [2]),
    ("chain20_k7", [20], 10, [7]), ("chain22_sz1_k5", [22], 10, [5]), ("chain24_k0", [24], 12, [0]),
    ("tri4x4_k12", [4, 4], 8, [1, 2]), ("tri3x4_k23", [3, 4], 6, [2, 3]), ("tri6x3_k12", [6, 3], 9, [1, 2]),
    ("tri4x5_k32", [4, 5], 10, [3, 2]),
]


def _sector_bonds(L):
    import repr_builders as R
    return R.chain_bonds(L[0]) if len(L) == 1 else R.triangular_bonds(*L)


@pytest.mark.parametrize("name,L,ndown,k", _SECTOR_CASES, ids=[c[0] for c in _SECTOR_CASES])
def test_device_sector_builder_is_bit_identical_to_the_reference_convention(oracle, name, L, ndown, k):
    """Representatives, row order, norms and every matrix element of generate_Ham_sparse_repr (src/model.cc:688-836)
    against tests/repr_builders.py, which is itself pinned bit for bit to matrices assembled by the compiled
    reference (tests/golden/repr_hashes.json)."""
    import repr_builders as R
    bonds = _sector_bonds(L)
    S, ia, ja, val = R.heisenberg_sector_upper_csr(L, ndown, k, bonds)
    sec = qb.Sector(L, ndown, k)
    assert sec.dim == S.n and sec.lin_order == S.lin_order and sec.zero_norm == int((S.nu == 0).sum())
    assert np.array_equal(sec.states().astype(np.uint64), S.states)
    assert np.array_equal(sec.norms(), S.nu)
    M = sec.heisenberg(bonds, flags=1)                       # QBGPU_KEEP_COMPLEX: compare complex values as assembled
    rowptr, col, v = M.download_expanded()
    eia, eja, ev = _expanded(S.n, ia, ja, val, oracle)
    assert M.dim == S.n and M.info.nnz_input == ja.size
    assert np.array_equal(rowptr, eia) and np.array_equal(col.astype(np.int64), eja)
    assert np.array_equal(v, ev)
    sec.free()


def test_device_sector_matches_the_golden_reference_matrix_and_E0(oracle):
    """The k=3 sector of the L=16 chain: same matrix as the one the reference assembled (golden), and its published
    E0 (examples/trans_symmetric/latt_chain/chain_Heisenberg_spin_half.cc:102-117) from the device Lanczos."""
    A, meta, ex = oracle.load_golden("heis16_k3")
    sec = qb.Sector([16], 8, [3])
    M = sec.heisenberg(_sector_bonds([16]), flags=1)
    rowptr, col, v = M.download_expanded()
    eia, eja, ev = oracle.expand_upper(A)
    assert np.array_equal(rowptr, eia) and np.array_equal(col.astype(np.int64), eja) and np.array_equal(v, ev)
    E = qb.locate_E0_lanczos(M, nev=1, ncv=0)["eigenvals"]
    assert abs(E[0] - meta["golden_E0"]) < 1e-8


def test_device_sector_real_momenta_are_stored_as_fp64_and_config2_style_sector_runs():
    """k = 0 gives a real matrix (demoted to fp64 values); chain L=24: 112,720 representatives in well under a second."""
    sec = qb.Sector([24], 12, [0])
    M = sec.heisenberg(_sector_bonds([24]))
    assert M.info.val_is_real == 1 and sec.zero_norm == 0 and sec.dim == 112720
    E = qb.locate_E0_lanczos(M, nev=1, ncv=0)["eigenvals"]
    assert abs(E[0] / 24 - (-0.4438)) < 2e-3         # Bethe-ansatz energy density -ln2 + 1/4 up to finite-size corrections


@pytest.mark.parametrize("L,ndown,k,bonds", [([16], 8, [3], "chain"), ([12], 6, [0], "chain"), ([4, 4], 8, [1, 2], "tri"),
                                             ([4, 4], 8, [2, 2], "tri"), ([6, 2], 6, [3, 1], "tri")])
def test_matrix_free_sector_product_equals_the_stored_sector_matrix(L, ndown, k, bonds):
    """model<T>::MultMv / MultMv2 with matrix_free == true, repr branch (src/model.cc:1016-1107): rows regenerated inside the
    product -- against the stored handle of the same sector (which is the reference's matrix bit for bit, tests above), sectors
    with zero-norm representatives (their fake diagonal, :1022-1025) included; then MultMv2's accumulate form and the fused loops."""
    import repr_builders as R
    bl = R.chain_bonds(L[0]) if bonds == "chain" else R.triangular_bonds(*L)
    sec = qb.Sector(L, ndown, k)
    Hs, Hf = sec.heisenberg(bl, flags=1), sec.heisenberg_matrix_free(bl)
    n = sec.dim
    assert Hf.dim == n and Hf.info.nnz_stored == 0
    rng = np.random.default_rng(5)
    x = rng.normal(size=n) + 1j * rng.normal(size=n)
    ys, yf = np.zeros(n, dtype=np.complex128), np.zeros(n, dtype=np.complex128)
    Hs.MultMv(x, ys); Hf.MultMv(x, yf)
    assert rel_l2(yf, ys) < TOL_MV
    y0 = rng.normal(size=n) + 1j * rng.normal(size=n)
    y2 = y0.copy()
    Hf.MultMv2(x, y2)
    assert rel_l2(y2, y0 + ys) < TOL_MV
    if n > 40:
        Es = qb.locate_E0_lanczos(Hs, nev=1, ncv=0)["eigenvals"][0]
        Ef = qb.locate_E0_lanczos(Hf, nev=1, ncv=0)["eigenvals"][0]
        assert abs(Es - Ef) <= TOL_E0 * abs(Es)
    del Hf, Hs
    sec.free()


def test_matrix_free_sector_reaches_the_published_E0(oracle):
    """The k=3 sector of the L=16 chain without a stored matrix: E0 of the reference's example
    (examples/trans_symmetric/latt_chain/chain_Heisenberg_spin_half.cc:102-117)."""
    A, meta, ex = oracle.load_golden("heis16_k3")
    sec = qb.Sector([16], 8, [3])
    Hf = sec.heisenberg_matrix_free(_sector_bonds([16]))
    y = np.zeros(A.dim, dtype=np.complex128)
    Hf.MultMv(oracle.vec_randomize(A.dim, 1), y)
    assert rel_l2(y, ex["y1"]) < TOL_MV                      # y1 = the compiled reference's csr_mat::MultMv on vec_randomize(seed 1)
    E = qb.locate_E0_lanczos(Hf, nev=1, ncv=0)["eigenvals"]
    assert abs(E[0] - meta["golden_E0"]) < 1e-8


# ------------------------------------------------------------------ Hubbard momentum sectors (electron orbital)
HUBBARD4X2_E0 = [-14.07605866, -10.50470669, -12.16861094, -12.19847764, -10.54300366, -14.03137587, -12.16861094, -12.19847764]


@pytest.mark.parametrize("L,nup,ndn,k", [([4, 2], 4, 4, [0, 0]), ([4, 2], 4, 4, [1, 0]), ([4, 2], 4, 4, [2, 1]), ([4, 2], 4, 4, [3, 1]),
                                         ([4, 2], 3, 4, [1, 1]), ([2, 2], 2, 2, [1, 0]), ([4, 3], 2, 3, [1, 2]), ([6], 3, 3, [2]),
                                         ([4, 3], 6, 6, [0, 0]), ([4, 3], 6, 6, [2, 1])])
def test_device_hubbard_sector_is_bit_identical_to_the_reference_assembly(oracle, L, nup, ndn, k):
    """Electron sectors on the device (qbgpu_sector_create_electron / _build_hubbard): representatives, row order, norms and
    every matrix element of generate_Ham_sparse_repr (src/model.cc:688-836) with the fermionic translation signs
    (src/basis.cc:593-620, 2134-2147) against tests/repr_builders_fermion.py, which is pinned bit for bit to matrices assembled
    by the compiled reference (qb_ref hubbard_k, tests/golden/repr_hashes.json)."""
    import repr_builders_fermion as F
    hops = F.square_hops(*L) if len(L) == 2 else [h for i in range(L[0]) for h in [(i, (i + 1) % L[0], 0), ((i + 1) % L[0], i, 0), (i, (i + 1) % L[0], 1), ((i + 1) % L[0], i, 1)]]
    S, ia, ja, val = F.hubbard_sector_upper_csr(L, nup, ndn, k, hops, 1.0, 1.1)
    sec = qb.ElectronSector(L, nup, ndn, k)
    assert sec.dim == S.n and sec.lin_order == S.lin_order and sec.zero_norm == int((S.nu == 0).sum())
    assert np.array_equal(sec.states().astype(np.uint64), S.states)
    assert np.array_equal(sec.norms(), S.nu)
    M = sec.hubbard(hops, 1.0, 1.1, flags=1)                 # QBGPU_KEEP_COMPLEX: compare complex values as assembled
    rowptr, col, v = M.download_expanded()
    eia, eja, ev = _expanded(S.n, ia, ja, val, oracle)
    assert M.dim == S.n and M.info.nnz_input == ja.size
    assert np.array_equal(rowptr, eia) and np.array_equal(col.astype(np.int64), eja)
    assert np.array_equal(v, ev)
    del M
    sec.free()


@pytest.mark.parametrize("idx", range(8))
def test_device_hubbard4x2_sector_energies_match_the_published_list(idx):
    """examples/trans_symmetric/latt_square/square_Fermi_Hubbard.cc:112-119 (E0_list index = 2 m + n): sector built and solved on
    the device (zero-norm representatives carry fake_pos on the diagonal and stay out of the way, as in the reference)."""
    import repr_builders_fermion as F
    m, n = idx // 2, idx % 2
    sec = qb.ElectronSector([4, 2], 4, 4, [m, n])
    M = sec.hubbard(F.square_hops(4, 2), 1.0, 1.1)
    E = qb.locate_E0_lanczos(M, nev=1, ncv=0)["eigenvals"]
    assert abs(E[0] - HUBBARD4X2_E0[idx]) < 1e-8
    del M
    sec.free()


def test_device_hubbard4x4_momentum_sectors_at_baseline_size():
    """All 16 momentum sectors of BASELINE config 3's model (4x4, 8 up, 8 down; about 10.4 M representatives each) assembled and
    solved on the device -- beyond the reference's own assembler in practice.  Size-independent properties: the live
    representatives of all sectors together are the 165,636,900 states of the full basis; no sector lies below the full-basis
    ground-state energy -20.497352266554 (BASELINE config 3, also produced by the compiled reference's stop rule on our matrix)
    and the lowest one reaches it."""
    import repr_builders_fermion as F
    hops = F.square_hops(4, 4)
    live, energies = 0, {}
    for m in range(4):
        for n in range(4):
            sec = qb.ElectronSector([4, 4], 8, 8, [m, n])
            live += sec.dim - sec.zero_norm
            if (m, n) in ((0, 0), (2, 2), (1, 0), (2, 0), (1, 1), (2, 1)):        # one of every class of the square's point group
                M = sec.hubbard(hops, 1.0, 1.1)
                energies[(m, n)] = qb.locate_E0_lanczos(M, nev=1, ncv=0)["eigenvals"][0]
                del M
            sec.free()
    assert live == 165636900
    E_full = -20.497352266554
    assert min(energies.values()) > E_full - 1e-8
    assert abs(min(energies.values()) - E_full) < 1e-8, energies


# ------------------------------------------------------------------ S^z_q between momentum sectors + dnmcs Lanczos (config 5)
def _dyn_golden(name):
    import json
    import os
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    return z, json.loads(str(z["meta"]))


@pytest.mark.parametrize("name", ["heis16_szq3", "heis16_szq8", "heis12_szq1"])
def test_sector_sz_operator_and_dynamic_lanczos_match_the_reference(name):
    """model::moprXvec_repr + measure_repr_dynamic (src/model.cc:1716-1846, 1897-1912) on the device against vectors and
    Lanczos coefficients produced by the compiled reference (oracle/make_golden.py dynamic)."""
    import repr_builders as R
    z, meta = _dyn_golden(name)
    L, q, k0, maxit = meta["L"], meta["q"], meta["k0"], meta["maxit"]
    s0, s1 = qb.Sector([L], L // 2, [k0]), qb.Sector([L], L // 2, [k0 - q])
    coef = R.szq_coefficients(L, q)
    y = s0.apply_sz(s1, coef, z["phi0"]).to_numpy()
    assert np.abs(y - z["Aphi0"]).max() < 1e-15
    H1 = s1.heisenberg(R.chain_bonds(L))
    hess = np.zeros(2 * maxit)
    m, norm = qb.measure_repr_dynamic(coef, s0, s1, H1, z["phi0"], maxit, hess)
    assert m == meta["dyn_steps"] and abs(norm - meta["dyn_norm"]) < 1e-14
    # S^z_q phi0 lives in a small symmetry sector (total spin 1): once its Krylov space is exhausted the recursion only
    # amplifies rounding, in the reference as well, so the comparison is on the leading coefficients
    k = min(m, 10)
    assert np.abs(hess[maxit:maxit + k] - z["dyn_a"][:k]).max() < 1e-10
    assert np.abs(hess[:k] - z["dyn_b"][:k]).max() < 1e-10


def test_config5_flow_on_the_device_end_to_end():
    """E0 and phi0 of the (Sz=0, k=0) sector by Lanczos + CG, S^z_q phi0 in the k=-q sector, dnmcs coefficients and KPM
    moments from it -- nothing leaves HBM between the steps.  E0, |S^z_q phi0| and the leading coefficients against the
    reference's own run of the same flow."""
    import repr_builders as R
    z, meta = _dyn_golden("heis16_szq3")
    L, q, maxit = 16, 3, 60
    s0, s1 = qb.Sector([L], 8, [0]), qb.Sector([L], 8, [-q])
    H0, H1 = s0.heisenberg(R.chain_bonds(L)), s1.heisenberg(R.chain_bonds(L))
    res = qb.locate_E0_lanczos(H0, nev=1, ncv=1, device_vectors=True)
    assert abs(res["eigenvals"][0] - meta["E0"]) < 1e-9
    phi0 = res["eigenvecs_device"][0]
    hess = np.zeros(2 * maxit)
    m, norm = qb.measure_repr_dynamic(R.szq_coefficients(L, q), s0, s1, H1, phi0, maxit, hess)
    assert abs(norm - meta["dyn_norm"]) < 1e-8
    assert np.abs(hess[maxit:maxit + 10] - z["dyn_a"][:10]).max() < 1e-6
    assert np.abs(hess[1:10] - z["dyn_b"][1:10]).max() < 1e-6


# ------------------------------------------------------------------ orbit assembler: arbitrary abelian translation groups (config 4)
def _full_sector_spectrum(nsites, ndown, bonds):
    M = qb.heisenberg(nsites, ndown, bonds)
    D = M.to_dense()
    return np.linalg.eigvalsh(D)


@pytest.mark.parametrize("A0,A1,ndown", [((2, 1), (-1, 3), 3), ((3, 1), (-1, 4), 6), ((3, 1), (-1, 3), 5), ((4, 0), (0, 3), 6),
                                         ((4, 0), (0, 3), 4)])
def test_orbit_sectors_partition_the_full_spectrum(A0, A1, ndown):
    """Tilted and untilted clusters, prime and composite group orders: the eigenvalues of all momentum sectors together
    are exactly the eigenvalues of the full Sz sector (multiset), and the sector dimensions add up."""
    from quantum_basis_b200.clusters import Cluster
    cl = Cluster(A0, A1)
    bonds, perms = cl.triangular_bonds(), cl.translations()
    full = _full_sector_spectrum(cl.det, ndown, bonds)
    ev, total = [], 0
    for m in cl.distinct_momenta():
        M = qb.heisenberg_orbit(cl.det, ndown, perms, cl.characters(m), bonds, flags=1)
        D = M.to_dense()
        assert np.abs(D - D.conj().T).max() == 0.0
        ev.append(np.linalg.eigvalsh(D))
        total += M.dim
    assert total == full.size
    ev = np.sort(np.concatenate(ev))
    assert np.abs(ev - full).max() < 1e-10


def test_orbit_sector_equals_reference_convention_sector_spectrum():
    """On an untilted cluster the orbit-minimum sector and the reference-convention sector (sectors.cu) are the same
    operator in two bases: identical spectra once the reference's artificial zero-norm eigenvalues (>= fake_pos) are set
    aside."""
    import repr_builders as R
    from quantum_basis_b200.clusters import Cluster
    cl = Cluster((4, 0), (0, 4))
    # same lattice, same bonds, momentum (1, 2) in both descriptions
    sec = qb.Sector([4, 4], 8, [1, 2])
    Href = sec.heisenberg(R.triangular_bonds(4, 4), flags=1).to_dense()
    wref = np.linalg.eigvalsh(Href)
    wref = wref[wref < 50.0]
    best = None
    for m in cl.distinct_momenta():
        M = qb.heisenberg_orbit(16, 8, cl.translations(), cl.characters(m), cl.triangular_bonds(), flags=1)
        if M.dim != wref.size:
            continue
        w = np.linalg.eigvalsh(M.to_dense())
        err = np.abs(w - wref).max()
        best = err if best is None else min(best, err)
    assert best is not None and best < 1e-10


def test_orbit_sector_product_matches_the_oracle_on_the_same_matrix(oracle):
    """SURVEY 8d for config 4: per-product parity against the CPU restatement on the same CSR (21-site tilted cluster)."""
    from oracle_lib import Csr
    from quantum_basis_b200.clusters import Cluster
    cl = Cluster((4, 1), (-1, 5))
    M = qb.heisenberg_orbit(cl.det, 10, cl.translations(), cl.characters((1, 0)), cl.triangular_bonds(), flags=1)
    rowptr, col, v = M.download_expanded()
    A = Csr(M.dim, rowptr, col.astype(np.int64), v, False)
    x = oracle.vec_randomize(M.dim, 1)
    x = x * np.exp(1j * np.linspace(0.0, 3.0, M.dim))
    y = np.zeros(M.dim, dtype=np.complex128)
    M.MultMv(x, y)
    yo = oracle.spmv(A, x)
    assert np.linalg.norm(y - yo) / np.linalg.norm(yo) < 1e-12


def test_config4_tilted_31_site_cluster_builds_and_is_hermitian():
    """BASELINE config 4: triangular 31-site cluster (A0 = [5,1], A1 = [-1,6]), Sz = +1/2 (15 down), a k != 0 sector.
    dim = C(31,15)/31 exactly (31 is prime: every orbit is full); <x, H y> = conj(<y, H x>); Lanczos converges."""
    from math import comb
    from quantum_basis_b200.clusters import Cluster
    cl = Cluster((5, 1), (-1, 6))
    M = qb.heisenberg_orbit(31, 15, cl.translations(), cl.characters((1, 0)), cl.triangular_bonds())
    n = M.dim
    assert n == comb(31, 15) // 31 == 9694845 and M.info.val_is_real == 0
    x = qb.vec_randomize(n, 1, device=True)
    y = qb.vec_randomize(n, 8, device=True)
    hx, hy = qb.DeviceVector(n), qb.DeviceVector(n)
    M.MultMv(x, hx); M.MultMv(y, hy)
    import ctypes as C
    d1 = (C.c_double * 2)(); d2 = (C.c_double * 2)()
    L = qb.lib()
    assert L.qbgpu_zdotc(n, C.c_void_p(x.ptr), C.c_void_p(hy.ptr), d1) == 0
    assert L.qbgpu_zdotc(n, C.c_void_p(hx.ptr), C.c_void_p(y.ptr), d2) == 0
    assert abs(complex(d1[0], d1[1]) - complex(d2[0], d2[1])) < 1e-12
    res = qb.locate_E0_lanczos(M, nev=1, ncv=0)
    assert -0.60 * 31 < res["eigenvals"][0] < -0.45 * 31          # triangular-lattice Heisenberg: about -0.55 J per site


@pytest.mark.parametrize("A0,A1,ndown,m", [((3, 1), (-1, 4), 6, (1, 0)), ((4, 0), (0, 3), 6, (1, 1)), ((4, 0), (0, 3), 4, (2, 0)),
                                           ((4, 1), (-1, 5), 10, (1, 0)), ((4, 1), (-1, 5), 9, (3, 2))])
def test_orbit_assembler_matches_its_cpu_restatement(oracle, A0, A1, ndown, m):
    """Representatives, structure and matrix elements of the orbit assembler against tests/orbit_builders.py (which is
    checked on the CPU by the spectrum-partition property): same representatives, same sparsity, values to 1e-14 (the
    device contracts w*chi + acc into an fma, the restatement rounds twice)."""
    import orbit_builders as OB
    from quantum_basis_b200.clusters import Cluster
    cl = Cluster(A0, A1)
    bonds, perms, chi = cl.triangular_bonds(), cl.translations(), cl.characters(m)
    reps, stab, ia, ja, val = OB.heisenberg_orbit_upper_csr(cl.det, ndown, perms, chi, bonds)
    M, states = qb.heisenberg_orbit(cl.det, ndown, perms, chi, bonds, flags=1, return_states=True)
    assert M.dim == reps.size and np.array_equal(states.astype(np.uint64), reps)
    rowptr, col, v = M.download_expanded()
    eia, eja, ev = _expanded(reps.size, ia, ja, val, oracle)
    assert np.array_equal(rowptr, eia) and np.array_equal(col.astype(np.int64), eja)
    assert np.abs(v - ev).max() < 1e-14


@pytest.mark.parametrize("case", ["hubbard4x3", "hubbard3x3", "heis20", "heis_square4x4"])
def test_term_coded_matrix_free_product_replays_the_walk_exactly(case):
    """QBGPU_MATFREE_TERMS: one byte per entry naming the Hamiltonian term; the product replays the row (column through
    the Lin tables, sign from the occupancy words) in the order of the neighbour walk, so it is bit-identical to the walk
    kernel and agrees with the stored matrix to rounding; the fused Lanczos gives the same E0."""
    mk = {"hubbard4x3": lambda **k: qb.hubbard(12, 6, 6, B.square_bonds(4, 3), 1.0, 1.1, **k),
          "hubbard3x3": lambda **k: qb.hubbard(9, 4, 5, B.square_bonds(3, 3), 0.7, 1.9, **k),
          "heis20": lambda **k: qb.heisenberg(20, 10, B.chain_bonds(20), 1.0, **k),
          "heis_square4x4": lambda **k: qb.heisenberg(16, 8, B.square_bonds(4, 4), 1.0, **k)}[case]
    for cplx in (True, False):
        Ms, Mw, Mt = mk(is_complex=cplx), mk(is_complex=cplx, matrix_free=True), mk(is_complex=cplx, matrix_free=True, flags=64)
        n = Ms.dim
        rng = np.random.default_rng(3)
        x = (rng.normal(size=n) + (1j * rng.normal(size=n) if cplx else 0.0)).astype(np.complex128 if cplx else np.float64)
        ys, yw, yt = (np.zeros_like(x) for _ in range(3))
        Ms.MultMv(x, ys); Mw.MultMv(x, yw); Mt.MultMv(x, yt)
        assert np.array_equal(yw, yt)
        assert np.linalg.norm(yt - ys) / np.linalg.norm(ys) < 1e-13
    e_s = qb.locate_E0_lanczos(mk(is_complex=True), nev=1, ncv=0)["eigenvals"][0]
    e_t = qb.locate_E0_lanczos(mk(is_complex=True, matrix_free=True, flags=64), nev=1, ncv=0)["eigenvals"][0]
    assert abs(e_s - e_t) < 1e-10 * max(1.0, abs(e_s))


_CHAIN16_E0 = [-7.142296361, -6.523407057, -5.990986863, -5.615175598, -5.451965668, -5.525353087, -5.823231143, -6.298652725,
               -6.872106678, -6.298652725, -5.823231143, -5.525353087, -5.451965668, -5.615175598, -5.990986863, -6.523407057]
_TRI4X4_E0 = {(0, 0): -8.555514918, (0, 1): -8.002263841, (0, 2): -7.944709784, (0, 3): -8.002263841, (1, 2): -7.588987242}


def test_device_sectors_reproduce_the_published_sector_energies():
    """The reference's example asserts (chain_Heisenberg_spin_half.cc:102-117, triangular_Heisenberg_spin_half.cc:135-139):
    E0 of all sixteen momentum sectors of the L = 16 chain and of five sectors of the 4x4 triangular cluster, each
    assembled on the device and solved by the fused device Lanczos with the reference's start vector and stop rule."""
    import repr_builders as R
    for k in range(16):
        sec = qb.Sector([16], 8, [k])
        E = qb.locate_E0_lanczos(sec.heisenberg(R.chain_bonds(16)), nev=1, ncv=0)["eigenvals"][0]
        assert abs(E - _CHAIN16_E0[k]) < 1e-8, (k, E)
        sec.free()
    for mn, e0 in _TRI4X4_E0.items():
        sec = qb.Sector([4, 4], 8, list(mn))
        E = qb.locate_E0_lanczos(sec.heisenberg(R.triangular_bonds(4, 4)), nev=1, ncv=0)["eigenvals"][0]
        assert abs(E - e0) < 1e-8, (mn, E)
        sec.free()


@pytest.mark.parametrize("name", ["kpm_heis16_k3", "kpm_tri4x4_k01", "kpm_hubbard4x2"])
def test_kpm_moments_pinned_to_the_references_product(oracle, name):
    """Chebyshev moments of the device loop (qbgpu_kpm_moments_z: two moments per product through the doubling identities)
    against the moments oracle/ref_driver.cc computed with the compiled reference's own csr_mat::MultMv and energy_scale
    (tests/golden/kpm_*.npz): 1e-9, BASELINE.json's bound."""
    import json
    z = np.load(os.path.join(oracle.GOLDEN_DIR, name + ".npz"))
    meta = json.loads(str(z["meta"]))
    A, m0, _ = oracle.load_golden(meta["matrix"])
    M = qb.csr_mat(A.dim, A.ia, A.ja, A.val, A.sym)
    phi = oracle.vec_randomize(A.dim, meta["seed"])
    mu = qb.kpm_moments(M, phi, meta["lo"], meta["hi"], meta["nmom"])
    assert np.abs(mu - z["moments"]).max() < 1e-9
    # the reference's bounds, on the device: 39 unconverged Lanczos steps, so the extreme Ritz values carry the amplified round-off
    # of the coefficients (measured: 4e-7 on the chain sector, < 1e-9 on the others); the moments above use the golden's own bounds
    lo, hi = qb.energy_scale(A.dim, M, np.zeros(2 * A.dim, dtype=np.complex128), 0.1, meta["iters"])
    assert abs(lo - meta["lo"]) < 1e-5 * abs(meta["lo"]) and abs(hi - meta["hi"]) < 1e-5 * abs(meta["hi"])


@pytest.mark.parametrize("kind", ["ordinary", "species", "species_matfree", "matfree"])
def test_hubbard4x3_against_the_references_own_run(oracle, kind):
    """BASELINE config 3's model at the largest size the reference itself assembles in seconds (4x3, N_up = N_dn = 6, dim
    853,776): every handle kind, generated on the device, against the digest of the compiled reference's run
    (tests/golden/hubbard4x3_digest.npz): sampled entries of y = MultMv(vec_randomize(1)) and |y| to 1e-12, the Lanczos step
    count, and E0 = -16.879382788684 to 1e-10."""
    import json
    import lin_builders as B
    from quantum_basis_b200 import _lib
    z = np.load(os.path.join(oracle.GOLDEN_DIR, "hubbard4x3_digest.npz"))
    meta = json.loads(str(z["meta"]))
    bonds = B.square_bonds(4, 3)
    kw = {"ordinary": {}, "species": dict(flags=_lib.SPECIES_ORDER), "species_matfree": dict(flags=_lib.SPECIES_ORDER, matrix_free=True),
          "matfree": dict(matrix_free=True)}[kind]
    M = qb.hubbard(12, 6, 6, bonds, 1.0, 1.1, **kw)
    n = M.dim
    assert n == meta["dim"]
    x = qb.vec_randomize(n, 1, device=True)
    y = qb.DeviceVector(n)
    M.MultMv(x, y)
    yh = y.to_numpy()
    assert np.linalg.norm(yh[z["idx"]] - z["y_at_idx"]) <= 1e-12 * np.linalg.norm(z["y_at_idx"])
    assert abs(np.linalg.norm(yh) - meta["y_norm"]) <= 1e-12 * meta["y_norm"]
    v = np.zeros(2 * n, dtype=np.complex128)
    v[:n] = oracle.vec_randomize(n, 1)
    hess = np.zeros(2000)
    m = qb.lanczos(0, 999, 1000, n, M, v, hess, "sr_val0")
    assert abs(m - meta["lanczos_steps"]) <= 1
    e0 = qb.hess_eigen(hess, 1000, m)[0][0]
    assert abs(e0 - meta["lanczos_E0"]) <= 1e-10 * abs(meta["lanczos_E0"])
    assert abs(e0 + 16.879382788684) < 1e-9
    k = 20
    assert np.abs(hess[1000:1000 + k] - z["lanczos_a"][:k]).max() < 1e-10 and np.abs(hess[1:k] - z["lanczos_b"][1:k]).max() < 1e-10


# ---------------------------------------------------------------------------------------------- native multi-GPU drivers
def _run_dist_check(nproc):
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = os.path.join(root, "scripts", "dist_native_check.py")
    if nproc == 1:
        cmd = [sys.executable, script, "4", "3", "6", "6"]
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
               "--master-port", "29533", script, "4", "3", "6", "6"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert res.returncode == 0 and lines, (res.stdout[-1500:], res.stderr[-1500:])
    import json
    out = json.loads(lines[-1])
    assert out["all_ranks_ok"], out
    return out


def test_native_dist_drivers_one_rank():
    """csrc/dist.cu (qbgpu_dist_*: sharded product, Lanczos with the reference's stop rule, eigenvec_CG, energy_scale, KPM
    moments) on ONE rank against the single-GPU entry points -- same loops, no peers (scripts/dist_native_check.py)."""
    out = _run_dist_check(1)
    assert abs(out["fp64_lanczos"]["E0"] + 16.879382788684) < 1e-9


def test_native_dist_drivers_two_ranks():
    """The same on TWO GPUs: peer-memory pulls, the push all-reduce kernel, E0 equal to the single-GPU run to 1e-10."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    out = _run_dist_check(2)
    assert abs(out["fp64_lanczos"]["E0"] - out["fp64_lanczos"]["E0_single"]) <= 1e-10 * abs(out["fp64_lanczos"]["E0_single"])
