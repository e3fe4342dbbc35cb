"""CPU checks of the kernel-route helpers (tests/kernel_routes.py): the case tables reach every route the predictor
names, and the per-row error bound accepts correct products and rejects a single wrong entry."""
import numpy as np
import pytest

import kernel_routes as K


def test_ordinary_case_table_covers_every_lane_count_and_value_type():
    table = K.ordinary_route_table()
    routes = {(kind, p["route"]) for (case, kind, fl), p in table.items()}
    for kind in K.VALUE_KINDS:
        for L in K.LANES:
            assert (kind, f"csr_vector_{L}") in routes
        assert (kind, "sjds") in routes
    for (case, kind, fl), p in table.items():
        if fl & K.FORMAT_CSR:
            assert case == f"lanes{p['lanes']}"                 # each lane case takes the lane count it is named for
    # the 256-value dictionary case of the GPU tests and its 257-value fall-back
    assert K.predict_ordinary(100, 10, K.NO_AUTOTUNE | K.VALUE_DICT, True, 256)["route"] == "sjds_dict"
    assert K.predict_ordinary(100, 10, K.NO_AUTOTUNE | K.VALUE_DICT, True, 257)["value_dict"] == 0
    assert K.predict_ordinary(100, 10, K.NO_AUTOTUNE | K.VALUE_DICT, False, None)["value_dict"] == 0


@pytest.mark.parametrize("lanes", K.LANES)
def test_lane_cases_have_the_special_row_lengths(lanes):
    n, ia, ja, val = K.lane_case(lanes)
    rp, col, v = K.expand(n, ia, ja, val)
    lens = set(np.diff(rp).tolist())
    assert {0, 1, lanes, 2 * lanes - 1, 2 * lanes, 2 * lanes + 1} <= lens
    assert K.lanes_for(int(rp[-1]), n) == lanes
    assert K.empty_slices(rp).size >= 1                       # a whole 32-row slice without entries
    # Hermitian: the expanded matrix equals its conjugate transpose
    import scipy.sparse as sp
    A = sp.csr_matrix((v, col, rp), shape=(n, n))
    assert abs(A - A.conj().T).max() == 0


def test_species_case_table_covers_every_pass1_route():
    table = K.species_route_table(lambda name: True)
    seen = {r for kinds in table.values() for routes in kinds.values() for r in routes}
    assert {"pass1_block_bulk_x", "pass1_block_thread_x", "pass1_plain", "periodic_meta", "no_periodic_meta", "empty_cross",
            "dn_dim_1", "n_below_32", "pass2_bulk", "packed"} <= seen
    assert "unpacked" in K.predict_species(4, 6, False, False)
    t = {name: table[name] for name in table}
    assert "pass1_block_thread_x" in t["4x3_1_4"]["fp64"] and "no_periodic_meta" in t["4x3_1_4"]["fp64"]
    assert "periodic_meta" in t["4x3_2_4"]["fp64"] and "pass1_block_thread_x" in t["4x3_2_4"]["fp64"]
    assert "pass1_block_bulk_x" in t["4x4_1_7"]["fp64"] and "pass1_plain" in t["4x4_1_7"]["complex"]
    assert "pass1_block_thread_x" in t["5x3_3_7"]["fp64"] and "pass1_block_bulk_x" in t["5x3_3_7"]["complex"]
    assert "pass1_plain" in t["6x3_1_9"]["fp64"] and "pass1_plain" in t["6x3_1_9"]["complex"]
    assert "empty_cross" in t["4x3_0_4"]["fp64"] and "dn_dim_1" in t["4x3_5_0"]["fp64"]
    assert "n_below_32" in t["2x2_1_2"]["fp64"] and "n_below_32" in t["4x3_0_0"]["fp64"]
    assert "periodic_meta" in t["4x4_2_1"]["fp64"]                          # gcd(32, 16) = 16: a period of 2 blocks
    # an 8-byte-aligned x turns the bulk copy off
    assert "pass1_block_thread_x" in K.predict_species(16, 11440, False, True, 1, x_aligned16=False)


def _random_csr(rng, n, per_row, cplx):
    lens = rng.integers(0, per_row + 1, n)
    rp = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = np.concatenate([np.sort(rng.choice(n, k, replace=False)) for k in lens]).astype(np.int64)
    v = rng.normal(size=rp[-1]) * np.exp(rng.uniform(-8, 8, rp[-1]))          # magnitudes over 7 decades
    if cplx:
        v = v + 1j * rng.normal(size=rp[-1])
    return rp, col, v


@pytest.mark.parametrize("cplx", [False, True])
def test_bound_accepts_the_long_double_and_fp64_products(oracle, cplx):
    from oracle_lib import Csr
    rng = np.random.default_rng(3)
    n = 3000
    rp, col, v = _random_csr(rng, n, 40, cplx)
    x = rng.normal(size=n) + (1j * rng.normal(size=n) if cplx else 0)
    ref = K.RowRef(rp, col, v, x)
    A = Csr(n, rp, col, v.astype(np.complex128), False)
    y_ld = oracle.spmv_ld(A, x)                                   # the oracle's long-double product, rounded to fp64
    assert K.row_errors(y_ld, ref, x, cplx=True)[0].size == 0
    import scipy.sparse as sp
    y64 = sp.csr_matrix((v, col, rp), shape=(n, n)) @ x           # plain fp64 sums in another order
    assert K.row_errors(y64, ref, x, cplx=cplx)[0].size == 0
    # epilogue with complex scalars, in fp64
    z = rng.normal(size=n) + 1j * rng.normal(size=n)
    a, g, b = 0.7 - 0.3j, 0.2 + 0.45j, -0.6 + 0.25j
    y = a * y64 + g * x + b * z
    assert K.row_errors(y, ref, x, z, a, g, b, cplx=True)[0].size == 0
    d = np.array([np.vdot(x, y).real, np.vdot(x, y).imag, np.vdot(y, y).real])
    K.assert_dots(d, x, y)


def _million_row_case(rng):
    n = 1_000_000
    rp, col, v = _random_csr(rng, n, 12, False)
    x = rng.normal(size=n)
    import scipy.sparse as sp
    y = sp.csr_matrix((v, col, rp), shape=(n, n)) @ x
    return n, rp, col, v, x, y


def test_bound_rejects_one_wrong_entry_in_a_million_rows():
    rng = np.random.default_rng(9)
    n, rp, col, v, x, y = _million_row_case(rng)
    ref = K.RowRef(rp, col, v, x)
    assert K.row_errors(y, ref, x, cplx=False)[0].size == 0
    r = int(np.argmax(np.diff(rp) >= 6))
    k = rp[r] + 3
    # a perturbed entry: the value in the last bits of its sixth significant digit
    y_bad = y.copy()
    y_bad[r] += 1e-6 * abs(v[k] * x[col[k]])
    bad, _ = K.row_errors(y_bad, ref, x, cplx=False)
    assert bad.tolist() == [r]
    assert np.linalg.norm(y_bad - y) / np.linalg.norm(y) < 1e-12               # invisible to a global relative l2
    # a dropped tail entry (the kernel's unpaired last entry)
    y_drop = y.copy()
    e = rp[r + 1] - 1
    y_drop[r] -= v[e] * x[col[e]]
    bad, _ = K.row_errors(y_drop, ref, x, cplx=False)
    assert bad.tolist() == [r]
    # an empty row written as anything but 0 / z
    er = int(np.argmax(np.diff(rp) == 0))
    y_e = y.copy(); y_e[er] = 1e-300
    assert K.row_errors(y_e, ref, x, cplx=False)[0].tolist() == [er]
