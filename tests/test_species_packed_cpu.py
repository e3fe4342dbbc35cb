"""CPU tests of the packed entry words of stored species-order handles (quantum_basis_b200/csrc/species.cu).

A stored handle built without a row range, with real values, keeps each entry of its two parts as one 32-bit word, column | code << cbits, where
cbits is the bit width of n - 1 and code indexes the part's table of distinct values.  qbgpu_debug_species_packed_host
applies the build's rules on the host; decoding its words must give back exactly the columns and the fp64 bit patterns of
the 12-byte parts that qbgpu_debug_species_host generates.  The device build is compared with the ordinary handle in
tests/test_gpu_species_packed.py.
"""
import ctypes as C

import numpy as np
import pytest

import lin_builders as lb
from quantum_basis_b200 import _lib

p = lambda a: C.c_void_p(a.ctypes.data)   # noqa: E731
null = C.c_void_p(0)


def _parts(ns, nup, ndn, bonds, t, U):
    L = _lib.lib()
    b = np.ascontiguousarray(np.asarray(bonds, dtype=np.int32).reshape(-1, 2))
    sizes = np.zeros(4, dtype=np.int64)
    _lib.check(L.qbgpu_debug_species_host(ns, nup, ndn, b.shape[0], p(b), t, U, 64, p(sizes), *([null] * 11)))
    Du, Dd, tu, td = (int(v) for v in sizes)
    n = Du * Dd
    rpl, rpc = np.empty(n + 1, np.int64), np.empty(n + 1, np.int64)
    cl, vl = np.empty(Du * (td + Dd), np.int32), np.empty(Du * (td + Dd))
    cc, vc = np.empty(Dd * tu, np.int32), np.empty(Dd * tu)
    _lib.check(L.qbgpu_debug_species_host(ns, nup, ndn, b.shape[0], p(b), t, U, 64, p(sizes), null,
                                          p(rpl), p(cl), p(vl), p(rpc), p(cc), p(vc), null, null, null, null))
    return b, n, (cl, vl), (cc, vc)


def _packed(ns, nup, ndn, b, t, U, cbits, nl, nc):
    out = np.zeros(5, np.int64)
    tl, tc = np.zeros(256), np.zeros(256)
    wl, wc = np.zeros(nl, np.uint32), np.zeros(nc, np.uint32)
    _lib.check(_lib.lib().qbgpu_debug_species_packed_host(ns, nup, ndn, b.shape[0], p(b), t, U, cbits, p(out), p(tl), p(wl), p(tc), p(wc)))
    return out, (tl, wl), (tc, wc)


@pytest.mark.parametrize("Lx,Ly,nup,ndn,t,U", [(4, 3, 6, 6, 1.0, 1.1), (4, 4, 3, 3, 1.0, 1.1), (4, 4, 2, 3, -0.7, 4.0), (4, 2, 3, 5, 1.0, 1.1)])
def test_packed_words_decode_to_the_stored_parts(Lx, Ly, nup, ndn, t, U):
    ns, bonds = Lx * Ly, lb.square_bonds(Lx, Ly)
    b, n, local, cross = _parts(ns, nup, ndn, bonds, t, U)
    out, *packed = _packed(ns, nup, ndn, b, t, U, 0, local[0].size, cross[0].size)
    cbits = int(out[0])
    assert cbits == max(1, (n - 1).bit_length())
    for k, ((col, val), (table, words)) in enumerate(zip((local, cross), packed)):
        nt = int(out[1 + k])
        assert nt == np.unique(val.view(np.uint64)).size
        assert out[3 + k] == 1                              # a handful of distinct values: every part of these sizes packs
        codes = (words >> cbits).astype(np.int64)
        assert codes.max() < nt
        assert np.array_equal((words & ((1 << cbits) - 1)).astype(np.int32), col)
        assert np.array_equal(table[codes].view(np.uint64), val.view(np.uint64))     # same fp64 bit patterns
        assert np.all(np.diff(table[:nt]) > 0)              # ordered by value (no -0.0 among these tables)
    # the local part holds the diagonal U*k and the down hops, the cross part only the up hops (+-t, +-2t on doubled bonds)
    assert out[1] > out[2] >= 2


def test_packed_selection_keeps_fp64_when_the_table_does_not_fit():
    ns, bonds = 12, lb.square_bonds(4, 3)
    b, n, local, cross = _parts(ns, 6, 6, bonds, 1.0, 1.1)
    for cbits in (28, 30, 31):                             # room for 16, 4 and 2 codes above the column
        out, (tl, wl), (tc, wc) = _packed(ns, 6, 6, b, 1.0, 1.1, cbits, local[0].size, cross[0].size)
        room = 1 << (32 - cbits)
        for k in range(2):
            assert out[3 + k] == (1 if out[1 + k] <= room else 0), (cbits, out)
    assert out[3] == 0 and out[4] == 1                      # cbits 31: 2 codes -- the cross part's +-t fit, the local table does not
    assert not wl.any()                                     # (no words for a part that keeps its fp64 values)
    assert np.array_equal((wc & 0x7FFFFFFF).astype(np.int32), cross[0])
