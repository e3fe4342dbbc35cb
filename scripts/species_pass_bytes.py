"""DRAM bytes of one reference-order product through a stored species-order handle (the step bench.py times on hubbard
workloads), pass by pass, for three layouts of the stored entries:
  12  separate int32 column and fp64 value (row shards, and every handle before entries were packed)
   5  int32 column plus a 1-byte value code in a side array
   4  one packed word per entry: column | code << cbits (handles built without a row range, real values)
Computed from the shapes alone (entry counts from the library's host twin, no device): what each kernel must read or write
at least once, assuming every gathered vector entry is read from DRAM once per pass (the tiled traversal of pass 2 keeps the
columns of a tile in L2).  Usage: python scripts/species_pass_bytes.py [Lx Ly NUP NDN]; prints one JSON object."""
import ctypes as C
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from quantum_basis_b200 import _lib                      # noqa: E402
from quantum_basis_b200.bench_support import square_bonds  # noqa: E402


def entry_counts(Lx, Ly, nup, ndn):
    b = np.ascontiguousarray(np.asarray(square_bonds(Lx, Ly), dtype=np.int32).reshape(-1, 2))
    sizes = np.zeros(4, dtype=np.int64)
    null = C.c_void_p(0)
    _lib.check(_lib.lib().qbgpu_debug_species_host(Lx * Ly, nup, ndn, b.shape[0], C.c_void_p(b.ctypes.data), 1.0, 1.1, 64,
                                                   C.c_void_p(sizes.ctypes.data), *([null] * 11)))
    Du, Dd, tu, td = (int(v) for v in sizes)
    return Du * Dd, Du * (td + Dd), Dd * tu


def pass_bytes(n, nnz_local, nnz_cross, entry_bytes):
    ns = (n + 31) // 32
    way_in = 16 * n + 4 * n + 8 * n            # complex x in the reference's order, perm, fp64 x in the internal order
    # pass 1: the matrix stream, x once (block by block into shared memory), y written; row metadata repeats (read from L2)
    p1 = nnz_local * entry_bytes + 8 * n + 8 * n
    # pass 2: the matrix stream, rowinfo + rowptr per slice + slice order, x gathered once, y read, perm_inv, complex y_ref written
    p2 = nnz_cross * entry_bytes + 4 * 32 * ns + 8 * ns + 4 * ns + 8 * n + 8 * n + 4 * n + 16 * n
    return {"way_in": way_in, "pass1": p1, "pass1_stream": nnz_local * entry_bytes, "pass2": p2,
            "pass2_stream": nnz_cross * entry_bytes, "total": way_in + p1 + p2}


def main():
    Lx, Ly, nup, ndn = (int(a) for a in sys.argv[1:5]) if len(sys.argv) >= 5 else (4, 4, 8, 8)
    n, zl, zc = entry_counts(Lx, Ly, nup, ndn)
    out = {"lattice": f"{Lx}x{Ly}", "nup": nup, "ndn": ndn, "n": n, "entries_local": zl, "entries_cross": zc,
           "cbits": max(1, (n - 1).bit_length()),
           "layouts": {f"{b}_bytes_per_entry": pass_bytes(n, zl, zc, b) for b in (12, 5, 4)}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
