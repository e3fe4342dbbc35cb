#!/usr/bin/env python
"""Every route of tests/test_gpu_krylov_boundary.py (tests/krylov_routes.py) on its seeded inputs, with host and device vectors,
through the real views and with QBGPU_NO_REAL_MODE=1, each output written to DIR/<handle kind>.npz -- so that two builds of
libqbgpu.so can be compared array by array.  One GPU.

  python scripts/krylov_routes_dump.py [--lib path/to/libqbgpu.so] DIR
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", help="the library to load instead of quantum_basis_b200/libqbgpu.so")
    ap.add_argument("out", help="output directory")
    args = ap.parse_args()
    from quantum_basis_b200 import _lib
    if args.lib:
        _lib.LIB_PATH = os.path.abspath(args.lib)            # before the first load
    import krylov_routes as K
    import quantum_basis_b200 as qb
    assert qb.lib().qbgpu_init(0) == 0, qb.lib().qbgpu_last_error()
    os.makedirs(args.out, exist_ok=True)
    for kind in K.KINDS:
        M = K.make(kind)
        X = K.inputs(M)
        res = {f"inputs/{k}": np.atleast_1d(v) for k, v in X.items()}
        for dev in (False, True):
            tag = "device" if dev else "host"
            res.update({f"{tag}/{k}": v for k, v in K.run(M, X, dev).items()})
            if kind in K.REAL_VALUED:
                res.update({f"{tag}/real_view/{k}": v for k, v in K.run(M.real_view(), X, dev).items()})
            os.environ["QBGPU_NO_REAL_MODE"] = "1"
            res.update({f"{tag}/no_real_mode/{k}": v for k, v in K.run(M, X, dev).items()})
            del os.environ["QBGPU_NO_REAL_MODE"]
        np.savez(os.path.join(args.out, kind + ".npz"), **{k.replace("/", "."): v for k, v in res.items()})
        print(f"{kind}: {len(res)} arrays", flush=True)
        M.destroy()


if __name__ == "__main__":
    main()
