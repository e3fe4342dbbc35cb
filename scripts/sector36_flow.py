#!/usr/bin/env python
"""36-site spin-1/2 momentum sectors on one GPU: enumeration, matrix-free product and Lanczos E0.

Runs the Heisenberg model on the 6x6 square lattice at (Sz = 0, k = (0, 0)) and on the chain L = 36 at k = 0 (64-bit
states, matrix-free product) and prints one JSON line: enumerate / norm / Lin-table check seconds, the product's median
and minimum over `--reps` timed products after `--warmup` untimed ones (x = vec_randomize seed 1; the sector's keys and
norms, 4 GB, and the two 4 GB vectors do not fit in L2), and Lanczos E0 to the reference's stop rule (steps, iterations
per second, time to solution), with the card's name and power limit read in the same run.

  python scripts/sector36_flow.py --out profiles/r05_sector36_flow.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import quantum_basis_b200 as qb  # noqa: E402
import bethe_chain  # noqa: E402
import repr_builders as R  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def run(name, L, bonds, reps, warmup, reference):
    lib = qb.lib()
    t0 = time.time()
    sec = qb.Sector(L, int(np.prod(L)) // 2, [0] * len(L))
    t_create = time.time() - t0
    H = sec.heisenberg_matrix_free(bonds)
    x = qb.vec_randomize(sec.dim, 1, device=True)
    y = qb.DeviceVector(sec.dim)
    for _ in range(warmup):
        H.MultMv(x, y)
    lib.qbgpu_synchronize()
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        H.MultMv(x, y)
        lib.qbgpu_synchronize()
        ts.append(time.perf_counter() - t)
    x.free(); y.free()
    t0 = time.time()
    res = qb.locate_E0_lanczos(H, nev=1, ncv=0)
    t_e0 = time.time() - t0
    E0 = res["eigenvals"][0]
    out = {"case": name, "L": L, "dim": sec.dim, "zero_norm": sec.zero_norm, "lin_order": sec.lin_order, "state_bits": sec.state_bits,
           "create_s": t_create, "enumerate_s": sec.enumerate_seconds, "lin_check_host_s": sec.lin_check_seconds, "norms_s": sec.norms_seconds,
           "product_median_s": float(np.median(ts)), "product_min_s": float(np.min(ts)), "timed_products": reps, "warmup_products": warmup,
           "lanczos_steps": res["lanczos_steps"], "lanczos_s": t_e0, "lanczos_iter_per_s": res["lanczos_steps"] / t_e0,
           "E0": E0, "E0_per_site": E0 / np.prod(L)}
    if reference is not None:
        out["E0_reference"], out["E0_rel_diff"] = reference[1], abs(E0 - reference[1]) / abs(reference[1])
        out["E0_reference_source"] = reference[0]
    del H
    sec.free()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--cases", default="square6x6,chain36")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    assert qb.lib().qbgpu_init(0) == 0
    result = {"card": card(), "cases": []}
    for c in a.cases.split(","):
        if c == "square6x6":
            result["cases"].append(run(c, [6, 6], R.square_bonds(6, 6), a.reps, a.warmup,
                                       ("E0/N = -0.678872, Schulz, Ziman & Poilblanc 1996", -0.678872 * 36)))
        elif c == "chain36":
            result["cases"].append(run(c, [36], R.chain_bonds(36), a.reps, a.warmup, ("Bethe ansatz", bethe_chain.ground_state_energy(36))))
        else:
            raise SystemExit(f"unknown case {c}")
    line = json.dumps(result)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
