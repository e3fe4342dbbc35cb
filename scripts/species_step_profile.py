#!/usr/bin/env python
"""Kernel split of the bench step on a stored species-order handle: torch.profiler (CUDA activities) around repeated
reference-order MultMv calls (device vectors, real content -- the fp64 passes and the fused way out), the same call
bench.py times.  Prints one JSON line: per kernel name the calls, the total and the mean time per call.

    python scripts/species_step_profile.py [workload] [reps] [out.json]
"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from torch.profiler import ProfilerActivity, profile

import bench
import quantum_basis_b200 as qb


def main():
    workload = sys.argv[1] if len(sys.argv) > 1 else "hubbard4x4"
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
    out = sys.argv[3] if len(sys.argv) > 3 else None
    L = qb.lib()
    assert L.qbgpu_init(0) == 0
    fam, p = bench.WORKLOADS[workload]
    M = qb.hubbard(p["Lx"] * p["Ly"], p["nup"], p["ndn"], bench.square_bonds(p["Lx"], p["Ly"]), p["t"], p["U"], flags=128)
    n = M.info.n
    x = qb.vec_randomize(n, 1, device=True)
    y = qb.DeviceVector(n)
    for _ in range(5):
        M.MultMv(x, y)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            M.MultMv(x, y)
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        k = kernels.setdefault(ev.name, {"calls": 0, "total_ms": 0.0})
        k["calls"] += 1
        k["total_ms"] += ev.time_range.elapsed_us() / 1e3
    for k in kernels.values():
        k["ms_per_call"] = k["total_ms"] / k["calls"]
    line = {"workload": workload, "n": n, "reps": reps, "gpu": torch.cuda.get_device_name(0),
            "step_ms": sum(k["total_ms"] for k in kernels.values()) / reps,
            "kernels": dict(sorted(kernels.items(), key=lambda kv: -kv[1]["total_ms"]))}
    print(json.dumps(line))
    if out:
        with open(out, "w") as f:
            json.dump(line, f, indent=1)


if __name__ == "__main__":
    main()
