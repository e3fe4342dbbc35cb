#!/usr/bin/env python
"""locate_E0_lanczos(nev = 2, ncv = 2) of BASELINE config 3 (Hubbard 4x4, 8+8, t = 1, U = 1.1) on N GPUs with the native
multi-GPU drivers: species-order shards, fp64 vectors through the real view.

    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29549 scripts/dist_locate_e0.py [--single]

Runs the four stages one by one through the public entry points, in the order and with the seeds of the one-call flow
(E0: sr_val0 Lanczos from vec_randomize(1); phi0: eigenvec_CG from vec_randomize(1); E1: sr_val1 Lanczos from vec_randomize(1)
projected off phi0; phi1: eigenvec_CG at E1 from vec_randomize(8)) with a wall clock around each, then the one-call flow
(NativeDist.locate_E0_lanczos) timed as a whole.  --single (N = 1 only): also the single-GPU csr.locate_E0_lanczos on the full
handle, its E1 and its time.  Prints one JSON line (rank 0) with the card's name and power limit read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import quantum_basis_b200 as qb
from quantum_basis_b200 import dist as qd
from quantum_basis_b200.bench_support import square_bonds

E0_CONFIG3 = -20.497352266554


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim, clk = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:                                   # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"not read ({e})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--single", action="store_true", help="N = 1: also the single-GPU csr.locate_E0_lanczos")
    ap.add_argument("--maxit", type=int, default=1000)
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    L = qb.lib()
    assert L.qbgpu_init(local_rank) == 0
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    assert L.qbgpu_set_stream(C.c_void_p(stream.cuda_stream)) == 0
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")

        def exchange(b):
            out = [None] * world
            dist.all_gather_object(out, b)
            return out

        def tmax(t):
            x = torch.tensor([t], dtype=torch.float64)
            dist.all_reduce(x, op=dist.ReduceOp.MAX)
            return float(x.item())

        def barrier():
            dist.barrier()

        def allsum(v):
            x = torch.tensor([v], dtype=torch.float64)
            dist.all_reduce(x)
            return float(x.item())
    else:
        exchange = lambda b: [b]          # noqa: E731
        tmax = allsum = lambda t: t       # noqa: E731
        barrier = lambda: None            # noqa: E731
    maxit = args.maxit
    ns, nup, ndn = 16, 8, 8
    bonds = square_bonds(4, 4)
    n = L.qbgpu_dim_hubbard(ns, nup, ndn)
    bounds, _ = qd.species_nnz_balanced_bounds(ns, nup, ndn, bonds, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    nloc = hi - lo
    out = {"workload": "hubbard4x4 8+8 (BASELINE config 3), species-order shards, fp64 vectors (real view)", "gpus": world, "n": n}
    if rank == 0:
        out.update(card())
    t0 = time.time()
    M = qb.hubbard(ns, nup, ndn, bonds, 1.0, 1.1, flags=128, rows=(lo, hi))
    shard = qd.SpeciesShard(qb, M, ns, nup, ndn, bonds, bounds, rank, world, real=True)
    D = qd.NativeDist(qb, n, bounds, rank, world, False, exchange)
    mode = os.environ.get("QB_DIST_MODE", "refined_needed_rows" if world > 1 else "plain_whole_slices")
    shard.install(D, mode, lanes=1)
    loc, cross = shard.local, shard.cross
    ref_rows = torch.empty(max(nloc, 1), dtype=torch.int32, device="cuda")
    assert L.qbgpu_species_ref_rows(ns, nup, ndn, lo, hi, C.c_void_p(ref_rows.data_ptr())) == 0, L.qbgpu_last_error()
    torch.cuda.synchronize()
    out["build_s"] = tmax(time.time() - t0)
    out["decomposition"] = mode
    rr = ref_rows.data_ptr()
    vb = 8 * max(nloc, 1)
    phi = torch.zeros(2 * max(nloc, 1), dtype=torch.float64, device="cuda")
    phi0, phi1 = phi.data_ptr(), phi.data_ptr() + vb
    work = [torch.zeros(max(nloc, 1), dtype=torch.float64, device="cuda") for _ in range(3)]
    wp = [w.data_ptr() for w in work]

    def seeded(dst, seed):
        D.randomize(0, seed, rr)
        if nloc:
            assert L.qbgpu_memcpy_d2d(C.c_void_p(dst), C.c_void_p(D.own(0)), nloc * 8) == 0

    def project_start():
        """X[0] <- vec_randomize(1) - <phi0, .> phi0, normalised (src/model.cc:1240-1252), with torch on the own slice"""
        D.randomize(0, 1, rr)
        x = torch.zeros(max(nloc, 1), dtype=torch.float64, device="cuda")
        if nloc:
            assert L.qbgpu_memcpy_d2d(C.c_void_p(x.data_ptr()), C.c_void_p(D.own(0)), nloc * 8) == 0
        p0 = phi[:max(nloc, 1)]
        h = allsum(float(torch.dot(p0[:nloc], x[:nloc]).item()) if nloc else 0.0)
        x.sub_(h * p0)
        nn = allsum(float(torch.dot(x[:nloc], x[:nloc]).item()) if nloc else 0.0)
        x.mul_(1.0 / np.sqrt(nn))
        if nloc:
            assert L.qbgpu_memcpy_d2d(C.c_void_p(D.own(0)), C.c_void_p(x.data_ptr()), nloc * 8) == 0
        torch.cuda.synchronize()
        D.barrier()

    def timed(fn):
        torch.cuda.synchronize(); barrier()
        t = time.time()
        r = fn()
        torch.cuda.synchronize(); barrier()
        return r, tmax(time.time() - t)

    # warm-up: every kernel of the loops has been loaded and launched once
    D.randomize(0, 1, rr)
    D.lanczos(loc, cross, 6, maxit, "sr_val0")
    seeded(phi0, 1)
    D.eigenvec_cg(loc, cross, E0_CONFIG3, phi0, *wp, maxit=2)
    project_start()
    D.lanczos_val1(loc, cross, phi0, 6, maxit)

    # the four stages, one by one
    D.randomize(0, 1, rr)
    (m0, h0), t_l0 = timed(lambda: D.lanczos(loc, cross, maxit - 1, maxit, "sr_val0"))
    E0 = float(qb.hess_eigen(h0, maxit, m0)[0][0])
    seeded(phi0, 1)
    (mc0, ac0), t_c0 = timed(lambda: D.eigenvec_cg(loc, cross, E0, phi0, *wp, maxit=maxit))
    project_start()
    (m1, h1), t_l1 = timed(lambda: D.lanczos_val1(loc, cross, phi0, maxit - 1, maxit))
    E1 = float(qb.hess_eigen(h1, maxit, m1)[0][0])
    seeded(phi1, 8)
    (mc1, ac1), t_c1 = timed(lambda: D.eigenvec_cg(loc, cross, E1, phi1, *wp, maxit=maxit))
    out["stages"] = {"E0": E0, "E1": E1, "gap": E1 - E0, "steps": [m0, mc0, m1, mc1], "cg_accuracy": [float(ac0), float(ac1)],
                     "seconds": {"lanczos_E0": t_l0, "cg_phi0": t_c0, "lanczos_E1": t_l1, "cg_phi1": t_c1},
                     "lanczos_it_per_s": {"E0_loop": m0 / t_l0, "E1_loop": m1 / t_l1},
                     "E1_loop_over_E0_loop_it_per_s": (m1 / t_l1) / (m0 / t_l0)}
    # the one-call flow
    got, t_flow = timed(lambda: D.locate_E0_lanczos(loc, cross, nev=2, ncv=2, maxit=maxit, ref_rows_ptr=rr))
    out["flow"] = {"E0": got["eigenvals"][0], "E1": got["eigenvals"][1], "gap": got["gap"],
                   "steps": [got["lanczos_steps"], got["cg_steps"], got["lanczos_steps_E1"], got["cg_steps_E1"]], "seconds": t_flow}
    out["E0_ok"] = bool(abs(got["eigenvals"][0] - E0_CONFIG3) < 1e-10 and abs(E0 - E0_CONFIG3) < 1e-10)
    out["timing"] = "wall clock from a device synchronise to a device synchronise, max over ranks; kernels warmed up by short runs"
    # QBGPU_VERBOSE phase breakdown of both loops (per-step device time of the phases; on stderr)
    os.environ["QBGPU_VERBOSE"] = "1"
    D.randomize(0, 1, rr)
    D.lanczos(loc, cross, maxit - 1, maxit, "sr_val0")
    project_start()
    D.lanczos_val1(loc, cross, phi0, maxit - 1, maxit)
    os.environ.pop("QBGPU_VERBOSE")
    D.destroy(); shard.destroy(); M.destroy()
    del work, phi
    if args.single and world == 1:
        torch.cuda.empty_cache()
        full = qb.hubbard(ns, nup, ndn, bonds, 1.0, 1.1, flags=128)
        r1, t1 = timed(lambda: qb.locate_E0_lanczos(full, nev=2, ncv=2, maxit=maxit))
        out["single_gpu_csr_locate_E0_lanczos"] = {"E0": float(r1["eigenvals"][0]), "E1": float(r1["eigenvals"][1]), "gap": float(r1["gap"]),
                                                   "steps": [int(r1["lanczos_steps"]), int(r1["cg_steps"]), int(r1["lanczos_steps_E1"]), int(r1["cg_steps_E1"])],
                                                   "seconds": t1, "timing": "includes the download of both eigenvectors to the host"}
        out["E1_vs_single_rel"] = float(abs(got["eigenvals"][1] - r1["eigenvals"][1]) / abs(r1["eigenvals"][1]))
        out["E1_ok"] = bool(out["E1_vs_single_rel"] <= 1e-8)
        full.destroy()
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sys.exit(0 if out["E0_ok"] and out.get("E1_ok", True) else 1)


if __name__ == "__main__":
    main()
