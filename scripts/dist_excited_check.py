#!/usr/bin/env python
"""E1 and the gap on N ranks: the sharded sr_val1 Lanczos (qbgpu_dist_lanczos_val1) and the four-stage flow
(qbgpu_dist_locate_e0_lanczos) against the single-GPU entry points:

    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29547 scripts/dist_excited_check.py

also runs with N = 1 (plain python).  Every rank builds its shard AND the full single-GPU handle of the same model (small
sizes) and checks
  1. loop parity: sr_val1 from the same phi0 and start vector as qb.lanczos(..., "sr_val1") -- steps within 1, the first 20
     a and b within 1e-10, E1 within 1e-10 relative -- on Hubbard 4x3 species shards (fp64 and complex vectors) and an
     ordinary complex row shard of the L = 16 Heisenberg chain; once more with QBGPU_DIST_SPECULATE=0, bit-identical;
  2. flow parity: locate_E0_lanczos(nev = 2, ncv = 2) against the single-GPU flow on Hubbard 4x3 (E0, E1, residuals and
     norms of phi0 and phi1, bit-identical eigenvalues and step counts on every rank);
  3. degenerate pairs: the tj12 golden (E0 = E1 = -9.762087307 by ARPACK, src/main_test.cc:207-208) as ordinary row shards,
     and a diagonal matrix with a doubly degenerate ground level; the gap and whether the orthonormalisation of phi1 against
     phi0 (src/model.cc:1302-1311) ran are recorded, and when it ran |<phi0|phi1>| < 1e-10 is required.  On tj12 the Lanczos
     flow does not find the degenerate partner, on one GPU as on the shards: the Krylov space of one start vector holds one
     direction of a degenerate level, and phi0 -- CG from the same vec_randomize(1) -- is that direction, so the start vector
     projected off phi0 has no component left in the level and E1 is the next level, -9.717157950726.  E1 is held to the
     single-GPU flow there, and the branch is covered by the diagonal case, where E1 = E0 to round-off;
  4. shapes (nev, ncv) = (1, 0), (1, 1) and the argument errors.
Prints one JSON line (rank 0) with all_ranks_ok and exits non-zero on a mismatch."""
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import quantum_basis_b200 as qb
from quantum_basis_b200 import dist as qd
from quantum_basis_b200.bench_support import square_bonds

E0_HUB43 = -16.879382788684          # the reference's value for Hubbard 4x3, 6+6, t = 1, U = 1.1
E_TJ12 = -9.762087307                 # src/main_test.cc:207-208: E0 = E1
LANCZOS_PRECISION = 2e-12
QBGPU_ERR_ARG = 1


def main():
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    device = local_rank % torch.cuda.device_count()          # more ranks than GPUs: ranks share a device (IPC on one GPU)
    torch.cuda.set_device(device)
    L = qb.lib()
    assert L.qbgpu_init(device) == 0
    stream = torch.cuda.Stream()                  # one stream for torch and the library (like dist_native_check.py)
    torch.cuda.set_stream(stream)
    assert L.qbgpu_set_stream(C.c_void_p(stream.cuda_stream)) == 0
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")                      # host-side plumbing only: handles, check sums, the verdict

        def exchange(b):
            out = [None] * world
            dist.all_gather_object(out, b)
            return out
    else:
        exchange = lambda b: [b]          # noqa: E731
    ok = True
    out = {"world": world}

    def check(name, cond, detail):
        nonlocal ok
        ok = ok and bool(cond)
        out[name] = detail if cond else {"FAILED": detail}
        if not cond:
            print(f"[dist_excited_check] rank {rank}: {name} FAILED: {detail}", file=sys.stderr, flush=True)

    def allsum(vals):
        t = torch.tensor([[complex(v).real, complex(v).imag] for v in vals], dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t)
        return [complex(a, b) for a, b in t.cpu().numpy()]

    def same_on_all_ranks(obj):
        if world == 1:
            return True
        allv = [None] * world
        dist.all_gather_object(allv, obj)
        return all(v == allv[0] for v in allv)

    def dev(arr, cplx):
        """this rank's rows as a device buffer of the vector type (at least one element: a valid pointer on an empty shard)"""
        a = np.ascontiguousarray(arr if cplx else np.real(arr), dtype=np.complex128 if cplx else np.float64)
        t = torch.zeros(max(a.size, 1) * (2 if cplx else 1), dtype=torch.float64, device="cuda")
        if a.size:
            t[:a.size * (2 if cplx else 1)] = torch.from_numpy(a.view(np.float64)).cuda()
        return t

    def residual(D, loc, rest, v_local, E):
        """(|H v - E v|, |v|) over all ranks, with the sharded product"""
        D.upload_own(0, v_local)
        y = torch.zeros((2 if D.complex else 1) * max(D.nloc, 1), dtype=torch.float64, device="cuda")
        D.mv(loc, rest, 0, y.data_ptr(), barrier=3)
        hv = y.cpu().numpy()
        hv = (hv.view(np.complex128) if D.complex else hv)[:D.nloc]
        s = allsum([np.linalg.norm(hv - E * v_local) ** 2, np.linalg.norm(v_local) ** 2])
        return float(np.sqrt(s[0].real)), float(np.sqrt(s[1].real))

    def overlap(a_local, b_local):
        return abs(allsum([np.vdot(a_local, b_local)])[0])

    def loop_parity(tag, D, loc, rest, full, n, rows_of, phi_ref):
        """sr_val1 on the shards vs qb.lanczos(..., "sr_val1") from the same phi0 and start vector"""
        x = qb.vec_randomize(n, 1)
        x = x - np.vdot(phi_ref, x) * phi_ref
        x /= np.linalg.norm(x)
        v = np.zeros(3 * n, dtype=np.complex128)
        v[:n], v[2 * n:] = x, phi_ref
        hs = np.zeros(2000)
        ms = qb.lanczos(0, 999, 1000, n, full, v, hs, "sr_val1")
        es = qb.hess_eigen(hs, 1000, ms)[0][0]
        phi = dev(rows_of(phi_ref), D.complex)
        runs = []
        for spec in (None, "0"):
            if spec is None:
                os.environ.pop("QBGPU_DIST_SPECULATE", None)
            else:
                os.environ["QBGPU_DIST_SPECULATE"] = spec
            D.upload_own(0, rows_of(x))
            D.barrier()
            runs.append(D.lanczos_val1(loc, rest, phi.data_ptr(), 999, 1000))
        os.environ.pop("QBGPU_DIST_SPECULATE", None)
        (m, h), (m2, h2) = runs
        e = qb.hess_eigen(h, 1000, m)[0][0]
        da = float(np.abs(h[1000:1020] - hs[1000:1020]).max())
        db = float(np.abs(h[1:21] - hs[1:21]).max())
        check(f"{tag}_val1_loop", abs(m - ms) <= 1 and da < 1e-10 and db < 1e-10 and abs(e - es) <= 1e-10 * abs(es),
              {"steps": m, "steps_single": int(ms), "E1": float(e), "E1_single": float(es), "max_da_first20": da, "max_db_first20": db})
        check(f"{tag}_val1_no_speculation_bit_identical", m2 == m and np.array_equal(h2, h), {"steps": m2})
        return float(e)

    def flow_checks(D, loc, rest, ref, ref_rows_ptr, e_tol):
        got = D.locate_E0_lanczos(loc, rest, nev=2, ncv=2, maxit=1000, ref_rows_ptr=ref_rows_ptr)
        E0, E1 = got["eigenvals"]
        E0s, E1s = ref["eigenvals"]
        r0, n0 = residual(D, loc, rest, got["eigenvecs"][0], E0)
        r1, n1 = residual(D, loc, rest, got["eigenvecs"][1], E1)
        keys = ("lanczos_steps", "cg_steps", "lanczos_steps_E1", "cg_steps_E1")
        steps = [got[k] for k in keys]
        same = same_on_all_ranks((float(E0).hex(), float(E1).hex(), steps))
        detail = {"E0": E0, "E1": E1, "gap": got["gap"], "E0_single": float(E0s), "E1_single": float(E1s), "gap_single": float(ref["gap"]),
                  "steps": steps, "steps_single": [int(ref[k]) for k in keys], "accuracies": [got["lanczos_accuracy"], got["cg_accuracy"], got["cg_accuracy_E1"]],
                  "residual_phi0": r0, "residual_phi1": r1, "norm_phi0": n0, "norm_phi1": n1, "identical_on_all_ranks": same}
        cond = (abs(E0 - E0s) <= 1e-10 * abs(E0s) and abs(E1 - E1s) <= e_tol * abs(E1s) and r0 < 1e-8 and r1 < 1e-8
                and abs(n0 - 1) < 1e-10 and abs(n1 - 1) < 1e-10 and same)
        return got, detail, cond

    # ------------------------------------------------------------------ Hubbard 4x3, 6+6: species-order shards
    ns, nup, ndn = 12, 6, 6
    bonds = square_bonds(4, 3)
    n = L.qbgpu_dim_hubbard(ns, nup, ndn)
    bounds, _ = qd.species_nnz_balanced_bounds(ns, nup, ndn, bonds, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    nloc = hi - lo
    full = qb.hubbard(ns, nup, ndn, bonds, 1.0, 1.1, flags=128)
    perm = full.native_perm()
    ref = qb.locate_E0_lanczos(full, nev=2, ncv=2)                          # single GPU, reference order
    ref10 = qb.locate_E0_lanczos(full, nev=1, ncv=0)
    ref11 = qb.locate_E0_lanczos(full, nev=1, ncv=1)

    def rows_int(vec):                                                       # this rank's rows in the internal order
        w = np.empty_like(vec)
        w[perm] = vec
        return w[lo:hi]

    ref_rows = torch.empty(max(nloc, 1), dtype=torch.int32, device="cuda")
    assert L.qbgpu_species_ref_rows(ns, nup, ndn, lo, hi, C.c_void_p(ref_rows.data_ptr())) == 0, L.qbgpu_last_error()
    M = qb.hubbard(ns, nup, ndn, bonds, 1.0, 1.1, flags=128, rows=(lo, hi))
    for tag, cplx in (("fp64", False), ("complex", True)):
        shard = qd.SpeciesShard(qb, M, ns, nup, ndn, bonds, bounds, rank, world, real=not cplx, gap=2)
        loc, cross = shard.local, shard.cross
        D = qd.NativeDist(qb, n, bounds, rank, world, cplx, exchange)
        shard.install(D, "rows2_needed_rows" if cplx else "refined_needed_rows", lanes=1)
        loop_parity(f"{tag}_hubbard4x3", D, loc, cross, full, n, lambda vec: rows_int(vec) if cplx else rows_int(vec).real, ref["eigenvecs"][0])
        got, detail, cond = flow_checks(D, loc, cross, ref, ref_rows.data_ptr(), 1e-8)
        check(f"{tag}_hubbard4x3_flow", cond and abs(got["eigenvals"][0] - E0_HUB43) < 1e-9, detail)
        if not cplx:
            # shapes: (1, 0) -> E0 only; (1, 1) -> E0 and phi0, both as the single-GPU mirror
            g10 = D.locate_E0_lanczos(loc, cross, nev=1, ncv=0, ref_rows_ptr=ref_rows.data_ptr())
            g11 = D.locate_E0_lanczos(loc, cross, nev=1, ncv=1, ref_rows_ptr=ref_rows.data_ptr())
            e10, e11 = g10["eigenvals"][0], g11["eigenvals"][0]
            dphi = allsum([np.abs(g11["eigenvecs"][0] - rows_int(ref11["eigenvecs"][0]).real).max() if nloc else 0.0])[0].real
            check("shape_1_0", len(g10["eigenvals"]) == 1 and g10["eigenvecs"] == [] and "cg_steps" not in g10
                  and abs(e10 - ref10["eigenvals"][0]) <= 1e-10 * abs(ref10["eigenvals"][0]) and g10["lanczos_steps"] > 0,
                  {"E0": e10, "E0_single": float(ref10["eigenvals"][0]), "steps": g10["lanczos_steps"]})
            check("shape_1_1", len(g11["eigenvals"]) == 1 and len(g11["eigenvecs"]) == 1 and "gap" not in g11 and dphi < 1e-8
                  and abs(e11 - ref11["eigenvals"][0]) <= 1e-10 * abs(ref11["eigenvals"][0]),
                  {"E0": e11, "cg_steps": g11["cg_steps"], "cg_steps_single": int(ref11["cg_steps"]), "sum_max_abs_dphi0": dphi})
            # argument errors: QBGPU_ERR_ARG and a message, before any collective work (every rank returns alike)
            w, st, ac = np.zeros(4), np.zeros(4, dtype=np.int64), np.zeros(4)
            buf = torch.zeros(2 * max(nloc, 1), dtype=torch.float64, device="cuda")
            m64 = C.c_int64(0)
            hs = np.zeros(2000)

            def flow_rc(nev, ncv, phi):
                rc = L.qbgpu_dist_locate_e0_lanczos(D.h, loc.handle, cross.handle, C.c_void_p(ref_rows.data_ptr()), nev, ncv, 1000,
                                                    C.c_void_p(w.ctypes.data), phi, C.c_void_p(st.ctypes.data), C.c_void_p(ac.ctypes.data))
                return rc, L.qbgpu_last_error().decode(errors="replace")
            errs = {"nev3": flow_rc(3, 2, C.c_void_p(buf.data_ptr())), "nev2_ncv0": flow_rc(2, 0, None),
                    "nev1_ncv2": flow_rc(1, 2, C.c_void_p(buf.data_ptr())), "ncv1_null_phi": flow_rc(1, 1, None)}
            rc = L.qbgpu_dist_lanczos_val1(D.h, loc.handle, cross.handle, None, 999, 1000, C.byref(m64), C.c_void_p(hs.ctypes.data), 1)
            errs["val1_null_phi0"] = (rc, L.qbgpu_last_error().decode(errors="replace"))
            rc = L.qbgpu_dist_lanczos(D.h, loc.handle, cross.handle, 999, 1000, C.byref(m64), C.c_void_p(hs.ctypes.data), b"sr_val1", 1)
            errs["dist_lanczos_sr_val1"] = (rc, L.qbgpu_last_error().decode(errors="replace"))
            check("argument_errors", all(r == QBGPU_ERR_ARG and len(msg) > 0 for r, msg in errs.values()), errs)
        D.destroy(); shard.destroy()
    M.destroy(); full.destroy()

    # ------------------------------------------------------------------ an ordinary complex row shard: Heisenberg chain L = 16
    Lc = 16
    cb = [(q, (q + 1) % Lc) for q in range(Lc)]
    nh = L.qbgpu_dim_heisenberg(Lc, Lc // 2)
    bh, _ = qd.equal_row_bounds(nh, world)
    fullh = qb.heisenberg(Lc, Lc // 2, cb, 1.0)
    refh = qb.locate_E0_lanczos(fullh, nev=1, ncv=1)
    S = qb.heisenberg(Lc, Lc // 2, cb, 1.0, rows=(bh[rank], bh[rank + 1]))
    D = qd.NativeDist(qb, nh, bh, rank, world, True, exchange)
    loop_parity("ordinary_heisenberg16", D, None, S, fullh, nh, lambda vec: vec[bh[rank]:bh[rank + 1]], refh["eigenvecs"][0])
    D.destroy(); S.destroy(); fullh.destroy()

    # ------------------------------------------------------------------ degenerate pairs, ordinary complex row shards
    import oracle_lib as O
    A, meta, _ = O.load_golden("tj12")
    dg = np.concatenate([[-1.0, -1.0], np.linspace(0.5, 8.0, 254)])          # doubly degenerate ground level, exactly
    diag = (256, np.arange(257, dtype=np.int64), np.arange(256, dtype=np.int64), dg.astype(np.complex128), True)
    cases = (("tj12", (A.dim, A.ia, A.ja, A.val, A.sym), (E_TJ12, None)), ("diag256", diag, (-1.0, -1.0)))
    for tag, (dim, ia, ja, val, sym), golden in cases:
        fullt = qb.csr_mat(dim, ia, ja, val, sym)
        reft = qb.locate_E0_lanczos(fullt, nev=2, ncv=2)
        bt, _ = qd.equal_row_bounds(dim, world)
        St = qb.csr_mat(dim, ia, ja, val, sym, rows=(bt[rank], bt[rank + 1]))
        D = qd.NativeDist(qb, dim, bt, rank, world, True, exchange)
        got = D.locate_E0_lanczos(None, St, nev=2, ncv=2)
        E0, E1 = got["eigenvals"]
        r0, _ = residual(D, None, St, got["eigenvecs"][0], E0)
        r1, _ = residual(D, None, St, got["eigenvecs"][1], E1)
        orth = got["gap"] < LANCZOS_PRECISION                                # the orthonormalisation of :1302-1311 ran
        ov = overlap(got["eigenvecs"][0], got["eigenvecs"][1])
        detail = {"E0": E0, "E1": E1, "gap": got["gap"], "E0_single": float(reft["eigenvals"][0]), "E1_single": float(reft["eigenvals"][1]),
                  "gap_single": float(reft["gap"]), "orthonormalised": bool(orth), "orthonormalised_single": bool(reft["gap"] < LANCZOS_PRECISION),
                  "overlap_phi0_phi1": ov, "residual_phi0": r0, "residual_phi1": r1,
                  "steps": [got[k] for k in ("lanczos_steps", "cg_steps", "lanczos_steps_E1", "cg_steps_E1")]}
        check(f"degenerate_{tag}", all((g is None or abs(e - g) < 1e-8) and abs(e - es) < 1e-8 for e, es, g in zip((E0, E1), reft["eigenvals"], golden))
              and r0 < 1e-7 and r1 < 1e-7 and (ov < 1e-10 if orth else True), detail)
        D.destroy(); St.destroy(); fullt.destroy()

    flag = torch.tensor([0 if ok else 1], dtype=torch.int32)
    if world > 1:
        dist.all_reduce(flag)
    out["all_ranks_ok"] = int(flag.item()) == 0
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 0 else 1)


if __name__ == "__main__":
    main()
