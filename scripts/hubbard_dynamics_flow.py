#!/usr/bin/env python
"""Hubbard dynamics in the momentum basis on one GPU: S^zz(q, omega), N(q, omega) and A(k, omega) of the half-filled square
cluster (default 4x4, t = 1, U = 1.1; the model of BASELINE config 3).

  1. E0 and phi0 in the k = (0,0) sector of (N/2, N/2) electrons: Lanczos + CG on the sector handle.
     ASSUMED: the ground state lies in k = (0,0) and is unique there.  The script does not check degeneracy across momenta;
     it reports E0 next to the full-basis value when one is given (--e0-full), and averaging over a ground-state manifold is
     left to the caller.
  2. For every q: S^z_q = sum_r e^{+i q.r}/(2 sqrt N) (n_up,r - n_dn,r) and n_q = sum_r e^{+i q.r}/sqrt N (n_up,r + n_dn,r) applied
     to phi0 (both land in the sector k = q, whose H is assembled once), then `maxit` dnmcs Lanczos steps from each vector.
  3. For every k: c_{k,up} phi0 (c_k = N^{-1/2} sum_r e^{-i k.r} c_r; sector (N_up - 1, N_dn, -k)) and c+_{k,up} phi0 (sector
     (N_up + 1, N_dn, +k)), each followed by `maxit` dnmcs steps: photoemission and inverse photoemission parts of A(k, omega).
One target sector and its H live at a time (a 10 M-row complex sector with its stored H takes several GB).  Prints one JSON line:
times per step (sector build, operator, Lanczos), norms, the first Lanczos coefficient and the sum rules
sum_k |c_k phi0|^2 = N_up and |c_k phi0|^2 + |c+_k phi0|^2 = 1.

  python scripts/hubbard_dynamics_flow.py --L 4 4 --maxit 200 --e0-full -20.497352266554
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import quantum_basis_b200 as qb  # noqa: E402


def square_hops(Lx, Ly):
    """Directed hops in the reference example's insertion order (site x + y Lx; per site the +x then the +y bond; per bond
    c+_up,i c_up,j ; c+_up,j c_up,i ; c+_dn,i c_dn,j ; c+_dn,j c_dn,i), as (to, from, spin)."""
    hops = []
    for x in range(Lx):
        for y in range(Ly):
            i = x + y * Lx
            for j in ((x + 1) % Lx + y * Lx, x + ((y + 1) % Ly) * Lx):
                hops += [(i, j, 0), (j, i, 0), (i, j, 1), (j, i, 1)]
    return hops


def gpu_description():
    """Name and power limit of the card the numbers were measured on (a read-only query)."""
    import subprocess
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown"


def plane_wave(Lx, Ly, k, sign):
    return np.array([np.exp(sign * 2j * np.pi * (k[0] * (r % Lx) / Lx + k[1] * (r // Lx) / Ly)) for r in range(Lx * Ly)])


def dynamic(apply, n, H, maxit):
    """apply(out) writes A phi0 into `out`; then measure_repr_dynamic's normalisation and the dnmcs Lanczos, timed apart."""
    lib = qb.lib()
    v = qb.DeviceVector(2 * n)
    v.zero()
    t0 = time.time()
    apply(v.view(0, n))
    t_op = time.time() - t0
    nr = C.c_double()
    qb._lib.check(lib.qbgpu_dznrm2(n, C.c_void_p(v.ptr), C.byref(nr)))
    rec = {"norm2": nr.value ** 2, "op_s": t_op, "dnmcs_steps": 0, "dnmcs_s": 0.0}
    if nr.value >= qb.lanczos_precision:
        qb._lib.check(lib.qbgpu_zscal(n, (C.c_double * 2)(1.0 / nr.value, 0.0), C.c_void_p(v.ptr)))
        hess = np.zeros(2 * maxit)
        t0 = time.time()
        m = qb.lanczos(0, maxit - 1, maxit, n, H, v, hess, "dnmcs")
        rec.update(dnmcs_steps=m, dnmcs_s=time.time() - t0, a0=hess[maxit], b1=hess[1] if m > 1 else 0.0)
    v.free()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--L", type=int, nargs=2, default=[4, 4])
    ap.add_argument("--t", type=float, default=1.0)
    ap.add_argument("--U", type=float, default=1.1)
    ap.add_argument("--maxit", type=int, default=200)
    ap.add_argument("--e0-full", type=float, default=None, help="full-basis ground-state energy to report E0 against")
    a = ap.parse_args()
    Lx, Ly = a.L
    N = Lx * Ly
    nup = ndn = N // 2
    assert qb.lib().qbgpu_init(0) == 0
    hops = square_hops(Lx, Ly)
    moms = [(m, n) for m in range(Lx) for n in range(Ly)]
    t_all = time.time()

    t0 = time.time()
    s0 = qb.ElectronSector([Lx, Ly], nup, ndn, [0, 0])
    H0 = s0.hubbard(hops, a.t, a.U)
    t_build0 = time.time() - t0
    t0 = time.time()
    res = qb.locate_E0_lanczos(H0, nev=1, ncv=1, device_vectors=True)
    phi0 = res["eigenvecs_device"][0]
    out = {"L": [Lx, Ly], "t": a.t, "U": a.U, "nup": nup, "ndn": ndn, "maxit": a.maxit, "gpu": gpu_description(), "dim_k0": s0.dim,
           "build_k0_s": t_build0, "E0": res["eigenvals"][0], "E0_and_phi0_s": time.time() - t0,
           "lanczos_steps": res["lanczos_steps"], "cg_steps": res["cg_steps"], "cg_accuracy": res["cg_accuracy"],
           "assumption": "ground state unique and at k = (0,0); no averaging over a ground-state manifold"}
    if a.e0_full is not None:
        out["E0_full_basis"] = a.e0_full

    def sector(nu, nd, k):
        t0 = time.time()
        s = qb.ElectronSector([Lx, Ly], nu, nd, list(k))
        H = s.hubbard(hops, a.t, a.U)
        return s, H, time.time() - t0

    out["q"] = []
    for q in moms:                                                   # S^zz(q, w) and N(q, w): both land in k = q
        s1, H1, tb = sector(nup, ndn, q)
        c = plane_wave(Lx, Ly, q, +1) / np.sqrt(N)
        rec = {"q": q, "dim": s1.dim, "zero_norm": s1.zero_norm, "build_s": tb}
        rec["szz"] = dynamic(lambda y: s0.apply_density(s1, 0.5 * c, -0.5 * c, phi0, out=y), s1.dim, H1, a.maxit)
        rec["nn"] = dynamic(lambda y: s0.apply_density(s1, c, c, phi0, out=y), s1.dim, H1, a.maxit)
        out["q"].append(rec)
        H1.destroy()
        s1.free()

    out["k"] = []
    for k in moms:                                                   # A(k, w), spin up: c_k phi0 and c+_k phi0
        rec = {"k": k}
        for name, d in (("c", -1), ("cdag", +1)):
            s1, H1, tb = sector(nup + d, ndn, (d * k[0] % Lx, d * k[1] % Ly))
            c = plane_wave(Lx, Ly, k, d) / np.sqrt(N)
            r = dynamic(lambda y: s0.apply_fermion(s1, c, phi0, create=d > 0, spin=0, out=y), s1.dim, H1, a.maxit)
            r.update(dim=s1.dim, build_s=tb)
            rec[name] = r
            H1.destroy()
            s1.free()
        out["k"].append(rec)

    pipi = [r for r in out["q"] if tuple(r["q"]) == (Lx // 2, Ly // 2)][0]
    out["szz_weight_pi_pi"] = pipi["szz"]["norm2"]
    out["sum_szz_weights"] = sum(r["szz"]["norm2"] for r in out["q"])        # = sum_r <(S^z_r)^2> = (N_e - 2 <doubly occupied sites>) / 4
    out["sum_k_c_up"] = sum(r["c"]["norm2"] for r in out["k"])               # = N_up
    out["max_dev_c_plus_cdag"] = max(abs(r["c"]["norm2"] + r["cdag"]["norm2"] - 1.0) for r in out["k"])
    out["total_s"] = time.time() - t_all
    out["build_s_total"] = t_build0 + sum(r["build_s"] for r in out["q"]) + sum(r[n]["build_s"] for r in out["k"] for n in ("c", "cdag"))
    out["op_s_total"] = sum(r[n]["op_s"] for r in out["q"] for n in ("szz", "nn")) + sum(r[n]["op_s"] for r in out["k"] for n in ("c", "cdag"))
    out["dnmcs_s_total"] = sum(r[n]["dnmcs_s"] for r in out["q"] for n in ("szz", "nn")) + sum(r[n]["dnmcs_s"] for r in out["k"] for n in ("c", "cdag"))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
