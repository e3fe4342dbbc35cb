#!/usr/bin/env python
"""bench.py -- H*v throughput of the B200-native path (BASELINE.json metric: H*v/sec and achieved HBM GB/s; Lanczos
iterations/s and E0 time-to-solution ride along as extra keys).

  python bench.py --gpus 1 --steps K --warmup W                       our arm, one GPU
  torchrun ... bench.py --gpus N --steps K --warmup W                  our arm, H row-sharded over N GPUs (strong scaling)
  python bench.py --impl reference --gpus N --steps K --warmup W       the reference's CPU implementation (oracle/_ref)
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR    also write what the last timed step computed (dump_outputs)

A step is one product y = H x (csr_mat::MultMv) on the workload named in config.workload.  Default workload =
BASELINE config 3, Fermi-Hubbard 4x4, N_up = N_dn = 8 (dim 165,636,900; 5.82e9 stored entries), generated directly in
HBM in the reference's basis order (the reference's own assembler cannot produce it, SURVEY F6).  `value` = products/s
with vectors resident in HBM; `e2e` = the same through the reference-facing call with HOST vectors (x H2D and y D2H
inside the timed region: what the ARPACK callback of src/lanczos.cc:476 pays).  The matrix is far larger than L2
(126 MB), so no L2 flush is needed between steps; smaller workloads flush L2 between timed products.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                  # the benchmark leaves the tree it runs from as it found it (it may be read-only)
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"          # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line

WORKLOADS = {
    # name: (family, params)
    "hubbard4x4": ("hubbard", dict(Lx=4, Ly=4, nup=8, ndn=8, t=1.0, U=1.1)),       # BASELINE config 3
    "hubbard4x3": ("hubbard", dict(Lx=4, Ly=3, nup=6, ndn=6, t=1.0, U=1.1)),       # CPU-sized sample of the same model
    "heis_chain20": ("heisenberg", dict(L=20)),                                     # BASELINE config 1
    "heis_chain24": ("heisenberg", dict(L=24)),
    "heis_chain28": ("heisenberg", dict(L=28)),
    "heis_chain30": ("heisenberg", dict(L=30)),
    # translation-symmetric sectors assembled on the device in the reference's representative convention (sectors.cu)
    "heis_chain32_k0": ("heisenberg_k", dict(L=32, k=0)),                           # BASELINE config 2
    "heis_chain28_k1": ("heisenberg_k", dict(L=28, k=1)),                           # one sector of BASELINE config 5
    "heis_chain24_k3": ("heisenberg_k", dict(L=24, k=3)),
    # tilted clusters: orbit-minimum representatives (orbit.cu); the reference cannot build these (SURVEY F5)
    "tri31_k10": ("orbit", dict(A0=(5, 1), A1=(-1, 6), ndown=15, m=(1, 0))),           # BASELINE config 4
    "tri21_k10": ("orbit", dict(A0=(4, 1), A1=(-1, 5), ndown=10, m=(1, 0))),
}
L2_BYTES = 126e6
# DRAM bytes per product (dram__bytes_read.sum + dram__bytes_write.sum) from the committed ncu captures, per workload
# the species step (profiles/r02_ncu_full_mv_reference_order_hubbard4x4.csv): way in 3.43 + 1.36, pass 1 38.90 + 1.29,
# pass 2 (writes the reference's order itself) 40.33 + 2.84 GB
TRAFFIC_NCU_SPECIES = {"hubbard4x4": 88150000000}
KERNEL_SHARES_SPECIES = {"hubbard4x4": {"to_native_tiled_kernel": 0.057, "sjds_block_smem_kernel": 0.474, "spmv_sjds_bulk_kernel": 0.469,
                                        "source": "profiles/r02_ncu_full_mv_reference_order_hubbard4x4.csv (ncu gpu__time_duration.sum: 0.95 / 7.80 / 7.71 ms)"}}
TRAFFIC_NCU = {"hubbard4x4": 133686405000,     # profiles/r01_ncu_full_spmv_sjds_hubbard4x4_details.csv: 131.03 GB read + 2.65 GB write
               "tri31_k10": 13300097712,       # profiles/r01_ncu_full_spmv_sjds_tri31_k10_details.csv: 13.14 GB read + 0.158 GB write
               "heis_chain32_k0": 8834161656}  # profiles/r01_ncu_full_spmv_sjds_heis_chain32_k0_details.csv: 8.53 GB read + 0.302 GB write


def square_bonds(Lx, Ly):
    site = lambda x, y: (x % Lx) + (y % Ly) * Lx   # noqa: E731
    b = []
    for x in range(Lx):
        for y in range(Ly):
            b += [(site(x, y), site(x + 1, y)), (site(x, y), site(x, y + 1))]
    return b


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  Samples come from NVML in a thread of this process (20 ms period,
    time-stamped; no process start-up inside a sub-second region); if NVML cannot be used, from an `nvidia-smi -lms` child.  The
    sampler is started before the warm-up; begin() / stop() mark the timed window and only samples inside it count (if the window
    was too short to catch one, the samples nearest to it are used and `samples_in_window` says 0)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t0, self.t1, self.max_mhz = index, [], None, None, None, None
        self._stop = threading.Event()
        self.source = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)

            def loop():
                while not self._stop.is_set():
                    try:
                        mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        mask = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                        self.rows.append((time.time(), mhz, {name for bit, name in self.REASONS if mask & bit}))
                    except Exception:
                        pass
                    self._stop.wait(0.02)
            threading.Thread(target=loop, daemon=True).start()
            self.source = "nvml"
            return
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            self.source = "nvidia-smi"
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            if len(r) >= 8 and r[1].replace(".", "").isdigit():
                if r[2].replace(".", "").isdigit():
                    self.max_mhz = max(self.max_mhz or 0.0, float(r[2]))
                names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
                self.rows.append((time.time(), float(r[1]), {n for n, v in zip(names, r[4:8]) if v.lower().startswith("active")}))

    def begin(self):
        self.t0 = time.time()

    def stop(self):
        self.t1 = time.time()
        time.sleep(0.03)                                   # (let a sample that straddles the end land)
        self._stop.set()
        if self.proc:
            self.proc.terminate()
        rows = list(self.rows)
        t0 = self.t0 if self.t0 is not None else 0.0
        inside = [r for r in rows if t0 <= r[0] <= self.t1 + 0.03]
        used = inside
        if not used and rows:                              # window shorter than the sampling period: the nearest samples
            used = sorted(rows, key=lambda r: min(abs(r[0] - t0), abs(r[0] - self.t1)))[:2]
        sm = sorted(r[1] for r in used)
        reasons = set()
        for r in used:
            reasons |= r[2]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(reasons),
                "samples": len(used), "samples_in_window": len(inside), "source": self.source}


def algorithmic_bytes(nnz, nrows_local, n, s_val, s_vec):
    """B_spmv = Z*(S_val+4) + 8*(rows+1) + (n + rows)*S_vec  (SURVEY section 8d; one compulsory read of x, one write of y)."""
    return nnz * (s_val + 4) + 8 * (nrows_local + 1) + (n + nrows_local) * s_vec


DUMP_ROWS = 1 << 21                 # rows of y written by --dump-outputs: 3 float64 arrays of at most 2 M entries = 48 MB
DUMP_SEED = 20261020


def dump_outputs(dirpath, y):
    """What a caller of the timed step receives: y = H x (complex128, the reference's order).  Written as DIR/y_rows.npy (row
    indices), DIR/y_real.npy and DIR/y_imag.npy, all float64: every row when dim <= DUMP_ROWS, else the rows drawn with the fixed
    seed DUMP_SEED (the same rows for every build of the same workload), so two builds can be compared output for output."""
    import numpy as np
    n = y.n
    rows = np.arange(n) if n <= DUMP_ROWS else np.unique(np.random.default_rng(DUMP_SEED).integers(0, n, size=DUMP_ROWS, dtype=np.int64))
    ys = y.to_numpy()[rows]
    os.makedirs(dirpath, exist_ok=True)
    np.save(os.path.join(dirpath, "y_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(dirpath, "y_real.npy"), np.ascontiguousarray(ys.real))
    np.save(os.path.join(dirpath, "y_imag.npy"), np.ascontiguousarray(ys.imag))


# ------------------------------------------------------------------------------------------------ reference arm
def _host_ram_available_gb():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) / 1e6
    except Exception:
        pass
    return 0.0


def run_reference(args, workload):
    """The reference's own CPU implementation (unmodified sources compiled under oracle/_ref) on this host's cores.

    Hubbard workloads: the reference's csr_mat<complex<double>> of the workload ITSELF (config 3: 2,992,506,660 stored entries,
    73 GB in the reference's ILP64 layout) is filled directly -- without the LIL intermediate the reference's assembler needs
    (> 140 GB, SURVEY F6; oracle/ref_driver.cc: hubbard_direct, pinned bit for bit to the reference's own assembly on 4x3) -- and
    every step is one csr_mat::MultMv of the reference: same config, measured, nothing scaled.  If the host cannot hold it
    (or QB_REF_SAMPLE=1), and for the other families: a bounded sample of the same model at the largest size the reference's
    own assembler builds in seconds; then `value` is the SAMPLE's measured rate, `config.workload` names the sample, and the
    figure scaled by stored entries to the full workload is reported separately as `scaled_value` (an extrapolation)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    fam, p = WORKLOADS[workload]
    cores = os.cpu_count() or 1
    if not O.have_qb_ref():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/qb_ref was not built (needs /root/reference at build time)"}))
        return
    nnz_upper_full = workload_upper_nnz(workload)
    base = {"metric": "H*v/sec", "unit": "H*v/s", "impl": "reference", "n_gpus": 0, "warmup": args.warmup, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64 (complex128 values and vectors, int64 indices)", "data": "synthetic"}
    kernel_note = "MKL replaced by the shim's restated mkl_sparse_z_mv (row-partitioned OpenMP), BLAS-1 = OpenBLAS"
    if fam == "hubbard" and not os.environ.get("QB_REF_SAMPLE"):
        from math import comb
        ns = p["Lx"] * p["Ly"]
        n = comb(ns, p["nup"]) * comb(ns, p["ndn"])
        need_gb = (24 * nnz_upper_full + 8 * n + 2 * 16 * n) / 1e9 * 1.03 + 4.0
        if _host_ram_available_gb() >= need_gb:
            steps, warm = max(1, args.steps), max(0, args.warmup)
            est = 0.65e-9 * nnz_upper_full * 16.0 / max(cores, 1)            # seconds per product at the measured ns/entry
            if est * (steps + warm) > 150.0:                                 # keep the arm within a few minutes
                warm = min(warm, 1)
                steps = max(3, int(150.0 / est) - warm)
            res = O.run_qb_ref(["hubbard_direct", p["Lx"], p["Ly"], p["nup"], p["ndn"], p["t"], p["U"], "--time-mv", steps, warm],
                               threads=cores, timeout=3000)
            t_step = res["mv_total_s"] / res["mv_reps"]
            value = 1.0 / t_step
            desc = (f"the workload itself: csr_mat<complex<double>> of {workload} (dim {res['dim']:,}, {res['nnz']:,} stored upper-triangle entries) filled "
                    f"directly in {res['build_seconds']:.0f} s (oracle/ref_driver.cc: hubbard_direct), {res['mv_reps']} x the reference's csr_mat::MultMv at "
                    f"{1e3 * t_step:.1f} ms each ({1e9 * t_step / res['nnz']:.2f} ns per stored entry); {kernel_note}")
            line = dict(base, value=value, steps=res["mv_reps"], warmup=warm, ms_per_step=1e3 * t_step,
                        config={"workload": workload, "dim": res["dim"], "reference_upper_entries": res["nnz"], "same_config_as_gpu_arm": True,
                                "requested_steps": args.steps, "host_build_seconds": res["build_seconds"]},
                        cpu_baseline={"value": value, "unit": "H*v/s", "cores": cores, "kind": "reference", "sample": desc},
                        e2e={"value": value, "unit": "H*v/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
            print(json.dumps(line))
            return
    if fam == "hubbard":
        sample_args = ["hubbard", 4, 3, 6, 6, p["t"], p["U"]]
        sample_name = "hubbard4x3"
        sample_desc = "Fermi-Hubbard 4x3, N_up=N_dn=6 (dim 853,776; 12,030,480 stored upper-triangle entries), reference-assembled"
    elif fam == "heisenberg_k":
        sample_args = ["heis_chain_k", 20, 0, p["k"] % 20]
        sample_name = f"heis_chain20_k{p['k'] % 20}"
        sample_desc = f"Heisenberg chain L=20, Sz=0, momentum sector k={p['k'] % 20}, reference-assembled"
    elif fam == "orbit":
        sample_args = ["tri_k", 4, 5, 0, 3, 2]
        sample_name = "tri4x5_k32"
        sample_desc = "triangular 4x5 Heisenberg, Sz=0, momentum sector (3,2) (complex csr_mat, the largest 2-D sector the reference assembles in seconds), reference-assembled"
    else:
        Ls = min(p["L"], 22)
        sample_args = ["heis_chain", Ls, "sz", 0]
        sample_name = f"heis_chain{Ls}"
        sample_desc = f"Heisenberg chain L={Ls}, Sz=0, reference-assembled"
    res = O.run_qb_ref(sample_args + ["--time-mv", max(1, args.steps), max(0, args.warmup)], threads=cores, timeout=3000)
    t_step = res["mv_total_s"] / res["mv_reps"]
    nnz_sample = res["nnz"]
    scale = nnz_upper_full / nnz_sample
    same = abs(scale - 1.0) < 1e-12
    value = 1.0 / t_step                          # the SAMPLE's measured rate; nothing scaled in value / ms_per_step
    line = dict(base, value=value, steps=res["mv_reps"], ms_per_step=1e3 * t_step,
                scaled_value=1.0 / (t_step * scale), scaled_ms_per_step=1e3 * t_step * scale,
                scaled_note=f"extrapolated x{scale:.1f} by stored entries from the sample to {workload}: an estimate, not a measurement",
                config={"workload": workload if same else sample_name, "sample": sample_desc, "sample_of": workload, "same_config_as_gpu_arm": same,
                        "scaled_by_stored_entries": scale},
                cpu_baseline={"value": value, "unit": "H*v/s", "cores": cores, "kind": "reference",
                              "sample": f"{sample_desc}; {res['mv_reps']} x csr_mat::MultMv at {1e3 * t_step:.2f} ms each "
                                        f"({1e9 * t_step / nnz_sample:.2f} ns per stored entry); {kernel_note}"},
                e2e={"value": value, "unit": "H*v/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
    print(json.dumps(line))


def hubbard_upper_nnz(Lx, Ly, nup, ndn):
    """Entries the reference stores (upper triangle incl. every diagonal) for the square-lattice Hubbard model: (Z + n) / 2."""
    from math import comb
    ns = Lx * Ly
    n = comb(ns, nup) * comb(ns, ndn)
    bonds = {tuple(sorted(b)) for b in square_bonds(Lx, Ly)}
    # each undirected bond, each spin: states with exactly one of the two sites occupied by that spin
    z_off = 0
    for _ in bonds:
        z_off += 2 * comb(ns - 2, nup - 1) * comb(ns, ndn) + 2 * comb(ns - 2, ndn - 1) * comb(ns, nup)
    return (z_off + n + n) // 2


def workload_upper_nnz(workload):
    """Entries the reference stores (upper triangle incl. every diagonal) for a workload: (Z + n) / 2."""
    from math import comb
    fam, p = WORKLOADS[workload]
    if fam in ("heisenberg_k", "orbit"):
        return _SECTOR_UPPER[workload]          # counted by the device assembler (qbgpu_matrix_info.nnz_input)
    if fam == "hubbard":
        return hubbard_upper_nnz(p["Lx"], p["Ly"], p["nup"], p["ndn"])
    L = p["L"]
    n = comb(L, L // 2)
    z_off = L * 2 * comb(L - 2, L // 2 - 1)
    return (z_off + n + n) // 2


_SECTOR_UPPER = {"heis_chain32_k0": 173901570, "heis_chain28_k1": 11831544, "heis_chain24_k3": 817580,    # from runs of the assembler
                 "tri31_k10": 242371008, "tri21_k10": 293829}
SECTOR_PHASES = {}


def cpu_baseline_sample(workload, max_entries=4.0e8):
    """The bounded sample the `cpu_baseline` leg times (qb_ref arguments, description).  Hubbard workloads: the SAME lattice and
    operator with fewer electrons -- N_up = N_dn lowered until the reference's csr_mat has at most `max_entries` stored entries
    (config 3: N_up = N_dn = 5, dim 19,079,424, 298,910,976 entries = 7.2 GB, far beyond the caches, so the time per stored entry
    is the large-matrix one; the 12 M entries of the 4x3 cluster gave 0.62 ns where config 3 itself takes 0.99) -- filled
    directly like the reference arm's matrix (oracle/ref_driver.cc: hubbard_direct).  A workload that is small enough is its
    own sample.  The other families: the largest instance of the same model the reference's assembler builds in seconds."""
    fam, p = WORKLOADS[workload]
    if fam == "hubbard":
        nu, nd = p["nup"], p["ndn"]
        while hubbard_upper_nnz(p["Lx"], p["Ly"], nu, nd) > max_entries and min(nu, nd) > 1:
            nu, nd = nu - 1, nd - 1
        return (["hubbard_direct", p["Lx"], p["Ly"], nu, nd, p["t"], p["U"]],
                f"Fermi-Hubbard {p['Lx']}x{p['Ly']}, N_up={nu}, N_dn={nd} (the workload's lattice and operator"
                + (")" if (nu, nd) == (p["nup"], p["ndn"]) else f" with fewer electrons; the workload has {p['nup']}, {p['ndn']})"))
    if fam == "heisenberg_k":
        return ["heis_chain_k", 20, 0, p["k"] % 20], f"Heisenberg chain L=20, Sz=0, momentum sector k={p['k'] % 20}, reference-assembled"
    if fam == "orbit":
        return ["tri_k", 4, 5, 0, 3, 2], "triangular 4x5 Heisenberg, Sz=0, momentum sector (3,2), reference-assembled"
    Ls = min(p["L"], 22)
    return ["heis_chain", Ls, "sz", 0], f"Heisenberg chain L={Ls}, Sz=0, reference-assembled"


def cpu_baseline_leg(workload, reps=5, warm=2):
    """`cpu_baseline` of the GPU arm's line: the compiled reference's csr_mat::MultMv (oracle/_ref) on this host's cores, on a
    bounded sample of the workload (cpu_baseline_sample), scaled to the metric's unit by stored entries and labelled so; the
    sample's own measured figures are in `sample_ms_per_product` / `sample_ns_per_entry`.  (`bench.py --impl reference` times the
    reference on the workload itself.)  Never raises: the baseline is informative and must not cost the GPU line."""
    cores = os.cpu_count() or 1
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        if not O.have_qb_ref():
            return {"value": None, "unit": "H*v/s", "cores": cores, "kind": "reference", "sample": "oracle/_ref/qb_ref not built"}
        sample_args, desc = cpu_baseline_sample(workload)
        res = O.run_qb_ref(sample_args + ["--time-mv", reps, warm], threads=cores, timeout=1200)
        t_step = res["mv_total_s"] / res["mv_reps"]
        scale = workload_upper_nnz(workload) / res["nnz"]
        return {"value": 1.0 / (t_step * scale), "unit": "H*v/s", "cores": cores, "kind": "reference",
                "sample_ms_per_product": 1e3 * t_step, "sample_ns_per_entry": 1e9 * t_step / res["nnz"], "scaled_by_stored_entries": scale,
                "sample": f"{desc}: dim {res['dim']:,}, {res['nnz']:,} stored upper-triangle entries, {res['mv_reps']} x the reference's "
                          f"csr_mat::MultMv at {1e3 * t_step:.2f} ms ({1e9 * t_step / res['nnz']:.2f} ns per stored entry)"
                          + ("" if abs(scale - 1.0) < 1e-12 else f", scaled x{scale:.2f} by stored entries to {workload}")
                          + f"; MKL replaced by the shim's restated mkl_sparse_z_mv, OpenMP {cores} threads"}
    except Exception as e:
        return {"value": None, "unit": "H*v/s", "cores": cores, "kind": "reference", "sample": f"failed: {e}"}


# ------------------------------------------------------------------------------------------------------ our arm
def build_matrix(qb, workload, row_range=None, flags=0):
    """BASELINE matrices generated directly in HBM (qbgpu_build_*), bit-identical to what the reference assembles."""
    fam, p = WORKLOADS[workload]
    import numpy as np
    L = qb.lib()
    h = C.c_void_p()
    lo, hi = (0, -1) if row_range is None else row_range
    if fam == "orbit":
        if row_range is not None:
            raise SystemExit("sector workloads are single-GPU in this round")
        from quantum_basis_b200.clusters import Cluster
        cl = Cluster(p["A0"], p["A1"])
        t0 = time.time()
        M = qb.heisenberg_orbit(cl.det, p["ndown"], cl.translations(), cl.characters(p["m"]), cl.triangular_bonds(), flags=flags)
        SECTOR_PHASES.update(enumerate_and_assemble_s=time.time() - t0, sites=cl.det)
        _SECTOR_UPPER[workload] = M.info.nnz_input
        return M
    if fam == "heisenberg_k":
        if row_range is not None:
            raise SystemExit("sector workloads are single-GPU in this round")
        n = p["L"]
        t0 = time.time()
        sec = qb.Sector([n], n // 2, [p["k"]])
        t1 = time.time()
        M = sec.heisenberg([(x, (x + 1) % n) for x in range(n)], flags=flags)
        SECTOR_PHASES.update(enumerate_representatives_s=sec.enumerate_seconds, norms_s=sec.norms_seconds, sector_total_s=t1 - t0,
                             assemble_and_expand_s=time.time() - t1, zero_norm=sec.zero_norm, lin_order=sec.lin_order)
        _SECTOR_UPPER[workload] = M.info.nnz_input
        sec.free()
        return M
    if fam == "hubbard":
        bonds = np.array(square_bonds(p["Lx"], p["Ly"]), dtype=np.int32).ravel()
        rc = L.qbgpu_build_hubbard(C.byref(h), p["Lx"] * p["Ly"], p["nup"], p["ndn"], len(bonds) // 2, bonds.ctypes.data,
                                   p["t"], p["U"], 1, flags, lo, hi)
    else:
        n = p["L"]
        bonds = np.array([(x, (x + 1) % n) for x in range(n)], dtype=np.int32).ravel()
        rc = L.qbgpu_build_heisenberg(C.byref(h), n, n // 2, n, bonds.ctypes.data, 1.0, 1, flags, lo, hi)
    if rc != 0:
        raise RuntimeError(L.qbgpu_last_error().decode())
    return qb.csr_mat._adopt(h, True)


def species_probe(args):
    """Child process of the single-GPU bench (hubbard workloads): the same H through the species-order handles
    (QBGPU_SPECIES_ORDER, csrc/species.cu) -- parity against the ordinary handle first, then timings.  Run in a process of
    its own because these kernels had not met hardware when they were committed: whatever happens here cannot touch the
    numbers of the main line.  Prints one JSON object."""
    os.environ.setdefault("QBGPU_MV_REAL_MODE", "1")       # opt-in fp64 route of MultMv on ORDINARY handles, for this child only
    import numpy as np
    import torch
    import quantum_basis_b200 as qb
    torch.cuda.set_device(0)
    L = qb.lib()
    assert L.qbgpu_init(0) == 0, L.qbgpu_last_error()
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    assert L.qbgpu_set_stream(C.c_void_p(stream.cuda_stream)) == 0
    fam, p = WORKLOADS[args.workload]
    ns = p["Lx"] * p["Ly"]
    peak, _ = measured_peak()
    out = {"workload": args.workload, "tile": os.environ.get("QBGPU_SPECIES_TILE", "default (stored 64, matrix-free 128)")}

    def timed(fn, steps):
        for _ in range(3):
            fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record(stream)
        for _ in range(steps):
            fn()
        b.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b) / steps

    def rel_err(ya, yref, n):
        """|ya - yref| / |yref| on the device (ya is overwritten)."""
        nr, nd = C.c_double(), C.c_double()
        assert L.qbgpu_dznrm2(n, C.c_void_p(yref.ptr), C.byref(nr)) == 0
        assert L.qbgpu_zaxpy(n, (C.c_double * 2)(-1.0, 0.0), C.c_void_p(yref.ptr), C.c_void_p(ya.ptr)) == 0
        assert L.qbgpu_dznrm2(n, C.c_void_p(ya.ptr), C.byref(nd)) == 0
        return nd.value / nr.value

    P = build_matrix(qb, args.workload, flags=2 | 8)          # ordinary handle, production layout, no autotune pass
    n, Z = P.info.n, P.info.nnz_stored
    x = qb.vec_randomize(n, 1, device=True)
    yref, y = qb.DeviceVector(n), qb.DeviceVector(n)
    # the complex product exactly as the main line measures it: through the fused entry point, which never takes the opt-in
    # fp64 route of MultMv (QBGPU_MV_REAL_MODE, set for this child below)
    one_, zero_ = (C.c_double * 2)(1.0, 0.0), (C.c_double * 2)(0.0, 0.0)
    assert L.qbgpu_spmv_fused(P.handle, C.c_void_p(x.ptr), None, C.c_void_p(yref.ptr), one_, zero_, zero_, None) == 0
    out["ordinary_ms"] = timed(lambda: L.qbgpu_spmv_fused(P.handle, C.c_void_p(x.ptr), None, C.c_void_p(y.ptr), one_, zero_, zero_, None),
                               max(3, args.steps // 2))
    # opt-in: MultMv on complex vectors without imaginary parts multiplies on fp64 copies (csrc/spmv.cu: mv_real_mode)
    try:
        P.MultMv(x, y)
        err = rel_err(y, yref, n)
        ms = timed(lambda: P.MultMv(x, y), max(3, args.steps // 2))
        B16 = algorithmic_bytes(Z, n, n, 8, 16)
        out["ordinary_real_mode"] = {"ms_per_product": ms, "rel_err_vs_complex_kernel": err, "achieved_GBs": B16 / ms / 1e6,
                                     "frac_of_measured_peak": B16 / ms / 1e6 / peak,
                                     "note": "complex128 x and y at the boundary; imag(x) == 0 detected, product on fp64 copies, result widened"}
    except Exception as e:
        out["ordinary_real_mode"] = {"error": str(e)[:300]}
    P.destroy()
    bonds = square_bonds(p["Lx"], p["Ly"])
    fused = L.qbgpu_spmv_fused
    one, zero = (C.c_double * 2)(1.0, 0.0), (C.c_double * 2)(0.0, 0.0)
    for kind in ("stored", "matrix_free"):
        r = {}
        out[kind] = r
        try:
            t0 = time.time()
            M = qb.hubbard(ns, p["nup"], p["ndn"], bonds, p["t"], p["U"], flags=128, matrix_free=(kind == "matrix_free"))
            torch.cuda.synchronize()
            r["build_s"] = time.time() - t0
            r["device_bytes"] = M.info.device_bytes
            M.MultMv(x, y)
            r["rel_err_vs_ordinary"] = rel_err(y, yref, n)
            r["parity_ok"] = bool(r["rel_err_vs_ordinary"] <= 1e-12)
            # (a) the reference-shaped call: vectors in the reference's order, permuted in and out around the two passes
            ms = timed(lambda: M.MultMv(x, y), args.steps)
            B16 = algorithmic_bytes(Z, n, n, 8, 16)
            r["reference_order_complex"] = {"ms_per_product": ms, "achieved_GBs": B16 / ms / 1e6, "frac_of_measured_peak": B16 / ms / 1e6 / peak}
            # (a') the same call on a vector WITH imaginary parts: no fp64 route, the complex passes
            xc = qb.vec_randomize(n, 2, device=True)
            assert L.qbgpu_zaxpy(n, (C.c_double * 2)(0.0, 1.0), C.c_void_p(x.ptr), C.c_void_p(xc.ptr)) == 0      # xc = r2 + i r1
            ms = timed(lambda: M.MultMv(xc, y), args.steps)
            r["reference_order_genuinely_complex"] = {"ms_per_product": ms, "achieved_GBs": B16 / ms / 1e6, "frac_of_measured_peak": B16 / ms / 1e6 / peak}
            xc.free()
            # (b) vectors kept in the internal order (what the Krylov loops do between their first and last step)
            xn, yn = M.to_native(x), qb.DeviceVector(n)
            ms = timed(lambda: fused(M.handle, C.c_void_p(xn.ptr), None, C.c_void_p(yn.ptr), one, zero, zero, None), args.steps)
            r["internal_order_complex"] = {"ms_per_product": ms, "achieved_GBs": B16 / ms / 1e6, "frac_of_measured_peak": B16 / ms / 1e6 / peak}
            if kind == "matrix_free":                         # pass-1 variants of the matrix-free product (csrc/species.cu)
                r["pass1_variants_complex_ms"] = {}
                for vname, vid in (("grid_stride", 0), ("row_ranges", 1), ("smem_staged", 2)):
                    assert L.qbgpu_debug_set_variant(1000 + vid) == 0
                    fused(M.handle, C.c_void_p(xn.ptr), None, C.c_void_p(yn.ptr), one, zero, zero, None)
                    xr_ = M.from_native(yn)
                    err = rel_err(xr_, yref, n)
                    xr_.free()
                    r["pass1_variants_complex_ms"][vname] = {"ms": timed(lambda: fused(M.handle, C.c_void_p(xn.ptr), None, C.c_void_p(yn.ptr), one, zero, zero, None), args.steps),
                                                             "rel_err_vs_ordinary": err}
                best = min(r["pass1_variants_complex_ms"].items(), key=lambda kv: kv[1]["ms"] if kv[1]["rel_err_vs_ordinary"] <= 1e-12 else 1e30)
                assert L.qbgpu_debug_set_variant(1000 + {"grid_stride": 0, "row_ranges": 1, "smem_staged": 2}[best[0]]) == 0
                r["pass1_variant_used_below"] = best[0]
            xn.free(); yn.free()
            # (c) fp64 vectors, internal order
            Mr = M.real_view()
            xr = qb.vec_randomize(n, 1, dtype=np.float64, device=True)
            yr = qb.DeviceVector(n, np.float64)
            ms = timed(lambda: fused(Mr.handle, C.c_void_p(xr.ptr), None, C.c_void_p(yr.ptr), one, zero, zero, None), args.steps)
            B8 = algorithmic_bytes(Z, n, n, 8, 8)
            r["internal_order_fp64"] = {"ms_per_product": ms, "achieved_GBs": B8 / ms / 1e6, "frac_of_measured_peak": B8 / ms / 1e6 / peak}
            xr.free(); yr.free()
            # (d) E0 through the reference-shaped Lanczos call
            v = qb.DeviceVector(2 * n)
            assert L.qbgpu_vec_randomize_z(n, C.c_void_p(v.ptr), 1) == 0
            hess = np.zeros(2000)
            torch.cuda.synchronize()
            tl = time.time()
            m = qb.lanczos(0, 999, 1000, n, M, v, hess, "sr_val0")
            torch.cuda.synchronize()
            tl = time.time() - tl
            ritz, _ = qb.hess_eigen(hess, 1000, m)
            r["lanczos"] = {"steps": m, "seconds": tl, "iters_per_s": m / tl, "E0": float(ritz[0])}
            v.free()
            M.destroy()
        except Exception as e:                               # keep what was measured so far
            r["error"] = str(e)[:500]
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("QB_WORKLOAD", "hubbard4x4"), choices=sorted(WORKLOADS))
    ap.add_argument("--no-lanczos", action="store_true", help="skip the E0 time-to-solution leg")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-species", action="store_true", help="skip the species-order probe (hubbard workloads, child process)")
    ap.add_argument("--layout", default="default", choices=["default", "ordinary", "species", "species-matfree"],
                    help="hubbard workloads, one GPU: which handle the main line measures.  default = species (the stored two-part "
                         "QBGPU_SPECIES_ORDER handle: same entries, same 12 bytes each, two passes); ordinary = the one-pass "
                         "sliced-jagged handle in the reference's order; species-matfree = nothing stored.  Same operator, same "
                         "calling convention everywhere: complex128 device vectors in the reference's order through MultMv")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="one GPU, our arm: after the timed steps write y = H x of the last one to DIR as .npy (float64; a fixed, "
                         "seeded sample of rows when the workload has more than %d)" % DUMP_ROWS)
    ap.add_argument("--species-probe", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.species_probe:
        return species_probe(args)
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs writes the products of our arm on one GPU")

    if args.impl == "reference":
        if rank == 0:
            run_reference(args, args.workload)
        return

    import numpy as np
    import torch
    import quantum_basis_b200 as qb
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libqbgpu has no CPU fallback")
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    L = qb.lib()
    assert L.qbgpu_init(local_rank) == 0, L.qbgpu_last_error()
    # the library adopts a torch stream so that torch.cuda.Event timing sees its kernels (the legacy default stream has
    # handle 0, which qbgpu_set_stream reads as "use your own stream": hence a dedicated non-default stream)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    assert L.qbgpu_set_stream(C.c_void_p(stream.cuda_stream)) == 0

    if world > 1:
        from quantum_basis_b200 import dist as qdist
        return qdist.bench_sharded(args, WORKLOADS, build_matrix, algorithmic_bytes, measured_peak, ClockSampler, workload_upper_nnz)

    # ---------------------------------------------------------------- single GPU
    t0 = time.time()
    fam_, p_ = WORKLOADS[args.workload]
    if args.layout == "default":
        args.layout = "species" if fam_ == "hubbard" else "ordinary"
    if args.layout == "ordinary":
        M = build_matrix(qb, args.workload)
    else:
        if fam_ != "hubbard":
            raise SystemExit("--layout species*: the species order exists for the Hubbard model only")
        M = qb.hubbard(p_["Lx"] * p_["Ly"], p_["nup"], p_["ndn"], square_bonds(p_["Lx"], p_["Ly"]), p_["t"], p_["U"],
                       flags=128, matrix_free=(args.layout == "species-matfree"))
    torch.cuda.synchronize()
    t_build = time.time() - t0
    inf = M.info
    n, Z = inf.n, inf.nnz_stored
    if Z == 0:                                   # matrix-free: the algorithmic bytes of SURVEY 8d refer to the stored operator
        Z = 2 * workload_upper_nnz(args.workload) - n
    s_val = 8 if inf.val_is_real else 16
    s_vec = 16
    B = algorithmic_bytes(Z, n, n, s_val, s_vec)
    need_flush = B < 2 * L2_BYTES
    flush_buf = torch.empty(int(256e6) // 4, dtype=torch.float32, device="cuda") if need_flush else None

    x = qb.vec_randomize(n, 1, device=True)
    y = qb.DeviceVector(n)
    sampler = ClockSampler(local_rank)
    sampler.start()                                         # running before the warm-up; begin() marks the timed window
    for _ in range(args.warmup):
        M.MultMv(x, y)
    torch.cuda.synchronize()
    L.qbgpu_kernel_launches(1)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    torch.cuda.synchronize()
    sampler.begin()
    wall0 = time.time()
    for k in range(args.steps):
        if need_flush:
            flush_buf.zero_()
        ev[k][0].record(stream)
        M.MultMv(x, y)
        ev[k][1].record(stream)
    torch.cuda.synchronize()
    wall = time.time() - wall0
    launches = int(L.qbgpu_kernel_launches(0))
    per_step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = sum(per_step_ms)
    clocks = sampler.stop()
    if args.dump_outputs:                                   # before any later leg reuses y
        dump_outputs(args.dump_outputs, y)
    ms_per_step = total_ms / args.steps
    value = 1e3 / ms_per_step
    peak, peak_src = measured_peak()
    achieved = B / (ms_per_step * 1e-3) / 1e9

    def time_products(mat, xv, yv, steps):
        for _ in range(3):
            mat.MultMv(xv, yv)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record(stream)
        for _ in range(steps):
            mat.MultMv(xv, yv)
        b.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b) / steps

    def roof(bytes_, ms):
        g = bytes_ / (ms * 1e-3) / 1e9
        return {"ms_per_product": ms, "products_per_s": 1e3 / ms, "algorithmic_bytes": bytes_, "achieved_GBs": g, "frac_of_measured_peak": g / peak}

    # ---------------------------------------------------------------- the same matrix with fp64 vectors (what the fused
    # Krylov loops run when H and the start vector are real) and with 1-byte dictionary-coded values (opt-in layout)
    extras = {}
    Md = None
    if inf.val_is_real and not need_flush:
        Mr = M.real_view()
        xr = qb.vec_randomize(n, 1, dtype=np.float64, device=True)
        yr = qb.DeviceVector(n, np.float64)
        extras["real_vectors"] = dict(S_val=s_val, S_vec=8, **roof(algorithmic_bytes(Z, n, n, s_val, 8), time_products(Mr, xr, yr, args.steps)))
        try:
            if args.layout != "ordinary":
                raise RuntimeError("skipped on species handles")
            Md = build_matrix(qb, args.workload, flags=16)
            if Md.info.value_dict:
                nd = Md.info.value_dict
                extras["value_dict_complex_vectors"] = dict(S_val=1, S_vec=16, dict_entries=nd, **roof(algorithmic_bytes(Z, n, n, 1, 16), time_products(Md, x, y, args.steps)))
                extras["value_dict_real_vectors"] = dict(S_val=1, S_vec=8, dict_entries=nd, **roof(algorithmic_bytes(Z, n, n, 1, 8), time_products(Md.real_view(), xr, yr, args.steps)))
        except Exception as e:
            Md = None
            extras["value_dict_error"] = str(e)
        xr.free(); yr.free()

    # ---------------------------------------------------------------- parity at the BASELINE size: sampled rows recomputed on the host
    # in long double from the Lin tables (qbgpu_debug_rows_host: the generators' own row function, pinned entry for entry to
    # matrices the compiled reference assembled) -- full-basis families only (the sector assemblers have no host twin)
    parity = None
    if fam_ in ("hubbard", "heisenberg"):
        M.MultMv(x, y)
        xh0, yh0 = x.to_numpy(), y.to_numpy()
        rng = np.random.default_rng(20261017)
        rows = np.unique(rng.integers(0, n, size=min(100000, n), dtype=np.int64))
        yr = np.zeros(2 * rows.size)
        if fam_ == "hubbard":
            bl = np.array(square_bonds(p_["Lx"], p_["Ly"]), dtype=np.int32).ravel()
            rc = L.qbgpu_debug_rows_host(1, p_["Lx"] * p_["Ly"], p_["nup"], p_["ndn"], len(bl) // 2, bl.ctypes.data, 0.0, p_["t"], p_["U"],
                                         rows.size, rows.ctypes.data, xh0.ctypes.data, 1, yr.ctypes.data)
        else:
            bl = np.array([(q, (q + 1) % p_["L"]) for q in range(p_["L"])], dtype=np.int32).ravel()
            rc = L.qbgpu_debug_rows_host(0, p_["L"], p_["L"] // 2, 0, len(bl) // 2, bl.ctypes.data, 1.0, 0.0, 0.0,
                                         rows.size, rows.ctypes.data, xh0.ctypes.data, 1, yr.ctypes.data)
        assert rc == 0, L.qbgpu_last_error()
        yr = yr.view(np.complex128)
        err = float(np.linalg.norm(yh0[rows] - yr) / np.linalg.norm(yr))
        parity = {"rows": int(rows.size), "rel_l2_error": err, "bound": 1e-12, "ok": bool(err <= 1e-12),
                  "how": "y = MultMv(x) of the timed handle against rows recomputed on the host in long double (Lin tables + the generators' row function)"}
        del xh0, yh0

    # ---------------------------------------------------------------- e2e: host vectors through the reference-facing call
    M.MultMv(x, y)
    xh_t = torch.empty(2 * n, dtype=torch.float64).pin_memory()
    yh_t = torch.empty(2 * n, dtype=torch.float64).pin_memory()
    xh = xh_t.numpy().view(np.complex128)
    yh = yh_t.numpy().view(np.complex128)
    xh[:] = x.to_numpy()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        M.MultMv(xh, yh)
    torch.cuda.synchronize()
    te = time.time()
    for _ in range(e2e_steps):
        M.MultMv(xh, yh)                  # H2D(x) + product + D2H(y), synchronous like the reference's call
    torch.cuda.synchronize()
    e2e_s = (time.time() - te) / e2e_steps
    y_dev = y.to_numpy()
    assert np.array_equal(y_dev, yh), "host-vector and device-vector products disagree"

    line = {"metric": "H*v/sec", "value": value, "unit": "H*v/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": args.workload, "dim": n, "stored_entries": Z, "reference_upper_entries": workload_upper_nnz(args.workload),
                       "S_val": s_val, "S_vec": s_vec,
                       "layout": ({"species": "species order: two sliced-jagged parts (diagonal + down hops | up hops), two passes",
                                   "species-matfree": "species order, matrix-free"}[args.layout]
                                  if args.layout != "ordinary" else "sliced-jagged" if inf.format == 8 else f"csr-vector lanes={inf.lanes}"),
                       "l2": "flush between steps" if need_flush else "inputs larger than L2", "matrix_bytes": inf.device_bytes,
                       "vectors": "complex128 x and y in the reference's order (the model<complex<double>> calling convention); x = vec_randomize(seed 1), "
                                  "imag == 0 like every vector of the reference's flows" + (": the species handle detects it while permuting and runs its two passes "
                                  "on fp64 copies (genuinely complex x: species_order.stored.reference_order_genuinely_complex)" if args.layout != "ordinary" else "")},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (TRAFFIC_NCU.get(args.workload) if args.layout == "ordinary" else TRAFFIC_NCU_SPECIES.get(args.workload) if args.layout == "species" else None),
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of the step's kernels in the committed ncu capture (profiles/), not measured in this run",
                         "algorithmic_bytes": B, "peak_source": peak_src, "frac_of_8TBs": achieved / 8000.0,
                         "kernel": ("kron_local_kernel + kron_cross_kernel" if args.layout == "species-matfree" else
                                    "one step = to_native_tiled_kernel (way in, checks imag == 0) + sjds_block_smem_kernel<double,double> (pass 1) + spmv_sjds_bulk_kernel<double,double,..,OUT> (pass 2, UBLKCP; writes y in the reference's order)"
                                    if args.layout == "species" else "spmv_sjds_kernel<double,double2>" if inf.format == 8 else "spmv_csr_vector_kernel"),
                         "kernel_shares_ncu": (KERNEL_SHARES_SPECIES.get(args.workload) if args.layout == "species" else None)},
            "e2e": {"value": 1.0 / e2e_s, "unit": "H*v/s", "h2d_bytes_per_step": n * s_vec, "d2h_bytes_per_step": n * s_vec,
                    "ms_per_step": 1e3 * e2e_s},
            "gpu_launches": launches, "clocks": clocks, "wall_s_timed_region": wall,
            "ms_per_step_median": sorted(per_step_ms)[len(per_step_ms) // 2], "ms_per_step_min": min(per_step_ms), "parity_sampled": parity,
            "host_phases": {"generate_matrix_s": t_build, "autotune_s": inf.autotune_seconds, **SECTOR_PHASES}}
    line.update(extras)

    # ---------------------------------------------------------------- Lanczos iterations/s and E0 time-to-solution
    if not args.no_lanczos:
        def lanczos_leg(mat, sv):
            v = qb.DeviceVector(2 * n)
            assert L.qbgpu_vec_randomize_z(n, C.c_void_p(v.ptr), 1) == 0
            hess = np.zeros(2000)
            qb.lanczos(0, 6, 1000, n, mat, v, hess, "sr_val0")            # warm-up: every kernel of the loop loaded and launched once
            assert L.qbgpu_vec_randomize_z(n, C.c_void_p(v.ptr), 1) == 0
            hess[:] = 0.0
            torch.cuda.synchronize()
            tl = time.time()
            m = qb.lanczos(0, 999, 1000, n, mat, v, hess, "sr_val0")      # the reference's call, stop rule included
            torch.cuda.synchronize()
            tl = time.time() - tl
            ritz, _ = qb.hess_eigen(hess, 1000, m)
            v.free()
            # real-mode loop: fp64 vectors when H and the start vector are real
            svec = 8 if inf.val_is_real else 16
            b_iter = Z * (sv + 4) + 8 * (n + 1) + 6 * n * svec
            return {"steps": m, "seconds": tl, "iters_per_s": m / tl, "E0": float(ritz[0]), "S_val": sv, "S_vec": svec,
                    "algorithmic_bytes_per_iter": b_iter, "achieved_GBs": b_iter * m / tl / 1e9,
                    "frac_of_measured_peak": b_iter * m / tl / 1e9 / peak}
        line["lanczos"] = lanczos_leg(M, s_val)
        if Md is not None and Md.info.value_dict:
            line["lanczos_value_dict"] = lanczos_leg(Md, 1)
    if Md is not None:
        Md.destroy()

    # ---------------------------------------------------------------- CPU baseline beside it (bounded sample)
    if not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline_leg(args.workload)

    # ---------------------------------------------------------------- species-order handles, in a process of their own
    # (hubbard workloads; everything above is already measured and this process gives its HBM back first)
    if WORKLOADS[args.workload][0] == "hubbard" and not args.no_species:
        try:
            M.destroy(); x.free(); y.free()
            del xh, yh, xh_t, yh_t, flush_buf
            torch.cuda.empty_cache()
            res = subprocess.run([sys.executable, os.path.abspath(__file__), "--species-probe", "--workload", args.workload,
                                  "--steps", str(max(5, min(args.steps, 20)))], capture_output=True, text=True, timeout=300)
            lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
            line["species_order"] = json.loads(lines[-1]) if lines else {"error": f"exit {res.returncode}: {res.stderr[-400:]}"}
        except Exception as e:
            line["species_order"] = {"error": str(e)[:400]}

    print(json.dumps(line))


if __name__ == "__main__":
    main()
