"""CPU checks of bench.py's contract (the driver parses these lines): the reference arm prints ONE JSON line with the keys the
contract names, our arm refuses to run without a device instead of falling back, and the byte formulas behind the roofline
match SURVEY section 8d's figures for BASELINE config 3."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout=900):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout,
                          env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))


def test_reference_arm_prints_one_contract_line(oracle):
    if not oracle.have_qb_ref():
        pytest.skip("oracle/_ref/qb_ref is not built (needs the reference's sources at build time)")
    r = _run(["--impl", "reference", "--steps", "2", "--warmup", "1", "--workload", "heis_chain20"])
    assert r.returncode == 0, r.stderr[-500:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1                                            # ONE line on stdout
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "impl", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"] == "H*v/sec" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["config"]["workload"] == "heis_chain20" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["warmup"] >= 3                                           # timing rule: at least three warm-up steps


def test_our_arm_needs_a_device_and_has_no_fallback():
    r = _run(["--steps", "1", "--warmup", "1", "--workload", "heis_chain20", "--no-cpu", "--no-lanczos"], timeout=300)
    assert r.returncode != 0
    assert "CUDA" in (r.stderr + r.stdout)
    assert not any(ln.startswith("{") for ln in r.stdout.splitlines())   # no number is printed


def test_steps_below_one_are_refused():
    r = _run(["--steps", "0", "--warmup", "1", "--workload", "heis_chain20", "--no-cpu", "--no-lanczos"], timeout=300)
    assert r.returncode != 0 and "--steps" in r.stderr
    assert not any(ln.startswith("{") for ln in r.stdout.splitlines())


def test_dump_outputs_writes_a_fixed_bounded_sample_of_y(tmp_path, monkeypatch):
    """--dump-outputs: y of the last timed step as float64 .npy files, every row of a small workload, a seeded sample of a large
    one (the same rows on every run), at most 64 MB in all."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    assert 3 * 8 * bench.DUMP_ROWS <= 64 << 20

    class HostY:                                                       # the two members of DeviceVector the dump reads
        def __init__(self, n):
            self.n = n
            self.v = np.arange(n) * (1.0 - 0.5j)

        def to_numpy(self):
            return self.v.copy()

    def dump(d, n):
        bench.dump_outputs(str(d), HostY(n))
        z = {k: np.load(str(d / f"y_{k}.npy")) for k in ("rows", "real", "imag")}
        assert all(a.dtype == np.float64 and a.shape == z["rows"].shape for a in z.values())
        assert np.array_equal(z["real"], z["rows"]) and np.array_equal(z["imag"], -0.5 * z["rows"])
        return z["rows"]

    assert np.array_equal(dump(tmp_path / "small", 1000), np.arange(1000))
    monkeypatch.setattr(bench, "DUMP_ROWS", 500)
    rows = dump(tmp_path / "a", 100000)
    assert 400 < rows.size <= 500 and np.all(np.diff(rows) > 0)
    assert np.array_equal(rows, dump(tmp_path / "b", 100000))


def test_byte_formulas_match_the_survey():
    sys.path.insert(0, ROOT)
    import bench
    n, Z = 165636900, 5819376420                                      # BASELINE config 3 (SURVEY 8a/8d)
    assert bench.workload_upper_nnz("hubbard4x4") == (Z + n) // 2 == 2992506660
    assert abs(bench.algorithmic_bytes(Z, n, n, 16, 16) / 1e9 - 123.0) < 0.1     # complex values, complex vectors
    assert abs(bench.algorithmic_bytes(Z, n, n, 8, 16) / 1e9 - 76.5) < 0.1       # real values, complex vectors
    assert abs(bench.algorithmic_bytes(Z, n, n, 8, 8) / 1e9 - 73.8) < 0.1        # real / real
    assert bench.workload_upper_nnz("heis_chain20") == 1157156                    # BASELINE config 1 (SURVEY 8a)


def test_cpu_baseline_sample_is_the_same_lattice_and_bounded(oracle):
    """The `cpu_baseline` leg of our arm: a bounded sample of the SAME model (for config 3 the 4x4 lattice with five electrons per
    species: 0.3 G stored entries, far beyond the caches), scaled by stored entries; small workloads are their own sample."""
    sys.path.insert(0, ROOT)
    import bench
    args, desc = bench.cpu_baseline_sample("hubbard4x4")
    assert args == ["hubbard_direct", 4, 4, 5, 5, 1.0, 1.1] and "fewer electrons" in desc
    assert bench.hubbard_upper_nnz(4, 4, 5, 5) == 298910976            # what the reference's csr_mat holds for it (qb_ref, measured)
    assert bench.hubbard_upper_nnz(4, 4, 6, 6) > 4.0e8                 # the next larger filling is over the bound
    assert bench.hubbard_upper_nnz(4, 3, 6, 6) == 12030480             # BASELINE.md section 3 (reference-assembled)
    args, desc = bench.cpu_baseline_sample("hubbard4x3")
    assert args == ["hubbard_direct", 4, 3, 6, 6, 1.0, 1.1] and "fewer" not in desc
    assert bench.cpu_baseline_sample("heis_chain32_k0")[0] == ["heis_chain_k", 20, 0, 0]
    if not oracle.have_qb_ref():                                       # no reference build: the leg says so instead of raising
        r = bench.cpu_baseline_leg("hubbard4x3", reps=2, warm=1)
        assert r["value"] is None and r["kind"] == "reference" and "not built" in r["sample"]
        return
    r = bench.cpu_baseline_leg("hubbard4x3", reps=2, warm=1)          # its own sample: nothing scaled
    assert r["kind"] == "reference" and r["value"] > 0 and r["scaled_by_stored_entries"] == 1.0 and "scaled x" not in r["sample"]
    assert abs(r["value"] - 1e3 / r["sample_ms_per_product"]) < 1e-9 * r["value"]
    r = bench.cpu_baseline_leg("heis_chain24")                         # a scaled sample says so
    assert r["value"] > 0 and r["scaled_by_stored_entries"] > 1.0 and "scaled x" in r["sample"]
