"""E1 and the gap on several GPUs: the sharded sr_val1 Lanczos (qbgpu_dist_lanczos_val1) and locate_E0_lanczos(nev = 2) in one
call (qbgpu_dist_locate_e0_lanczos), against the single-GPU entry points (scripts/dist_excited_check.py), and the C++ example
with NEV = 2 against the Python flow."""
import json
import os
import re
import shutil
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E0_HUB43 = -16.879382788684


def _run_check(nproc):
    script = os.path.join(ROOT, "scripts", "dist_excited_check.py")
    if nproc == 1:
        cmd = [sys.executable, script]
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
               "--master-port", "29547", script]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert res.returncode == 0 and lines, (res.stdout[-3000:], res.stderr[-3000:])
    out = json.loads(lines[-1])
    assert out["all_ranks_ok"], out
    return out


@pytest.fixture(scope="module")
def one_rank():
    return _run_check(1)


def _check_common(out):
    flow = out["fp64_hubbard4x3_flow"]
    assert abs(flow["E0"] - E0_HUB43) < 1e-9
    assert flow["identical_on_all_ranks"]
    for tag in ("fp64_hubbard4x3", "complex_hubbard4x3", "ordinary_heisenberg16"):
        assert out[f"{tag}_val1_no_speculation_bit_identical"]["steps"] == out[f"{tag}_val1_loop"]["steps"]
    # The orthonormalisation of a degenerate pair (src/model.cc:1302-1311) is never taken on the tj12 golden: its E0 is
    # doubly degenerate (ARPACK), but phi0 -- CG from the Lanczos start vector's seed -- is the one direction of that level in
    # the start vector's Krylov space, so the re-orthogonalised run finds the next level (E1 = -9.717157950726, on one GPU
    # as on the shards; the script holds E1 to the single-GPU flow there).  The diagonal case takes the branch: E1 = E0 to
    # round-off.  The script requires |<phi0|phi1>| < 1e-10 whenever the branch runs.
    assert not out["degenerate_tj12"]["orthonormalised"] and abs(out["degenerate_tj12"]["E0"] + 9.762087307) < 1e-8
    assert out["degenerate_diag256"]["orthonormalised"]
    assert out["degenerate_diag256"]["overlap_phi0_phi1"] < 1e-10


def test_dist_excited_one_rank(one_rank):
    """sr_val1 loop and the four-stage flow on ONE rank (same loops, no peers) against the single-GPU entry points."""
    _check_common(one_rank)


def test_dist_excited_two_ranks():
    """The same on TWO GPUs: the projection travels through the push all-reduce, every rank takes the same branch."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    out = _run_check(2)
    _check_common(out)
    assert out["world"] == 2


def test_dist_lanczos_example_nev2_matches_python_flow(tmp_path, one_rank):
    """examples/dist_lanczos.cc with NEV = 2 on two GPUs (on one where only one is present; plain C++,
    qbgpu_dist_locate_e0_lanczos) gives the E0 and E1 of the Python flow on the same model (Hubbard 4x3, 6+6, fp64 vectors
    through the real view)."""
    import torch
    ngpus = min(2, torch.cuda.device_count())
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    exe = tmp_path / "dist_lanczos"
    libdir = os.path.join(ROOT, "quantum_basis_b200")
    subprocess.run([gxx, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "dist_lanczos.cc"),
                    "-o", str(exe), "-L", libdir, "-lqbgpu", "-Wl,-rpath," + libdir], check=True)
    r = subprocess.run([str(exe), str(ngpus), "4", "3", "6", "6", "2"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout, r.stderr)
    m = re.search(r"E0 = (\S+)\s+E1 = (\S+)\s+gap = (\S+)", r.stdout)
    assert m, r.stdout
    e0, e1 = float(m.group(1)), float(m.group(2))
    flow = one_rank["fp64_hubbard4x3_flow"]
    assert abs(e0 - flow["E0"]) <= 1e-10 * abs(flow["E0"])
    assert abs(e1 - flow["E1"]) <= 1e-8 * abs(flow["E1"])
