"""A/B drop-in test on the GPU box: the reference's OWN lanczos<T,MAT> / eigenvec_CG<T,MAT> templates (compiled from the
unmodified src/lanczos.cc into oracle/_ref/qb_ab) instantiated over the GPU adaptor include/qbgpu_csr_mat.hpp."""
import json
import os
import subprocess

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QB_AB = os.path.join(ROOT, "oracle", "_ref", "qb_ab")


@pytest.mark.parametrize("name", ["tri4x4_k01", "hubbard4x2", "heis16_full"])
def test_reference_templates_over_the_gpu_adaptor(oracle, name, tmp_path):
    if not os.path.exists(QB_AB):
        pytest.skip("oracle/_ref/qb_ab not built (make -C oracle ab; needs the reference's sources at build time)")
    A, meta, ex = oracle.load_golden(name)
    f = str(tmp_path / "H.qbcsr")
    out = str(tmp_path / "ab.json")
    oracle.write_qbcsr(f, A)
    subprocess.run([QB_AB, f, out], check=True, stdout=subprocess.DEVNULL, timeout=900)
    r = json.load(open(out))
    e0 = meta["lanczos_E0"]
    assert r["ref_cpu_steps"] == meta["lanczos_steps"]                      # the reference on the CPU, as recorded
    assert abs(r["ref_cpu_E0"] - e0) <= 1e-12 * abs(e0)
    assert abs(r["ref_loop_gpu_mv_E0"] - e0) <= 1e-10 * abs(e0)             # reference loop, GPU products
    assert abs(r["ref_loop_gpu_mv_steps"] - meta["lanczos_steps"]) <= 2
    assert abs(r["fused_gpu_E0"] - e0) <= 1e-10 * abs(e0)                   # fused device loop, same argument list
    assert abs(r["fused_gpu_steps"] - meta["lanczos_steps"]) <= 2
    assert r["cg_accu"] < 2e-12 and r["cg_residual"] < 1e-9                 # reference CG loop, GPU products
