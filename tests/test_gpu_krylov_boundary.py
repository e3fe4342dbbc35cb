"""The vector boundary of the whole-loop Krylov drivers (csrc/krylov.cu: begin / end): host staging, real mode and the species
order's permutation must not change a bit of what the loops compute.  On an ordinary handle with real values (hubbard4x2), one
with complex values (tri4x4_k01) and the species-order handles, stored and matrix-free (hub3x3_45), every driver -- Lanczos
sr_val0 / sr_val1 / dnmcs / resumed with its stop state, eigenvec_CG fresh and resumed, energy_scale, KPM -- is held to:
- host and device vectors give identical bits;
- real mode (a complex-API call on real values with real inputs) gives the bits of the fp64 call on qbgpu_real_view, widened;
- the complex loop taken on its own (complex start vector, resumed CG, complex E0) gives the bits of the run forced complex
  by QBGPU_NO_REAL_MODE."""
import numpy as np
import pytest

import krylov_routes as K

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=K.KINDS)
def case(request):
    M = K.make(request.param)
    yield request.param, M, K.inputs(M)
    M.destroy()


def same_bits(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def test_host_and_device_vectors_give_identical_bits(case):
    kind, M, X = case
    host, dev = K.run(M, X, dev=False), K.run(M, X, dev=True)
    assert sorted(host) == sorted(dev)
    for key in host:
        assert same_bits(host[key], dev[key]), key
    assert host["lanczos_sr_val0/m"][0] > 3 and np.isfinite(host["cg/v"]).all() and np.isfinite(host["kpm/mu"]).all()


def test_real_mode_equals_the_real_view(case):
    kind, M, X = case
    if kind not in K.REAL_VALUED:
        pytest.skip("complex values: no real mode")
    # energy_scale only without an internal order: there the start vector is drawn in the loop's type (see krylov.cu)
    routes = {"lanczos_sr_val0", "lanczos_sr_val1", "lanczos_dnmcs", "lanczos_resumed", "cg", "kpm"}
    if not kind.startswith("hub3x3"):
        routes.add("energy_scale")
    Mr = M.real_view()
    for dev in (False, True):
        z, d = K.run(M, X, dev, routes), K.run(Mr, X, dev, routes)
        assert sorted(z) == sorted(d) and {k.split("/")[0] for k in z} == routes
        for key in z:
            want = d[key].astype(np.complex128) if z[key].dtype == np.complex128 else d[key]
            assert same_bits(z[key], want), (dev, key)


def test_complex_loop_equals_the_forced_complex_run(case, monkeypatch):
    kind, M, X = case
    routes = {"lanczos_complex_start", "cg_resumed", "cg_complex_E0"}
    for dev in (False, True):
        auto = K.run(M, X, dev, routes)
        monkeypatch.setenv("QBGPU_NO_REAL_MODE", "1")
        forced = K.run(M, X, dev, routes)
        monkeypatch.delenv("QBGPU_NO_REAL_MODE")
        assert sorted(auto) == sorted(forced) and {k.split("/")[0] for k in auto} == routes
        for key in auto:
            assert same_bits(auto[key], forced[key]), (dev, key)
