"""Seeded calls of the whole-loop Krylov drivers (Lanczos, eigenvec_CG, energy_scale, KPM moments) on every route of their
vector boundary: host or device vectors, real mode or the complex loop, handles with and without an internal order.  Shared by
tests/test_gpu_krylov_boundary.py and scripts/krylov_routes_dump.py (TEST INFRASTRUCTURE)."""
import ctypes as C

import numpy as np

import oracle_lib as O
import quantum_basis_b200 as qb
from gpu_species_common import _case
from quantum_basis_b200 import _lib

# an ordinary handle with real values, one with complex values, and the species-order handles (stored and matrix-free)
KINDS = ("hubbard4x2", "tri4x4_k01", "hub3x3_45_stored", "hub3x3_45_matfree")
REAL_VALUED = ("hubbard4x2", "hub3x3_45_stored", "hub3x3_45_matfree")
MAXIT = 200
SEED = 20261020


def make(kind):
    if kind in ("hubbard4x2", "tri4x4_k01"):
        A, _, _ = O.load_golden(kind)
        return qb.csr_mat(A.dim, A.ia, A.ja, A.val, A.sym)
    mk = _case("hub3x3_45")[-1]
    return mk(mf=kind.endswith("matfree"))


def inputs(M):
    """Seeded start vectors for the complex-API handle M, and the E0 / spectral bounds the CG and KPM calls use."""
    n = M.dim
    rng = np.random.default_rng(SEED)
    unit = lambda a: a / np.linalg.norm(a)    # noqa: E731
    X = {"x0": unit(rng.standard_normal(n)), "phi": unit(rng.standard_normal(n)),
         "xc": unit(rng.standard_normal(n) + 1j * rng.standard_normal(n))}
    v = np.zeros(2 * n, dtype=np.complex128)
    v[:n] = X["x0"]
    hess = np.zeros(2 * MAXIT)
    m = qb.lanczos(0, MAXIT - 1, MAXIT, n, M, v, hess, "sr_val0")
    X["E0"] = float(qb.hess_eigen(hess, MAXIT, m)[0][0])
    X["lo"], X["hi"] = qb.energy_scale(n, M, np.zeros(2 * n, dtype=np.complex128), 0.1, 40)
    # the state of a CG run after 6 steps, from which every resumed CG call starts (the same inputs on every route: the
    # fresh steps themselves may run in real mode)
    cg = [X["x0"].astype(np.complex128)] + [np.zeros(n, dtype=np.complex128) for _ in range(3)]
    X["cg6_m"], _ = qb.eigenvec_CG(n, 6, 0, M, X["E0"], *cg)
    X["cg6_v"], X["cg6_r"], X["cg6_p"], X["cg6_pp"] = cg
    return X


def _p(a):
    return C.c_void_p(a.ptr) if isinstance(a, qb.DeviceVector) else C.c_void_p(a.ctypes.data)


def _check(rc):
    assert rc == 0, qb.lib().qbgpu_last_error()


class _Caller:
    """The drivers' C entry points on host (numpy) or device vectors of the handle's API type."""

    def __init__(self, M, dev):
        self.M, self.dev, self.z, self.L = M, dev, M.is_complex, qb.lib()
        self.where = _lib.QBGPU_DEVICE if dev else _lib.QBGPU_HOST
        self.dtype = np.complex128 if self.z else np.float64

    def vec(self, *parts):
        a = np.zeros(sum(p.size for p in parts), dtype=self.dtype)
        a[:] = np.concatenate(parts) if self.z else np.concatenate(parts).real
        return qb.DeviceVector.from_numpy(a) if self.dev else a

    @staticmethod
    def get(a):
        if isinstance(a, qb.DeviceVector):
            out = a.to_numpy()
            a.free()
            return out
        return a

    def lanczos(self, v, k, np_, purpose, hess, stop=None):
        m = C.c_int64(0)
        f = self.L.qbgpu_lanczos_resume_z if self.z else self.L.qbgpu_lanczos_resume_d
        _check(f(self.M.handle, k, np_, MAXIT, C.byref(m), _p(v), _p(hess), purpose.encode(), self.where, None if stop is None else _p(stop)))
        return m.value

    def cg(self, m, E0, v, r, p, pp, maxit=MAXIT):
        mm, accu = C.c_int64(m), C.c_double(0.0)
        if self.z:
            e = (C.c_double * 2)(complex(E0).real, complex(E0).imag)
            _check(self.L.qbgpu_eigenvec_cg_z(self.M.handle, maxit, C.byref(mm), e, C.byref(accu), _p(v), _p(r), _p(p), _p(pp), self.where))
        else:
            _check(self.L.qbgpu_eigenvec_cg_d(self.M.handle, maxit, C.byref(mm), float(E0), C.byref(accu), _p(v), _p(r), _p(p), _p(pp), self.where))
        return mm.value, accu.value

    def energy_scale(self, v):
        lo, hi = C.c_double(), C.c_double()
        f = self.L.qbgpu_energy_scale_z if self.z else self.L.qbgpu_energy_scale_d
        _check(f(self.M.handle, _p(v), C.byref(lo), C.byref(hi), 0.1, 40, self.where))
        return lo.value, hi.value

    def kpm(self, phi, lo, hi, nmom=40):
        mu = np.zeros(nmom)
        f = self.L.qbgpu_kpm_moments_z if self.z else self.L.qbgpu_kpm_moments_d
        _check(f(self.M.handle, _p(phi), lo, hi, nmom, _p(mu), self.where))
        return mu


def run(M, X, dev, routes=None):
    """Every route on handle M (complex API, or the fp64 API of a real view: then the real parts of the inputs), with host
    (dev=False) or device vectors.  Returns {route/output: ndarray}; `routes` limits the routes run."""
    c = _Caller(M, dev)
    n = M.dim
    zero = np.zeros(n)
    out = {}

    def put(route, **arrays):
        for k, a in arrays.items():
            out[f"{route}/{k}"] = np.atleast_1d(np.asarray(c.get(a)))

    def want(route):
        return routes is None or route in routes

    for route, purpose, np_, parts in (("lanczos_sr_val0", "sr_val0", MAXIT - 1, (X["x0"], zero)),
                                       ("lanczos_sr_val1", "sr_val1", MAXIT - 1, (X["x0"], zero, X["phi"])),
                                       ("lanczos_dnmcs", "dnmcs", 30, (X["x0"], zero)),
                                       ("lanczos_complex_start", "sr_val0", MAXIT - 1, (X["xc"], zero))):
        if want(route) and (c.z or route != "lanczos_complex_start"):
            v, hess = c.vec(*parts), np.zeros(2 * MAXIT)
            m = c.lanczos(v, 0, np_, purpose, hess)
            put(route, m=m, hess=hess, v=v)
    if want("lanczos_resumed"):                     # 12 steps, then the rest from the handed-back vectors and stop state
        v, hess, stop = c.vec(X["x0"], zero), np.zeros(2 * MAXIT), np.zeros(4)
        m1 = c.lanczos(v, 0, 12, "sr_val0", hess, stop)
        put("lanczos_resumed", m1=m1, hess1=hess.copy(), stop1=stop.copy())
        v = c.vec(c.get(v))
        m = c.lanczos(v, m1, MAXIT - 1 - m1, "sr_val0", hess, stop)
        put("lanczos_resumed", m=m, hess=hess, stop=stop, v=v)
    if want("cg"):
        v, r, p, pp = c.vec(X["x0"]), c.vec(zero), c.vec(zero), c.vec(zero)
        m, accu = c.cg(0, X["E0"], v, r, p, pp)
        put("cg", m=m, accu=accu, v=v, r=r, p=p, pp=pp)
    if want("cg_resumed"):                          # on from (v, r, p) of step cg6_m
        v, r, p, pp = (c.vec(X["cg6_" + s]) for s in ("v", "r", "p", "pp"))
        m, accu = c.cg(X["cg6_m"], X["E0"], v, r, p, pp)
        put("cg_resumed", m=m, accu=accu, v=v, r=r, p=p, pp=pp)
    if want("cg_complex_E0") and c.z:
        v, r, p, pp = c.vec(X["x0"]), c.vec(zero), c.vec(zero), c.vec(zero)
        m, accu = c.cg(0, complex(X["E0"], 1e-3), v, r, p, pp, maxit=20)
        put("cg_complex_E0", m=m, accu=accu, v=v, r=r, p=p, pp=pp)
    if want("energy_scale"):
        v = c.vec(zero, zero)
        lo, hi = c.energy_scale(v)
        put("energy_scale", lo=lo, hi=hi, v=v)
    if want("kpm"):
        phi = c.vec(X["x0"])
        put("kpm", mu=c.kpm(phi, X["lo"], X["hi"]))
        c.get(phi)
    return out
