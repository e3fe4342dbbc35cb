"""Host-side mirror of the reference's interface for the H*v path, over the C ABI (include/qbgpu.h).

Names, argument meaning and error behaviour follow the reference so that parity tests read like its own:
  csr_mat.MultMv / MultMv2 / to_dense   reference src/sparse.cc:262-315 (qbasis.h:976-1021)
  lanczos                               src/lanczos.cc:134-266
  eigenvec_CG                           src/lanczos.cc:281-341
  hess_eigen                            src/lanczos.cc:355-390
  energy_scale                          src/kpm.cc:45-88
  vec_randomize                         src/miscellaneous.cc:371-388
  locate_E0_lanczos                     src/model.cc:1124-1316 (the csr_mat branch; model's bookkeeping stays host-side)
Host vectors are numpy arrays (complex128 / float64); device-resident vectors are DeviceVector.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import QbgpuError, check, lib

lanczos_precision = 2e-12      # reference src/miscellaneous.cc:47


def _ptr(a):
    if isinstance(a, DeviceVector):
        return C.c_void_p(a.ptr)
    return C.c_void_p(a.ctypes.data)


def _where(*arrs):
    dev = [isinstance(a, DeviceVector) for a in arrs]
    if all(dev):
        return _lib.QBGPU_DEVICE
    if not any(dev):
        return _lib.QBGPU_HOST
    raise QbgpuError("mixing host and device vectors in one call")


def _host_vec(a, dtype, n=None, name="vector"):
    if not isinstance(a, np.ndarray) or a.dtype != dtype or not a.flags["C_CONTIGUOUS"]:
        raise QbgpuError(f"{name} must be a C-contiguous numpy array of dtype {np.dtype(dtype).name}")
    if n is not None and a.size < n:
        raise QbgpuError(f"{name} has {a.size} entries, needs {n}")
    return a


class DeviceVector:
    """A vector resident in HBM (qbgpu_malloc)."""

    def __init__(self, n, dtype=np.complex128):
        self.n = int(n)
        self.dtype = np.dtype(dtype)
        p = C.c_void_p()
        check(lib().qbgpu_malloc(C.byref(p), self.n * self.dtype.itemsize))
        self.ptr = p.value
        self._owned = True

    @classmethod
    def from_numpy(cls, a):
        a = np.ascontiguousarray(a)
        v = cls(a.size, a.dtype)
        check(lib().qbgpu_memcpy_h2d(C.c_void_p(v.ptr), C.c_void_p(a.ctypes.data), a.nbytes))
        return v

    def view(self, offset, n):
        """A non-owning window [offset, offset+n) (e.g. one column of the reference's v[] workspace)."""
        w = object.__new__(DeviceVector)
        w.n, w.dtype, w.ptr, w._owned, w._parent = int(n), self.dtype, self.ptr + offset * self.dtype.itemsize, False, self
        return w

    def clone(self):
        """A new device vector with the same contents (device-to-device copy)."""
        v = DeviceVector(self.n, self.dtype)
        check(lib().qbgpu_memcpy_d2d(C.c_void_p(v.ptr), C.c_void_p(self.ptr), self.n * self.dtype.itemsize))
        return v

    def to_numpy(self):
        out = np.empty(self.n, dtype=self.dtype)
        check(lib().qbgpu_memcpy_d2h(C.c_void_p(out.ctypes.data), C.c_void_p(self.ptr), out.nbytes))
        return out

    def zero(self):
        check(lib().qbgpu_memset0(C.c_void_p(self.ptr), self.n * self.dtype.itemsize))

    def free(self):
        if self._owned and self.ptr:
            lib().qbgpu_free(C.c_void_p(self.ptr))
            self.ptr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def vec_disk_write(filename, x):
    """vec_disk_write (src/miscellaneous.cc:437-468): int64 n, the raw elements, CRC-32 of both (boost::crc_32_type, the
    zlib polynomial) -- the file format of the reference's checkpoints and saved eigenvectors, so vectors computed here
    can be picked up by a CPU run of the reference and vice versa.  x: host array or DeviceVector (float64 / complex128)."""
    import struct
    import zlib
    a = x.to_numpy() if isinstance(x, DeviceVector) else np.ascontiguousarray(x)
    if a.dtype not in (np.float64, np.complex128):
        raise QbgpuError("vec_disk_write: float64 or complex128")
    head = struct.pack("<q", a.size)
    crc = zlib.crc32(a.tobytes(), zlib.crc32(head)) & 0xFFFFFFFF
    with open(filename, "wb") as f:
        f.write(head)
        f.write(a.tobytes())
        f.write(struct.pack("<I", crc))
    return 0


def vec_disk_read(filename, n, dtype=np.complex128, device=False):
    """vec_disk_read (src/miscellaneous.cc:391-434): returns the vector, or None where the reference returns 1 (missing
    file, wrong size, wrong n, checksum mismatch)."""
    import os
    import struct
    import zlib
    dt = np.dtype(dtype)
    if not os.path.exists(filename) or os.path.getsize(filename) != 8 + dt.itemsize * n + 4:
        return None
    with open(filename, "rb") as f:
        b = f.read()
    if struct.unpack("<q", b[:8])[0] != n or struct.unpack("<I", b[-4:])[0] != (zlib.crc32(b[:-4]) & 0xFFFFFFFF):
        return None
    a = np.frombuffer(b, dtype=dt, count=n, offset=8).copy()
    return DeviceVector.from_numpy(a) if device else a


class csr_mat:
    """Device-resident counterpart of the reference's csr_mat<T> (qbasis.h:976-1021).

    Constructed from the reference's own arrays: ``dim``, ``ia[dim+1]``, ``ja[nnz]`` (int64), ``val[nnz]`` (float64 ->
    csr_mat<double>, complex128 -> csr_mat<complex<double>>) and ``sym`` (upper triangle only).  The arrays are
    uploaded once, like the MKL handle the reference creates in its constructors (src/sparse.cc:129,258).
    """

    def __init__(self, dim, ia, ja, val, sym, flags=0, rows=None):
        ia = np.ascontiguousarray(ia, dtype=np.int64)
        ja = np.ascontiguousarray(ja, dtype=np.int64)
        val = np.ascontiguousarray(val)
        if val.dtype not in (np.float64, np.complex128):
            raise QbgpuError("val must be float64 or complex128")
        if ia.size != dim + 1:
            raise QbgpuError("ia must have dim+1 entries")
        self.dim = int(dim)
        self.sym = bool(sym)
        self.dtype = val.dtype
        self.is_complex = val.dtype == np.complex128
        h = C.c_void_p()
        L = lib()
        rs, re = C.c_void_p(ia.ctypes.data), C.c_void_p(ia.ctypes.data + 8)
        if rows is None:
            f = L.qbgpu_create_zcsr if self.is_complex else L.qbgpu_create_dcsr
            check(f(C.byref(h), dim, rs, re, C.c_void_p(ja.ctypes.data), C.c_void_p(val.ctypes.data), int(self.sym), flags))
        else:
            f = L.qbgpu_create_zcsr_shard if self.is_complex else L.qbgpu_create_dcsr_shard
            check(f(C.byref(h), dim, rs, re, C.c_void_p(ja.ctypes.data), C.c_void_p(val.ctypes.data), int(self.sym), flags,
                    int(rows[0]), int(rows[1])))
        self.handle = h

    @classmethod
    def _adopt(cls, handle, is_complex):
        self = object.__new__(cls)
        self.handle = handle
        self.is_complex = bool(is_complex)
        self.dtype = np.dtype(np.complex128 if is_complex else np.float64)
        info = self.info
        self.dim = info.n
        self.sym = True
        return self

    @property
    def info(self):
        inf = _lib.MatrixInfo()
        check(lib().qbgpu_matrix_get_info(self.handle, C.byref(inf)))
        return inf

    @property
    def nrows_local(self):
        inf = self.info
        return inf.row_hi - inf.row_lo

    def dimension(self):
        return self.dim

    def real_view(self):
        """A csr_mat<double>-typed view on the same device arrays (only when the stored values are real)."""
        h = C.c_void_p()
        check(lib().qbgpu_real_view(self.handle, C.byref(h)))
        v = csr_mat._adopt(h, False)
        v._parent = self                                   # keep the owner alive
        return v

    # y = alpha*H*x + beta*y : what csr_mat::MultMv2 asks of mkl_sparse_?_mv (src/sparse.cc:287)
    def _mv(self, alpha, x, beta, y):
        if self.handle is None:
            raise QbgpuError("matrix was destroyed")
        where = _where(x, y)
        if where == _lib.QBGPU_HOST:
            _host_vec(x, self.dtype, self.dim, "x")
            _host_vec(y, self.dtype, self.nrows_local, "y")
        if self.is_complex:
            a = (C.c_double * 2)(alpha.real, alpha.imag)
            b = (C.c_double * 2)(beta.real, beta.imag)
            check(lib().qbgpu_zmv(self.handle, a, _ptr(x), b, _ptr(y), where))
        else:
            check(lib().qbgpu_dmv(self.handle, float(complex(alpha).real), _ptr(x), float(complex(beta).real), _ptr(y), where))

    def MultMv2(self, x, y):
        """y = H*x + y (src/sparse.cc:262-289)."""
        self._mv(complex(1.0), x, complex(1.0), y)

    def MultMv(self, x, y):
        """y = H*x (src/sparse.cc:291-297)."""
        self._mv(complex(1.0), x, complex(0.0), y)

    def has_internal_order(self):
        """True for QBGPU_SPECIES_ORDER handles: the fused low-level entry points then work in the handle's internal order,
        the reference-shaped ones (MultMv, lanczos, ...) keep the reference's."""
        f = C.c_int(0)
        check(lib().qbgpu_native_order(self.handle, C.byref(f)))
        return bool(f.value)

    def species_parts(self):
        """(local, cross): the two parts of a stored species-order handle or row shard as handles of their own (views).  The
        local part's gathers never leave the handle's own rows -- on a shard it needs no remote data."""
        a, b = C.c_void_p(), C.c_void_p()
        check(lib().qbgpu_species_parts(self.handle, C.byref(a), C.byref(b)))
        return csr_mat._adopt(a, True), csr_mat._adopt(b, True)

    def native_perm(self):
        """perm[r] = internal index of the reference's basis state r (species-order handles)."""
        p = np.empty(self.dim, dtype=np.int32)
        check(lib().qbgpu_native_perm(self.handle, _ptr(p)))
        return p

    def to_native(self, x, out=None):
        """Device vector in the reference's order -> the handle's internal order (out of place)."""
        out = out if out is not None else DeviceVector(x.n, x.dtype)
        check(lib().qbgpu_vec_to_native(self.handle, _ptr(x), _ptr(out)))
        return out

    def from_native(self, x, out=None):
        out = out if out is not None else DeviceVector(x.n, x.dtype)
        check(lib().qbgpu_vec_from_native(self.handle, _ptr(x), _ptr(out)))
        return out

    def to_dense(self):
        """Column-major dense copy, returned as an (n, n) array with out[row, col] (src/sparse.cc:299-315)."""
        out = np.zeros(self.dim * self.dim, dtype=self.dtype)
        check(lib().qbgpu_to_dense(self.handle, C.c_void_p(out.ctypes.data)))
        return out.reshape(self.dim, self.dim).T

    def download_expanded(self):
        inf = self.info
        nloc = inf.row_hi - inf.row_lo
        rowptr = np.zeros(nloc + 1, dtype=np.int64)
        col = np.zeros(inf.nnz_stored, dtype=np.int32)
        val = np.zeros(inf.nnz_stored, dtype=np.float64 if inf.val_is_real else np.complex128)
        check(lib().qbgpu_download_expanded(self.handle, C.c_void_p(rowptr.ctypes.data), C.c_void_p(col.ctypes.data),
                                            C.c_void_p(val.ctypes.data)))
        return rowptr, col, val

    def destroy(self):
        """Explicitly free the device copy (csr_mat::destroy, src/sparse.cc:150-169)."""
        if getattr(self, "handle", None) is not None:
            check(lib().qbgpu_destroy(self.handle))
            self.handle = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def _bond_array(bonds):
    b = np.ascontiguousarray(np.asarray(bonds, dtype=np.int32).reshape(-1, 2))
    return b, b.shape[0]


def heisenberg(nsites, ndown, bonds, J=1.0, is_complex=True, flags=0, rows=None, matrix_free=False):
    """Spin-1/2 Heisenberg model H = J sum_<ij> S_i.S_j in the sector with `ndown` down spins (Sz_total = nsites/2 - ndown),
    in the reference's Lin-table basis order.  Stored (the matrix model::generate_Ham_sparse_full would assemble,
    src/model.cc:619-686, generated directly in HBM) or matrix_free (the counterpart of model::MultMv2 with
    matrix_free == true, src/model.cc:942-1109).  Returns a csr_mat."""
    b, nb = _bond_array(bonds)
    h = C.c_void_p()
    lo, hi = (0, -1) if rows is None else (int(rows[0]), int(rows[1]))
    f = lib().qbgpu_create_matfree_heisenberg if matrix_free else lib().qbgpu_build_heisenberg
    check(f(C.byref(h), nsites, ndown, nb, C.c_void_p(b.ctypes.data), float(J), int(is_complex), flags, lo, hi))
    return csr_mat._adopt(h, is_complex)


def hubbard(nsites, nup, ndn, bonds, t=1.0, U=0.0, is_complex=True, flags=0, rows=None, matrix_free=False):
    """Single-orbital Fermi-Hubbard model H = -t sum_<ij>,s (c+_is c_js + h.c.) + U sum_i n_up n_dn with N_up, N_dn fixed,
    in the reference's Lin-table basis order and fermion-sign convention (src/basis.cc:2717-2731).  Stored or
    matrix_free as for heisenberg().  flags | SPECIES_ORDER: same operator and calling convention, vectors kept
    internally in (up configuration, down configuration) order and multiplied in two passes (include/qbgpu.h)."""
    b, nb = _bond_array(bonds)
    h = C.c_void_p()
    lo, hi = (0, -1) if rows is None else (int(rows[0]), int(rows[1]))
    f = lib().qbgpu_create_matfree_hubbard if matrix_free else lib().qbgpu_build_hubbard
    check(f(C.byref(h), nsites, nup, ndn, nb, C.c_void_p(b.ctypes.data), float(t), float(U), int(is_complex), flags, lo, hi))
    return csr_mat._adopt(h, is_complex)


def heisenberg_orbit(nsites, ndown, perms, chi, bonds, J=1.0, flags=0, return_states=False):
    """Spin-1/2 Heisenberg model in the sector of a one-dimensional irrep of an abelian symmetry group given as site
    permutations `perms[t][s]` (element 0 the identity) with characters `chi[t]`: orbit-minimum representatives, no
    reference counterpart (tilted clusters, SURVEY F5).  Returns a csr_mat (and the representatives)."""
    pa = np.ascontiguousarray(perms, dtype=np.int32)
    ca = np.ascontiguousarray(chi, dtype=np.complex128)
    if pa.ndim != 2 or pa.shape[1] != nsites or ca.size != pa.shape[0]:
        raise QbgpuError("perms must be [ntrans, nsites] with one character per group element")
    b, nb = _bond_array(bonds)
    h = C.c_void_p()
    from math import comb
    cap = comb(nsites, ndown) if return_states else 0
    st = np.empty(max(1, cap), dtype=np.uint32)
    check(lib().qbgpu_build_heisenberg_orbit(C.byref(h), nsites, ndown, pa.shape[0], C.c_void_p(pa.ctypes.data), C.c_void_p(ca.ctypes.data),
                                             nb, C.c_void_p(b.ctypes.data), float(J), flags,
                                             C.c_void_p(st.ctypes.data) if return_states else None, cap))
    M = csr_mat._adopt(h, True)
    return (M, st[:M.dim].copy()) if return_states else M


class Sector:
    """One (Sz, momentum) sector of a spin-1/2 model on an untilted lattice: the device counterpart of
    model::fill_Weisse_table + enumerate_basis_repr (src/model.cc:205-249, 275-487).  Representatives, their order and
    their norms are the reference's; `heisenberg()` assembles generate_Ham_sparse_repr's matrix (src/model.cc:688-836)
    directly in HBM and returns a csr_mat."""

    def __init__(self, L, ndown, momentum):
        La = np.ascontiguousarray(L, dtype=np.int32)
        ka = np.ascontiguousarray(momentum, dtype=np.int32)
        if La.size != ka.size:
            raise QbgpuError("momentum needs one integer per lattice direction")
        self._h = C.c_void_p()
        check(lib().qbgpu_sector_create(C.byref(self._h), int(La.size), C.c_void_p(La.ctypes.data), int(ndown), C.c_void_p(ka.ctypes.data)))
        info = _lib.SectorInfo()
        check(lib().qbgpu_sector_get_info(self._h, C.byref(info)))
        self.dim, self.zero_norm, self.nsites, self.lin_order = info.dim, info.zero_norm, info.nsites, bool(info.lin_order)
        self.enumerate_seconds, self.norms_seconds = info.enumerate_seconds, info.norms_seconds

    def states(self):
        """Bit patterns of the representatives in row order (bit s set = site s down)."""
        out = np.empty(self.dim, dtype=np.uint32)
        check(lib().qbgpu_sector_states(self._h, C.c_void_p(out.ctypes.data)))
        return out

    def norms(self):
        """norm_repr of the reference (src/basis.cc:2104-2202): orbit size, or 0 when the momentum kills the state."""
        out = np.empty(self.dim, dtype=np.float64)
        check(lib().qbgpu_sector_norms(self._h, C.c_void_p(out.ctypes.data)))
        return out

    def heisenberg(self, bonds, J=1.0, fake_pos=100.0, flags=0):
        b, nb = _bond_array(bonds)
        h = C.c_void_p()
        check(lib().qbgpu_sector_build_heisenberg(self._h, C.byref(h), nb, C.c_void_p(b.ctypes.data), float(J), float(fake_pos), flags))
        return csr_mat._adopt(h, True)

    def heisenberg_matrix_free(self, bonds, J=1.0, fake_pos=100.0):
        """The handle of model<T>::MultMv2 with matrix_free == true on this sector (src/model.cc:1016-1107): no stored entries,
        rows regenerated inside every product.  Keeps the sector alive for as long as the handle lives."""
        b, nb = _bond_array(bonds)
        h = C.c_void_p()
        check(lib().qbgpu_sector_matfree_heisenberg(self._h, C.byref(h), nb, C.c_void_p(b.ctypes.data), float(J), float(fake_pos)))
        m = csr_mat._adopt(h, True)
        m._sector = self
        return m

    def apply_sz(self, new_sector, coef, x, out=None):
        """model::moprXvec_repr (src/model.cc:1716-1846) for A = sum_r coef[r] S^z_r: x (DeviceVector or host array in this
        sector) -> DeviceVector in `new_sector` (written into `out` when given)."""
        cf = np.ascontiguousarray(coef, dtype=np.complex128)
        if cf.size != self.nsites:
            raise QbgpuError("one coefficient per site")
        xd = x if isinstance(x, DeviceVector) else DeviceVector.from_numpy(np.ascontiguousarray(x, dtype=np.complex128))
        y = out if out is not None else DeviceVector(self.dim)
        check(lib().qbgpu_sector_apply_sz(self._h, new_sector._h, C.c_void_p(cf.ctypes.data), C.c_void_p(xd.ptr), C.c_void_p(y.ptr)))
        return y

    def apply_ladder(self, new_sector, coef, x, lower=True, out=None):
        """The off-diagonal branch of model::moprXvec_repr (src/model.cc:1762-1834) for A = sum_r coef[r] S^-_r (lower=True:
        `new_sector` has one more down spin) or sum_r coef[r] S^+_r (lower=False): x in this sector -> DeviceVector in
        `new_sector`."""
        cf = np.ascontiguousarray(coef, dtype=np.complex128)
        if cf.size != self.nsites:
            raise QbgpuError("one coefficient per site")
        xd = x if isinstance(x, DeviceVector) else DeviceVector.from_numpy(np.ascontiguousarray(x, dtype=np.complex128))
        y = out if out is not None else DeviceVector(new_sector.dim)
        check(lib().qbgpu_sector_apply_ladder(self._h, new_sector._h, int(bool(lower)), C.c_void_p(cf.ctypes.data), C.c_void_p(xd.ptr), C.c_void_p(y.ptr)))
        return y

    def free(self):
        if self._h:
            lib().qbgpu_sector_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class ElectronSector(Sector):
    """One (N_up, N_dn, momentum) sector of single-orbital electrons on an untilted lattice (at most 16 sites): the device
    counterpart of model::fill_Weisse_table + enumerate_basis_repr for the reference's "electron" orbital (two bits per site,
    bit 0 up, bit 1 down), fermionic translation signs included (src/basis.cc:593-620, 2134-2147).  `hubbard()` assembles
    generate_Ham_sparse_repr's matrix (src/model.cc:688-836) for the Hubbard model directly in HBM -- the momentum-resolved
    flow of examples/trans_symmetric/latt_square/square_Fermi_Hubbard.cc."""

    def __init__(self, L, nup, ndn, momentum):
        La = np.ascontiguousarray(L, dtype=np.int32)
        ka = np.ascontiguousarray(momentum, dtype=np.int32)
        if La.size != ka.size:
            raise QbgpuError("momentum needs one integer per lattice direction")
        self._h = C.c_void_p()
        check(lib().qbgpu_sector_create_electron(C.byref(self._h), int(La.size), C.c_void_p(La.ctypes.data), int(nup), int(ndn), C.c_void_p(ka.ctypes.data)))
        info = _lib.SectorInfo()
        check(lib().qbgpu_sector_get_info(self._h, C.byref(info)))
        self.dim, self.zero_norm, self.nsites, self.lin_order = info.dim, info.zero_norm, info.nsites, bool(info.lin_order)
        self.enumerate_seconds, self.norms_seconds = info.enumerate_seconds, info.norms_seconds

    def hubbard(self, hops, t=1.0, U=1.1, fake_pos=100.0, flags=0):
        """hops: directed (to, from, spin) triples in the order of the caller's add_Ham calls."""
        h3 = np.ascontiguousarray(np.asarray(hops, dtype=np.int32).reshape(-1, 3))
        h = C.c_void_p()
        check(lib().qbgpu_sector_build_hubbard(self._h, C.byref(h), int(h3.shape[0]), C.c_void_p(h3.ctypes.data), float(t), float(U), float(fake_pos), flags))
        return csr_mat._adopt(h, True)

    # model::moprXvec_repr (src/model.cc:1716-1846) for one-site electron operators, x in this sector -> DeviceVector in
    # `new_sector` (written into `out` when given).  Coefficients e^{+i q.r} move a vector from momentum K to K + q;
    # c_k = N^{-1/2} sum_r e^{-i k.r} c_r moves it from K to K - k.  See include/qbgpu.h for the sign and norm rules.
    def _coef(self, c):
        cf = np.ascontiguousarray(c, dtype=np.complex128)
        if cf.size != self.nsites:
            raise QbgpuError("one coefficient per site")
        return cf

    def _xy(self, new_sector, x, out):
        xd = x if isinstance(x, DeviceVector) else DeviceVector.from_numpy(np.ascontiguousarray(x, dtype=np.complex128))
        if xd.n < self.dim:
            raise QbgpuError("x must hold the dimension of this sector")
        y = out if out is not None else DeviceVector(new_sector.dim)
        if y.n < new_sector.dim:
            raise QbgpuError("out must hold the dimension of the new sector")
        return xd, y

    def apply_density(self, new_sector, cu, cd, x, out=None):
        """A = sum_r cu[r] n_up,r + cd[r] n_dn,r (S^z_q: cd = -cu; charge density n_q: cd = cu); `new_sector` has the same
        particle numbers."""
        a, b = self._coef(cu), self._coef(cd)
        xd, y = self._xy(new_sector, x, out)
        check(lib().qbgpu_sector_apply_density(self._h, new_sector._h, C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data),
                                               C.c_void_p(xd.ptr), C.c_void_p(y.ptr)))
        return y

    def apply_spin_flip(self, new_sector, c, x, lower=True, out=None):
        """A = sum_r c[r] c+_{r,dn} c_{r,up} (lower=True, S^-: `new_sector` has N_up - 1, N_dn + 1) or its S^+ counterpart."""
        cf = self._coef(c)
        xd, y = self._xy(new_sector, x, out)
        check(lib().qbgpu_sector_apply_spin_flip(self._h, new_sector._h, int(bool(lower)), C.c_void_p(cf.ctypes.data),
                                                 C.c_void_p(xd.ptr), C.c_void_p(y.ptr)))
        return y

    def apply_fermion(self, new_sector, c, x, create=False, spin=0, out=None):
        """A = sum_r c[r] c_{r,spin} (create=False: `new_sector` has one electron fewer of that spin) or sum_r c[r] c+_{r,spin};
        spin 0 is up, 1 is down."""
        cf = self._coef(c)
        xd, y = self._xy(new_sector, x, out)
        check(lib().qbgpu_sector_apply_fermion(self._h, new_sector._h, int(bool(create)), int(spin), C.c_void_p(cf.ctypes.data),
                                               C.c_void_p(xd.ptr), C.c_void_p(y.ptr)))
        return y


def measure_repr_dynamic(coef, sec_old, sec_new, mat_new, phi0, maxit, hessenberg, op="sz"):
    """model<T>::measure_repr_dynamic (src/model.cc:1897-1912) for A = sum_r coef[r] S^z_r (op="sz"), S^-_r ("s-") or
    S^+_r ("s+"), everything on the device: vec = A phi0 mapped into sec_new (moprXvec_repr), norm = |vec|, then
    lanczos(0, maxit-1, maxit, ..., "dnmcs") from vec/norm on `mat_new`.  Returns (m, norm); hessenberg[2*maxit] receives
    b in [0, m) and a in [maxit, maxit+m)."""
    n = sec_new.dim
    v = DeviceVector(2 * n)
    v.zero()
    if op == "sz":
        sec_old.apply_sz(sec_new, coef, phi0, out=v.view(0, n))
    elif op in ("s-", "s+"):
        sec_old.apply_ladder(sec_new, coef, phi0, lower=(op == "s-"), out=v.view(0, n))
    else:
        raise QbgpuError("op must be 'sz', 's-' or 's+'")
    nr = C.c_double()
    check(lib().qbgpu_dznrm2(n, C.c_void_p(v.ptr), C.byref(nr)))
    if abs(nr.value) < lanczos_precision:
        v.free()
        return 0, nr.value
    check(lib().qbgpu_zscal(n, (C.c_double * 2)(1.0 / nr.value, 0.0), C.c_void_p(v.ptr)))
    m = lanczos(0, maxit - 1, maxit, n, mat_new, v, hessenberg, "dnmcs")
    v.free()
    return m, nr.value


def measure_repr_dynamic_electron(op, coefs, sec_old, sec_new, mat_new, phi0, maxit, hessenberg):
    """model<T>::measure_repr_dynamic (src/model.cc:1897-1912) for one-site electron operators between ElectronSectors:
    vec = A phi0 mapped into sec_new, norm = |vec|, then lanczos(0, maxit-1, maxit, ..., "dnmcs") from vec/norm on `mat_new`.
      op = "density":             coefs = (cu, cd)     A = sum_r cu[r] n_up,r + cd[r] n_dn,r
      op = "s-" / "s+":           coefs = c            A = sum_r c[r] c+_{r,dn} c_{r,up} / c+_{r,up} c_{r,dn}
      op = "c_up" / "c_dn":       coefs = c            A = sum_r c[r] c_{r,s}
      op = "cdag_up" / "cdag_dn": coefs = c            A = sum_r c[r] c+_{r,s}
    Returns (m, norm) like measure_repr_dynamic; hessenberg[2*maxit] receives b in [0, m) and a in [maxit, maxit+m).  With
    norm below lanczos_precision nothing is run and m = 0."""
    n = sec_new.dim
    v = DeviceVector(2 * n)
    v.zero()
    y = v.view(0, n)
    if op == "density":
        cu, cd = coefs
        sec_old.apply_density(sec_new, cu, cd, phi0, out=y)
    elif op in ("s-", "s+"):
        sec_old.apply_spin_flip(sec_new, coefs, phi0, lower=(op == "s-"), out=y)
    elif op in ("c_up", "c_dn", "cdag_up", "cdag_dn"):
        sec_old.apply_fermion(sec_new, coefs, phi0, create=op.startswith("cdag"), spin=int(op.endswith("dn")), out=y)
    else:
        v.free()
        raise QbgpuError("op must be 'density', 's-', 's+', 'c_up', 'c_dn', 'cdag_up' or 'cdag_dn'")
    nr = C.c_double()
    check(lib().qbgpu_dznrm2(n, C.c_void_p(v.ptr), C.byref(nr)))
    if abs(nr.value) < lanczos_precision:
        v.free()
        return 0, nr.value
    check(lib().qbgpu_zscal(n, (C.c_double * 2)(1.0 / nr.value, 0.0), C.c_void_p(v.ptr)))
    m = lanczos(0, maxit - 1, maxit, n, mat_new, v, hessenberg, "dnmcs")
    v.free()
    return m, nr.value


def continued_fraction(a, b, z):
    """G(z) = 1 / (z - a_0 - b_1^2 / (z - a_1 - b_2^2 / ...)) from Lanczos coefficients a[0..m), b[0..m) (b[0] unused): the
    evaluation of the reference's examples/trans_absent/latt_chain/plot_sqw.py:77-89.  With the dnmcs coefficients of
    A phi0 / |A phi0| and z = E0 + omega + i eta, -|A phi0|^2 Im G / pi is the broadened spectral weight of A at omega."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    z = np.asarray(z)
    g = np.zeros(z.shape, dtype=np.complex128)
    for j in range(len(a) - 1, -1, -1):
        g = 1.0 / (z - a[j] - (b[j + 1] ** 2 * g if j + 1 < len(a) else 0.0))
    return g


def full_apply_diag(kind, nsites, n0, n1, coef0, coef1, x, out=None):
    """model::moprXvec_full (src/model.cc:1468-1538) for one-site diagonal operators on a full-basis vector in the reference's
    Lin order: kind "heisenberg" (A = sum_r coef0[r] S^z_r, n0 = ndown) or "hubbard" (A = sum_r coef0[r] n_up,r + coef1[r] n_dn,r).
    x: DeviceVector or host array (complex128) -> DeviceVector."""
    k = {"heisenberg": 0, "hubbard": 1}[kind]
    c0 = np.ascontiguousarray(coef0, dtype=np.complex128)
    c1 = np.ascontiguousarray(coef1 if coef1 is not None else np.zeros(nsites), dtype=np.complex128)
    if c0.size != nsites or c1.size != nsites:
        raise QbgpuError("one coefficient per site")
    xd = x if isinstance(x, DeviceVector) else DeviceVector.from_numpy(np.ascontiguousarray(x, dtype=np.complex128))
    y = out if out is not None else DeviceVector(xd.n)
    check(lib().qbgpu_full_apply_diag(k, nsites, n0, n1, C.c_void_p(c0.ctypes.data), C.c_void_p(c1.ctypes.data),
                                      C.c_void_p(xd.ptr), C.c_void_p(y.ptr)))
    return y


def measure_full_dynamic(kind, nsites, n0, n1, coef0, coef1, mat, phi0, maxit, hessenberg):
    """model<T>::measure_full_dynamic (src/model.cc:1697-1712) for one-site diagonal operators (e.g. S^z_q of the Hubbard
    model: coef1 = -coef0), everything on the device: vec = A phi0, norm = |vec|, then lanczos(0, maxit-1, maxit, ..., "dnmcs")
    from vec/norm on `mat` (a full-basis handle in the reference's order, ordinary or species).  Returns (m, norm)."""
    n = mat.dim
    v = DeviceVector(2 * n)
    v.zero()
    full_apply_diag(kind, nsites, n0, n1, coef0, coef1, phi0, out=v.view(0, n))
    nr = C.c_double()
    check(lib().qbgpu_dznrm2(n, C.c_void_p(v.ptr), C.byref(nr)))
    if abs(nr.value) < lanczos_precision:
        v.free()
        return 0, nr.value
    check(lib().qbgpu_zscal(n, (C.c_double * 2)(1.0 / nr.value, 0.0), C.c_void_p(v.ptr)))
    m = lanczos(0, maxit - 1, maxit, n, mat, v, hessenberg, "dnmcs")
    v.free()
    return m, nr.value


def measure_vrnl_dynamic(vec_new, mat, maxit, hessenberg):
    """model<T>::measure_vrnl_dynamic (src/model.cc:2132-2143) from the point where the device path starts: `mat` is the handle
    of HamMat_csr_vrnl[sec] (assembled on the host by generate_Ham_sparse_vrnl, src/model.cc:839-924, and uploaded like any other
    csr_mat -- host assembly is outside the hot path) and `vec_new` = moprXgs_vrnl(Bq) = N * Aq |phi> (host array or DeviceVector,
    complex128, length dim).  norm = |vec_new|; if it is not below lanczos_precision: lanczos(0, maxit-1, maxit, m, dim, HamMat,
    vec_new / norm, hessenberg, "dnmcs").  Returns (m, norm)."""
    n = mat.dim
    v = DeviceVector(2 * n)
    v.zero()
    src = vec_new if isinstance(vec_new, DeviceVector) else DeviceVector.from_numpy(np.ascontiguousarray(vec_new, dtype=np.complex128))
    if src.n < n:
        raise QbgpuError("vec_new must hold dim entries")
    check(lib().qbgpu_zaxpy(n, (C.c_double * 2)(1.0, 0.0), C.c_void_p(src.ptr), C.c_void_p(v.ptr)))      # v[:dim] = vec_new (v is zero)
    if src is not vec_new:
        src.free()
    nr = C.c_double()
    check(lib().qbgpu_dznrm2(n, C.c_void_p(v.ptr), C.byref(nr)))
    if abs(nr.value) < lanczos_precision:
        v.free()
        return 0, nr.value
    check(lib().qbgpu_zscal(n, (C.c_double * 2)(1.0 / nr.value, 0.0), C.c_void_p(v.ptr)))
    m = lanczos(0, maxit - 1, maxit, n, mat, v, hessenberg, "dnmcs")
    v.free()
    return m, nr.value


def vec_randomize(n, seed=1, dtype=np.complex128, device=False):
    """src/miscellaneous.cc:371-388, generated on the device."""
    v = DeviceVector(n, dtype)
    f = lib().qbgpu_vec_randomize_z if np.dtype(dtype) == np.complex128 else lib().qbgpu_vec_randomize_d
    check(f(n, C.c_void_p(v.ptr), seed))
    if device:
        return v
    out = v.to_numpy()
    v.free()
    return out


def hess_eigen(hessenberg, maxit, m, order="sr"):
    """src/lanczos.cc:355-390 -> (ritz[m], s[m, m]) with s[:, j] the j-th Ritz vector."""
    if order.lower() not in ("sr", "sa"):
        raise QbgpuError("only order 'sr' is implemented")
    hess = _host_vec(np.ascontiguousarray(hessenberg, dtype=np.float64), np.float64, 2 * maxit, "hessenberg")
    ritz = np.zeros(m)
    s = np.zeros(m * m)
    check(lib().qbgpu_hess_eigen(_ptr(hess), maxit, m, _ptr(ritz), _ptr(s)))
    return ritz, s.reshape(m, m).T


def lanczos(k, np_, maxit, dim, mat, v, hessenberg, purpose):
    """lanczos<T,MAT>(k, np, maxit, m, dim, mat, v, hessenberg, purpose); returns m (src/lanczos.cc:134-266)."""
    if dim != mat.dim:
        raise QbgpuError("dim does not match the matrix")
    hess = _host_vec(hessenberg, np.float64, 2 * maxit, "hessenberg")
    nvec = 3 if "val1" in purpose else 2
    where = _where(v)
    if where == _lib.QBGPU_HOST:
        _host_vec(v, mat.dtype, nvec * dim, "v")
    m = C.c_int64(0)
    f = lib().qbgpu_lanczos_z if mat.is_complex else lib().qbgpu_lanczos_d
    check(f(mat.handle, k, np_, maxit, C.byref(m), _ptr(v), _ptr(hess), purpose.encode(), where))
    return m.value


def eigenvec_CG(dim, maxit, m, mat, E0, v, r, p, pp):
    """eigenvec_CG<T,MAT>(dim, maxit, m, mat, E0, accu, v, r, p, pp); returns (m, accu) (src/lanczos.cc:281-341)."""
    if dim != mat.dim:
        raise QbgpuError("dim does not match the matrix")
    where = _where(v, r, p, pp)
    if where == _lib.QBGPU_HOST:
        for name, a in (("v", v), ("r", r), ("p", p), ("pp", pp)):
            _host_vec(a, mat.dtype, dim, name)
    mm = C.c_int64(m)
    accu = C.c_double(0.0)
    if mat.is_complex:
        e = (C.c_double * 2)(complex(E0).real, complex(E0).imag)
        check(lib().qbgpu_eigenvec_cg_z(mat.handle, maxit, C.byref(mm), e, C.byref(accu), _ptr(v), _ptr(r), _ptr(p), _ptr(pp), where))
    else:
        check(lib().qbgpu_eigenvec_cg_d(mat.handle, maxit, C.byref(mm), float(E0), C.byref(accu), _ptr(v), _ptr(r), _ptr(p), _ptr(pp), where))
    return mm.value, accu.value


def eigenvec_CG_stepwise(dim, maxit, m, mat, E0, v, r, p, pp):
    """The reference's eigenvec_CG loop (src/lanczos.cc:293-332) kept on the HOST, its body replaced by the step-level entry points
    qbgpu_cg_restart / qbgpu_cg_step -- what a maintainer does who wants to keep the loop (logging, checkpoints) and move only the
    arithmetic.  Device vectors in the handle's own order and element type; starts at m == 0.  Returns (m, accu); the same
    kernels in the same order as eigenvec_CG, hence the same bits (when that one does not switch to fp64 vectors)."""
    if dim != mat.dim or m != 0:
        raise QbgpuError("eigenvec_CG_stepwise: dim must match the matrix and m must be 0")
    if _where(v, r, p, pp) != _lib.QBGPU_DEVICE:
        raise QbgpuError("eigenvec_CG_stepwise: device vectors only")
    L = lib()
    sc = DeviceVector(8, np.float64)
    sc.zero()
    e = (C.c_double * 2)(complex(E0).real, complex(E0).imag)
    accu, vn = C.c_double(0.0), C.c_double(0.0)
    nrm = L.qbgpu_dznrm2 if mat.is_complex else L.qbgpu_dnrm2
    while m < maxit:
        if accu.value < lanczos_precision:                                   # :295
            check(nrm(dim, _ptr(v), C.byref(vn)))
            if m == 0 or abs(vn.value - 1.0) > lanczos_precision:            # :297 re-normalise and restart
                check(L.qbgpu_cg_restart(mat.handle, e, _ptr(sc), _ptr(v), _ptr(r), _ptr(p), C.byref(vn), C.byref(accu)))
                m += 1
                if accu.value < lanczos_precision:                           # :315
                    break
            else:
                break                                                        # :317
        else:
            check(L.qbgpu_cg_step(mat.handle, e, _ptr(sc), _ptr(v), _ptr(r), _ptr(p), _ptr(pp), C.byref(accu)))      # :320-330
            m += 1
    sc.free()
    return m, accu.value


def kpm_moments_stepwise(mat, phi, lo, hi, nmom):
    """kpm_moments as a host loop over qbgpu_cheb_step (one fused product per two moments); phi: a device vector in the handle's
    order and element type.  Same products and epilogue sums as qbgpu_kpm_moments_*."""
    if _where(phi) != _lib.QBGPU_DEVICE:
        raise QbgpuError("kpm_moments_stepwise: device vectors only")
    L = lib()
    n = mat.dim
    T = [phi.clone(), DeviceVector(n, phi.dtype)]
    nprod = nmom // 2 + 1
    dots = DeviceVector(4 * (nprod + 1), np.float64)
    dots.zero()
    for k in range(nprod):
        cur, nxt = T[k % 2], T[(k + 1) % 2]
        check(L.qbgpu_cheb_step(mat.handle, lo, hi, int(k == 0), _ptr(cur), _ptr(nxt), _ptr(nxt), C.c_void_p(dots.ptr + 8 * 4 * (k + 1))))
    h = dots.to_numpy()
    nn = C.c_double(0.0)
    check((L.qbgpu_dznrm2 if mat.is_complex else L.qbgpu_dnrm2)(n, _ptr(phi), C.byref(nn)))
    mu0, mu1 = nn.value ** 2, h[4]
    mu = np.zeros(nmom)
    for j in range(nmom):
        if j == 0:
            mu[j] = mu0
        elif j == 1:
            mu[j] = mu1
        elif j % 2 == 0:
            mu[j] = 2.0 * h[4 * (j // 2) + 2] - mu0                          # mu_{2k+2} = 2 |T_{k+1}|^2 - mu_0
        else:
            mu[j] = 2.0 * h[4 * ((j - 1) // 2 + 1)] - mu1                    # mu_{2k+1} = 2 <T_k, T_{k+1}> - mu_1
    for t in T:
        t.free()
    dots.free()
    return mu


def energy_scale(dim, mat, v, extend=0.1, iters=128):
    """energy_scale<T,MAT>(dim, mat, v, lo, hi, extend, iters); returns (lo, hi) (src/kpm.cc:45-88)."""
    where = _where(v)
    if where == _lib.QBGPU_HOST:
        _host_vec(v, mat.dtype, 2 * dim, "v")
    lo, hi = C.c_double(), C.c_double()
    f = lib().qbgpu_energy_scale_z if mat.is_complex else lib().qbgpu_energy_scale_d
    check(f(mat.handle, _ptr(v), C.byref(lo), C.byref(hi), extend, iters, where))
    return lo.value, hi.value


def kpm_moments(mat, phi, lo, hi, nmom):
    """Chebyshev moments mu_k = <phi|T_k((H-c)/s)|phi> (new functionality; the reference has none, SURVEY F1)."""
    where = _where(phi)
    if where == _lib.QBGPU_HOST:
        _host_vec(phi, mat.dtype, mat.dim, "phi")
    mu = np.zeros(nmom)
    f = lib().qbgpu_kpm_moments_z if mat.is_complex else lib().qbgpu_kpm_moments_d
    check(f(mat.handle, _ptr(phi), lo, hi, nmom, _ptr(mu), where))
    return mu


def iram(dim, mat, v0, nev, ncv, maxit, order="sr"):
    """iram<T,MAT>(dim, mat, v0, nev, ncv, maxit, order, nconv, eigenvals, eigenvecs) (src/lanczos.cc:497-603): ARPACK's
    implicitly restarted Arnoldi with every product served by mat.MultMv on ARPACK's own HOST work vectors -- the
    reverse-communication callback of src/lanczos.cc:426,476.  ARPACK itself stays on the host, as in the reference
    (arpack-ng there; here scipy's bundled ARPACK, driven through scipy.sparse.linalg.eigsh).  dim <= 30 falls back to
    dense diagonalisation of mat.to_dense() like src/lanczos.cc:508-542.  Returns (nconv, eigenvals, eigenvecs[:, j])."""
    if nev <= 0 or nev >= dim - 1:
        raise ValueError("0 < nev < N-1 should be satisfied.")                  # src/lanczos.cc:502
    if maxit < 20:
        raise ValueError("maxit should not be smaller than 20!")               # :504
    order = order.upper()
    which = {"SR": "SA", "SA": "SA", "LR": "LA", "LA": "LA", "SM": "SM", "LM": "LM"}.get(order)
    if which is None:
        raise ValueError("Invalid argument orderC.")
    if dim <= 30:
        w, U = np.linalg.eigh(mat.to_dense())
        idx = {"SA": np.argsort(w), "LA": np.argsort(-w), "SM": np.argsort(np.abs(w)), "LM": np.argsort(-np.abs(w))}[which][:nev]
        return nev, w[idx], U[:, idx]
    from scipy.sparse.linalg import LinearOperator, eigsh
    nprod = [0]

    def matvec(x):
        x = np.ascontiguousarray(x, dtype=mat.dtype).ravel()
        y = np.empty(dim, dtype=mat.dtype)
        mat.MultMv(x, y)                                                         # host pointers in, host pointers out
        nprod[0] += 1
        return y

    A = LinearOperator((dim, dim), matvec=matvec, dtype=mat.dtype)
    w, U = eigsh(A, k=nev, which=which, ncv=ncv, maxiter=maxit, tol=0.0)         # tol <= 0: machine precision (:405,452)
    key = {"SA": w, "LA": -w, "SM": np.abs(w), "LM": -np.abs(w)}[which]
    idx = np.argsort(key, kind="stable")                                         # the reference's post-sort, :583-595
    iram.last_products = nprod[0]
    return len(w), w[idx], U[:, idx]


def trlan(mat, nev, ncv, maxit=0, tol=0.0, vectors=True, largest=False):
    """Device-resident thick-restart Lanczos (qbgpu_trlan): the `nev` lowest (or, largest=True, highest) eigenpairs with
    `ncv` basis vectors in HBM.  Returns (nconv, eigenvals[nev], eigenvecs[n, nev] or None, products)."""
    w = np.zeros(nev)
    U = np.zeros(mat.dim * nev, dtype=mat.dtype) if vectors else None
    nconv, nprod = C.c_int(0), C.c_int(0)
    f = lib().qbgpu_trlan_largest if largest else lib().qbgpu_trlan
    check(f(mat.handle, nev, ncv, maxit, tol, C.byref(nconv), C.byref(nprod), _ptr(w),
            _ptr(U) if vectors else None, _lib.QBGPU_HOST))
    return nconv.value, w, (U.reshape(nev, mat.dim).T if vectors else None), nprod.value


def herm_eigen(a):
    """Host dense Hermitian eigensolver used by trlan for the projected matrix (complex Jacobi)."""
    a = np.asarray(a, dtype=np.complex128)
    m = a.shape[0]
    acm = np.asfortranarray(a).ravel(order="F").copy()
    w = np.zeros(m)
    s = np.zeros(m * m, dtype=np.complex128)
    check(lib().qbgpu_herm_eigen(m, _ptr(acm), _ptr(w), _ptr(s)))
    return w, s.reshape(m, m, order="F")


def locate_E0_iram(mat, nev=2, ncv=6, maxit=0, device_resident=False):
    """The csr_mat branch of model<T>::locate_E0_iram (src/model.cc:1320-1366): returns dict(eigenvals, eigenvecs, nconv, gap).
    device_resident=False: ARPACK on the host calling MultMv per product (the reference's data flow);
    device_resident=True: the same contract served by the thick-restart Lanczos that keeps the basis in HBM."""
    if not (nev > 0 and ncv > nev + 1):
        raise QbgpuError("need nev > 0 and ncv > nev + 1")                        # the reference's asserts, :1337-1338
    if maxit <= 0:
        maxit = nev * 100                                                        # :1339
    if device_resident and mat.dim > 30:
        nconv, w, U, nprod = trlan(mat, nev, ncv, maxit)
        out = {"eigenvals": list(w), "eigenvecs": [U[:, j].copy() for j in range(nev)], "nconv": nconv, "products": nprod}
        if nev > 1:
            out["gap"] = w[1] - w[0]
        return out
    v0 = np.ones(mat.dim, dtype=mat.dtype)                                       # :1352 (ARPACK ignores it with info = 0)
    nconv, w, U = iram(mat.dim, mat, v0, nev, ncv, maxit, "sr")
    out = {"eigenvals": list(w), "eigenvecs": [U[:, j].copy() for j in range(U.shape[1])], "nconv": nconv}
    if nconv > 1:
        out["gap"] = w[1] - w[0]
    return out


def locate_Emax_iram(mat, nev=2, ncv=6, maxit=0, device_resident=False, fake_pos=100.0):
    """The csr_mat branch of model<T>::locate_Emax_iram (src/model.cc:1370-1422): the highest eigenpairs (order "lr");
    Emax = the first eigenvalue below fake_pos (momentum sectors carry artificial diagonal entries >= fake_pos for their
    zero-norm representatives, src/model.cc:737-740, 1417-1421).  Returns dict(eigenvals, eigenvecs, nconv, Emax)."""
    if not (nev > 0 and ncv > nev + 1):
        raise QbgpuError("need nev > 0 and ncv > nev + 1")                        # the reference's asserts, :1388-1389
    if maxit <= 0:
        maxit = nev * 100                                                        # :1390
    if device_resident and mat.dim > 30:
        nconv, w, U, nprod = trlan(mat, nev, ncv, maxit, largest=True)
        vecs = [U[:, j].copy() for j in range(nev)]
    else:
        v0 = np.ones(mat.dim, dtype=mat.dtype)                                   # :1403
        nconv, w, U = iram(mat.dim, mat, v0, nev, ncv, max(maxit, 20), "lr")
        vecs = [U[:, j].copy() for j in range(U.shape[1])]
    if nconv <= 0:
        raise QbgpuError("locate_Emax_iram: nothing converged")                   # the reference's assert, :1413
    emax = w[0]
    for e in w[:max(nconv, 1)]:                                                  # :1417-1421
        if e < fake_pos:
            emax = e
            break
    return {"eigenvals": list(w), "eigenvecs": vecs, "nconv": nconv, "Emax": emax}


def locate_E0_lanczos(mat, nev=1, ncv=1, maxit=1000, device_vectors=False):
    """The csr_mat branch of model<T>::locate_E0_lanczos (src/model.cc:1124-1316): E0 by simple Lanczos, ground-state
    vector by CG, optionally E1 (re-orthogonalised Lanczos) and its vector.  Everything stays on the device; returns a
    dict with eigenvals, eigenvecs (host arrays), step counts and accuracies."""
    if not (0 < nev <= 2 and nev - 1 <= ncv <= nev):
        raise QbgpuError("need 0 < nev <= 2 and nev-1 <= ncv <= nev")          # the reference's assert, :1141
    n, dt, seed = mat.dim, mat.dtype, 1
    out = {"eigenvals": [], "eigenvecs": []}
    v = DeviceVector((5 if ncv == 2 else 4 if ncv > 0 else 2) * n, dt)
    col = lambda j: v.view(j * n, n)                                           # noqa: E731
    rnd = lib().qbgpu_vec_randomize_z if mat.is_complex else lib().qbgpu_vec_randomize_d
    check(rnd(n, C.c_void_p(col(0).ptr), seed))                                # :1165
    hess = np.zeros(2 * maxit)
    m = lanczos(0, maxit - 1, maxit, n, mat, v, hess, "sr_val0")               # :1176-1181
    ritz, s = hess_eigen(hess, maxit, m)
    E0 = ritz[0]
    out["eigenvals"].append(E0)
    out["lanczos_steps"] = m
    out["lanczos_accuracy"] = abs(hess[m] * s[m - 1, 0])
    if ncv == 0:
        return out
    check(rnd(n, C.c_void_p(col(2).ptr), seed))                                # :1209
    mcg, accu = eigenvec_CG(n, maxit, 0, mat, E0, col(2), col(0), col(1), col(3))   # :1216-1217
    out["cg_steps"], out["cg_accuracy"] = mcg, accu
    if nev == 2:                                                               # :1233-1265
        check(rnd(n, C.c_void_p(col(0).ptr), seed))
        L = lib()
        if mat.is_complex:
            d = (C.c_double * 2)()
            check(L.qbgpu_zdotc(n, C.c_void_p(col(2).ptr), C.c_void_p(col(0).ptr), d))
            na = (C.c_double * 2)(-d[0], -d[1])
            check(L.qbgpu_zaxpy(n, na, C.c_void_p(col(2).ptr), C.c_void_p(col(0).ptr)))
            nr = C.c_double()
            check(L.qbgpu_dznrm2(n, C.c_void_p(col(0).ptr), C.byref(nr)))
            check(L.qbgpu_zscal(n, (C.c_double * 2)(1.0 / nr.value, 0.0), C.c_void_p(col(0).ptr)))
        else:
            d = C.c_double()
            check(L.qbgpu_ddot(n, C.c_void_p(col(2).ptr), C.c_void_p(col(0).ptr), C.byref(d)))
            check(L.qbgpu_daxpy(n, -d.value, C.c_void_p(col(2).ptr), C.c_void_p(col(0).ptr)))
            nr = C.c_double()
            check(L.qbgpu_dnrm2(n, C.c_void_p(col(0).ptr), C.byref(nr)))
            check(L.qbgpu_dscal(n, 1.0 / nr.value, C.c_void_p(col(0).ptr)))
        hess[:] = 0.0
        m1 = lanczos(0, maxit - 1, maxit, n, mat, v, hess, "sr_val1")
        ritz, s = hess_eigen(hess, maxit, m1)
        out["eigenvals"].append(ritz[0])
        out["gap"] = ritz[0] - E0
        out["lanczos_steps_E1"] = m1
    out["eigenvecs"].append(col(2).to_numpy())
    if device_vectors:                       # keep phi0 in HBM for what follows (moprXvec / measure_*_dynamic)
        out["eigenvecs_device"] = [col(2).clone()]
    if ncv == 2:                                                               # :1275-1315
        check(rnd(n, C.c_void_p(col(3).ptr), seed + 7))
        mcg1, accu1 = eigenvec_CG(n, maxit, 0, mat, out["eigenvals"][1], col(3), col(0), col(1), col(4))
        out["cg_steps_E1"], out["cg_accuracy_E1"] = mcg1, accu1
        v1 = col(3).to_numpy()
        if out["gap"] < lanczos_precision:                                     # orthogonalise a degenerate pair, :1302-1311
            v0 = out["eigenvecs"][0]
            v1 = v1 - np.vdot(v0, v1) * v0
            v1 /= np.linalg.norm(v1)
        out["eigenvecs"].append(v1)
    v.free()
    return out
