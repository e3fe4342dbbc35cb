"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol include/qbgpu.h declares,
fails loudly without a GPU (no CPU fallback), and the host-only helpers work."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import quantum_basis_b200 as qb
from quantum_basis_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "qbgpu.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(qbgpu_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def L():
    if not os.path.exists(qb.LIB_PATH):
        qb.build_library()
    return qb.lib()


def test_every_declared_symbol_is_exported_and_bound(L):
    decl = declared_symbols()
    assert len(decl) > 40
    for name in decl:
        assert hasattr(L, name), f"{name} declared in include/qbgpu.h but not exported by libqbgpu.so"
    assert sorted(_lib.EXPORTS) == decl, "python binding table and header disagree"


def test_debug_set_variant_accepts_only_the_species_pass1_variants(L):
    try:
        for vid in (1000, 1001, 1002):
            assert L.qbgpu_debug_set_variant(vid) == 0
        for vid in (0, 45, 999, 1003, 2001, 3020):
            assert L.qbgpu_debug_set_variant(vid) == 1, vid             # QBGPU_ERR_ARG
            assert f"unknown id {vid} ".encode() in L.qbgpu_last_error()
    finally:
        assert L.qbgpu_debug_set_variant(1000) == 0


def test_library_is_sm100a_only():
    import subprocess
    out = subprocess.run(["cuobjdump", "--list-elf", qb.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_no_gpu_means_loud_failure_not_fallback(L):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    rc = L.qbgpu_init(0)
    assert rc == 2
    assert b"no CUDA device" in L.qbgpu_last_error()
    ia = np.array([0, 1, 2], dtype=np.int64); ja = np.array([0, 1], dtype=np.int64); val = np.ones(2)
    with pytest.raises(qb.QbgpuError):
        qb.csr_mat(2, ia, ja, val, True)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "quantum_basis_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".hpp", ".h", ".cc")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle_lib" not in txt and "qb_oracle" not in txt and "libqb_oracle" not in txt, f


def test_sector_dimensions(L):
    from math import comb
    assert L.qbgpu_dim_heisenberg(20, 10) == comb(20, 10) == 184756          # BASELINE config 1
    assert L.qbgpu_dim_hubbard(16, 8, 8) == comb(16, 8) ** 2 == 165636900    # BASELINE config 3
    assert L.qbgpu_dim_hubbard(8, 4, 4) == 4900
    assert L.qbgpu_dim_heisenberg(15, 7) == comb(15, 7)


def test_partition_rows_balances_expanded_nnz(L, oracle):
    A, meta, ex = oracle.load_golden("hubbard4x2")
    ia_full, _, _ = oracle.expand_upper(A)
    for parts in (1, 2, 3, 8):
        b = np.zeros(parts + 1, dtype=np.int64)
        rc = L.qbgpu_partition_rows(A.dim, A.ia.ctypes.data, A.ia.ctypes.data + 8, A.ja.ctypes.data, 1, parts, b.ctypes.data)
        assert rc == 0
        assert b[0] == 0 and b[-1] == A.dim and np.all(np.diff(b) >= 0)
        per = np.diff(ia_full[b])
        assert per.sum() == ia_full[-1]
        assert per.max() - per.min() <= 2 * np.diff(ia_full).max() + 1


def test_hess_eigen_host(L):
    rng = np.random.default_rng(3)
    m, maxit = 60, 100
    hess = np.zeros(2 * maxit)
    hess[1:m + 1] = rng.uniform(0.2, 1.5, m)
    hess[maxit:maxit + m] = rng.normal(size=m)
    ritz, s = qb.hess_eigen(hess, maxit, m)
    Tm = np.diag(hess[maxit:maxit + m]) + np.diag(hess[1:m], 1) + np.diag(hess[1:m], -1)
    w = np.linalg.eigvalsh(Tm)
    assert np.abs(ritz - w).max() < 1e-12
    assert np.abs(Tm @ s - s * ritz[None, :]).max() < 1e-12
    with pytest.raises(qb.QbgpuError):
        qb.hess_eigen(hess, maxit, maxit)          # the reference asserts m < maxit (src/lanczos.cc:358)


def test_herm_eigen_host(L):
    rng = np.random.default_rng(4)
    for m in (1, 2, 3, 8, 24):
        X = rng.normal(size=(m, m)) + 1j * rng.normal(size=(m, m))
        A = X + X.conj().T
        if m == 8:                                   # a degenerate pair and a real-symmetric case
            A = np.diag([1.0, 1.0, 2.0, 3.0, 3.0, 3.0, -1.0, 0.5]).astype(np.complex128)
            Q, _ = np.linalg.qr(X); A = Q @ A @ Q.conj().T
        w, S = qb.herm_eigen(A)
        assert np.abs(w - np.linalg.eigvalsh(A)).max() < 1e-12 * max(1.0, np.abs(A).max())
        assert np.abs(A @ S - S * w[None, :]).max() < 1e-11 * max(1.0, np.abs(A).max())
        assert np.abs(S.conj().T @ S - np.eye(m)).max() < 1e-12


def test_hess_smallest_matches_full_solve(L, oracle):
    import ctypes as C
    rng = np.random.default_rng(8)
    for m in (1, 2, 3, 10, 77, 300):
        maxit = 512
        hess = np.zeros(2 * maxit)
        hess[1:m + 1] = rng.uniform(1e-3, 3.0, m)
        hess[maxit:maxit + m] = rng.normal(size=m) * 5
        t = C.c_double()
        assert L.qbgpu_hess_smallest(hess.ctypes.data, maxit, m, C.byref(t)) == 0
        Tm = np.diag(hess[maxit:maxit + m]) + np.diag(hess[1:m], 1) + np.diag(hess[1:m], -1)
        w0 = np.linalg.eigvalsh(Tm)[0]
        assert abs(t.value - w0) <= 4e-15 * max(1.0, abs(w0))
    # a real Lanczos tridiagonal (converged ground state, tiny couplings at the end)
    A, meta, ex = oracle.load_golden("hubbard4x2")
    a, b = ex["lanczos_a"], ex["lanczos_b"]
    m = len(a); maxit = 1000
    hess = np.zeros(2 * maxit); hess[:m + 1] = b; hess[maxit:maxit + m] = a
    t = C.c_double()
    assert L.qbgpu_hess_smallest(hess.ctypes.data, maxit, m, C.byref(t)) == 0
    assert abs(t.value - meta["lanczos_E0"]) <= 1e-13 * abs(meta["lanczos_E0"])


def test_vector_files_are_the_reference_format(tmp_path, oracle):
    """vec_disk_write / vec_disk_read (src/miscellaneous.cc:391-468): a file written by the compiled reference
    (tests/golden/vec70_seed3.qbvec = vec_randomize(70, seed 3)) is read back, and a file written here is byte-identical."""
    import os
    import quantum_basis_b200 as qb
    g = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vec70_seed3.qbvec")
    x = qb.vec_disk_read(g, 70)
    assert x is not None and np.abs(x - oracle.vec_randomize(70, 3)).max() < 1e-15
    assert qb.vec_disk_read(g, 71) is None and qb.vec_disk_read(g, 70, dtype=np.float64) is None
    out = str(tmp_path / "v.qbvec")
    qb.vec_disk_write(out, x)
    assert open(out, "rb").read() == open(g, "rb").read()
    bad = bytearray(open(g, "rb").read()); bad[100] ^= 1
    open(out, "wb").write(bytes(bad))
    assert qb.vec_disk_read(out, 70) is None                      # checksum mismatch -> the reference's return 1


def test_cpp_adaptor_compiles_links_and_fails_loudly_without_a_gpu(tmp_path):
    """include/qbgpu_csr_mat.hpp (csr_mat<T> and sector) against libqbgpu.so with the image's g++: every entry point it
    uses exists, and without a device the constructors throw std::runtime_error -- never a silent fallback."""
    import shutil
    import subprocess
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "adaptor.cc"
    src.write_text('''
#include <cstdio>
#include "qbgpu_csr_mat.hpp"
int main() {
    int thrown = 0;
    try { qbgpu::sector s({16}, 8, {3}); auto H = s.heisenberg({0, 1, 1, 2}); std::printf("dim %lld\\n", (long long)H.dimension()); }
    catch (const std::runtime_error &e) { std::printf("sector: %s\\n", e.what()); thrown++; }
    long long ia[3] = {0, 1, 2}, ja[2] = {0, 1};
    std::complex<double> val[2] = {1.0, 2.0};
    try { qbgpu::csr_mat<std::complex<double>> A(2, 2, true, val, ja, ia); std::complex<double> x[2] = {1.0, 1.0}, y[2]; A.MultMv(x, y); std::printf("y %g %g\\n", y[0].real(), y[1].real()); }
    catch (const std::runtime_error &e) { std::printf("csr_mat: %s\\n", e.what()); thrown++; }
    return thrown;
}
// every member of both instantiations compiles and links (never called: argc is never 1000)
template <typename T> static void touch(int argc) {
    if (argc != 1000) return;
    qbgpu::csr_mat<T> A;
    T *v = nullptr; double *d = nullptr; double lo = 0, hi = 1, accu = 0; int64_t m = 0; int nconv = 0;
    A.MultMv(v, v); A.MultMv2(v, v); (void)A.to_dense();
    A.lanczos(0, 1, 2, m, v, d, "sr_val0"); A.eigenvec_CG(2, m, T(0), accu, v, v, v, v); A.energy_scale(v, lo, hi, 0.1, 8);
    (void)A.kpm_moments(v, lo, hi, 4); A.iram_device(1, 4, 10, "sr", nconv, d, v);
    (void)A.cg_restart(T(0), d, v, v, v); (void)A.cg_step(T(0), d, v, v, v, v); A.cheb_step(lo, hi, true, v, v, v, d);
}
template void touch<double>(int);
template void touch<std::complex<double>>(int);
''')
    exe = tmp_path / "adaptor"
    libdir = os.path.join(root, "quantum_basis_b200")
    subprocess.run([gxx, "-std=c++17", "-O1", "-I", os.path.join(root, "include"), str(src), "-o", str(exe), "-L", libdir, "-lqbgpu",
                    "-Wl,-rpath," + libdir], check=True)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([str(exe)], capture_output=True, text=True, env=env)
    assert r.returncode == 2, r.stdout + r.stderr               # both constructors threw
    assert "sector:" in r.stdout and "csr_mat:" in r.stdout and "failed" in r.stdout


@pytest.mark.parametrize("src,args", [("chain_heisenberg_momentum.cc", ["12"]), ("square_fermi_hubbard.cc", ["4", "2", "4", "4"])])
def test_cpp_example_builds_against_the_library(tmp_path, src, args):
    """The reference's chain and square-lattice Hubbard examples through the C++ adaptor compile and link; without a device
    they stop with the library's error message and a non-zero status."""
    import shutil
    import subprocess
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = tmp_path / "example"
    libdir = os.path.join(root, "quantum_basis_b200")
    subprocess.run([gxx, "-std=c++17", "-O1", "-I", os.path.join(root, "include"), os.path.join(root, "examples", src),
                    "-o", str(exe), "-L", libdir, "-lqbgpu", "-Wl,-rpath," + libdir], check=True)
    r = subprocess.run([str(exe)] + args, capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 2 and "no CUDA device" in r.stderr


def test_multi_gpu_cpp_example_builds_against_the_library(tmp_path):
    """examples/dist_lanczos.cc (E0 on N GPUs from plain C++ over the qbgpu_dist_* entries) compiles and links against the header
    and the library as they are; without a device every rank stops with the library's message and the program reports failure."""
    import shutil
    import subprocess
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = tmp_path / "dist_lanczos"
    libdir = os.path.join(root, "quantum_basis_b200")
    subprocess.run([gxx, "-std=c++17", "-O1", "-I", os.path.join(root, "include"), os.path.join(root, "examples", "dist_lanczos.cc"),
                    "-o", str(exe), "-L", libdir, "-lqbgpu", "-Wl,-rpath," + libdir], check=True)
    r = subprocess.run([str(exe), "2"], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), timeout=120)
    assert r.returncode != 0 and "no CUDA device" in r.stderr
