"""ctypes loader for libqbgpu.so (the C ABI declared in include/qbgpu.h).  Fails loudly when the library is missing."""
import ctypes as C
import os
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libqbgpu.so")
CSRC_DIR = os.path.join(PKG_DIR, "csrc")

QBGPU_HOST, QBGPU_DEVICE = 0, 1
KEEP_COMPLEX, NO_AUTOTUNE, FORMAT_CSR, FORMAT_SELL, VALUE_DICT, MATFREE_TERMS, SPECIES_ORDER = 1, 2, 4, 8, 16, 64, 128


class QbgpuError(RuntimeError):
    """Non-zero status from libqbgpu (the adaptor's analogue of the std::runtime_error thrown at
    reference src/sparse.cc:130,259,288)."""


class SectorInfo(C.Structure):
    _fields_ = [("dim", C.c_int64), ("zero_norm", C.c_int64), ("nsites", C.c_int), ("lin_order", C.c_int),
                ("enumerate_seconds", C.c_double), ("norms_seconds", C.c_double)]


class MatrixInfo(C.Structure):
    _fields_ = [("n", C.c_int64), ("row_lo", C.c_int64), ("row_hi", C.c_int64), ("nnz_stored", C.c_int64),
                ("nnz_input", C.c_int64), ("val_is_real", C.c_int), ("value_dict", C.c_int), ("api_is_complex", C.c_int), ("format", C.c_int),
                ("lanes", C.c_int), ("device_bytes", C.c_int64), ("upload_seconds", C.c_double),
                ("convert_seconds", C.c_double), ("autotune_seconds", C.c_double)]


def build_library(verbose=False):
    """Compile every CUDA source for sm_100a into quantum_basis_b200/libqbgpu.so (nvcc cross-compiles without a GPU)."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.run(["make", "-j8", "-C", CSRC_DIR], check=True, stdout=out)
    return LIB_PATH


_lib = None
vp, i64, dbl = C.c_void_p, C.c_int64, C.c_double
_SIGS = {
    "qbgpu_init": [C.c_int], "qbgpu_finalize": [], "qbgpu_device_count": [C.POINTER(C.c_int)],
    "qbgpu_set_stream": [vp], "qbgpu_synchronize": [],
    "qbgpu_create_dcsr": [C.POINTER(vp), i64, vp, vp, vp, vp, C.c_int, C.c_int],
    "qbgpu_create_zcsr": [C.POINTER(vp), i64, vp, vp, vp, vp, C.c_int, C.c_int],
    "qbgpu_create_dcsr_shard": [C.POINTER(vp), i64, vp, vp, vp, vp, C.c_int, C.c_int, i64, i64],
    "qbgpu_create_zcsr_shard": [C.POINTER(vp), i64, vp, vp, vp, vp, C.c_int, C.c_int, i64, i64],
    "qbgpu_destroy": [vp], "qbgpu_matrix_get_info": [vp, C.POINTER(MatrixInfo)], "qbgpu_to_dense": [vp, vp],
    "qbgpu_download_expanded": [vp, vp, vp, vp],
    "qbgpu_partition_rows": [i64, vp, vp, vp, C.c_int, C.c_int, vp],
    "qbgpu_dmv": [vp, dbl, vp, dbl, vp, C.c_int], "qbgpu_zmv": [vp, vp, vp, vp, vp, C.c_int],
    "qbgpu_host_register": [vp, C.c_size_t], "qbgpu_host_unregister": [vp],
    "qbgpu_malloc": [C.POINTER(vp), C.c_size_t], "qbgpu_free": [vp], "qbgpu_memcpy_h2d": [vp, vp, C.c_size_t],
    "qbgpu_memcpy_d2h": [vp, vp, C.c_size_t], "qbgpu_memcpy_d2d": [vp, vp, C.c_size_t], "qbgpu_memset0": [vp, C.c_size_t],
    "qbgpu_vec_randomize_d": [i64, vp, C.c_uint32], "qbgpu_vec_randomize_z": [i64, vp, C.c_uint32],
    "qbgpu_zdotc": [i64, vp, vp, vp], "qbgpu_ddot": [i64, vp, vp, vp], "qbgpu_dznrm2": [i64, vp, vp],
    "qbgpu_dnrm2": [i64, vp, vp], "qbgpu_zaxpy": [i64, vp, vp, vp], "qbgpu_daxpy": [i64, dbl, vp, vp],
    "qbgpu_zscal": [i64, vp, vp], "qbgpu_dscal": [i64, dbl, vp],
    "qbgpu_lanczos_d": [vp, i64, i64, i64, C.POINTER(i64), vp, vp, C.c_char_p, C.c_int],
    "qbgpu_lanczos_z": [vp, i64, i64, i64, C.POINTER(i64), vp, vp, C.c_char_p, C.c_int],
    "qbgpu_lanczos_resume_d": [vp, i64, i64, i64, C.POINTER(i64), vp, vp, C.c_char_p, C.c_int, vp],
    "qbgpu_lanczos_resume_z": [vp, i64, i64, i64, C.POINTER(i64), vp, vp, C.c_char_p, C.c_int, vp],
    "qbgpu_eigenvec_cg_d": [vp, i64, C.POINTER(i64), dbl, C.POINTER(dbl), vp, vp, vp, vp, C.c_int],
    "qbgpu_eigenvec_cg_z": [vp, i64, C.POINTER(i64), vp, C.POINTER(dbl), vp, vp, vp, vp, C.c_int],
    "qbgpu_energy_scale_d": [vp, vp, C.POINTER(dbl), C.POINTER(dbl), dbl, i64, C.c_int],
    "qbgpu_energy_scale_z": [vp, vp, C.POINTER(dbl), C.POINTER(dbl), dbl, i64, C.c_int],
    "qbgpu_kpm_moments_d": [vp, vp, dbl, dbl, i64, vp, C.c_int],
    "qbgpu_kpm_moments_z": [vp, vp, dbl, dbl, i64, vp, C.c_int],
    "qbgpu_hess_eigen": [vp, i64, i64, vp, vp], "qbgpu_herm_eigen": [C.c_int, vp, vp, vp], "qbgpu_hess_smallest": [vp, i64, i64, C.POINTER(dbl)],
    "qbgpu_trlan": [vp, C.c_int, C.c_int, C.c_int, dbl, C.POINTER(C.c_int), C.POINTER(C.c_int), vp, vp, C.c_int],
    "qbgpu_trlan_largest": [vp, C.c_int, C.c_int, C.c_int, dbl, C.POINTER(C.c_int), C.POINTER(C.c_int), vp, vp, C.c_int],
    "qbgpu_spmv_fused": [vp, vp, vp, vp, vp, vp, vp, vp],
    "qbgpu_lanczos_step_a": [vp, vp, vp, vp], "qbgpu_lanczos_step_a_part": [vp, vp, vp, vp, C.c_int, C.c_int],
    "qbgpu_split_columns": [vp, C.c_int, vp, vp, C.c_int], "qbgpu_debug_set_variant": [C.c_int], "qbgpu_real_view": [vp, C.POINTER(vp)],
    "qbgpu_ipc_export": [vp, vp], "qbgpu_ipc_open": [vp, C.POINTER(vp)], "qbgpu_ipc_close": [vp],
    "qbgpu_peer_pull_async": [C.c_int, C.c_int, vp, vp, C.c_size_t], "qbgpu_peer_wait": [C.c_int], "qbgpu_ring_prepare": [vp, C.c_int, C.c_int, i64, C.POINTER(vp)], "qbgpu_peer_ring_reset": [],
    "qbgpu_peer_pull_flag": [C.c_int, C.c_int, vp, vp, C.c_size_t, C.c_int], "qbgpu_peer_ring_status": [vp], "qbgpu_peer_pull_sm": [C.c_int, C.c_int, vp, vp, C.c_size_t, C.c_int], "qbgpu_lanczos_step_b": [vp, vp, vp, vp],
    "qbgpu_lanczos_step_c": [vp, vp, vp, i64],
    "qbgpu_cg_restart": [vp, vp, vp, vp, vp, vp, C.POINTER(dbl), C.POINTER(dbl)],
    "qbgpu_cg_step": [vp, vp, vp, vp, vp, vp, vp, C.POINTER(dbl)],
    "qbgpu_cheb_step": [vp, dbl, dbl, C.c_int, vp, vp, vp, vp],
    "qbgpu_build_heisenberg": [C.POINTER(vp), C.c_int, C.c_int, C.c_int, vp, dbl, C.c_int, C.c_int, i64, i64],
    "qbgpu_build_hubbard": [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, vp, dbl, dbl, C.c_int, C.c_int, i64, i64],
    "qbgpu_create_matfree_heisenberg": [C.POINTER(vp), C.c_int, C.c_int, C.c_int, vp, dbl, C.c_int, C.c_int, i64, i64],
    "qbgpu_create_matfree_hubbard": [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, vp, dbl, dbl, C.c_int, C.c_int, i64, i64],
    "qbgpu_sector_create": [C.POINTER(vp), C.c_int, vp, C.c_int, vp], "qbgpu_sector_destroy": [vp],
    "qbgpu_sector_get_info": [vp, C.POINTER(SectorInfo)], "qbgpu_sector_states": [vp, vp], "qbgpu_sector_norms": [vp, vp],
    "qbgpu_sector_build_heisenberg": [vp, C.POINTER(vp), C.c_int, vp, dbl, dbl, C.c_int],
    "qbgpu_sector_matfree_heisenberg": [vp, C.POINTER(vp), C.c_int, vp, dbl, dbl],
    "qbgpu_sector_create_electron": [C.POINTER(vp), C.c_int, vp, C.c_int, C.c_int, vp],
    "qbgpu_sector_build_hubbard": [vp, C.POINTER(vp), C.c_int, vp, dbl, dbl, dbl, C.c_int],
    "qbgpu_sector_apply_sz": [vp, vp, vp, vp, vp], "qbgpu_sector_apply_ladder": [vp, vp, C.c_int, vp, vp, vp],
    "qbgpu_sector_apply_density": [vp, vp, vp, vp, vp, vp], "qbgpu_sector_apply_spin_flip": [vp, vp, C.c_int, vp, vp, vp],
    "qbgpu_sector_apply_fermion": [vp, vp, C.c_int, C.c_int, vp, vp, vp],
    "qbgpu_full_apply_diag": [C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp],
    "qbgpu_debug_full_apply_diag_host": [C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp],
    "qbgpu_native_order": [vp, C.POINTER(C.c_int)], "qbgpu_vec_to_native": [vp, vp, vp], "qbgpu_vec_from_native": [vp, vp, vp],
    "qbgpu_native_perm": [vp, vp], "qbgpu_species_parts": [vp, C.POINTER(vp), C.POINTER(vp)],
    "qbgpu_dist_create": [C.POINTER(vp), C.c_int, C.c_int, i64, vp, C.c_int], "qbgpu_dist_export": [vp, vp], "qbgpu_dist_connect": [vp, vp],
    "qbgpu_dist_destroy": [vp], "qbgpu_dist_own": [vp, C.c_int, C.POINTER(vp), C.POINTER(i64)], "qbgpu_dist_full": [vp, C.c_int, C.POINTER(vp)],
    "qbgpu_dist_set_parts": [vp, C.c_int, vp, C.c_int, vp], "qbgpu_dist_set_pull_plan": [vp, C.c_int, vp, vp, vp, C.c_int],
    "qbgpu_species_split_cross": [vp, C.c_int, vp, vp], "qbgpu_row_view": [vp, i64, i64, i64, C.c_int, C.POINTER(vp)],
    "qbgpu_dist_set_wait_points": [vp, C.c_int, vp],
    "qbgpu_dist_barrier": [vp], "qbgpu_dist_allreduce": [vp, vp, C.c_int], "qbgpu_dist_randomize": [vp, C.c_int, C.c_uint32, vp],
    "qbgpu_species_ref_rows": [C.c_int, C.c_int, C.c_int, i64, i64, vp],
    "qbgpu_dist_mv": [vp, vp, vp, C.c_int, vp, C.c_int],
    "qbgpu_dist_lanczos": [vp, vp, vp, i64, i64, C.POINTER(i64), vp, C.c_char_p, C.c_int],
    "qbgpu_dist_energy_scale": [vp, vp, vp, vp, C.POINTER(dbl), C.POINTER(dbl), dbl, i64],
    "qbgpu_dist_kpm_moments": [vp, vp, vp, dbl, dbl, i64, vp],
    "qbgpu_dist_eigenvec_cg": [vp, vp, vp, i64, C.POINTER(i64), vp, C.POINTER(dbl), vp, vp, vp, vp],
    "qbgpu_debug_rows_host": [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, dbl, dbl, dbl, i64, vp, vp, C.c_int, vp],
    "qbgpu_debug_species_parts_host": [C.c_int, C.c_int, C.c_int, C.c_int, vp, dbl, dbl, C.c_int, i64, i64, C.c_int, vp, vp, vp, vp],
    "qbgpu_debug_species_host": [C.c_int, C.c_int, C.c_int, C.c_int, vp, dbl, dbl, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp],
    "qbgpu_debug_species_packed_host": [C.c_int, C.c_int, C.c_int, C.c_int, vp, dbl, dbl, C.c_int, vp, vp, vp, vp, vp],
    "qbgpu_build_heisenberg_orbit": [C.POINTER(vp), C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, vp, dbl, C.c_int, vp, i64],
}
_RESTYPES = {"qbgpu_last_error": C.c_char_p, "qbgpu_version": C.c_char_p, "qbgpu_kernel_launches": C.c_int64,
             "qbgpu_dim_heisenberg": C.c_int64, "qbgpu_dim_hubbard": C.c_int64}
EXPORTS = sorted(list(_SIGS) + ["qbgpu_last_error", "qbgpu_version", "qbgpu_kernel_launches", "qbgpu_dim_heisenberg",
                                "qbgpu_dim_hubbard"])


def lib():
    """Load libqbgpu.so.  Raises if it has not been built: there is no fallback implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise QbgpuError(f"{LIB_PATH} is missing: build it with __graft_entry__.build() or "
                         f"`make -C quantum_basis_b200/csrc` (no CPU fallback exists)")
    L = C.CDLL(LIB_PATH)
    for name, args in _SIGS.items():
        f = getattr(L, name)
        f.argtypes = args
        f.restype = C.c_int
    L.qbgpu_last_error.argtypes = []
    L.qbgpu_version.argtypes = []
    L.qbgpu_kernel_launches.argtypes = [C.c_int]
    L.qbgpu_dim_heisenberg.argtypes = [C.c_int, C.c_int]
    L.qbgpu_dim_hubbard.argtypes = [C.c_int, C.c_int, C.c_int]
    for name, rt in _RESTYPES.items():
        getattr(L, name).restype = rt
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise QbgpuError(f"libqbgpu status {rc}: {lib().qbgpu_last_error().decode(errors='replace')}")
