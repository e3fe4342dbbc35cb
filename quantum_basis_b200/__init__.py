"""quantum_basis_b200 -- B200-native H*v path for wztzjhn/quantum_basis.

The product is the C-ABI shared library ``libqbgpu.so`` (hand-written sm_100a CUDA, include/qbgpu.h).  This package
is the thin host-side mirror of the reference's interface for that path (``csr_mat`` with ``MultMv``/``MultMv2``,
``lanczos``, ``eigenvec_CG``, ``energy_scale``, ``locate_E0_lanczos``) over ctypes, plus the multi-GPU driver in
``dist``.  There is no CPU fallback: importing works anywhere, computing needs a CUDA device and the built library.
"""
from ._lib import lib, QbgpuError, build_library, LIB_PATH  # noqa: F401
from .csr import (csr_mat, lanczos, eigenvec_CG, eigenvec_CG_stepwise, energy_scale, kpm_moments, kpm_moments_stepwise, hess_eigen, vec_randomize,  # noqa: F401
                  locate_E0_lanczos, locate_E0_iram, locate_Emax_iram, iram, trlan, herm_eigen, heisenberg, hubbard, heisenberg_orbit, Sector, ElectronSector, measure_repr_dynamic, measure_repr_dynamic_electron, continued_fraction, measure_full_dynamic, measure_vrnl_dynamic, full_apply_diag, vec_disk_write, vec_disk_read, DeviceVector, lanczos_precision)
from . import ckpt  # noqa: F401,E402  (reference-format Lanczos checkpoints, src/ckpt.cc)
