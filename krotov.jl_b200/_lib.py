"""ctypes binding of ``libkrotov_cuda.so`` (C ABI in ``include/krotov_cuda.h``).

The library is the product's only compute path.  There is no CPU fallback: if the shared
object is missing this module raises ``ImportError`` on first use, and every entry point
raises ``KrotovCudaError`` on a non-zero status."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# KROTOV_CUDA_LIB points at another build of the same library (A/B experiments); the default is the in-tree build
LIB_PATH = os.environ.get("KROTOV_CUDA_LIB") or os.path.join(_HERE, "libkrotov_cuda.so")

KROTOV_OK = 0
ERR_NAMES = {1: "KROTOV_ERR_ARG", 2: "KROTOV_ERR_CUDA", 3: "KROTOV_ERR_STATE", 4: "KROTOV_ERR_UNSUPPORTED",
             5: "KROTOV_ERR_TIMEOUT", 6: "KROTOV_ERR_NOMEM"}
GEN_DENSE_COLMAJOR, GEN_CSR = 0, 1
FORWARD, BACKWARD = 0, 1
CHI_HOST, CHI_SM, CHI_SS, CHI_RE = 0, 1, 2, 3
PATH_WARP, PATH_DENSE, PATH_SPARSE = 1, 2, 3
PROP_CHEBY, PROP_EXPMV = 0, 1  # enum krotov_propagator (Problem.propagator)
# enum krotov_kernel (Info.kernel)
(KERNEL_TINY, KERNEL_PREG, KERNEL_SEQ_PREG, KERNEL_PAIR, KERNEL_RELOAD, KERNEL_DMMA_STREAM, KERNEL_DENSE_SWEEP,
 KERNEL_SPARSE_SWEEP, KERNEL_SPARSE_STREAM, KERNEL_TAYLOR) = range(1, 11)
COMM_DESC_BYTES = 256

# every symbol include/krotov_cuda.h declares that returns a status code or a string (tests check the .so exports all
# of them); krotov_live_device_objects returns a count and is bound below
EXPORTS = [
    "krotov_abi_version", "krotov_create", "krotov_destroy", "krotov_last_error", "krotov_get_info",
    "krotov_set_cheby", "krotov_set_taylor", "krotov_set_amplitudes", "krotov_set_amplitude_saturation", "krotov_set_control_terms", "krotov_forward", "krotov_set_chi", "krotov_set_chi_coeffs", "krotov_iterate",
    "krotov_get_states", "krotov_get_tau", "krotov_get_storage", "krotov_get_profile", "krotov_comm_export", "krotov_comm_connect",
    "krotov_group_connect", "krotov_group_iterate",
    "krotov_hermitian_extremes", "krotov_envelope_extremes", "krotov_envelope_extremes_device",
]


class KrotovCudaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libkrotov_cuda: {ERR_NAMES.get(code, code)}: {msg}")
        self.code = code
        self.detail = msg


class Problem(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("d", C.c_int32), ("n_traj", C.c_int32), ("n_ctrl", C.c_int32),
        ("n_steps", C.c_int32), ("n_gen", C.c_int32), ("gen_format", C.c_int32), ("nnz", C.c_int32),
        ("tlist", C.c_void_p), ("gen_of_traj", C.c_void_p), ("csr_rowptr", C.c_void_p), ("csr_colind", C.c_void_p),
        ("gen_values", C.c_void_p), ("term_present", C.c_void_p), ("psi0", C.c_void_p), ("target", C.c_void_p),
        ("weight", C.c_void_p), ("update_shape", C.c_void_p), ("lambda_a", C.c_void_p),
        ("functional", C.c_int32), ("n_traj_global", C.c_int32), ("store_fw", C.c_int32), ("device", C.c_int32),
        ("force_path", C.c_int32), ("replicated_forward", C.c_int32), ("propagator", C.c_int32),
        ("reserved", C.c_int32 * 5),
    ]


class Info(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("path", C.c_int32), ("ell_width", C.c_int32), ("nnz_union", C.c_int32),
        ("grid_blocks", C.c_int32), ("block_threads", C.c_int32), ("m_fw", C.c_int32), ("m_bw", C.c_int32),
        ("sm_count", C.c_int32), ("exchange", C.c_int32),
        ("launches_total", C.c_int64), ("launches_last", C.c_int64), ("ms_last", C.c_double),
        ("ms_last_backward", C.c_double), ("hbm_bytes_state", C.c_int64), ("fallback_steps", C.c_int64),
        ("graph_replays", C.c_int64), ("ms_rank_wait", C.c_double), ("kernel", C.c_int32), ("lanes_per_traj", C.c_int32),
        ("reserved", C.c_int64 * 2),
    ]


_lib = None


def lib():
    """Load the shared library (once).  Fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` at the repo root. "
            "krotov_jl_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, dbl = C.c_void_p, C.c_int, C.c_double
    L.krotov_abi_version.restype = i32
    L.krotov_create.argtypes = [C.POINTER(Problem), C.POINTER(vp)]
    L.krotov_destroy.argtypes = [vp]
    L.krotov_last_error.argtypes = [vp]
    L.krotov_last_error.restype = C.c_char_p
    L.krotov_get_info.argtypes = [vp, C.POINTER(Info)]
    L.krotov_set_cheby.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, vp, i32]
    L.krotov_set_taylor.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, i32]
    L.krotov_set_amplitudes.argtypes = [vp, i32, vp, vp]
    L.krotov_set_amplitude_saturation.argtypes = [vp, vp]
    L.krotov_set_control_terms.argtypes = [vp, vp]
    L.krotov_forward.argtypes = [vp, vp]
    L.krotov_set_chi.argtypes = [vp, vp]
    L.krotov_set_chi_coeffs.argtypes = [vp, vp]
    L.krotov_iterate.argtypes = [vp, vp, vp, vp]
    L.krotov_get_states.argtypes = [vp, vp]
    L.krotov_get_tau.argtypes = [vp, vp]
    L.krotov_get_storage.argtypes = [vp, i32, i32, i32, i32, vp]
    L.krotov_get_profile.argtypes = [vp, i32, vp]
    L.krotov_comm_export.argtypes = [vp, vp]
    L.krotov_comm_connect.argtypes = [vp, i32, i32, vp]
    L.krotov_group_connect.argtypes = [vp, i32]
    L.krotov_group_iterate.argtypes = [vp, i32, vp, vp, vp]
    L.krotov_hermitian_extremes.argtypes = [i32, i32, vp, vp, vp, i32]
    L.krotov_envelope_extremes.argtypes = [i32, i32, i32, vp, vp, i32, vp, vp, vp, i32]
    L.krotov_envelope_extremes_device.argtypes = [vp, i32, vp, vp, vp]
    for name in EXPORTS:
        if name not in ("krotov_last_error",):
            getattr(L, name).restype = i32
    L.krotov_last_error.restype = C.c_char_p
    L.krotov_live_device_objects.argtypes = []
    L.krotov_live_device_objects.restype = C.c_int64
    _lib = L
    return L


def hermitian_extremes(stack, n_threads=0):
    """``(e_min, e_max)`` of every matrix of a stack of complex Hermitian matrices through the library's threaded
    host solver (``krotov_hermitian_extremes``)."""
    import numpy as np

    a = np.ascontiguousarray(stack, np.complex128)
    n, d = a.shape[0], a.shape[-1]
    lo, hi = np.empty(n, np.float64), np.empty(n, np.float64)
    rc = lib().krotov_hermitian_extremes(n, d, a.ctypes.data_as(C.c_void_p), lo.ctypes.data_as(C.c_void_p),
                                         hi.ctypes.data_as(C.c_void_p), int(n_threads))
    if rc != KROTOV_OK:
        raise KrotovCudaError(rc, "krotov_hermitian_extremes: bad argument")
    return lo, hi


def envelope_extremes(H0s, Hcs, corners, n_threads=0):
    """``(e_min, e_max)`` per generator over the amplitude corners: ``H0s`` (n_gen, d, d), ``Hcs`` (L, n_gen, d, d),
    ``corners`` (n_corner, L) -- ``krotov_envelope_extremes``."""
    import numpy as np

    H0s = np.ascontiguousarray(H0s, np.complex128)
    Hcs = np.ascontiguousarray(Hcs, np.complex128)
    amps = np.ascontiguousarray(corners, np.float64)
    n_gen, d = H0s.shape[0], H0s.shape[-1]
    n_ctrl = Hcs.shape[0] if Hcs.size else 0
    lo, hi = np.empty(n_gen, np.float64), np.empty(n_gen, np.float64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    rc = lib().krotov_envelope_extremes(n_gen, d, n_ctrl, p(H0s), p(Hcs), amps.shape[0], p(amps), p(lo), p(hi),
                                        int(n_threads))
    if rc != KROTOV_OK:
        raise KrotovCudaError(rc, "krotov_envelope_extremes: bad argument")
    return lo, hi
