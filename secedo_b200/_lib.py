"""ctypes binding of secedo_b200/libsecedo_b200.so — the C ABI declared in include/secedo_b200.h.

This is the reference-side binding shape (INTEGRATION.md shows the same calls from C++). The
library is loaded eagerly and loudly: there is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsecedo_b200.so")

MAX_CLASS = 64
N_PLANES = 9
NO_POS = 16383
NO_POS_WIDE = 0xFFFFFFFF
NORMALIZATIONS = {"ADD_MIN": 0, "EXPONENTIATE": 1, "SCALE_MAX_1": 2}
PATHS = {"auto": 0, "scatter": 1, "gemm": 2}
PATH_NAMES = {v: k for k, v in PATHS.items()}


class SgpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"secedo_b200 error {code}: {msg}")
        self.code = code


class Stats(C.Structure):
    _fields_ = [
        ("n_loci", C.c_uint64), ("n_entries", C.c_uint64), ("n_reads", C.c_uint64),
        ("n_dropped_entries", C.c_uint64), ("n_multi_reads", C.c_uint64), ("n_tail_reads", C.c_uint64),
        ("n_pairs_first", C.c_uint64), ("n_pairs_multi", C.c_uint64),
        ("path_used", C.c_int32), ("n_span_splits", C.c_int32),
        ("ms_link", C.c_float), ("ms_first_order", C.c_float), ("ms_multi", C.c_float), ("ms_epilogue", C.c_float),
        ("ms_stage", C.c_float), ("ms_gemm", C.c_float), ("gemm_launches", C.c_uint64),
    ]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}
        d["path_used"] = PATH_NAMES.get(d["path_used"], str(d["path_used"]))
        return d


class SpectralStats(C.Structure):
    _fields_ = [
        ("outer_iterations", C.c_uint32), ("block", C.c_uint32), ("matvec_columns", C.c_uint64),
        ("matvec_launches", C.c_uint64), ("launches", C.c_uint64), ("max_residual", C.c_double),
        ("lower_bound", C.c_double), ("ms_laplacian", C.c_float), ("ms_solver", C.c_float), ("ms_matvec", C.c_float),
        ("reserved", C.c_uint32),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class EigenvalueStats(C.Structure):
    _fields_ = [
        ("launches", C.c_uint64), ("ms_laplacian", C.c_float), ("ms_tridiagonal", C.c_float), ("ms_bisection", C.c_float),
        ("bytes_matvec", C.c_uint64), ("reserved", C.c_uint32),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class SynthParams(C.Structure):
    _fields_ = [
        ("n_cells", C.c_uint32), ("n_chr", C.c_uint32), ("loci_per_chr", C.c_uint32), ("n_clones", C.c_uint32),
        ("spacing", C.c_uint32), ("reserved", C.c_uint32),
        ("coverage", C.c_float), ("frac_somatic", C.c_float), ("frac_germline", C.c_float), ("theta", C.c_float),
        ("p_multi", C.c_float), ("p_mate", C.c_float), ("p_mate_mismatch", C.c_float), ("reserved2", C.c_float),
        ("seed", C.c_uint64),
    ]


_vp = C.c_void_p
_u8p, _u16p, _u32p, _u64p = (C.POINTER(t) for t in (C.c_uint8, C.c_uint16, C.c_uint32, C.c_uint64))
_i32p, _f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)

# name -> (restype, argtypes); every symbol include/secedo_b200.h declares
SIGNATURES = {
    "sgpu_init": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "sgpu_shutdown": (None, [_vp]),
    "sgpu_last_error": (C.c_char_p, [_vp]),
    "sgpu_set_stream": (C.c_int, [_vp, _vp]),
    "sgpu_synchronize": (C.c_int, [_vp]),
    "sgpu_launch_count": (C.c_uint64, [_vp]),
    "sgpu_tensor_times": (C.c_int, [_vp, C.POINTER(C.c_float), C.POINTER(C.c_uint64)]),
    "sgpu_set_option": (C.c_int, [_vp, C.c_char_p, C.c_int]),
    "sgpu_synth_pileup": (C.c_int, [_vp, C.POINTER(SynthParams), C.POINTER(_vp)]),
    "sgpu_pileup_upload": (C.c_int, [_vp, C.c_uint32, _vp, _vp, _vp, _vp, _vp, C.POINTER(_vp)]),
    "sgpu_pileup_upload_async": (C.c_int, [_vp, C.c_uint32, _vp, _vp, _vp, _vp, _vp, C.POINTER(_vp)]),
    "sgpu_pileup_upload_lazy_async": (C.c_int, [_vp, C.c_uint32, _vp, _vp, _vp, _vp, _vp, C.POINTER(_vp)]),
    "sgpu_pileup_from_bin": (C.c_int, [_vp, C.c_uint32, _vp, _vp, _vp, C.c_uint32, C.c_uint32, _vp, _vp, C.POINTER(_vp),
                                       _u32p, _u32p]),
    "sgpu_pileup_upload_wide": (C.c_int, [_vp, C.c_uint32, _vp, _vp, _vp, _vp, _vp, C.POINTER(_vp)]),
    "sgpu_pileup_upload_wide_async": (C.c_int, [_vp, C.c_uint32, _vp, _vp, _vp, _vp, _vp, C.POINTER(_vp)]),
    "sgpu_pileup_download_wide": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sgpu_pileup_is_wide": (C.c_int, [_vp]),
    "sgpu_pileup_wrap_device": (C.c_int, [_vp, C.c_uint32, _vp, _vp, _vp, _vp, _vp, C.POINTER(_vp)]),
    "sgpu_pileup_dims": (C.c_int, [_vp, _u32p, _u64p, _u64p]),
    "sgpu_pileup_download": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sgpu_pileup_free": (None, [_vp, _vp]),
    "sgpu_is_significant": (C.c_int, [_vp, _vp, C.c_uint64, C.c_double, C.c_int, _vp]),
    "sgpu_filter": (C.c_int, [_vp, _vp, _vp, C.c_uint32, C.c_double, C.c_int, C.POINTER(_vp), _f64p]),
    "sgpu_similarity": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, _vp, C.c_uint32, C.c_double, C.c_double,
                                  C.c_double, C.c_uint32, C.c_int, C.c_int, _vp, C.POINTER(Stats)]),
    "sgpu_counts_create": (C.c_int, [_vp, C.c_uint32, C.POINTER(_vp)]),
    "sgpu_counts_zero": (C.c_int, [_vp, _vp]),
    "sgpu_counts_free": (None, [_vp, _vp]),
    "sgpu_counts_accumulate": (C.c_int, [_vp, _vp, _vp, C.c_uint32, _vp, C.c_uint32, C.c_double, C.c_double,
                                         C.c_double, C.c_uint32, C.c_int, C.POINTER(Stats)]),
    "sgpu_counts_accumulate_range": (C.c_int, [_vp, _vp, _vp, C.c_uint32, _vp, C.c_uint32, C.c_double, C.c_double,
                                               C.c_double, C.c_uint32, _vp, _vp, _vp, C.c_int, C.POINTER(Stats)]),
    "sgpu_chromosome_cutoff": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, _vp, _vp, _vp]),
    "sgpu_counts_buffers": (C.c_int, [_vp, C.POINTER(_vp), _u64p, C.POINTER(_vp), _u64p, C.POINTER(_vp), _u64p]),
    "sgpu_counts_set_layout": (C.c_int, [_vp, _vp, C.c_int, C.c_int]),
    "sgpu_counts_pack": (C.c_int, [_vp, _vp, C.POINTER(_vp), _u64p]),
    "sgpu_counts_unpack": (C.c_int, [_vp, _vp]),
    "sgpu_counts_pack_range": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.POINTER(_vp), _u64p]),
    "sgpu_counts_unpack_range": (C.c_int, [_vp, _vp, C.c_int, C.c_int]),
    "sgpu_counts_sparse_pack": (C.c_int, [_vp, _vp, C.c_int, C.POINTER(_vp), C.POINTER(_vp), _u64p]),
    "sgpu_counts_sparse_add": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_uint64]),
    "sgpu_counts_download": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "sgpu_similarity_finalize": (C.c_int, [_vp, _vp, C.c_uint32, C.c_double, C.c_double, C.c_double, C.c_int, _vp,
                                           C.POINTER(Stats)]),
    "sgpu_similarity_finalize_async": (C.c_int, [_vp, _vp, C.c_uint32, C.c_double, C.c_double, C.c_double, C.c_int, _vp]),
    "sgpu_output_wait": (C.c_int, [_vp]),
    "sgpu_slab_raw": (C.c_int, [_vp, _vp, _vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_double, C.c_double,
                                C.c_double, C.POINTER(_vp)]),
    "sgpu_slab_finalize": (C.c_int, [_vp, _vp, C.c_int, _vp, C.POINTER(_vp)]),
    "sgpu_slab_range": (C.c_int, [_vp, _u64p, _u64p]),
    "sgpu_counts_ipc_handle": (C.c_int, [_vp, _vp, C.c_int, _vp]),
    "sgpu_ipc_open": (C.c_int, [_vp, _vp, C.POINTER(_vp)]),
    "sgpu_ipc_close": (C.c_int, [_vp, _vp]),
    "sgpu_host_register": (C.c_int, [_vp, _vp, C.c_uint64, C.POINTER(_vp)]),
    "sgpu_host_unregister": (C.c_int, [_vp, _vp]),
    "sgpu_counts_checksum": (C.c_int, [_vp, _vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _u64p]),
    "sgpu_multi_init": (C.c_int, [_vp, C.c_int, C.POINTER(_vp)]),
    "sgpu_multi_shutdown": (None, [_vp]),
    "sgpu_multi_last_error": (C.c_char_p, [_vp]),
    "sgpu_multi_size": (C.c_int, [_vp]),
    "sgpu_multi_ctx": (_vp, [_vp, C.c_int]),
    "sgpu_multi_similarity": (C.c_int, [_vp, C.c_uint32, _vp, _vp, _vp, _vp, _vp, C.c_uint32, C.c_uint32, _vp, C.c_uint32,
                                        C.c_double, C.c_double, C.c_double, C.c_uint32, C.c_int, C.c_int, _vp, C.POINTER(Stats)]),
    "sgpu_log_probs": (C.c_int, [_vp, C.c_double, C.c_double, C.c_double, C.c_uint32, C.c_uint32, _vp, _vp]),
    "sgpu_expectation_maximization": (C.c_int, [_vp, _vp, _vp, C.c_uint32, C.c_double, _vp, C.c_uint32, C.c_uint32, _u32p,
                                                C.POINTER(C.c_float)]),
    "sgpu_laplacian": (C.c_int, [_vp, _vp, C.c_uint32, _vp]),
    "sgpu_spectral_embedding": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_double, _vp, _vp, C.POINTER(SpectralStats)]),
    "sgpu_similarity_finalize_spectral": (C.c_int, [_vp, _vp, C.c_uint32, C.c_double, C.c_double, C.c_double, C.c_int, _vp,
                                                    C.c_uint32, C.c_double, _vp, _vp, C.POINTER(Stats),
                                                    C.POINTER(SpectralStats)]),
    "sgpu_laplacian_eigenvalues": (C.c_int, [_vp, _vp, C.c_uint32, _vp, C.POINTER(EigenvalueStats)]),
    "sgpu_similarity_finalize_eigenvalues": (C.c_int, [_vp, _vp, C.c_uint32, C.c_double, C.c_double, C.c_double, C.c_int, _vp,
                                                       _vp, C.POINTER(Stats), C.POINTER(EigenvalueStats)]),
    "sgpu_spectral_matvec": (C.c_int, [_vp, _vp, C.c_uint32, C.c_int, _vp, _vp, C.c_double, C.c_double, C.c_double, _vp]),
}

_lib = None


def load() -> C.CDLL:
    """Load the CUDA library; raises if it has not been built (``python -m secedo_b200.build``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m secedo_b200.build` "
                "(or __graft_entry__.build()). secedo_b200 has no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
