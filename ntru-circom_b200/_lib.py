"""ctypes binding of libntru_b200.so (include/ntru_b200.h).

There is no CPU fallback: if the shared library is missing it is built with nvcc,
and if that is impossible, or no CUDA device is present, the calls raise.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_int, c_int8, c_long, c_size_t, c_uint8, c_uint16, c_uint32, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
#: NTRU_B200_LIB points the harness at another build of the library (A/B runs, the NTRU_TRACE build)
LIB_PATH = os.environ.get("NTRU_B200_LIB") or os.path.join(_HERE, "libntru_b200.so")

NTRU_OK = 0
NTRU_E_PARAM, NTRU_E_LENGTH, NTRU_E_NOKEY, NTRU_E_CUDA = -1, -2, -3, -4
NTRU_E_NCCL, NTRU_E_NOMEM, NTRU_E_UNSUPPORTED = -5, -6, -7
NTRU_OPT_PATH, NTRU_OPT_CHUNK_ROWS, NTRU_OPT_TIMING, NTRU_OPT_DR, NTRU_OPT_DEC1_FORM, NTRU_OPT_SCHEDULE, NTRU_OPT_EPILOGUE = 1, 2, 3, 5, 6, 7, 8
NTRU_OPT_IMMA_FORM = 9
KERNEL_KINDS = ["enc_tensor", "dec1_tensor", "dec2_tensor", "enc_core", "dec_core", "sum", "other", "enc_imma", "dec_imma",
                "muldiv", "pack", "inverse", "check"]
#: verdict bits of the witness checks (ntru_check_*)
NTRU_CHECK_SATISFIED, NTRU_CHECK_CANONICAL, NTRU_CHECK_DOMAIN = 1, 2, 4
PATH_AUTO, PATH_CUDA_CORE, PATH_TENSOR, PATH_IMMA = 0, 1, 2, 3

#: every symbol include/ntru_b200.h declares: name -> (restype, argtypes)
_P = c_void_p
SYMBOLS = {
    "ntru_create": (c_int, [POINTER(c_void_p), c_int, c_int, c_int, c_int]),
    "ntru_destroy": (None, [_P]),
    "ntru_last_error": (c_char_p, [_P]),
    "ntru_strerror": (c_char_p, [c_int]),
    "ntru_set_option": (c_int, [_P, c_int, c_long]),
    "ntru_pitch": (c_int, [_P]),
    "ntru_launch_count": (c_uint64, [_P]),
    "ntru_last_path": (c_int, [_P]),
    "ntru_timing_read": (c_int, [_P, c_int, POINTER(ctypes.c_double), POINTER(c_uint64)]),
    "ntru_timing_reset": (c_int, [_P]),
    "ntru_set_public_key": (c_int, [_P, _P]),
    "ntru_set_private_key": (c_int, [_P, _P, _P]),
    "ntru_encrypt_batch": (c_int, [_P, c_size_t, _P, _P, _P, _P, _P, _P]),
    "ntru_encrypt_batch_wide": (c_int, [_P, c_size_t, _P, _P, _P, _P, _P, _P]),
    "ntru_encrypt_batch_keys": (c_int, [_P, c_size_t, _P, _P, _P, _P, _P, _P, _P]),
    "ntru_set_rng_key": (c_int, [_P, _P, c_uint64]),
    "ntru_rng_next_row": (c_uint64, [_P]),
    "ntru_decrypt_batch": (c_int, [_P, c_size_t, _P, _P, _P, _P, _P, _P]),
    "ntru_decrypt_batch_keys": (c_int, [_P, c_size_t, _P, _P, _P, _P, _P, _P, _P, _P]),
    "ntru_packed_elems": (c_int, [_P, c_int, c_int]),
    "ntru_encrypt_batch_packed": (c_int, [_P, c_size_t, _P, _P, _P, _P, _P, _P]),
    "ntru_decrypt_batch_packed": (c_int, [_P, c_size_t, _P, _P, _P, _P, _P, _P]),
    "ntru_sum": (c_int, [_P, c_size_t, _P, _P]),
    "ntru_sum_allreduce": (c_int, [_P, c_size_t, _P, _P]),
    "ntru_pack_output": (c_int, [_P, c_size_t, _P, c_int, c_int, ctypes.c_uint32, _P]),
    "ntru_unpack_input": (c_int, [_P, c_size_t, _P, c_int, ctypes.c_uint32, c_int, _P, c_int]),
    "ntru_get_params": (c_int, [_P, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "ntru_keygen_batch": (c_int, [_P, c_size_t, _P, _P, _P, _P, _P, _P]),
    "ntru_keygen_dev": (c_int, [_P, c_size_t, _P, _P, _P, _P, _P, _P]),
    "ntru_generate_keys_dev": (c_int, [_P, c_size_t, c_int, c_int, _P, _P, _P, _P, _P]),
    "ntru_pack_geometry": (c_int, [ctypes.c_uint32, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "ntru_pack_output_dev": (c_int, [_P, c_size_t, _P, c_int, c_int, c_size_t, ctypes.c_uint32, _P]),
    "ntru_unpack_input_dev": (c_int, [_P, c_size_t, _P, c_int, ctypes.c_uint32, c_int, _P, c_int, c_size_t]),
    "ntru_verify_keys_batch": (c_int, [_P, c_size_t, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "ntru_muldiv_dev": (c_int, [_P, c_size_t, _P, _P, c_int, _P, _P]),
    "ntru_check_encrypt_dev": (c_int, [_P, c_size_t, _P, c_size_t, _P, _P, _P, _P, _P]),
    "ntru_check_decrypt_dev": (c_int, [_P, c_size_t, _P, _P, c_size_t, _P, _P, _P, _P, _P, _P]),
    "ntru_check_inverse_dev": (c_int, [_P, c_size_t, c_int, _P, _P, _P, _P, _P]),
    "ntru_check_encrypt_batch": (c_int, [_P, c_size_t, _P, c_int, _P, _P, _P, _P, _P]),
    "ntru_check_decrypt_batch": (c_int, [_P, c_size_t, _P, _P, c_int, _P, _P, _P, _P, _P, _P]),
    "ntru_check_inverse_batch": (c_int, [_P, c_size_t, c_int, _P, _P, _P, _P, _P]),
    "ntru_encrypt_dev": (c_int, [_P, c_size_t, _P, _P, _P, _P, _P, _P]),
    "ntru_decrypt_dev": (c_int, [_P, c_size_t, _P, _P, _P, _P, _P, _P, _P, _P]),
    "ntru_sum_partial_dev": (c_int, [_P, c_size_t, _P, _P]),
    "ntru_sum_finalize_dev": (c_int, [_P, _P, _P]),
    "ntru_sample_r_dev": (c_int, [_P, c_size_t, c_int, c_uint64, _P]),
    "ntru_xchg_create": (c_int, [_P, c_int, c_int, _P]),
    "ntru_xchg_connect": (c_int, [_P, _P]),
    "ntru_sum_allreduce_dev": (c_int, [_P, c_size_t, _P, _P]),
    "ntru_xchg_destroy": (c_int, [_P]),
    "ntru_stream": (c_void_p, [_P]),
    "ntru_set_stream": (c_int, [_P, _P]),
    "ntru_sync": (c_int, [_P]),
    "ntru_host_alloc": (c_void_p, [c_size_t]),
    "ntru_host_free": (None, [_P]),
}

_lib = None


class NtruError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libntru_b200: {msg} (code {code})")
        self.code = code


def load() -> ctypes.CDLL:
    """Load (building first if needed) the CUDA library.  Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build   # nvcc; raises RuntimeError when nvcc is absent
        _build.build()
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)     # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
