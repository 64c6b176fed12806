"""ctypes binding of libquip_b200.so (the C ABI declared in include/quip_b200.h).

There is no CPU fallback: if the shared library is missing or a launch fails, callers get an
exception carrying quip_last_error().
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libquip_b200.so')

QUIP_FLAG_SYMMETRIC = 1
WS_HEADER_BYTES = 16 * 1024


ABI_VERSION = 2


class QuipPass(C.Structure):
    _fields_ = [('p', C.c_int32), ('nblk', C.c_int32), ('strided', C.c_int32), ('shared', C.c_int32),
                ('factors', C.c_void_p), ('factors_frag', C.c_void_p)]


class QuipSide(C.Structure):
    _fields_ = [('n', C.c_int32), ('npass', C.c_int32), ('passes', QuipPass * 2), ('idx', C.c_void_p),
                ('inv_idx', C.c_void_p)]


class QuipLinearDesc(C.Structure):
    _fields_ = [('K', C.c_int32), ('N', C.c_int32), ('bits', C.c_int32), ('flags', C.c_int32),
                ('qweight', C.c_void_p), ('scales', C.c_void_p), ('zeros', C.c_void_p), ('bias', C.c_void_p),
                ('inv_scale', C.c_void_p), ('V', QuipSide), ('U', QuipSide)]


# name -> (restype, argtypes); every symbol include/quip_b200.h declares
EXPORTS = {
    'quip_qlinear_forward': (C.c_int, [C.POINTER(QuipLinearDesc), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                       C.c_size_t, C.c_void_p]),
    'quip_qlinear_workspace_bytes': (C.c_int, [C.POINTER(QuipLinearDesc), C.c_int64, C.POINTER(C.c_size_t)]),
    'quip_qgemm': (C.c_int, [C.POINTER(QuipLinearDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                             C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    'quip_rowsum': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    'quip_gather': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_void_p]),
    'quip_rot_pass': (C.c_int, [C.POINTER(QuipPass), C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int,
                                C.c_void_p]),
    'quip_rmsnorm': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_float,
                               C.c_void_p]),
    'quip_rope': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                            C.c_void_p]),
    'quip_silu_mul': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'quip_vecquant_matmul': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                       C.c_void_p]),
    'quip_ldlq_block': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32,
                                  C.c_int32, C.c_void_p]),
    'quip_greedy_block': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p]),
    'quip_hessian_accumulate': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    'quip_silu_mul_gather': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    'quip_decode_attention': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                        C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p,
                                        C.c_size_t, C.c_void_p]),
    'quip_decode_attention_workspace_bytes': (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_size_t)]),
    'quip_pack_codes': (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    'quip_unpack_codes': (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    'quip_convert_ref': (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    'quip_packed_words': (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    'quip_config': (C.c_int, [C.c_char_p, C.c_int]),
    'quip_timing_enable': (C.c_int, [C.c_int]),
    'quip_timing_reset': (C.c_int, []),
    'quip_timing_read': (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_double),
                                   C.POINTER(C.c_double)]),
    'quip_last_error': (C.c_char_p, []),
    'quip_abi_version': (C.c_int, []),
    'quip_launch_count': (C.c_int64, []),
}

_lib = None


class QuipError(RuntimeError):
    pass


def load():
    """Load the library once; raises (loudly) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise QuipError(f'{LIB_PATH} not found: build it with `python -m quip_b200.build` '
                            '(there is no CPU fallback for the packed path)')
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.quip_abi_version() != ABI_VERSION:
            raise QuipError('libquip_b200.so ABI version mismatch')
        _lib = lib
    return _lib


def check(code):
    if code != 0:
        raise QuipError(f'quip_b200 error {code}: {load().quip_last_error().decode()}')


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())
