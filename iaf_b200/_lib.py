"""ctypes binding of include/iaf_b200.h.  There is no fallback: if the shared library is
missing or a call fails, the caller gets an exception."""
import ctypes as C
import os

from .build import LIB

IAF_MAX_HIDDEN = 4
IAF_MAX_HEADS = 2

VARIANTS = {"tf": 0, "theano": 1}
NLS = {None: 0, "None": 0, "none": 0, "elu": 1, "softplus": 2, "relu": 3, "tanh": 4, "leakyrelu": 5}
PATHS = {"auto": 0, "simt": 1, "tc": 2}
PATH_NAMES = {1: "simt", 2: "tc"}
ENTRIES = {"multiconv": 0, "step": 1, "layer": 2}

OK, ERR_BAD_ARG, ERR_BAD_SHAPE, ERR_UNSUPPORTED, ERR_CUDA, ERR_NOT_PACKED, ERR_NO_DEVICE = 0, -1, -2, -3, -4, -5, -6


class IafDesc(C.Structure):
    _fields_ = [("variant", C.c_int), ("n_z", C.c_int), ("n_hidden", C.c_int),
                ("hidden", C.c_int * IAF_MAX_HIDDEN), ("n_heads", C.c_int), ("head", C.c_int * IAF_MAX_HEADS),
                ("H", C.c_int), ("W", C.c_int), ("nl", C.c_int), ("path", C.c_int)]


# every symbol include/iaf_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "iaf_plan_create": (C.c_int, [C.POINTER(_P), C.POINTER(IafDesc)]),
    "iaf_plan_destroy": (None, [_P]),
    "iaf_pack_weights": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), _P]),
    "iaf_multiconv_fwd": (C.c_int, [_P, _P, _P, C.POINTER(_P), C.c_int, _P]),
    "iaf_step_fwd": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "iaf_step_fwd_host": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "iaf_step_submit_host": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int]),
    "iaf_host_wait": (C.c_int, [_P]),
    "iaf_layer_fwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "iaf_step_bwd": (C.c_int, [_P, _P, _P, C.POINTER(_P), C.POINTER(_P), _P, _P, _P, _P, _P, C.POINTER(_P), C.POINTER(_P),
                               C.POINTER(_P), C.c_int, _P]),
    "iaf_step_fwd_train": (C.c_int, [_P, _P, _P, _P, _P, _P, C.POINTER(_P), C.c_int, _P]),
    "iaf_step_bwd_saved": (C.c_int, [_P, _P, _P, _P, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), _P, _P, _P, _P, _P,
                                     C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.c_int, _P]),
    "iaf_layer_bwd": (C.c_int, [_P] * 7 + [C.POINTER(_P), C.POINTER(_P)] + [_P] * 10 + [C.POINTER(_P)] * 3 + [C.c_int, _P]),
    "iaf_multiconv_fwd_train": (C.c_int, [_P, _P, _P, C.POINTER(_P), C.POINTER(_P), C.c_int, _P]),
    "iaf_multiconv_bwd_saved": (C.c_int, [_P, _P, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), _P, _P,
                                          C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.c_int, _P]),
    "iaf_multiconv_bwd": (C.c_int, [_P, _P, _P, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), _P, _P, C.POINTER(_P),
                                    C.POINTER(_P), C.POINTER(_P), C.c_int, _P]),
    "iaf_multiconv_init": (C.c_int, [_P, _P, _P, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P),
                                     C.POINTER(_P), _P, C.c_int, _P]),
    "iaf_strerror": (C.c_char_p, [C.c_int]),
    "iaf_last_cuda_error": (C.c_char_p, []),
    "iaf_version": (C.c_int, []),
    "iaf_plan_path": (C.c_int, [_P]),
    "iaf_plan_path_for_entry": (C.c_int, [_P, C.c_int]),
    "iaf_plan_bwd_path": (C.c_int, [_P]),
    "iaf_plan_launch_count": (C.c_uint64, [_P]),
    "iaf_plan_algorithmic_bytes": (C.c_size_t, [_P, C.c_int]),
    "iaf_plan_algorithmic_flops": (C.c_double, [_P, C.c_int]),
}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            raise RuntimeError(
                "libiaf_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'`; "
                "iaf_b200 has no CPU or PyTorch fallback." % LIB)
        L = C.CDLL(LIB)
        for name, (res, args) in SYMBOLS.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(status):
    if status == OK:
        return
    L = lib()
    msg = L.iaf_strerror(status).decode()
    if status == ERR_CUDA:
        msg += ": " + L.iaf_last_cuda_error().decode()
    if status in (ERR_BAD_ARG, ERR_BAD_SHAPE):
        raise ValueError("iaf_b200: " + msg)
    if status == ERR_UNSUPPORTED:
        raise NotImplementedError("iaf_b200: " + msg)
    raise RuntimeError("iaf_b200: " + msg)
