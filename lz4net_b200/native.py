"""ctypes binding of liblz4b200.so (the C ABI in include/lz4b200.h).

This is the Python twin of the managed stub a lz4net maintainer would write (INTEGRATION.md): plain pointers and
sizes, nothing torch-specific.  It fails loudly when the library is missing -- there is no CPU path to fall back to.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "liblz4b200.so")

MODE_FAST, MODE_HC = 0, 1
MEM_HOST, MEM_DEVICE = 0, 1
OK, E_ARG, E_NODEVICE, E_CUDA, E_NOMEM, E_FORMAT = 0, -1, -2, -3, -4, -5

# every symbol include/lz4b200.h declares: (name, restype, argtypes)
_P, _I, _L, _U64 = C.c_void_p, C.c_int, C.c_int64, C.c_uint64
SIGNATURES = {
    "lz4b200_version": (_I, []),
    "lz4b200_last_error": (C.c_char_p, []),
    "lz4b200_device_count": (_I, []),
    "lz4b200_create": (_I, [C.POINTER(_P), _I]),
    "lz4b200_destroy": (None, [_P]),
    "lz4b200_synchronize": (_I, [_P]),
    "lz4b200_compress_bound": (_I, [_I]),
    "lz4b200_encode_batch": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int32, _I, _I, _P]),
    "lz4b200_decode_batch": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int32, _I, _I, _P]),
    "lz4b200_encode_batch_packed": (_I, [_P, _P, _P, _P, _P, _P, _L, _P, _P, C.c_int32, _I]),
    "lz4b200_compact": (_I, [_P, _P, _P, _P, _P, _P, C.c_int32, _P]),
    "lz4b200_compress_limitedOutput": (_I, [_P, _P, _I, _I]),
    "lz4b200_compressHC_limitedOutput": (_I, [_P, _P, _I, _I]),
    "lz4b200_uncompress": (_I, [_P, _P, _I, _I]),
    "lz4b200_uncompress_unknownOutputSize": (_I, [_P, _P, _I, _I]),
    "lz4b200_stream_bound": (_L, [_L, C.c_int32]),
    "lz4b200_stream_encode": (_L, [_P, _P, _L, C.c_int32, _I, _P, _L]),
    "lz4b200_stream_decoded_size": (_L, [_P, _L]),
    "lz4b200_stream_decode": (_L, [_P, _P, _L, _P, _L]),
    "lz4b200_stream_encode_device": (_L, [_P, _P, _L, C.c_int32, _I, _P, _L, _P]),
    "lz4b200_stream_decoded_size_device": (_L, [_P, _P, _L, _P]),
    "lz4b200_stream_decode_device": (_L, [_P, _P, _L, _P, _L, _P]),
    "lz4b200_wrap": (_I, [_P, _P, C.c_int32, _I, _P, C.c_int32]),
    "lz4b200_unwrap_size": (_I, [_P, C.c_int32]),
    "lz4b200_unwrap": (_I, [_P, _P, C.c_int32, _P, C.c_int32]),
    "lz4b200_wrap_batch": (_I, [_P, _P, _P, _P, _I, _P, _P, _P, _P, C.c_int32]),
    "lz4b200_unwrap_batch": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int32]),
    "lz4b200_host_register": (_I, [_P, _L]),
    "lz4b200_peer_copy": (_I, [_P, _P, _L, _P]),
    "lz4b200_host_unregister": (_I, [_P]),
    "lz4b200_synth_fill": (_I, [_P, _P, _L, C.c_int32, _I, _U64, _L, _P]),
    "lz4b200_set_option": (_I, [_P, C.c_char_p, _L]),
    "lz4b200_get_option": (_I, [_P, C.c_char_p, C.POINTER(_L)]),
    "lz4b200_launch_count": (_L, [_P]),
}

_lib = None


class Lz4B200Error(RuntimeError):
    pass


def lib():
    """Load the native library (once).  Raises if it has not been built: build with `python -m lz4net_b200.build`."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise Lz4B200Error(f"{SO_PATH} is missing: the CUDA extension is not built (python -m lz4net_b200.build). "
                               "lz4net_b200 has no CPU fallback.")
        l = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)          # AttributeError here = the library does not export what the header declares
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def last_error() -> str:
    return lib().lz4b200_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != OK:
        raise Lz4B200Error(f"{what} failed with status {rc}: {last_error()}")
