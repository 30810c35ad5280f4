"""ctypes binding of include/csic.h -- the same C ABI a Scala (Panama/JNI) host would bind.

The library is built in-tree by csrc/build.sh (`__graft_entry__.build()`).  If it is missing the
import fails loudly: there is no Python or CPU fallback for the pixel path.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# CSIC_LIB_PATH lets tools/ A/B two builds of the library on the same GPU box; default is the in-tree build.
LIB_PATH = os.environ.get("CSIC_LIB_PATH") or os.path.join(_HERE, "libcsic.so")


class CsicParams(ctypes.Structure):
    """`csic_params` (include/csic.h) == the ImageCompressorTop constructor surface
    (reference: src/main/scala/jpeg/ImageCompressorTop.scala:11-25)."""
    _fields_ = [("width", ctypes.c_int32), ("height", ctypes.c_int32),
                ("chroma_a", ctypes.c_int32), ("chroma_b", ctypes.c_int32),
                ("y_bits", ctypes.c_int32), ("cb_bits", ctypes.c_int32), ("cr_bits", ctypes.c_int32),
                ("factor", ctypes.c_int32), ("op", ctypes.c_int32 * 3),
                ("round_mode", ctypes.c_int32), ("pool_mode", ctypes.c_int32), ("out_format", ctypes.c_int32),
                ("in_format", ctypes.c_int32), ("reserved", ctypes.c_int32)]


# every symbol include/csic.h declares (tests/test_abi.py checks header <-> library <-> this table)
_PP = ctypes.POINTER(CsicParams)
_vp, _i32, _i64, _sz, _int = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t, ctypes.c_int
_cp = ctypes.c_char_p
PROTOTYPES = {
    "csic_abi_version": (_int, []),
    "csic_params_default": (_int, [_i32, _i32, _PP]),
    "csic_params_from_image_processor": (_int, [_i32, _i32, _i32, _i32, _i32, _PP]),
    "csic_params_from_legacy": (_int, [_i32, _i32, _i32, _i32, _i32, _PP]),
    "csic_validate": (_int, [_PP, ctypes.c_char_p, _sz]),
    "csic_out_shape": (_int, [_PP, ctypes.POINTER(_i32), ctypes.POINTER(_i32), ctypes.POINTER(_sz), ctypes.POINTER(_sz)]),
    "csic_planar_shape": (_int, [_PP, ctypes.POINTER(_i32), ctypes.POINTER(_i32), ctypes.POINTER(_sz), ctypes.POINTER(_sz)]),
    "csic_parse_step": (_int, [_cp]),
    "csic_strerror": (_cp, [_int]),
    "csic_last_error": (_cp, []),
    "csic_device_count": (_int, []),
    "csic_create": (_int, [_int, ctypes.POINTER(_vp)]),
    "csic_destroy": (_int, [_vp]),
    "csic_process_device": (_int, [_vp, _PP, _vp, _sz, _vp, _vp]),
    "csic_process_device_pitched": (_int, [_vp, _PP, _vp, _sz, _sz, _sz, _vp, _sz, _sz, _vp]),
    "csic_expand_planar_device": (_int, [_vp, _PP, _vp, _sz, _vp, _i32, _vp]),
    "csic_process_band": (_int, [_vp, _PP, _vp, _sz, _vp, _i32, _i32, _vp]),
    "csic_band_input_rows": (_int, [_PP, _i32, _i32, ctypes.POINTER(_i32), ctypes.POINTER(_i32)]),
    "csic_process_host": (_int, [_vp, _PP, _vp, _sz, _vp]),
    "csic_process_host_band": (_int, [_vp, _PP, _vp, _sz, _vp, _i32, _i32]),
    "csic_multi_create": (_int, [ctypes.POINTER(_int), _int, ctypes.POINTER(_vp)]),
    "csic_multi_destroy": (_int, [_vp]),
    "csic_multi_size": (_int, [_vp]),
    "csic_multi_process_host": (_int, [_vp, _PP, _vp, _sz, _vp]),
    "csic_multi_set_option": (_int, [_vp, _int, _i64]),
    "csic_multi_host_bytes": (_int, [_vp, ctypes.POINTER(ctypes.c_uint64), _int]),
    "csic_host_alloc": (_int, [_sz, ctypes.POINTER(_vp)]),
    "csic_host_free": (_int, [_vp]),
    "csic_synchronize": (_int, [_vp]),
    "csic_set_option": (_int, [_vp, _int, _i64]),
    "csic_host_bytes": (_int, [_vp, ctypes.POINTER(ctypes.c_uint64)]),
    "csic_last_kernel": (_int, [_vp, ctypes.POINTER(_i32), ctypes.POINTER(_i64)]),
    "csic_last_walk": (_int, [_vp, ctypes.POINTER(_i32)]),
}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(csrc/build.sh).  The pixel pipeline has no Python/CPU fallback.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib
