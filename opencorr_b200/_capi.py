"""ctypes binding of the C ABI in include/opencorr_b200.h (libopencorr_b200.so).

The library is hand-written CUDA for sm_100a; there is no CPU path.  Loading works without a
GPU (so the symbol table can be checked), but ocb_create() fails loudly.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OCB_LIB_PATH") or os.path.join(_HERE, "lib", "libopencorr_b200.so")  # override: A/B builds

OCB_OK = 0
OCB_ERR_CUDA = -1
OCB_ERR_ARG = -2
OCB_ERR_STATE = -3
OCB_ERR_UNSUPPORTED = -4

_vp = ctypes.c_void_p
_i = ctypes.c_int
_f = ctypes.c_float
_sz = ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/opencorr_b200.h one to one
SIGNATURES = {
    "ocb_device_count": (_i, []),
    "ocb_create": (_vp, [_i]),
    "ocb_create_multi": (_vp, [_vp, _i]),
    "ocb_member_count": (_i, [_vp]),
    "ocb_member": (_vp, [_vp, _i]),
    "ocb_host_register": (_i, [_vp, _sz]),
    "ocb_host_unregister": (_i, [_vp]),
    "ocb_host_alloc": (_vp, [_sz]),
    "ocb_host_alloc_on": (_vp, [_vp, _sz]),
    "ocb_host_free": (None, [_vp]),
    "ocb_destroy": (None, [_vp]),
    "ocb_last_error": (ctypes.c_char_p, [_vp]),
    "ocb_set_stream": (_i, [_vp, _vp]),
    "ocb_use_own_stream": (_i, [_vp]),
    "ocb_sync": (_i, [_vp]),
    "ocb_launch_count": (ctypes.c_longlong, [_vp]),
    "ocb_last_launch": (ctypes.c_char_p, [_vp]),
    "ocb_set_images_2d": (_i, [_vp, _vp, _vp, _i, _i, _i]),
    "ocb_set_images_3d": (_i, [_vp, _vp, _vp, _i, _i, _i]),
    "ocb_set_images_2d_u8": (_i, [_vp, _vp, _vp, _i, _i]),
    "ocb_set_images_3d_u8": (_i, [_vp, _vp, _vp, _i, _i, _i]),
    "ocb_set_images_2d_dev": (_i, [_vp, _vp, _vp, _i, _i]),
    "ocb_set_images_3d_dev": (_i, [_vp, _vp, _vp, _i, _i, _i]),
    "ocb_fftcc2d": (_i, [_vp, _vp, _sz, _i, _i]),
    "ocb_fftcc3d": (_i, [_vp, _vp, _sz, _i, _i, _i]),
    "ocb_fftcc2d_dev": (_i, [_vp, _vp, _sz, _i, _i]),
    "ocb_fftcc3d_dev": (_i, [_vp, _vp, _sz, _i, _i, _i]),
    "ocb_icgn2d_prepare": (_i, [_vp]),
    "ocb_icgn3d_prepare": (_i, [_vp]),
    "ocb_icgn2d1": (_i, [_vp, _vp, _sz, _i, _i, _f, _f]),
    "ocb_icgn2d2": (_i, [_vp, _vp, _sz, _i, _i, _f, _f]),
    "ocb_icgn3d1": (_i, [_vp, _vp, _sz, _i, _i, _i, _f, _f]),
    "ocb_icgn2d1_dev": (_i, [_vp, _vp, _sz, _i, _i, _f, _f]),
    "ocb_icgn2d2_dev": (_i, [_vp, _vp, _sz, _i, _i, _f, _f]),
    "ocb_icgn3d1_dev": (_i, [_vp, _vp, _sz, _i, _i, _i, _f, _f]),
    "ocb_icgn2d_ex": (_i, [_vp, _i, _vp, _sz, _i, _i, _f, _f, _vp, _i]),
    "ocb_icgn2d_ex_dev": (_i, [_vp, _i, _vp, _sz, _i, _i, _f, _f, _vp]),
    "ocb_iclm2d": (_i, [_vp, _i, _vp, _sz, _i, _i, _f, _f, _f, _f, _f]),
    "ocb_iclm2d_dev": (_i, [_vp, _i, _vp, _sz, _i, _i, _f, _f, _f, _f, _f]),
    "ocb_epipolar_search2d": (_i, [_vp, _vp, _sz, _vp, _vp, _vp, _i, _i, _i, _i, _f, _f]),
    "ocb_epipolar_search2d_dev": (_i, [_vp, _vp, _sz, _vp, _vp, _vp, _i, _i, _i, _i, _f, _f]),
    "ocb_strain2d": (_i, [_vp, _vp, _sz, _f, _i, _f, _i]),
    "ocb_strain3d": (_i, [_vp, _vp, _sz, _f, _i, _f, _i]),
    "ocb_strain2ds": (_i, [_vp, _vp, _sz, _f, _i, _f, _i]),
    "ocb_strain2ds_dev": (_i, [_vp, _vp, _sz, _f, _i, _f, _i]),
    "ocb_strain2d_single": (_i, [_vp, _vp, _sz, _sz, _f, _i, _f, _i]),
    "ocb_strain3d_single": (_i, [_vp, _vp, _sz, _sz, _f, _i, _f, _i]),
    "ocb_strain2d_dev": (_i, [_vp, _vp, _sz, _f, _i, _f, _i]),
    "ocb_strain3d_dev": (_i, [_vp, _vp, _sz, _f, _i, _f, _i]),
    "ocb_nr2d_prepare": (_i, [_vp]),
    "ocb_nr2d1": (_i, [_vp, _vp, _sz, _i, _i, _f, _f]),
    "ocb_nr2d1_dev": (_i, [_vp, _vp, _sz, _i, _i, _f, _f]),
    "ocb_get_tables_3d": (_i, [_vp, _vp, _vp, _vp, _vp]),
}

_lib = None


class OpenCorrB200Error(RuntimeError):
    """A C-ABI call returned a non-zero status (the C++ shim throws std::string instead)."""

    def __init__(self, code, message):
        super().__init__("opencorr_b200 error %d: %s" % (code, message))
        self.code = code


def load():
    """Load libopencorr_b200.so; raises if the CUDA extension has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise OpenCorrB200Error(
                OCB_ERR_STATE,
                "CUDA extension %s is missing - run `python -m opencorr_b200.build` "
                "(there is no CPU fallback)" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error(ctx=None):
    return load().ocb_last_error(ctx).decode("utf-8", "replace")


def check(rc, ctx=None):
    if rc != OCB_OK:
        raise OpenCorrB200Error(rc, last_error(ctx))
