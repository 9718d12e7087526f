"""Builds tests/user_functor/my_simplex_objectives.cu OUT OF TREE (a temporary directory, the user's own nvcc command line) the way
tests/user_functor_lib.py builds my_objectives.cu, and loads it: the four simplex test objectives register their launch tables, and with
them their batched simplex launchers, at load time."""
import user_functor_lib

MYS_F_NEGATIVE, MYS_F_QUANTIZED, MYS_F_SIGNED_ZERO, MYS_F_NAN_REGION = 1401, 1402, 1403, 1404
NAMES = {MYS_F_NEGATIVE: "negative", MYS_F_QUANTIZED: "quantized", MYS_F_SIGNED_ZERO: "signed_zero", MYS_F_NAN_REGION: "nan_region"}

_lib = None


def build_and_load():
    """compile once per process; returns the ctypes handle of the user's library"""
    global _lib
    if _lib is None:
        _lib = user_functor_lib.build_user_library("my_simplex_objectives.cu", with_host_lib=False)
        assert _lib.my_simplex_registration_status() == 0
    return _lib
