"""Builds the CPU stand-in of the host-logic tests extended by pnol_simplex_batch (tests/host_logic_simplex_batch.cpp) with the
unmodified host sources, the way tests/host_logic_bfgs_batch_lib.py builds the BFGS one, and loads it (ctypes, RTLD_LOCAL)."""
import ctypes as C
import glob
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

_lib = None


def build_and_load():
    """compile once per process; None when there is no g++"""
    global _lib
    if _lib is not None:
        return _lib
    cxx = shutil.which("g++")
    if cxx is None:
        return None
    so = os.path.join(tempfile.mkdtemp(prefix="pnol_host_logic_simplex_batch_"), "libpnol_host_logic_simplex_batch.so")
    host = os.path.join(ROOT, "parallelnonlinearoptimizationlibrary_b200", "host")
    # -Bsymbolic: the library's own pnol_* definitions win over a product library another test may have loaded RTLD_GLOBAL
    subprocess.check_call([cxx, "-std=c++17", "-O2", "-fPIC", "-ffp-contract=off", "-w", "-shared", "-Wl,-Bsymbolic", "-I" + os.path.join(ROOT, "include"),
                           "-I" + host] + sorted(glob.glob(os.path.join(host, "*.cpp"))) +
                          [os.path.join(HERE, "host_logic_simplex_batch.cpp"), os.path.join(ROOT, "oracle", "pnol_oracle.cpp"), "-o", so])
    lib = C.CDLL(so, mode=C.RTLD_LOCAL)
    lib.pnolhost_last_error.restype = C.c_char_p
    lib.pnolhost_last_evaluations.restype = C.c_longlong
    lib.standin_simplex_irregular_sorts.restype = C.c_longlong
    lib.pnol_stream_uniform.restype = C.c_double
    lib.pnol_stream_uniform.argtypes = [C.c_uint64, C.c_uint64, C.c_double]
    _lib = lib
    return lib
