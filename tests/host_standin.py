"""Builds the CPU stand-ins of the C-ABI that the host-logic tests link the unmodified host sources
(parallelnonlinearoptimizationlibrary_b200/host/*.cpp) against, each once per process into a temporary directory:

- base_path(): oracle/host_logic_device.cpp alone, the C-ABI without the analytic derivatives and the batch entry points;
- load(): tests/host_logic_standin.cpp, the base extended by them, loaded (ctypes, RTLD_LOCAL).

Both return None when there is no g++."""
import ctypes as C
import glob
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

_paths = {}
_lib = None


def _build(standin):
    if standin not in _paths:
        cxx = shutil.which("g++")
        if cxx is None:
            return None
        name = os.path.splitext(os.path.basename(standin))[0]
        so = os.path.join(tempfile.mkdtemp(prefix="pnol_%s_" % name), "lib%s.so" % name)
        host = os.path.join(ROOT, "parallelnonlinearoptimizationlibrary_b200", "host")
        # -Bsymbolic: the library's own pnol_* definitions win over a product library another test may have loaded RTLD_GLOBAL
        subprocess.check_call([cxx, "-std=c++17", "-O2", "-fPIC", "-ffp-contract=off", "-w", "-shared", "-Wl,-Bsymbolic", "-I" + os.path.join(ROOT, "include"),
                               "-I" + host] + sorted(glob.glob(os.path.join(host, "*.cpp"))) +
                              [standin, os.path.join(ROOT, "oracle", "pnol_oracle.cpp"), "-o", so])
        _paths[standin] = so
    return _paths[standin]


def base_path():
    """the path of the base stand-in's library, not loaded"""
    return _build(os.path.join(ROOT, "oracle", "host_logic_device.cpp"))


def load():
    """the extended stand-in's library"""
    global _lib
    if _lib is None:
        so = _build(os.path.join(HERE, "host_logic_standin.cpp"))
        if so is None:
            return None
        lib = C.CDLL(so, mode=C.RTLD_LOCAL)
        lib.pnolhost_last_error.restype = C.c_char_p
        lib.pnolhost_last_evaluations.restype = C.c_longlong
        lib.standin_simplex_irregular_sorts.restype = C.c_longlong
        lib.pnol_stream_uniform.restype = C.c_double
        lib.pnol_stream_uniform.argtypes = [C.c_uint64, C.c_uint64, C.c_double]
        lib.pnolhost_set_hinv_mode(0)          # PNOL_HINV_LITERAL: the reference's two matrix products
        _lib = lib
    return _lib
