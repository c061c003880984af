"""Host builds of the test scaffolding: a tests/*_host.cpp (which compiles a header of subproc_b200/csrc/ with g++) or a
reference in C (tests/*_oracle.c) as a shared object, built once per process into a temporary directory and loaded
with ctypes.

C++ is compiled with -std=c++17, not gnu++17: g++ then contracts no float expression, and only the explicit fmaf
fuses, as on the device."""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
_DIR = tempfile.mkdtemp(prefix="host_build_")
atexit.register(shutil.rmtree, _DIR, True)

_libs = {}


def load(source, defines=()):
    """ctypes.CDLL of tests/<source> compiled with -D<d> for each d in defines (e.g. "OBE_MAX_EMPTIES=12")"""
    key = (source, tuple(defines))
    if key not in _libs:
        out = os.path.join(_DIR, "lib%d.so" % len(_libs))
        cc, std, libs = ("gcc", "-std=c99", ["-lm"]) if source.endswith(".c") else ("g++", "-std=c++17", [])
        subprocess.check_call([cc, "-O2", std, "-shared", "-fPIC"] + ["-D" + d for d in defines] +
                              [os.path.join(HERE, source), "-o", out] + libs)
        _libs[key] = ctypes.CDLL(out)
    return _libs[key]
