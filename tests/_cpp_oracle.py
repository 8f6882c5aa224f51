"""TEST INFRASTRUCTURE -- compiles a CPU restatement (tests/*_oracle.cpp) on first use into a temporary directory of its own
and loads it."""
import ctypes as C
import os
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))


def load(name, argtypes):
    """tests/<name>.cpp built as libsvr_<name>.so, with argtypes {function name: [ctypes types]} set."""
    out = os.path.join(tempfile.mkdtemp(prefix=f"svr_{name}_"), f"libsvr_{name}.so")
    # the flags of oracle/Makefile's cpu target (the distro compiler: it has libgomp)
    subprocess.check_call(["/usr/bin/g++", "-O3", "-fopenmp", "-fno-fast-math", "-shared", "-fPIC", "-o", out, os.path.join(HERE, f"{name}.cpp")])
    lib = C.CDLL(out)
    for fn, types in argtypes.items():
        getattr(lib, fn).argtypes = types
    return lib
