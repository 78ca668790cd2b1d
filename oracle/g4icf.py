"""ctypes binding of the integer-coded float mapping of the CPU oracle (oracle/g4o_icf.cpp).  TEST INFRASTRUCTURE ONLY.

The two functions restate the ICF mapping as the ICF feature request gives it (GvrsElementSpecificationIntCodedFloat /
GvrsElementIntCodedFloat); no reference fixture pins it beyond exactly representable values.  The source is compiled on
first use with the flags of the rest of the oracle (-ffp-contract=off: the float32 subtraction and multiplication must not
be fused) into a temporary directory, so that nothing is written into the tree.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "g4o_icf.cpp")
INT4_NULL_CODE = -(2**31)
_lib = None


def build():
    """Compiles g4o_icf.cpp (once per source version) and returns the path of the shared object."""
    src = open(_SRC, "rb").read()
    out_dir = os.path.join(tempfile.gettempdir(), "g4icf-%d" % os.getuid())
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libg4icf-%s.so" % hashlib.sha256(src).hexdigest()[:16])
    if not os.path.exists(so):
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=out_dir)
        os.close(fd)
        cxx = os.environ.get("CXX", "g++")
        subprocess.check_call([cxx, "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra", "-shared",
                               "-o", tmp, _SRC])
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.g4o_icf_to_int.argtypes = [C.c_void_p, C.c_long, C.c_float, C.c_float, C.c_int32, C.c_void_p]
        L.g4o_icf_to_float.argtypes = [C.c_void_p, C.c_long, C.c_float, C.c_float, C.c_int32, C.c_float, C.c_void_p]
        _lib = L
    return _lib


def icf_to_int(values, scale, offset=0.0, fill_int=INT4_NULL_CODE):
    """float -> code: NaN -> fill_int; else (int) Math.floor((double)((v - offset) * scale) + 0.5) (float32 subtract and
    multiply, double + 0.5 and floor, Java's saturating cast).  Same shape as `values`, int32."""
    v = np.ascontiguousarray(values, dtype=np.float32)
    out = np.empty(v.shape, np.int32)
    lib().g4o_icf_to_int(v.ctypes.data, v.size, float(scale), float(offset), int(fill_int), out.ctypes.data)
    return out


def icf_to_float(codes, scale, offset=0.0, fill_int=INT4_NULL_CODE, fill_value=float("nan")):
    """code -> float: fill_int -> fill_value; else (float) code / scale + offset in float32.  Same shape as `codes`."""
    k = np.ascontiguousarray(codes, dtype=np.int32)
    out = np.empty(k.shape, np.float32)
    lib().g4o_icf_to_float(k.ctypes.data, k.size, float(scale), float(offset), int(fill_int), float(fill_value), out.ctypes.data)
    return out
