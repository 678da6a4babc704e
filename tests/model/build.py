"""Builds tests/model/deflate_model.cpp into a shared library (g++) and binds it.  TEST INFRASTRUCTURE.

The library goes to a per-user directory under the system temporary directory, named after a hash of its sources, so
that a read-only checkout can run the tests and concurrent runs never load a half-written file."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "deflate_model.cpp")
HDR = os.path.join(HERE, "..", "..", "hmse_b200", "csrc", "deflate_core.h")


class Params(C.Structure):
    _fields_ = [("hash_bytes", C.c_int), ("chain_own", C.c_int), ("chain_dict", C.c_int), ("lazy", C.c_int),
                ("too_far", C.c_int), ("dict_hash_bits", C.c_int), ("mode", C.c_int), ("min_len", C.c_int), ("hist", C.c_int),
                ("prev0", C.c_int)]


_libs = {}


def build(force=False):
    h = hashlib.sha256()
    for p in (SRC, HDR):
        with open(p, "rb") as f:
            h.update(f.read())
    key = h.hexdigest()[:16]
    if key in _libs and not force:
        return _libs[key]
    out_dir = os.path.join(tempfile.gettempdir(), "hmse_deflate_model_%d" % os.getuid())
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, "libdeflate_model_%s.so" % key)
    if force or not os.path.exists(out):
        tmp = "%s.%d.tmp" % (out, os.getpid())
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", tmp, SRC])
        os.replace(tmp, out)
    lib = C.CDLL(out)
    lib.model_compress.restype = C.c_int64
    lib.model_compress.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(Params), C.c_void_p,
                                   C.c_uint64, C.c_void_p]
    lib.model_compress_long.restype = C.c_int64
    lib.model_compress_long.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.POINTER(Params), C.c_int,
                                        C.c_void_p, C.c_uint64]
    _libs[key] = lib
    return lib
