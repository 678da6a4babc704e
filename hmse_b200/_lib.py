"""ctypes binding of libhmse_b200.so (the C ABI in include/hmse.h).  There is no fallback:
if the library is missing or a call fails, an exception is raised."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libhmse_b200.so")

HMSE_OK, HMSE_E_INVAL, HMSE_E_CAPACITY, HMSE_E_CUDA, HMSE_E_NOMEM, HMSE_E_NCCL = 0, -1, -2, -3, -4, -5
ABI_VERSION = 6


class HmseError(RuntimeError):
    def __init__(self, code: int, text: str):
        super().__init__("hmse error %d: %s" % (code, text))
        self.code = code


class CdcCfg(C.Structure):
    _fields_ = [("min_size", C.c_uint32), ("avg_size", C.c_uint32), ("max_size", C.c_uint32),
                ("reserved", C.c_uint32), ("mask_s", C.c_uint64), ("mask_l", C.c_uint64),
                ("gear", C.c_uint64 * 256)]


class ComposeSrc(C.Structure):
    _fields_ = [("d_layout", C.c_void_p), ("d_index", C.c_void_p), ("d_pointers", C.c_void_p), ("d_store", C.c_void_p),
                ("d_delta_store", C.c_void_p), ("n", C.c_uint64), ("m", C.c_uint64), ("n_delta", C.c_uint64)]


class CorpusCfg(C.Structure):
    _fields_ = [("seed", C.c_uint32), ("dup_thr", C.c_uint32), ("near_thr", C.c_uint32), ("n_lex", C.c_uint32),
                ("pick_tries", C.c_uint32)]


_P, _U64, _U32, _I = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
_PU64 = C.POINTER(C.c_uint64)

# name -> (restype, argtypes); every symbol include/hmse.h declares
SIGNATURES = {
    "hmse_abi_version": (_I, []),
    "hmse_create": (_I, [_I, C.POINTER(_P)]),
    "hmse_destroy": (None, [_P]),
    "hmse_last_error": (C.c_char_p, [_P]),
    "hmse_scratch_bytes": (_U64, [_P]),
    "hmse_guard_check": (_I, [_P]),
    "hmse_chunk": (_I, [_P, _P, _U64, C.POINTER(CdcCfg), _P, _U64, _PU64, _P]),
    "hmse_chunk_files": (_I, [_P, _P, _U64, _P, _U64, C.POINTER(CdcCfg), _P, _U64, _PU64, _P, _P]),
    "hmse_chunk_scan": (_I, [_P, _P, _U64, C.POINTER(CdcCfg), _P]),
    "hmse_chunk_resolve": (_I, [_P, _P, _U64, _U64, _I, _U64, _P, _U64, _PU64, _PU64, _P]),
    "hmse_chunk_candidates": (_I, [_P, _P, _P, _U64, _P]),
    "hmse_chunk_last_rounds": (_I, [_P]),
    "hmse_digest": (_I, [_P, _P, _U64, _P, _U64, _P, _P]),
    "hmse_dedup": (_I, [_P, _P, _U64, _P, _P, _P]),
    "hmse_dedup_select": (_I, [_P, _P, _U64, _P, _U64, _PU64, _P]),
    "hmse_dedup_begin": (_I, [_P, _U64, _P]),
    "hmse_dedup_append": (_I, [_P, _P, _U64, _U64, _P, _P, _P]),
    "hmse_timing": (_I, [_P, _I]),
    "hmse_timing_ms": (_I, [_P, _I, C.POINTER(C.c_float)]),
    "hmse_launch_count": (_U64, [_P]),
    "hmse_compress_stats": (_I, [_P, _PU64, C.POINTER(C.c_float), C.POINTER(C.c_uint32)]),
    "hmse_dedup_partition": (_I, [_P, _P, _U64, _U64, _U32, _P, _P, _PU64, _P]),
    "hmse_dedup_records": (_I, [_P, _P, _U64, _P, _P]),
    "hmse_dedup_scatter": (_I, [_P, _P, _P, _U64, _U64, _P, _P, _P]),
    "hmse_compress_bound": (_U64, [_U64]),
    "hmse_compress": (_I, [_P, _P, _U64, _P, _P, _U64, _P, _U32, _I, _P, _U64, _P, _PU64, _P]),
    "hmse_compress_pack": (_I, [_P, _P, _U64, _P, _U64, _P]),
    "hmse_debug_deflate_prof": (_I, [_PU64, _I]),
    "hmse_index_build": (_I, [_P, _P, _P, _U64, _P, _U64, _U64, _P, _U64, _P, _P, _P, _P]),
    "hmse_index_build_l4": (_I, [_P, _P, _P, _P, _U64, _U64, _P, _U64, _P, _P, _P, _P, _P, _P, _P, _U64, _PU64, _P]),
    "hmse_segment_copy": (_I, [_P, _P, _P, _P, _P, _U64, _P]),
    "hmse_inflate": (_I, [_P, _P, _P, _U64, _P, _U32, _P, _P, _P, _PU64, _P]),
    "hmse_read_layout_bytes": (_U64, [_U64, _U64, _U64]),
    "hmse_read_open": (_I, [_P, _P, _U64, _P, _U64, _U64, _P, _U64, _U64, _U64, _P, _U32, _P, _U64, _P]),
    "hmse_read": (_I, [_P, _P, _U64, _U64, _U64, _P, _P, _P, _U32, _P, _U64, _P, _U64, _P, _PU64, _P, _PU64, _PU64, _P]),
    "hmse_compose": (_I, [_P, C.POINTER(ComposeSrc), _U32, _P, _U64, _U64, _P, _P, _U64, _P, _U64, _P, _U64, _PU64, _P]),
    "hmse_compress_known": (_I, [_P, C.POINTER(ComposeSrc), _P, _U64, _P, _P, _P, _U64, _P, _U32, _I, _P, _U64, _P, _PU64, _P,
                                 _PU64, _P]),
    "hmse_compress_known_pack": (_I, [_P, _P, _U64, _P, _U64, _P]),
    "hmse_minhash": (_I, [_P, _P, _U64, _P, _U64, _P, _U32, _P, _P]),
    "hmse_minhash_select": (_I, [_P, _P, _U64, _P, _P, _U64, _P, _U32, _P, _P]),
    "hmse_lsh_keys": (_I, [_P, _P, _U64, _U32, _U32, _P, _P]),
    "hmse_lsh_buckets": (_I, [_P, _P, _U64, _U32, _U64, _P, _P, _P, _P]),
    "hmse_delta_bases": (_I, [_P, _P, _P, _P, _U64, _U32, _U64, _P, _U32, _P, _P]),
    "hmse_delta_encode": (_I, [_P, _P, _U64, _P, _U64, _P, _P, _U64, _P, _PU64, _P]),
    "hmse_delta_apply": (_I, [_P, _P, _P, _U64, _P, _U64, _P, _P, _P, _P, _P, _PU64, _P]),
    "hmse_comm_unique_id": (_I, [_P]),
    "hmse_comm_init": (_I, [_P, _P, _I, _I]),
    "hmse_comm_destroy": (_I, [_P]),
    "hmse_comm_info": (_I, [_P, _P, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "hmse_allgather_u64": (_I, [_P, _P, _PU64, _PU64, _P]),
    "hmse_chunk_sharded": (_I, [_P, _P, _P, _U64, _U64, _I, C.POINTER(CdcCfg), _P, _U64, _PU64, _PU64, _PU64, _PU64, _P]),
    "hmse_dedup_global": (_I, [_P, _P, _P, _U64, _U64, _P, _P, _P]),
    "hmse_lsh_exchange": (_I, [_P, _P, _P, _U64, _U32, _P, _U64, _PU64, _PU64, C.POINTER(_U32), _P]),
    "hmse_alltoallv": (_I, [_P, _P, _P, _PU64, _P, _PU64, _U32, _U64, _P]),
    "hmse_delta_heads": (_I, [_P, _P, _P, _P, _U64, _U32, _U64, _P, _P, _P]),
    "hmse_delta_votes": (_I, [_P, _P, _U64, _U32, _U64, _U32, _I, _P, _P, _P, _P]),
    "hmse_delta_encode_ext": (_I, [_P, _P, _U64, _P, _U64, _P, _P, _P, _U64, _P, _U64, _P, _PU64, _P]),
    "hmse_exchange_stats": (_I, [_P, _PU64, C.POINTER(_I)]),
    "hmse_corpus_lengths": (_I, [_P, C.POINTER(CorpusCfg), _P, _U64, _U64, _P, _P]),
    "hmse_corpus_render": (_I, [_P, C.POINTER(CorpusCfg), _P, _P, _U64, _U64, _P, _U64, _U64, _P, _P]),
}

_lib = None


def load() -> C.CDLL:
    """Loads the in-tree shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s is missing - build it with `python -m hmse_b200.build` (nvcc, sm_100a); "
                              "hmse_b200 has no CPU fallback" % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the build is stale
            fn.restype = res
            fn.argtypes = args
        if lib.hmse_abi_version() != ABI_VERSION:
            raise ImportError("libhmse_b200.so ABI %d != binding ABI %d" % (lib.hmse_abi_version(), ABI_VERSION))
        _lib = lib
    return _lib
