"""ctypes binding of libfrisk_b200.so (C ABI: include/frisk_b200.h).

The library is built in-tree by ``frisk_b200/csrc/Makefile`` (``__graft_entry__.build()``).
There is no CPU fallback: a missing library raises ImportError-like RuntimeError here, and
every device entry point raises when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("FRISK_B200_LIB") or os.path.join(HERE, "libfrisk_b200.so")   # override: load another build (A/B of two commits in one GPU call)

OK, E_INVALID, E_UNSUPPORTED, E_CUDA, E_NO_DEVICE, E_CAPACITY, E_FORMAT = 0, -1, -2, -3, -4, -5, -6
ROW_KLD_ZERODIV, ROW_GC_ZERODIV, ROW_LOG_DOMAIN, ROW_EXCLUDED = 1, 2, 4, 8
MAX_K = 12
MAX_WINDOW = 0x7FFFFFFF
MAX_BACKGROUNDS = 8                                       # FRISK_B200_MAX_BACKGROUNDS
FORMAT = {"text": 0, "bgzf": 1, "gzip": 2, "2bit": 3}     # FRISK_FORMAT_*

_p = C.c_void_p
_u64 = C.c_uint64
_i = C.c_int

# name -> (restype, argtypes); mirrors include/frisk_b200.h one to one
PROTOTYPES = {
    "frisk_b200_strerror": (C.c_char_p, [_i]),
    "frisk_b200_last_cuda_error": (C.c_char_p, []),
    "frisk_b200_abi_version": (_i, []),
    "frisk_b200_device_count": (_i, []),
    "frisk_b200_table_size": (_u64, [_i, _i]),
    "frisk_b200_fasta_scan": (_i, [_p, _u64, _u64, _p, _p, _p, _p, _p, _p]),
    "frisk_b200_pack_layout": (_i, [_p, _u64, _p, _p]),
    "frisk_b200_pack": (_i, [_p, _p, _p, _p, _p, _u64, _u64, _p, _p, _p, _p, _i]),
    "frisk_b200_windows": (_i, [_p, _p, _u64, _i, _i, _i, _u64, _p, _p, _p, _p, _p, _p]),
    "frisk_b200_format_rows": (_i, [_p, _p, _p, _p, _p, _p, _p, _u64, _i, _p, _u64, _p, _i]),
    "frisk_b200_hmm2_fit": (_i, [_p, _u64, _i, C.c_double, C.c_double, _p, _p, _p, _p]),
    "frisk_b200_hmm2_viterbi": (_i, [_p, _u64, _p, _p, _p, _p, _p]),
    "frisk_b200_background": (_i, [_p, _p, _p, _u64, _u64, _i, _i, _p, _p]),
    "frisk_b200_finalize_tables": (_i, [_p, _i, _i, _p, _p, _p]),
    "frisk_b200_finalize_tables_peers": (_i, [_p, _p, _i, _i, _u64, _i, _i, _p, _p, _p]),
    "frisk_b200_finalize_ivom": (_i, [_p, _p, _p, _i, _i, _u64, _i, _i, C.c_int64, _p, _p, _p, _p]),
    "frisk_b200_kld": (_i, [_p, _p, _u64, _p, _p]),
    "frisk_b200_feature_slots": (_i, [_i, _i, _p, _p]),
    "frisk_b200_region_features": (_i, [_p, _p, _p, _p, _u64, _i, _i, _p, _u64, _p, _p]),
    "frisk_b200_score_occupancy": (_i, [_i, C.c_uint32, C.POINTER(_i), C.POINTER(_i)]),
    "frisk_b200_set_option": (_i, [C.c_char_p, _i]),
    "frisk_b200_genome_ivom": (_i, [_p, _i, _i, C.c_int64, _p, _p]),
    "frisk_b200_score": (_i, [_p, _p, _p, _p, _p, _u64, C.c_uint32, _p, _i, _i, _i, _p, _p, _p, _p]),
    "frisk_b200_run_host": (_i, [_p, _p, _p, _u64, _p, _p, _p, _u64, _p, _p, _u64, C.c_uint32, _i, _i, _i, _i,
                                 C.c_int64, _p, _p, _p, _p, _p]),
    "frisk_b200_plane_sparse": (_i, [_p, _u64, _u64, _p, _p, _p]),
    "frisk_b200_run_host_sparse": (_i, [_p, _p, _p, _u64, _p, _u64, _p, _p, _p, _u64, _p, _u64, _p, _p, _u64, C.c_uint32,
                                        _i, _i, _i, _i, C.c_int64, _p, _p, _p, _p, _p]),
    "frisk_b200_run_host_peers": (_i, [_p, _p, _p, _u64, _p, _u64, _p, _p, _u64, C.c_uint32, _i, _i, _i, _i, C.c_int64,
                                       _p, _p, _p, _i, _i, _u64, _p, _p, _p, _p, _p]),
    "frisk_b200_run_resident": (_i, [_p, _p, _p, _u64, _p, _p, _p, _u64, _p, _p, _u64, C.c_uint32, _i, _i, _i, _i,
                                     C.c_int64, _p, _p, _p, _p, _p]),
    "frisk_b200_fasta_open": (_i, [_p, _u64, _p, C.POINTER(C.c_void_p), C.POINTER(_u64), C.POINTER(_u64), _p]),
    "frisk_b200_fasta_records": (_i, [_p, _p, _p, _p, _p]),
    "frisk_b200_fasta_pack": (_i, [_p, _p, _p, _p, _p]),
    "frisk_b200_fasta_close": (_i, [_p, _p]),
    "frisk_b200_fasta_open_stats": (_i, [_p]),
    "frisk_b200_run_fasta": (_i, [_p, _u64, _p, _u64, _i, _i, _i, _i, _i, _i, _i, _u64, _p, _p, _p, _p, C.POINTER(_u64),
                                  C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _p]),
    "frisk_b200_windows_device": (_i, [_p, _p, _u64, _i, _i, _i, _u64, _p, _p, _p, _p, _p]),
    "frisk_b200_fasta_info": (_i, [_p, C.POINTER(_u64), C.POINTER(_u64), _p]),
    "frisk_b200_bgzf_blocks": (_i, [_p, _u64, _u64, _p, _p, _p, _p, C.POINTER(_u64), C.POINTER(_u64)]),
    "frisk_b200_bgzf_inflate": (_i, [_p, _p, _p, _p, _p, _u64, _u64, _p, _p, _p]),
    "frisk_b200_bgzf_inflate_host": (_i, [_p, _p, _p, _p, _p, _u64, _u64, _p, _p, _p]),
    "frisk_b200_fasta_open_bgzf": (_i, [_p, _u64, _p, C.POINTER(C.c_void_p), C.POINTER(_u64), C.POINTER(_u64), _p]),
    "frisk_b200_run_fasta_bgzf": (_i, [_p, _u64, _p, _u64, _i, _i, _i, _i, _i, _i, _i, _u64, _p, _p, _p, _p, C.POINTER(_u64),
                                       C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _p]),
    "frisk_b200_fasta_name_text": (_i, [_p, C.POINTER(C.c_void_p), C.POINTER(_u64)]),
    "frisk_b200_gzip_member": (_i, [_p, _u64, C.POINTER(_u64), C.POINTER(_u64), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "frisk_b200_gzip_inflate": (_i, [_p, _u64, _p, _u64, C.POINTER(_u64), _p, _p]),
    "frisk_b200_gzip_inflate_host": (_i, [_p, _u64, _p, _u64, C.POINTER(_u64), _p, _p]),
    "frisk_b200_fasta_open_gzip": (_i, [_p, _u64, _p, C.POINTER(C.c_void_p), C.POINTER(_u64), C.POINTER(_u64), _p]),
    "frisk_b200_run_fasta_gzip": (_i, [_p, _u64, _p, _u64, _i, _i, _i, _i, _i, _i, _i, _u64, _p, _p, _p, _p, C.POINTER(_u64),
                                       C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _p]),
    "frisk_b200_2bit_records": (_i, [_p, _u64, _u64, _p, _p, _p, C.POINTER(_u64), C.POINTER(_u64)]),
    "frisk_b200_2bit_unpack_host": (_i, [_p, _u64, _u64, _p, _p, _p, _p]),
    "frisk_b200_fasta_open_2bit": (_i, [_p, _u64, _p, C.POINTER(C.c_void_p), C.POINTER(_u64), C.POINTER(_u64), _p]),
    "frisk_b200_run_2bit": (_i, [_p, _u64, _p, _u64, _i, _i, _i, _i, _i, _i, _i, _u64, _p, _p, _p, _p, C.POINTER(_u64),
                                 C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _p]),
    "frisk_b200_fasta_planes": (_i, [_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "frisk_b200_background_open": (_i, [_p, _i, _i, C.c_int64, _p, C.POINTER(C.c_void_p)]),
    "frisk_b200_background_run": (_i, [_p, _p, _u64, _i, _i, _i, _i, _i, _u64, _p, _p, C.POINTER(_u64), C.POINTER(C.c_void_p), _p]),
    "frisk_b200_background_score": (_i, [_p, _p, _p, _p, _u64, _p, _p, _u64, C.c_uint32, _i, _p, _p, _p]),
    "frisk_b200_background_run_many": (_i, [_p, _i, _p, _u64, _i, _i, _i, _i, _i, _u64, _p, _p, C.POINTER(_u64),
                                            C.POINTER(C.c_void_p), _p]),
    "frisk_b200_background_score_many": (_i, [_p, _i, _p, _p, _p, _u64, _p, _p, _u64, C.c_uint32, _i, _p, _p, _p]),
    "frisk_b200_background_close": (_i, [_p, _p]),
    "frisk_b200_last_run_timing": (_i, [C.POINTER(C.c_float), _i, C.POINTER(_i)]),
    "frisk_b200_score_sweep": (_i, [_p, _p, _p, _p, _p, _u64, C.c_uint32, _p, _i, _i, _p, _p, _p]),
    "frisk_b200_score_kernel_name": (_i, [_i, _i, C.c_uint32, C.c_char_p, _u64]),
    "frisk_b200_release_workspace": (_i, []),
    "frisk_b200_device_alloc": (_i, [C.POINTER(C.c_void_p), _u64]),
    "frisk_b200_device_free": (_i, [_p]),
    "frisk_b200_set_device": (_i, [_i]),
    "frisk_b200_host_alloc": (_i, [C.POINTER(C.c_void_p), _u64]),
    "frisk_b200_host_free": (_i, [_p]),
    "frisk_b200_bench_smem_atomics": (_i, [_i, _i, _i, C.POINTER(C.c_float), _p]),
    "frisk_b200_bench_l2_gather": (_i, [_i, _i, _u64, _i, C.POINTER(C.c_float), _p]),
    "frisk_b200_bench_smem_loads": (_i, [_i, _i, _i, C.POINTER(C.c_float), _p]),
}

_LIB = None


class FriskError(RuntimeError):
    def __init__(self, code: int, where: str, detail: str = ""):
        self.code = code
        super().__init__("%s failed: %s%s" % (where, _strerror(code), (" -- " + detail) if detail else ""))


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(frisk_b200 has no CPU fallback)" % SO_PATH)
        L = C.CDLL(SO_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)          # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if L.frisk_b200_abi_version() != 2:
            raise RuntimeError("libfrisk_b200.so ABI version mismatch")
        _LIB = L
    return _LIB


def _strerror(code: int) -> str:
    try:
        return lib().frisk_b200_strerror(code).decode()
    except Exception:
        return "error %d" % code


def check(code: int, where: str) -> None:
    if code != OK:
        detail = lib().frisk_b200_last_cuda_error().decode() if code == E_CUDA else ""
        raise FriskError(code, where, detail)


def device_count() -> int:
    return int(lib().frisk_b200_device_count())


def require_device() -> None:
    if device_count() <= 0:
        raise FriskError(E_NO_DEVICE, "frisk_b200")


def table_size(kmin: int, kmax: int) -> int:
    return int(lib().frisk_b200_table_size(kmin, kmax))
