"""ctypes binding of libsgcount_cuda.so (include/sgcount_cuda.h).

The library is built in-tree by ``__graft_entry__.build()`` (sgcount_b200/csrc/Makefile).
There is no fallback: if the shared object is missing or no CUDA device answers, every
call raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SGC_CUDA_LIB overrides the path (A/B timing of two builds; tuning only)
SO_PATH = os.environ.get("SGC_CUDA_LIB") or os.path.join(_HERE, "lib", "libsgcount_cuda.so")

OK = 0
ERR_INVALID_ARG = 1
ERR_CUDA = 2
ERR_DUPLICATE_SEQUENCE = 3
ERR_NON_ACGT_LIBRARY = 4
ERR_K_UNSUPPORTED = 5
ERR_READ_TOO_SHORT = 6
ERR_NAN_ENTROPY = 7
ERR_EMPTY_READER = 8
ERR_TOO_MANY_GUIDES = 9
ERR_BATCH_TOO_LARGE = 10
ERR_NCCL = 11
ERR_GZIP = 12
ERR_FASTQ_FORMAT = 13

RC_BITTRICK = 0
RC_KEEP_N = 1


class SgcError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"[sgc {code}] {msg}")
        self.code = code


class LibraryInfo(C.Structure):
    _fields_ = [
        ("n_guides", C.c_uint32),
        ("k", C.c_uint32),
        ("with_permutations", C.c_int32),
        ("device", C.c_int32),
        ("n_variants", C.c_uint64),
        ("n_ambiguous", C.c_uint64),
        ("n_slots", C.c_uint64),
        ("table_bytes", C.c_uint64),
        ("build_ms", C.c_double),
        ("front_left_out", C.c_uint64),
        ("opaque", C.c_int32),
    ]


class LaunchInfo(C.Structure):
    _fields_ = [
        ("grid", C.c_uint32),
        ("block", C.c_uint32),
        ("smem_bytes", C.c_uint32),
        ("kernel", C.c_uint32),
        ("launches_total", C.c_uint64),
        ("replicas", C.c_uint32),
        ("hot_guides", C.c_uint32),
    ]


class UnmatchedInfo(C.Structure):
    _fields_ = [
        ("unmatched", C.c_uint64),
        ("short_reads", C.c_uint64),
        ("non_acgt", C.c_uint64),
        ("overflow", C.c_uint64),
        ("distinct", C.c_uint64),
    ]


class PairInfo(C.Structure):
    _fields_ = [
        ("total", C.c_uint64),
        ("listed", C.c_uint64),
        ("recombined", C.c_uint64),
        ("first_only", C.c_uint64),
        ("second_only", C.c_uint64),
        ("neither", C.c_uint64),
        ("overflow", C.c_uint64),
        ("distinct", C.c_uint64),
    ]


# every symbol include/sgcount_cuda.h declares: name -> (restype, argtypes)
_vp, _u32, _u64, _int = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
SIGNATURES = {
    "sgc_last_error": (C.c_char_p, []),
    "sgc_abi_version": (_int, []),
    "sgc_device_count": (_int, [C.POINTER(_int)]),
    "sgc_device_memory": (_int, [_int, C.POINTER(_u64), C.POINTER(_u64)]),
    "sgc_host_alloc": (_int, [C.POINTER(_vp), C.c_size_t]),
    "sgc_host_free": (_int, [_vp]),
    "sgc_library_create": (_int, [_int, _vp, _u32, _u32, _int, C.POINTER(_vp)]),
    "sgc_library_destroy": (None, [_vp]),
    "sgc_library_get_info": (_int, [_vp, C.POINTER(LibraryInfo)]),
    "sgc_library_lookup": (_int, [_vp, _vp, _u64, _vp, _vp]),
    "sgc_position_counts": (_int, [_int, _vp, _u64, _vp, _u32, _u32, _u64, _vp, _u32, C.POINTER(_u32)]),
    "sgc_offset_detect": (_int, [_vp, _vp, _u64, _vp, _u32, _u32, _u64, C.POINTER(_int), C.POINTER(_u32)]),
    "sgc_span_geometry": (_int, [_u32, _u32, _int, _u32, _int, C.POINTER(_u32), C.POINTER(_u32), C.POINTER(_u32)]),
    "sgc_span_geometry_shift": (_int, [_u32, _u32, _int, _u32, _u32, C.POINTER(_u32), C.POINTER(_u32),
                                        C.POINTER(_u32)]),
    "sgc_counter_create": (_int, [_vp, _int, _u32, _int, _int, _vp, _vp, C.POINTER(_vp)]),
    "sgc_counter_destroy": (None, [_vp]),
    "sgc_counter_submit": (_int, [_vp, _vp, _u64, _vp, _u32, _u32, _u64]),
    "sgc_counter_submit_device": (_int, [_vp, _vp, _u64, _vp, _u32, _u32, _u64, _vp]),
    "sgc_counter_set_replicas": (_int, [_vp, _u32]),
    "sgc_counter_set_max_shift": (_int, [_vp, _u32]),
    "sgc_counter_set_unmatched_report": (_int, [_vp, _u64]),
    "sgc_counter_unmatched": (_int, [_vp, _u64, _vp, _vp, C.POINTER(_u64), C.POINTER(UnmatchedInfo)]),
    "sgc_unmatched_report_bytes": (_int, [_u64, C.POINTER(_u64)]),
    "sgc_counter_sync": (_int, [_vp]),
    "sgc_counter_wait_copies": (_int, [_vp, _u32]),
    "sgc_reduce_counts": (_int, [C.POINTER(_vp), _int, _int]),
    "sgc_reduce_prepare": (_int, [C.POINTER(_int), _int]),
    "sgc_counter_reset": (_int, [_vp]),
    "sgc_counter_finish": (_int, [_vp, _vp, C.POINTER(_u64), C.POINTER(_u64)]),
    "sgc_counter_state": (_int, [_vp, C.POINTER(_vp), C.POINTER(_u64)]),
    "sgc_fastq_stream_create": (_int, [_vp, _u32, _u32, _u32, C.POINTER(_vp)]),
    "sgc_fastq_stream_destroy": (None, [_vp]),
    "sgc_fastq_stream_submit": (_int, [_vp, _vp, _vp, _vp, _u32]),
    "sgc_fastq_stream_submit_range": (_int, [_vp, _vp, _vp, _vp, _u32, _u32, _u32, _int]),
    "sgc_fastq_stream_submit_member": (_int, [_vp, _vp, _u64]),
    "sgc_fastq_stream_member_stats": (_int, [_vp, C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u64)]),
    "sgc_fastq_stream_submit_gzip": (_int, [_vp, _vp, _u64]),
    "sgc_fastq_stream_submit_gzip_split": (_int, [C.POINTER(_vp), _u32, _vp, _u64]),
    "sgc_fastq_stream_scratch_bound": (_int, [_int, _u64, _u64, _u32, _u32, C.POINTER(_u64)]),
    "sgc_fastq_stream_submit_text": (_int, [_vp, _vp, _u64, _int]),
    "sgc_fastq_stream_text_scratch_bound": (_int, [_u32, _u32, C.POINTER(_u64)]),
    "sgc_fastq_stream_gzip_members": (_int, [_vp, C.POINTER(_u64)]),
    "sgc_fastq_stream_finish": (_int, [_vp, C.POINTER(_u64)]),
    "sgc_counter_launch_info": (_int, [_vp, C.POINTER(LaunchInfo)]),
    "sgc_pair_counter_create": (_int, [_vp, _vp, _vp, _vp, _u64, _u64, C.POINTER(_vp)]),
    "sgc_pair_counter_destroy": (None, [_vp]),
    "sgc_pair_counter_submit": (_int, [_vp, _vp, _u64, _vp, _u32, _u32, _vp, _u64, _vp, _u32, _u32, _u64]),
    "sgc_pair_counter_submit_device": (_int, [_vp, _vp, _u64, _vp, _u32, _u32, _vp, _u64, _vp, _u32, _u32, _u64]),
    "sgc_pair_counter_wait_copies": (_int, [_vp, _u32]),
    "sgc_pair_counter_finish": (_int, [_vp, _vp, C.POINTER(PairInfo)]),
    "sgc_pair_counter_recombinants": (_int, [_vp, _u64, _vp, _vp, _vp, C.POINTER(_u64)]),
    "sgc_pair_counter_reset": (_int, [_vp]),
    "sgc_pair_counter_bytes": (_int, [_u64, _u64, C.POINTER(_u64)]),
}

_lib = None


def load() -> C.CDLL:
    """Loads the shared object (no CUDA call is made)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(
                f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback for the sgcount CUDA path)")
        lib = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            if os.environ.get("SGC_CUDA_LIB") and not hasattr(lib, name):
                continue  # A/B timing against an older build (tuning only)
            fn = getattr(lib, name)  # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        if lib.sgc_abi_version() != 2:
            raise ImportError("libsgcount_cuda.so ABI version mismatch")
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != OK:
        raise SgcError(rc, load().sgc_last_error().decode(errors="replace"))
