"""The staggered-read rule (max_shift S >= 2) for the tests: three statements of it that check each
other and the device.  TEST INFRASTRUCTURE, NOT PRODUCT.

* ``assign`` / ``count``: tests/shift_oracle.cpp, a literal loop over positions with byte-string
  lookups through the CPU oracle's Library and Permuter (oracle/oracle.h), compiled on first use
  into a temporary directory and linked against oracle/liboracle.so;
* ``literal_assign_shift``: the same loop in Python over the literal Permuter of oracle_py;
* ``closed_form_assign_shift``: the same loop over oracle_py's closed-form lookup.

S = 1 is the reference's Centered/Plus/Minus recursion and goes to the oracle unchanged (orc_assign,
orc_counter_new).  S >= 2 tries offset + d for d = 0, +1, -1, ..., +S, -S in the coordinates of the
trimmed read; the first window that yields a guide wins; a window that does not fit is skipped."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from typing import Dict, List, Optional, Sequence

import numpy as np

from oracle import oracle as orc
from oracle import oracle_py as P

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "shift_oracle.cpp")
_lib = None


def lib() -> C.CDLL:
    """tests/shift_oracle.cpp built against oracle/liboracle.so (outside the tree: a temporary directory)"""
    global _lib
    if _lib is None:
        oracle_so = orc.build()
        orc.lib()
        with open(_SRC, "rb") as f:
            tag = hashlib.sha1(f.read() + str(os.path.getmtime(oracle_so)).encode()).hexdigest()[:12]
        out_dir = os.path.join(tempfile.gettempdir(), f"sgc_shift_oracle_{os.getuid()}_{tag}")
        so = os.path.join(out_dir, "libshift_oracle.so")
        if not os.path.exists(so):
            os.makedirs(out_dir, exist_ok=True)
            tmp = so + f".{os.getpid()}"
            oracle_dir = os.path.dirname(oracle_so)
            subprocess.run([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-o", tmp,
                            _SRC, oracle_so, f"-Wl,-rpath,{oracle_dir}"], check=True, capture_output=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        vp = C.c_void_p
        L.shift_assign.restype = C.c_int64
        L.shift_assign.argtypes = [vp, vp, vp, C.c_size_t, C.c_int, C.c_uint64, C.c_uint32, C.c_int]
        L.shift_assign_records.restype = None
        L.shift_assign_records.argtypes = [vp, vp, vp, C.c_int, C.c_uint64, C.c_uint32, C.c_int, C.c_int, vp]
        _lib = L
    return _lib


def assign(library: orc.Library, permuter: Optional[orc.Permuter], read: bytes, offset: orc.Offset,
           rc_mode: int = orc.RC_BITTRICK, max_shift: int = 1) -> int:
    """one read -> library index or -1"""
    if max_shift < 2:
        return orc.assign(library, permuter, read, offset, True, rc_mode)
    return int(lib().shift_assign(library._h, permuter._h if permuter else None, C.c_char_p(read), len(read),
                                  int(offset.reverse), offset.index, max_shift, rc_mode))


def count(records: orc.Records, library: orc.Library, permuter: Optional[orc.Permuter], offset: orc.Offset,
          rc_mode: int = orc.RC_BITTRICK, max_shift: int = 1, n_threads: int = 8):
    """(assignments, counts by library index, total_reads, matched_reads) of a record set.  Counts are
    by index (the tests' libraries have one alias per sequence)."""
    if max_shift < 2:
        c = orc.Counter.new(records, library, permuter, offset, rc_mode=rc_mode, n_threads=n_threads,
                            want_assignments=True)
        return c.assignments, c.counts_by_index(), c.total_reads(), c.matched_reads()
    a = np.empty(len(records), dtype=np.int32)
    lib().shift_assign_records(records._h, library._h, permuter._h if permuter else None, int(offset.reverse),
                               offset.index, max_shift, rc_mode, n_threads, a.ctypes.data)
    counts = np.bincount(a[a >= 0], minlength=len(library)).astype(np.uint64)
    return a, counts, len(a), int((a >= 0).sum())


def shift_order(max_shift: int) -> List[int]:
    """displacements tried: 0, +1, -1, ..., +S, -S"""
    out = [0]
    for d in range(1, max_shift + 1):
        out += [d, -d]
    return out


def literal_assign_shift(read: bytes, library: Dict[bytes, bytes], permuter: Optional[P.LiteralPermuter],
                         reverse: bool, offset: int, size: int, max_shift: int, bittrick: bool = True) -> Optional[bytes]:
    """-> alias or None, over the literal Permuter (S = 1: oracle_py.literal_assign)"""
    if max_shift < 2:
        return P.literal_assign(read, library, permuter, reverse, offset, size, True, bittrick)
    src = P.rev_comp(read, bittrick) if reverse else read
    for d in shift_order(max_shift):
        lo = offset + d
        if lo < 0 or lo + size > len(src):
            continue
        token = src[lo:lo + size]
        if token in library:
            return library[token]
        if permuter is not None:
            parent = permuter.contains(token)
            if parent is not None and parent in library:
                return library[parent]
    return None


def closed_form_assign_shift(read: bytes, lib_seqs: Sequence[bytes], with_permuter: bool, reverse: bool,
                             offset: int, max_shift: int, bittrick: bool = True) -> int:
    """-> library index or -1, over the closed-form lookup (S = 1: oracle_py.closed_form_assign)"""
    if max_shift < 2:
        return P.closed_form_assign(read, lib_seqs, with_permuter, reverse, offset, True, bittrick)
    size = len(lib_seqs[0])
    src = P.rev_comp(read, bittrick) if reverse else read
    for d in shift_order(max_shift):
        lo = offset + d
        if lo < 0 or lo + size > len(src):
            continue
        hit = P.closed_form_lookup(src[lo:lo + size], lib_seqs, with_permuter)
        if hit >= 0:
            return hit
    return -1
