"""Host-side mirror of the reference's hot-path interface over the C ABI.

Same names and argument meaning as /root/reference/src:
    Library.from_reader        library.rs:17     Permuter.new           permutes.rs:47
    Offset.Forward / Reverse   offsetter.rs:10   entropy_offset(_group) offsetter.rs:167,185
    Counter.new / get_value / total_reads / matched_reads               counter.rs:36,71,239,244
Everything that touches reads runs in libsgcount_cuda.so on the GPU; this module only
marshals buffers.  (The production host is the C++ program in sgcount_b200/host; this mirror
exists so the parity tests read like the reference's unit tests.)
"""
from __future__ import annotations

import ctypes as C
import gzip
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

from . import _cabi
from ._cabi import SgcError, check  # noqa: F401


@dataclass(frozen=True)
class Offset:
    """offsetter.rs:10-34"""

    reverse: bool
    index: int

    @staticmethod
    def Forward(i: int) -> "Offset":
        return Offset(False, int(i))

    @staticmethod
    def Reverse(i: int) -> "Offset":
        return Offset(True, int(i))

    def is_forward(self) -> bool:
        return not self.reverse

    def is_reverse(self) -> bool:
        return self.reverse

    def __repr__(self):
        return f"{'Reverse' if self.reverse else 'Forward'}({self.index})"


class ReadBatch:
    """Sequence lines as the kernels consume them: newline-terminated, either fixed stride
    (every read the same length) or with uint32 line offsets."""

    def __init__(self, lines: np.ndarray, n_reads: int, line_off: Optional[np.ndarray] = None,
                 stride: int = 0, read_len: int = 0, ids: Optional[List[bytes]] = None):
        self.lines = np.ascontiguousarray(lines, dtype=np.uint8)
        self.line_off = None if line_off is None else np.ascontiguousarray(line_off, dtype=np.uint32)
        self.n_reads = int(n_reads)
        self.stride = int(stride)
        self.read_len = int(read_len)
        self.ids = ids

    def __len__(self):
        return self.n_reads

    @staticmethod
    def from_seqs(seqs: Sequence[bytes], ids: Optional[List[bytes]] = None, force_offsets: bool = False) -> "ReadBatch":
        n = len(seqs)
        lens = {len(s) for s in seqs}
        buf = np.frombuffer(b"".join(s + b"\n" for s in seqs), dtype=np.uint8)
        if len(lens) == 1 and not force_offsets:
            ln = lens.pop()
            return ReadBatch(buf, n, None, ln + 1, ln, ids)
        off = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum([len(s) + 1 for s in seqs], out=off[1:])
        if n and off[-1] >= 2**32:
            raise ValueError("a variable-length batch must stay below 4 GiB")
        return ReadBatch(buf, n, off.astype(np.uint32), 0, 0, ids)

    def seq(self, i: int) -> bytes:
        if self.line_off is None:
            a = i * self.stride
            return self.lines[a:a + self.read_len].tobytes()
        return self.lines[int(self.line_off[i]):int(self.line_off[i + 1]) - 1].tobytes()

    def take(self, n: int) -> "ReadBatch":
        """Iterator::take(n) (offsetter.rs:173,197)"""
        n = min(n, self.n_reads)
        if self.line_off is None:
            return ReadBatch(self.lines[:n * self.stride], n, None, self.stride, self.read_len)
        end = int(self.line_off[n]) if n else 0
        return ReadBatch(self.lines[:end], n, self.line_off[:n + 1], 0, 0)

    def _args(self):
        off = None if self.line_off is None else self.line_off.ctypes.data
        return (self.lines.ctypes.data, self.lines.nbytes, off, self.stride, self.read_len, self.n_reads)


def read_fastx(path: str) -> ReadBatch:
    """fxread::initialize_reader restated for the test mirror (gzip iff *.gz; '>' = 2-line
    FASTA, '@' = 4-line FASTQ; ids without the marker, sequences raw)."""
    opener = gzip.open if path.endswith(".gz") else open
    with opener(path, "rb") as f:
        lines = f.read().split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()
    if not lines:
        return ReadBatch(np.zeros(0, np.uint8), 0, None, 1, 0, [])
    step = {b">": 2, b"@": 4}[lines[0][:1]]
    ids = [l[1:] for l in lines[0::step]]
    return ReadBatch.from_seqs(lines[1::step], ids)


class _Handle:
    """Owns one sgc_library."""

    def __init__(self, seqs: Sequence[bytes], with_permutations: bool, device: int):
        lib = _cabi.load()
        n = len(seqs)
        k = len(seqs[0]) if n else 0
        flat = np.frombuffer(b"".join(seqs), dtype=np.uint8)
        self.ptr = C.c_void_p()
        check(lib.sgc_library_create(device, flat.ctypes.data, n, k, int(with_permutations), C.byref(self.ptr)))
        self.k = k
        self.n = n
        self.device = device

    def info(self) -> _cabi.LibraryInfo:
        out = _cabi.LibraryInfo()
        check(_cabi.load().sgc_library_get_info(self.ptr, C.byref(out)))
        return out

    def lookup(self, tokens: Sequence[bytes]):
        n = len(tokens)
        flat = np.frombuffer(b"".join(tokens), dtype=np.uint8)
        assert flat.size == n * self.k
        idx = np.empty(n, dtype=np.int32)
        kind = np.empty(n, dtype=np.uint8)
        check(_cabi.load().sgc_library_lookup(self.ptr, flat.ctypes.data, n, idx.ctypes.data, kind.ctypes.data))
        return idx, kind

    def __del__(self):
        try:
            if getattr(self, "ptr", None):
                _cabi.load().sgc_library_destroy(self.ptr)
                self.ptr = None
        except Exception:  # interpreter shutdown
            pass


class Library:
    """library.rs:9-99.  Sequences and aliases stay on the host (they are the table's row
    labels); the device holds the packed table."""

    def __init__(self, seqs: List[bytes], aliases: List[bytes], device: int = 0):
        if len({len(s) for s in seqs}) > 1:
            raise SgcError(-1, "Library sequence sizes are inconsistent")  # library.rs:83
        self._seqs = list(seqs)
        self._aliases = list(aliases)
        self.device = device
        self._exact = _Handle(self._seqs, False, device)  # duplicate / non-ACGT checks happen here

    @staticmethod
    def from_reader(reader: ReadBatch, device: int = 0) -> "Library":
        seqs = [reader.seq(i) for i in range(len(reader))]
        ids = reader.ids if reader.ids is not None else [b"seq.%d" % i for i in range(len(reader))]
        return Library(seqs, ids, device)

    def __len__(self):
        return len(self._seqs)

    def size(self) -> int:
        return len(self._seqs[0])

    def contains(self, token: bytes) -> Optional[bytes]:
        """library.rs:34-40"""
        if len(token) != self.size():
            return None
        idx, _ = self._exact.lookup([token])
        return None if idx[0] < 0 else self._aliases[idx[0]]

    def keys(self) -> List[bytes]:
        return list(self._seqs)

    def values(self) -> List[bytes]:
        return list(self._aliases)


class Permuter:
    """permutes.rs:34-158: the unambiguous one-mismatch variants, as the unified device table."""

    def __init__(self, library: Library):
        self._library = library
        self._handle = _Handle(library._seqs, True, library.device)

    @staticmethod
    def new(library: Library) -> "Permuter":
        return Permuter(library)

    def lookup(self, tokens: Sequence[bytes]):
        """(index, kind) arrays of the composed Library -> Permuter lookup"""
        return self._handle.lookup(tokens)

    def contains(self, token: bytes) -> Optional[bytes]:
        """Parent sequence of a one-mismatch token (permutes.rs:55-57).  Library members
        report None: the reference consults the Library first, so what Permuter::contains
        says about them is never observed (and depends on hash order)."""
        idx, kind = self._handle.lookup([token])
        return self._library._seqs[idx[0]] if kind[0] == 2 else None

    def info(self):
        return self._handle.info()


def span_geometry(k: int, read_len: int, offset: Offset, position_recursion: bool = True):
    """sgc_span_geometry: (start, length) of the span of a `read_len`-byte read — the guide window
    and the byte either side that Counter::assign may look at (counter.rs:164-174) — and the Offset
    under which a counter treats span records as reads with the same outcome."""
    start, length, idx = C.c_uint32(), C.c_uint32(), C.c_uint32()
    check(_cabi.load().sgc_span_geometry(k, read_len, int(offset.reverse), offset.index, int(position_recursion),
                                         C.byref(start), C.byref(length), C.byref(idx)))
    return start.value, length.value, Offset(offset.reverse, idx.value)


def span_batch(reader: ReadBatch, k: int, offset: Offset, position_recursion: bool = True, out: Optional[np.ndarray] = None):
    """Fixed-length reads cut down to span records of stride round_up(length, 8): what a host that
    frames its own records sends instead of whole lines.  Returns (ReadBatch of spans, Offset)."""
    assert reader.line_off is None, "span records need fixed-length reads"
    start, length, span_offset = span_geometry(k, reader.read_len, offset, position_recursion)
    stride = (length + 7) & ~7
    n = reader.n_reads
    rows = reader.lines[:n * reader.stride].reshape(n, reader.stride)
    if out is None:
        out = np.zeros(n * stride, dtype=np.uint8)
    spans = out[:n * stride].reshape(n, stride)
    spans[:, :length] = rows[:, start:start + length]
    return ReadBatch(out[:n * stride], n, None, stride, length), span_offset


def reduce_counts(shards: Sequence["Counter"], root: int = 0) -> None:
    """Sum of the read shards' count vectors into shards[root] (sgc_reduce_counts: NCCL across
    devices, a fold kernel within one) — count.rs:136's collect for a sample cut into shards."""
    arr = (C.c_void_p * len(shards))(*[c._ptr for c in shards])
    check(_cabi.load().sgc_reduce_counts(arr, len(shards), int(root)))
    for c in shards:
        c._result = None


def reduce_prepare(devices: Sequence[int]) -> None:
    """sgc_reduce_prepare: NCCL communicators for these devices; every later reduce_counts of the
    process then goes through NCCL (without it, devices are summed with peer copies)"""
    arr = (C.c_int * len(devices))(*devices)
    check(_cabi.load().sgc_reduce_prepare(arr, len(devices)))


def position_counts(reader: ReadBatch, device: int = 0) -> np.ndarray:
    """offsetter.rs:55-79 on the device -> uint32[size][4]"""
    lib = _cabi.load()
    size = C.c_uint32()
    check(lib.sgc_position_counts(device, *reader._args(), None, 0, C.byref(size)))
    out = np.zeros((size.value, 4), dtype=np.uint32)
    check(lib.sgc_position_counts(device, *reader._args(), out.ctypes.data, size.value, C.byref(size)))
    return out


def entropy_offset(library: Library, reader: ReadBatch, subsample: int = 5000) -> Offset:
    """offsetter.rs:167-180 for one sample (the library entropy lives in the handle)"""
    sub = reader.take(subsample)
    rev, idx = C.c_int(), C.c_uint32()
    check(_cabi.load().sgc_offset_detect(library._exact.ptr, *sub._args(), C.byref(rev), C.byref(idx)))
    return Offset(bool(rev.value), int(idx.value))


def entropy_offset_group(library: Library, readers: Sequence[ReadBatch], subsample: int = 5000) -> List[Offset]:
    """offsetter.rs:185-210"""
    return [entropy_offset(library, r, subsample) for r in readers]


class Counter:
    """counter.rs:17-252"""

    def __init__(self, library: Library, permuter: Optional[Permuter], offset: Offset,
                 position_recursion: bool = True, rc_mode: int = _cabi.RC_BITTRICK,
                 stream: Optional[int] = None, d_state: Optional[int] = None):
        self._library = library
        self._handle = permuter._handle if permuter is not None else library._exact
        self._ptr = C.c_void_p()
        check(_cabi.load().sgc_counter_create(self._handle.ptr, int(offset.reverse), offset.index,
                                              int(position_recursion), rc_mode, stream, d_state, C.byref(self._ptr)))
        self._result = None

    def __del__(self):
        try:
            if getattr(self, "_ptr", None):
                _cabi.load().sgc_counter_destroy(self._ptr)
                self._ptr = None
        except Exception:  # interpreter shutdown
            pass

    @staticmethod
    def new(reader: ReadBatch, library: Library, permuter: Optional[Permuter], offset: Offset,
            size: Optional[int] = None, position_recursion: bool = True, **kw) -> "Counter":
        """Counter::new (counter.rs:36-66): counts the whole reader."""
        assert size is None or size == library.size()
        c = Counter(library, permuter, offset, position_recursion, **kw)
        c.submit(reader)
        c.finish()
        return c

    def submit(self, reader: ReadBatch) -> None:
        """host batch: H2D copies inside the call's pipeline"""
        check(_cabi.load().sgc_counter_submit(self._ptr, *reader._args()))
        self._result = None

    def submit_device(self, d_lines: int, n_bytes: int, n_reads: int, stride: int = 0, read_len: int = 0,
                      d_line_off: Optional[int] = None, d_assign_out: Optional[int] = None) -> None:
        check(_cabi.load().sgc_counter_submit_device(self._ptr, d_lines, n_bytes, d_line_off, stride, read_len,
                                                     n_reads, d_assign_out))
        self._result = None

    def set_replicas(self, replicas: int) -> None:
        """override the skew plan: 0 = automatic (default), 1 = never, >1 = that many copies of the
        count vector"""
        check(_cabi.load().sgc_counter_set_replicas(self._ptr, int(replicas)))

    def wait_copies(self, keep_in_flight: int = 0) -> None:
        check(_cabi.load().sgc_counter_wait_copies(self._ptr, int(keep_in_flight)))

    def sync(self) -> None:
        check(_cabi.load().sgc_counter_sync(self._ptr))

    def reset(self) -> None:
        check(_cabi.load().sgc_counter_reset(self._ptr))
        self._result = None

    def finish(self):
        if self._result is None:
            counts = np.zeros(len(self._library), dtype=np.uint64)
            total, matched = C.c_uint64(), C.c_uint64()
            check(_cabi.load().sgc_counter_finish(self._ptr, counts.ctypes.data, C.byref(total), C.byref(matched)))
            self._result = (counts, int(total.value), int(matched.value))
        return self._result

    def state(self):
        """(device pointer, words) of counts[n] + total + matched"""
        p, n = C.c_void_p(), C.c_uint64()
        check(_cabi.load().sgc_counter_state(self._ptr, C.byref(p), C.byref(n)))
        return p.value, int(n.value)

    def launch_info(self) -> _cabi.LaunchInfo:
        out = _cabi.LaunchInfo()
        check(_cabi.load().sgc_counter_launch_info(self._ptr, C.byref(out)))
        return out

    def counts_by_index(self) -> np.ndarray:
        return self.finish()[0]

    def get_value(self, alias: bytes) -> int:
        """counter.rs:71-76: results are keyed by alias; sequences sharing one are summed"""
        counts = self.finish()[0]
        return int(sum(int(c) for c, a in zip(counts, self._library._aliases) if a == alias))

    def total_reads(self) -> int:
        return self.finish()[1]

    def matched_reads(self) -> int:
        return self.finish()[2]

    def fraction_mapped(self) -> float:
        return self.matched_reads() / self.total_reads()


def bgzf_blocks(blob: bytes):
    """(begin offsets [n + 1], ISIZE [n]) of the blocks of a BGZF file (the 'BC' extra subfield
    holds the block size - 1), or None when the bytes are not BGZF."""
    begin, isize, pos, n = [], [], 0, len(blob)
    while pos < n:
        if n - pos < 28 or blob[pos:pos + 4] != b"\x1f\x8b\x08\x04":
            return None
        xlen = int.from_bytes(blob[pos + 10:pos + 12], "little")
        extra, bsize, at = blob[pos + 12:pos + 12 + xlen], None, 0
        while at + 4 <= len(extra):
            slen = int.from_bytes(extra[at + 2:at + 4], "little")
            if extra[at:at + 2] == b"BC" and slen == 2:
                bsize = int.from_bytes(extra[at + 4:at + 6], "little") + 1
            at += 4 + slen
        if bsize is None or pos + bsize > n:
            return None
        begin.append(pos)
        isize.append(int.from_bytes(blob[pos + bsize - 4:pos + bsize], "little"))
        pos += bsize
    begin.append(pos)
    return np.array(begin, dtype=np.uint64), np.array(isize, dtype=np.uint32)


class FastqStream:
    """sgc_fastq_stream: BGZF blocks of a FASTQ (or one single-member gzip file) inflated, framed and counted on the device.
    read_len > 0: fixed-length reads, `counter` created with the span Offset of span_geometry();
    read_len == 0: reads of any length, `counter` an ordinary counter."""

    def __init__(self, counter: Counter, read_len: int, span_start: int, span_len: int):
        self._counter = counter
        self._ptr = C.c_void_p()
        check(_cabi.load().sgc_fastq_stream_create(counter._ptr, read_len, span_start, span_len, C.byref(self._ptr)))

    def __del__(self):
        try:
            if getattr(self, "_ptr", None):
                _cabi.load().sgc_fastq_stream_destroy(self._ptr)
                self._ptr = None
        except Exception:  # interpreter shutdown
            pass

    def submit(self, blob: np.ndarray, begin: np.ndarray, isize: np.ndarray) -> None:
        """one wave: blocks begin[i]..begin[i+1] of `blob` (uint8), consecutive, in file order"""
        begin = np.ascontiguousarray(begin, dtype=np.uint64)
        isize = np.ascontiguousarray(isize, dtype=np.uint32)
        assert len(begin) == len(isize) + 1
        check(_cabi.load().sgc_fastq_stream_submit(self._ptr, blob.ctypes.data, begin.ctypes.data, isize.ctypes.data, len(isize)))
        self._counter._result = None

    def submit_member(self, blob: np.ndarray) -> None:
        """a whole single-member gzip file (uint8), decoded in parallel pieces on the device; call once,
        then finish().  SgcError(ERR_GZIP) when the device declines it (count it on the host instead)"""
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        check(_cabi.load().sgc_fastq_stream_submit_member(self._ptr, blob.ctypes.data, len(blob)))
        self._counter._result = None

    def submit_gzip(self, blob: np.ndarray) -> None:
        """a whole gzip file (uint8) of one or more members, BGZF included, decoded in parallel pieces on
        the device; call once, then finish().  SgcError(ERR_GZIP) when the device declines it (count it
        on the host instead)"""
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        check(_cabi.load().sgc_fastq_stream_submit_gzip(self._ptr, blob.ctypes.data, len(blob)))
        self._counter._result = None

    def gzip_members(self) -> int:
        """members decoded by submit_gzip (1 after submit_member)"""
        v = C.c_uint64()
        check(_cabi.load().sgc_fastq_stream_gzip_members(self._ptr, C.byref(v)))
        return int(v.value)

    def member_stats(self) -> tuple:
        """(candidate pieces, pieces on the chain of block boundaries, candidates run past) of submit_member
        or submit_gzip, summed over the members"""
        v = [C.c_uint64() for _ in range(3)]
        check(_cabi.load().sgc_fastq_stream_member_stats(self._ptr, *[C.byref(x) for x in v]))
        return tuple(int(x.value) for x in v)

    def finish(self) -> int:
        n = C.c_uint64()
        check(_cabi.load().sgc_fastq_stream_finish(self._ptr, C.byref(n)))
        self._counter._result = None
        return int(n.value)


def submit_gzip_split(streams: Sequence[FastqStream], blob: np.ndarray) -> None:
    """one whole gzip file (uint8), as FastqStream.submit_gzip, decoded by several fresh streams together
    (sgc_fastq_stream_submit_gzip_split), on one device or several; wave k of the text goes to
    streams[k % len(streams)].  Then sum the streams' counters with reduce_counts and call finish() on
    every stream: their records add up to the file's.  SgcError(ERR_GZIP) when the device declines it
    (every stream has then failed: count the file on the host instead)"""
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    arr = (C.c_void_p * len(streams))(*[s._ptr for s in streams])
    check(_cabi.load().sgc_fastq_stream_submit_gzip_split(arr, len(streams), blob.ctypes.data, len(blob)))
    for s in streams:
        s._counter._result = None


def device_memory(device: int = 0):
    """(free, total) bytes of a device's memory"""
    free, total = C.c_uint64(), C.c_uint64()
    check(_cabi.load().sgc_device_memory(int(device), C.byref(free), C.byref(total)))
    return int(free.value), int(total.value)


def fastq_stream_scratch_bound(bgzf: bool, gz_bytes: int, text_bytes: int, read_len: int, span_len: int) -> int:
    """the most device scratch one FastqStream allocates (sgc_fastq_stream_scratch_bound): BGZF waves of at most
    gz_bytes / text_bytes, or a gzip file of gz_bytes whose text is text_bytes (0: unknown)"""
    out = C.c_uint64()
    check(_cabi.load().sgc_fastq_stream_scratch_bound(1 if bgzf else 0, int(gz_bytes), int(text_bytes), int(read_len),
                                                      int(span_len), C.byref(out)))
    return int(out.value)
