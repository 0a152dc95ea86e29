"""sgcount_b200 — B200-native (sm_100a) read->guide matching and counting path of sgcount.

The product is libsgcount_cuda.so (C ABI: include/sgcount_cuda.h) plus the C++ host in
sgcount_b200/host.  This package is the thin ctypes mirror the tests and bench.py drive.
"""
from ._cabi import SgcError  # noqa: F401
from .api import (Counter, FastqStream, bgzf_blocks, device_memory, fastq_stream_scratch_bound, Library, Offset, Permuter, ReadBatch, entropy_offset,  # noqa: F401
                  entropy_offset_group, position_counts, read_fastx, reduce_counts, reduce_prepare, span_batch, span_geometry,
                  submit_gzip_split)
