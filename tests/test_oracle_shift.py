"""The staggered-read rule (max_shift S >= 2) without a device: its C++ statement over the oracle's
lookups (tests/shift_oracle.cpp) and its two Python statements check each other, S = 1 is the
reference's Counter::assign, and the span geometry of the new entry point equals the old one at S = 1.

S >= 2 is this project's own specification (the reference only has S = 1), so it cannot be pinned
to reference vectors; two independent statements of it must agree instead."""
import random

import numpy as np
import pytest

from oracle import oracle as O
from oracle import oracle_py as P

import shift_oracle as SO

BASES = b"ACGT"


def _rand_seq(rng, n, alphabet=BASES):
    return bytes(rng.choice(alphabet) for _ in range(n))


def _library(rng, n, k):
    seqs = set()
    while len(seqs) < n:
        seqs.add(_rand_seq(rng, k))
    return sorted(seqs)


def _mutate(rng, s, n_mut, alphabet=b"ACGTN"):
    s = bytearray(s)
    for _ in range(n_mut):
        i = rng.randrange(len(s))
        s[i] = rng.choice([c for c in alphabet if c != s[i]])
    return bytes(s)


def _reads(rng, lib, k, offset, max_shift, reverse, bittrick, n_reads):
    """reads with a guide (exact, one mismatch, one N, or two mismatches) planted at offset + d for
    |d| <= S + 1 in the trimmed read's coordinates, junk reads, N-rich reads, windows flush with
    either end of the read and reads shorter than offset + k"""
    out = []
    for _ in range(n_reads):
        kind = rng.random()
        d = rng.randint(-max_shift - 1, max_shift + 1)
        start = max(0, offset + d)
        if kind < 0.1:
            length = rng.randint(max(1, k - 2), offset + k)  # shorter than offset + k
        elif kind < 0.2:
            length = start + k  # window flush with the read's end
        else:
            length = max(start + k, offset + k) + rng.randint(0, max_shift + 3)
        read = bytearray(_rand_seq(rng, length, b"ACGTN" if rng.random() < 0.1 else BASES))
        if kind >= 0.05 and start + k <= length:
            g = rng.choice(lib)
            r = rng.random()
            g = g if r < 0.5 else _mutate(rng, g, 1 if r < 0.85 else 2)
            read[start:start + k] = g
            if rng.random() < 0.3:  # a second, different guide elsewhere: the order decides
                s2 = rng.randint(0, max(0, length - k))
                read[s2:s2 + k] = rng.choice(lib)
        read = bytes(read)
        if reverse:  # what is stored is the reverse complement of the trimmed read
            read = P.rev_comp(read, bittrick)
        out.append(read)
    return out


@pytest.mark.parametrize("max_shift", [2, 3, 8, 16])
@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("rc_mode", [O.RC_BITTRICK, O.RC_KEEP_N])
@pytest.mark.parametrize("permuter", [True, False])
def test_oracle_equals_python_twin(max_shift, reverse, rc_mode, permuter):
    rng = random.Random(hash((max_shift, reverse, rc_mode, permuter)) & 0xFFFF)
    k = rng.choice([5, 8, 12, 20])
    lib_seqs = _library(rng, 40, k)
    records = O.Records.from_seqs(lib_seqs)
    library = O.Library.from_reader(records)
    perm = O.Permuter.new(library) if permuter else None
    lit_perm = P.LiteralPermuter(lib_seqs) if permuter else None
    lib_map = {s: library.alias_at(i) for i, s in enumerate(lib_seqs)}
    bittrick = rc_mode == O.RC_BITTRICK
    for offset in (0, 1, max_shift - 1, max_shift + 2):
        reads = _reads(rng, lib_seqs, k, offset, max_shift, reverse, bittrick, 150)
        off = O.Offset(reverse, offset)
        assignments, counts, total, matched = SO.count(O.Records.from_seqs(reads), library, perm, off, rc_mode=rc_mode,
                                                       max_shift=max_shift)
        want = []
        for i, read in enumerate(reads):
            got = SO.assign(library, perm, read, off, rc_mode=rc_mode, max_shift=max_shift)
            closed = SO.closed_form_assign_shift(read, lib_seqs, permuter, reverse, offset, max_shift, bittrick)
            literal = SO.literal_assign_shift(read, lib_map, lit_perm, reverse, offset, k, max_shift, bittrick)
            assert got == closed, (read, offset)
            assert (literal is None) == (got < 0)
            if got >= 0:
                assert literal == library.alias_at(got)
            assert assignments[i] == got
            want.append(got)
        want = np.array(want)
        assert total == len(reads)
        assert matched == int((want >= 0).sum())
        assert np.array_equal(counts, np.bincount(want[want >= 0], minlength=len(lib_seqs)).astype(np.uint64))


def test_order_of_positions():
    """a one-mismatch hit at +1 beats an exact hit at +2, +d beats -d, and a window that does not
    fit is skipped rather than ending the search"""
    lib_seqs = [b"ACGTACGT", b"TTGGCCAA", b"GATTACAG", b"TGATTACC"]
    library = O.Library.from_reader(O.Records.from_seqs(lib_seqs))
    perm = O.Permuter.new(library)

    def both(read, offset, S, with_perm):
        got = SO.assign(library, perm if with_perm else None, bytes(read), O.Offset(False, offset), max_shift=S)
        assert got == SO.closed_form_assign_shift(bytes(read), lib_seqs, with_perm, False, offset, S)
        return got

    read = bytearray(b"C" * 30)
    read[7:15] = b"GATTACAG"  # d = +2: exact guide 2; d = +1 reads TGATTACA, one mismatch of guide 3
    read[6] = ord("T")
    assert both(read, 5, 2, True) == 3
    assert both(read, 5, 2, False) == 2
    read = bytearray(b"C" * 30)
    read[10:18] = b"TTGGCCAA"  # d = +5
    read[0:8] = b"ACGTACGT"  # d = -5
    assert both(read, 5, 5, False) == 1
    read[10:18] = b"C" * 8
    assert both(read, 5, 5, False) == 0
    # offset 3, S = 8: d = -4 .. -8 do not fit; the search goes on to +5 .. +8
    read = bytearray(b"C" * 30)
    read[10:18] = b"ACGTACGT"  # d = +7
    assert both(read, 3, 8, False) == 0
    # the Centered window does not fit the read, a window before it does
    read = b"CC" + b"TTGGCCAA" + b"C"
    assert both(read, 4, 2, False) == 1
    assert O.assign(library, None, read, O.Offset(False, 4)) == -1


@pytest.mark.parametrize("reverse", [False, True])
def test_shift_one_is_todays_assign(reverse):
    rng = random.Random(7 + reverse)
    k = 10
    lib_seqs = _library(rng, 30, k)
    library = O.Library.from_reader(O.Records.from_seqs(lib_seqs))
    perm = O.Permuter.new(library)
    for offset in (0, 1, 3):
        reads = _reads(rng, lib_seqs, k, offset, 1, reverse, True, 300)
        off = O.Offset(reverse, offset)
        a = O.Counter.new(O.Records.from_seqs(reads), library, perm, off, want_assignments=True)
        b = SO.count(O.Records.from_seqs(reads), library, perm, off, max_shift=1)
        assert np.array_equal(a.assignments, b[0])
        assert np.array_equal(a.counts_by_index(), b[1])
        for read in reads:
            assert SO.assign(library, perm, read, off, max_shift=1) == O.assign(library, perm, read, off)
            assert SO.closed_form_assign_shift(read, lib_seqs, True, reverse, offset, 1) == \
                O.assign(library, perm, read, off)


def _geometry(fn, *args):
    import ctypes as C
    start, length, idx = C.c_uint32(), C.c_uint32(), C.c_uint32()
    rc = fn(*args, C.byref(start), C.byref(length), C.byref(idx))
    return rc, (start.value, length.value, idx.value) if rc == 0 else None


def test_span_geometry_shift_one_equals_span_geometry():
    """no device needed: the library loads and the geometry is host arithmetic"""
    from sgcount_b200 import _cabi
    lib = _cabi.load()
    for k in (1, 5, 16, 20, 30):
        for read_len in range(k, k + 12):
            for offset in range(0, read_len - k + 3):
                for rev in (0, 1):
                    old = _geometry(lib.sgc_span_geometry, k, read_len, rev, offset, 1)
                    new = _geometry(lib.sgc_span_geometry_shift, k, read_len, rev, offset, 1)
                    assert old == new, (k, read_len, offset, rev)


def test_span_geometry_shift_holds_every_window():
    """S >= 2: the span records hold exactly the windows the read holds, and the call fails only
    when none fits"""
    from sgcount_b200 import _cabi
    lib = _cabi.load()
    for S in (2, 5, 16):
        for k in (4, 20):
            for read_len in range(max(1, k - 3), k + 2 * S + 3):
                for offset in range(0, read_len + S):
                    for rev in (0, 1):
                        rc, geo = _geometry(lib.sgc_span_geometry_shift, k, read_len, rev, offset, S)
                        fits = [d for d in range(-S, S + 1) if 0 <= offset + d and offset + d + k <= read_len]
                        assert (rc == 0) == bool(fits), (S, k, read_len, offset)
                        if rc:
                            assert rc == _cabi.ERR_INVALID_ARG
                            continue
                        start, length, span_off = geo
                        assert start + length <= read_len
                        in_span = [d for d in range(-S, S + 1) if 0 <= span_off + d and span_off + d + k <= length]
                        assert in_span == fits
                        # the same bytes: window d of the span is window d of the read
                        lo = read_len - start - length if rev else start
                        assert lo + span_off == offset
    for bad in (0, 17):
        rc, _ = _geometry(lib.sgc_span_geometry_shift, 20, 40, 0, 5, bad)
        assert rc == _cabi.ERR_INVALID_ARG
