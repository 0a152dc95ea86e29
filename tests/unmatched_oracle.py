"""The unmatched report stated for the tests.  TEST INFRASTRUCTURE, NOT PRODUCT.

For every read the oracle leaves unmatched (assignment -1) the window at the offset is sliced exactly as
the reference slices its first lookup: trimmed[o : o + k], where trimmed is the read in Forward and
seq_rev_comp(read) under the counter's rc_mode in Reverse, whatever the recursion and max_shift.  Such a
read is `short` when o + k exceeds its length, `non_acgt` when the window has a byte outside A, C, G, T,
and otherwise its window is tallied by its bytes.  The assignments come from the CPU oracle
(oracle.Counter.new(..., want_assignments=True)) and, for max_shift >= 2, from tests/shift_oracle.py."""
from __future__ import annotations

from collections import Counter as Tally
from typing import List, Optional, Sequence, Tuple

import numpy as np

from oracle import oracle as orc

import shift_oracle


def assignments(seqs: Sequence[bytes], guides: Sequence[bytes], with_perm: bool, offset: orc.Offset,
                rc_mode: int = orc.RC_BITTRICK, max_shift: int = 1, recursion: bool = True) -> np.ndarray:
    """the oracle's per-read library index or -1"""
    recs = orc.Records.from_seqs(list(seqs))
    olib = orc.Library.from_reader(orc.Records.from_seqs(list(guides)))
    operm = orc.Permuter.new(olib) if with_perm else None
    if max_shift >= 2:
        return shift_oracle.count(recs, olib, operm, offset, rc_mode=rc_mode, max_shift=max_shift)[0]
    return orc.Counter.new(recs, olib, operm, offset, position_recursion=recursion, rc_mode=rc_mode, n_threads=8,
                           want_assignments=True).assignments


def report(seqs: Sequence[bytes], assign: Sequence[int], k: int, offset: orc.Offset,
           rc_mode: int = orc.RC_BITTRICK) -> Tuple[Tally, dict]:
    """(window bytes -> count, {unmatched, short_reads, non_acgt}) of the unmatched reads"""
    windows: Tally = Tally()
    tally = {"unmatched": 0, "short_reads": 0, "non_acgt": 0}
    o = offset.index
    for seq, a in zip(seqs, assign):
        if a >= 0:
            continue
        tally["unmatched"] += 1
        trimmed = orc.seq_rev_comp(seq, rc_mode) if offset.reverse else seq
        if o + k > len(trimmed):
            tally["short_reads"] += 1
            continue
        w = trimmed[o:o + k]
        if w.strip(b"ACGT"):
            tally["non_acgt"] += 1
        else:
            windows[w] += 1
    return windows, tally


def ordered(windows: Tally) -> List[Tuple[bytes, int]]:
    """report order: count descending, then window bytes ascending"""
    return sorted(windows.items(), key=lambda kv: (-kv[1], kv[0]))


def statement(seqs: Sequence[bytes], guides: Sequence[bytes], with_perm: bool, offset: orc.Offset,
              rc_mode: int = orc.RC_BITTRICK, max_shift: int = 1, recursion: bool = True,
              assign: Optional[np.ndarray] = None):
    """(ordered windows, tallies, assignments) of a sample"""
    if assign is None:
        assign = assignments(seqs, guides, with_perm, offset, rc_mode, max_shift, recursion)
    windows, tally = report(seqs, assign, len(guides[0]), offset, rc_mode)
    return ordered(windows), tally, assign
