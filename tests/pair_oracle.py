"""The dual-guide pair rule stated for the tests.  TEST INFRASTRUCTURE, NOT PRODUCT.

Mate m of pair i gets a_m[i]: what that mate's counter assigns to the read alone, taken from the CPU oracle
(tests/unmatched_oracle.assignments: oracle.Counter.new, or tests/shift_oracle.py for max_shift >= 2).
Construct j is (first[j], second[j]).  Every pair falls into one class:
  listed       a1 >= 0, a2 >= 0 and (a1, a2) is construct j  -> counted on j
  recombined   a1 >= 0, a2 >= 0 and (a1, a2) is not listed    -> tallied by (a1, a2) in the report
  first_only   a1 >= 0, a2 < 0;   second_only   a1 < 0, a2 >= 0;   neither   a1 < 0, a2 < 0."""
from __future__ import annotations

from collections import Counter as Tally
from typing import List, Sequence, Tuple

import numpy as np

import unmatched_oracle

CLASSES = ("listed", "recombined", "first_only", "second_only", "neither")


def classify(a1: Sequence[int], a2: Sequence[int], pairs: Sequence[Tuple[int, int]]):
    """(construct counts uint64[len(pairs)], {total and the five classes}, Tally of recombinant (a1, a2))"""
    index = {}
    for j, (f, s) in enumerate(pairs):
        assert (int(f), int(s)) not in index, "duplicate construct"
        index[(int(f), int(s))] = j
    counts = np.zeros(len(pairs), dtype=np.uint64)
    tally = dict.fromkeys(CLASSES, 0)
    recombinants: Tally = Tally()
    for x, y in zip(a1, a2):
        x, y = int(x), int(y)
        if x >= 0 and y >= 0:
            j = index.get((x, y))
            if j is None:
                tally["recombined"] += 1
                recombinants[(x, y)] += 1
            else:
                tally["listed"] += 1
                counts[j] += 1
        elif x >= 0:
            tally["first_only"] += 1
        elif y >= 0:
            tally["second_only"] += 1
        else:
            tally["neither"] += 1
    tally["total"] = sum(tally[c] for c in CLASSES)
    return counts, tally, recombinants


def ordered(recombinants: Tally) -> List[Tuple[int, int, int]]:
    """report order: count descending, then (first, second) ascending"""
    return [(a, b, n) for (a, b), n in sorted(recombinants.items(), key=lambda kv: (-kv[1], kv[0]))]


def mate_assignments(seqs, guides, with_perm, offset, rc_mode=0, max_shift=1, recursion=True) -> np.ndarray:
    return unmatched_oracle.assignments(seqs, guides, with_perm, offset, rc_mode, max_shift, recursion)
