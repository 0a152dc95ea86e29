"""The pair rule (tests/pair_oracle.py) on the CPU: its invariants on random assignments, and the device
memory a pair counter declares, which needs no GPU."""
import numpy as np
import pytest

import sgcount_b200 as sg
from sgcount_b200 import _cabi

import pair_oracle as PO


@pytest.mark.parametrize("seed", range(5))
def test_statement_invariants(seed):
    rng = np.random.default_rng(1000 + seed)
    n1, n2, n = 40, 30, 20_000
    pairs = sorted({(int(a), int(b)) for a, b in zip(rng.integers(0, n1, 300), rng.integers(0, n2, 300))})
    a1 = np.where(rng.random(n) < 0.8, rng.integers(0, n1, n), -1)
    a2 = np.where(rng.random(n) < 0.7, rng.integers(0, n2, n), -1)
    listed = rng.random(n) < 0.5  # half the pairs on a listed construct
    pick = rng.integers(0, len(pairs), n)
    a1[listed] = [pairs[j][0] for j in pick[listed]]
    a2[listed] = [pairs[j][1] for j in pick[listed]]
    counts, tally, rec = PO.classify(a1, a2, pairs)
    assert tally["total"] == n == sum(tally[c] for c in PO.CLASSES)
    assert tally["listed"] == int(counts.sum())
    assert tally["recombined"] == sum(rec.values())
    # mate 1's marginal matched reads
    assert tally["listed"] + tally["recombined"] + tally["first_only"] == int((a1 >= 0).sum())
    assert tally["listed"] + tally["recombined"] + tally["second_only"] == int((a2 >= 0).sum())
    assert tally["neither"] == int(((a1 < 0) & (a2 < 0)).sum())
    assert not set(rec) & set(pairs)
    rows = PO.ordered(rec)
    assert [(-c, a, b) for a, b, c in rows] == sorted((-c, a, b) for a, b, c in rows)


def test_duplicate_construct_is_refused_by_the_statement():
    with pytest.raises(AssertionError):
        PO.classify([0], [0], [(1, 2), (1, 2)])


def test_pair_counter_bytes():
    small = sg.pair_counter_bytes(1, 0)
    assert small >= 2 * (1 << 24) * 4  # both mates' assignment scratch
    # table slots: the power of two >= 2 n_pairs, 12 bytes each, then 8 bytes per construct count
    assert sg.pair_counter_bytes(1000, 0) - small == (2048 - 2) * 12 + 999 * 8
    assert sg.pair_counter_bytes(1000, 64) - sg.pair_counter_bytes(1000, 0) == 64 * 16
    for n_pairs, capacity in ((0, 0), ((1 << 26) + 1, 0), (10, (1 << 26) + 1)):
        with pytest.raises(sg.SgcError) as e:
            sg.pair_counter_bytes(n_pairs, capacity)
        assert e.value.code == _cabi.ERR_INVALID_ARG
