"""The unmatched report's statement (tests/unmatched_oracle.py) on the CPU: the known answers of the
example fixtures, the sum invariant on random samples, and the CLI's --unmatched-report flag surface."""
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as orc

import unmatched_oracle as U
from helpers import make_library, make_reads

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")


def records(path):
    r = orc.Records.from_path(path)
    return [r.seq(i) for i in range(len(r))]


@pytest.fixture(scope="module")
def guides(example_dir):
    return records(os.path.join(example_dir, "library.fasta.gz"))


def test_diff_sequence_has_one_window(example_dir, guides):
    """the 101 @nonsense reads never match and share their window at Forward(5)"""
    seqs = records(os.path.join(example_dir, "diff.sequence.fastq.gz"))
    windows, tally, _ = U.statement(seqs, guides, True, orc.Offset.Forward(5))
    assert windows == [(b"CTAGGGACCACAGCCATTAT", 101)]
    assert tally == {"unmatched": 101, "short_reads": 0, "non_acgt": 0}


def test_offset_clipped_has_one_short_read(example_dir, guides):
    seqs = records(os.path.join(example_dir, "offset_clipped.fastq.gz"))
    windows, tally, _ = U.statement(seqs, guides, True, orc.Offset.Forward(5))
    assert windows == []
    assert tally == {"unmatched": 1, "short_reads": 1, "non_acgt": 0}


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("max_shift", [1, 4])
def test_sum_invariant(reverse, max_shift):
    """total - matched = short + non_acgt + the window counts, and every window is k bytes over A, C, G, T"""
    rng = np.random.default_rng(0xB17 + 2 * max_shift + reverse)
    k = 20
    guides = make_library(rng, 300, k)
    seqs = make_reads(rng, guides, 4000, 40, 6, reverse=reverse, variable=True, junk=0.2)
    for i in rng.choice(len(seqs), 400, replace=False):  # two Ns: no lookup settles such a window
        row = bytearray(seqs[i])
        for p in rng.integers(0, max(len(row), 1), 2):
            if len(row):
                row[p] = ord("N")
        seqs[i] = bytes(row)
    off = orc.Offset(reverse, 6)
    for rc_mode in (orc.RC_BITTRICK, orc.RC_KEEP_N):
        windows, tally, assign = U.statement(seqs, guides, True, off, rc_mode, max_shift)
        assert tally["unmatched"] == int((assign < 0).sum()) > 0
        assert tally["unmatched"] == tally["short_reads"] + tally["non_acgt"] + sum(c for _, c in windows)
        assert tally["short_reads"] > 0 and tally["non_acgt"] > 0
        assert all(len(w) == k and not w.strip(b"ACGT") for w, _ in windows)
        assert windows == sorted(windows, key=lambda kv: (-kv[1], kv[0]))


def test_reverse_windows_are_in_library_orientation():
    """a reverse read whose stored window is the reverse complement of a non-member reports the non-member"""
    guides = [b"ACGTACGTAC", b"GGGGCCCCAA"]
    window = b"AAAACCCGGT"
    read = b"TT" + window + b"GG"
    stored = orc.seq_rev_comp(read, orc.RC_KEEP_N)
    windows, tally, _ = U.statement([stored], guides, True, orc.Offset.Reverse(2), orc.RC_KEEP_N)
    assert windows == [(window, 1)] and tally["unmatched"] == 1


@pytest.fixture(scope="module")
def built():
    if not os.path.exists(BIN):
        import __graft_entry__ as g

        g.build()
    assert os.path.exists(BIN)


def test_cli_usage_lists_the_flag(built):
    p = subprocess.run([BIN, "--help"], capture_output=True, text=True, timeout=60)
    assert p.returncode == 0 and "--unmatched-report <PATH>" in p.stdout


def test_cli_flag_needs_a_value(built):
    p = subprocess.run([BIN, "-l", "x", "-i", "y", "--unmatched-report"], capture_output=True, text=True, timeout=60)
    assert p.returncode == 1
    assert "a value is required for '--unmatched-report'" in p.stderr
