"""A gzip file decoded in pieces and cut into WAVES whose windows are relayed through F_k and W_k, the
way sgc_fastq_stream_submit_gzip_split spreads one file over several streams (csrc/inflate_core.h
"waves on several streams": relay_symbol, wave_front, compose_window, settle_symbol), run serially by
sgcount_b200/lib/member_core_test with its fifth argument.  Whatever the wave count, the piece size and
the members, the result is the exact bytes zlib gives or a decline; damaged input is an error or a
decline."""
import random
import struct
import subprocess
import zlib

import pytest

from test_host_inflate import fnv, member
from test_member_inflate_core import EXE, fastq_random_qualities
from test_multi_member_inflate_core import built  # noqa: F401  (builds the helper once)

WAVES = [1, 2, 3, 7]
STRATEGIES = [(1, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_DEFAULT_STRATEGY),
              (6, zlib.Z_FILTERED), (6, zlib.Z_HUFFMAN_ONLY)]


def run(path, piece, skew, waves):
    p = subprocess.run([EXE, str(path), str(piece), str(int(skew)), "1", str(waves)], capture_output=True, text=True, timeout=300)
    return p.returncode, p.stdout.strip()


def cut(data, m, rng):
    at = sorted(rng.randrange(len(data) + 1) for _ in range(m - 1))
    return [data[a:b] for a, b in zip([0] + at, at + [len(data)])]


def expect(path, data, n_members, pieces, waves=WAVES, may_decline=False):
    passed = 0
    for piece in pieces:
        for skew in (False, True):
            for w in waves:
                rc, out = run(path, piece, skew, w)
                if rc == 3 and may_decline:
                    continue
                assert rc == 0, (path.name, piece, skew, w, rc, out)
                f = out.split()
                assert " ".join(f[:2]) == fnv(data), (path.name, piece, skew, w)
                assert int(f[5]) == n_members, (path.name, piece, skew, w, out)
                passed += 1
    return passed


@pytest.mark.parametrize("level,strategy", STRATEGIES)
def test_waves_equal_zlib(tmp_path, level, strategy):
    """small blocks (memLevel 1) and small pieces: waves of a few KiB, so that a wave's window is made
    of several waves in front of it and composes through several F_k"""
    data = fastq_random_qualities(600, seed=level * 7 + strategy)
    path = tmp_path / "one.gz"
    path.write_bytes(member(data, level, strategy, memlevel=1))
    # (Huffman-only blocks have no matches; fixed-code runs may leave no candidate: a decline is allowed)
    assert expect(path, data, 1, (300, 2000, 32768), may_decline=True) > 0
    expect(path, data, 1, (300,), waves=(40,), may_decline=True)


@pytest.mark.parametrize("m", [1, 2, 5, 64])
def test_members_over_waves(tmp_path, m):
    rng = random.Random(m)
    data = fastq_random_qualities(900, seed=m)
    parts = cut(data, m, rng)
    blob = b"".join(member(p, rng.choice([1, 6, 9]), zlib.Z_DEFAULT_STRATEGY, memlevel=rng.choice([1, 8])) for p in parts)
    path = tmp_path / "members.gz"
    path.write_bytes(blob)
    assert expect(path, data, m, (300, 4096), may_decline=True) > 0


def test_waves_shorter_than_the_window(tmp_path):
    data = fastq_random_qualities(400, seed=5)  # ~65 KB of text: 7 and 20 waves of under 32 KiB
    path = tmp_path / "short.gz"
    path.write_bytes(member(data, 6, zlib.Z_DEFAULT_STRATEGY, memlevel=1))
    assert expect(path, data, 1, (200, 600), waves=(3, 7, 20)) == 12


def test_member_start_on_a_wave_boundary(tmp_path):
    """two members of equal text and two waves: the second wave starts exactly at the second member"""
    data = fastq_random_qualities(800, seed=9)
    half = data[:len(data) // 2]
    path = tmp_path / "two.gz"
    for memlevel in (1, 8):
        path.write_bytes(member(half, 6, zlib.Z_DEFAULT_STRATEGY, memlevel) * 2)
        assert expect(path, half * 2, 2, (500, 1 << 20), waves=(2, 4)) == 8


def test_damaged_input_is_never_other_bytes(tmp_path):
    rng = random.Random(21)
    data = fastq_random_qualities(1200, seed=21)
    parts = cut(data, 3, rng)
    ms = [member(p, 6, zlib.Z_DEFAULT_STRATEGY, memlevel=1) for p in parts]
    blob = b"".join(ms)
    mid = len(ms[0]) + len(ms[1])
    cases = {"cut_last_body": blob[:len(blob) - len(ms[-1]) // 2], "no_last_trailer": blob[:-8],
             "bad_crc_middle": blob[:mid - 8] + struct.pack("<I", zlib.crc32(parts[1]) ^ 1) + blob[mid - 4:],
             "trailing_garbage": blob + b"garbage!"}
    for i in range(12):
        b = bytearray(blob)
        b[rng.randrange(len(b))] ^= 1 << rng.randrange(8)
        cases[f"flip{i}"] = bytes(b)
    for label, bad in cases.items():
        (tmp_path / "bad.gz").write_bytes(bad)
        try:
            out, rest = b"", bad
            while rest:
                d = zlib.decompressobj(31)
                out += d.decompress(rest)
                assert d.eof
                rest = d.unused_data
            same = out == data
        except (zlib.error, AssertionError):
            same = False
        for piece in (300, 4096):
            for w in (2, 7):
                rc, out = run(tmp_path / "bad.gz", piece, False, w)
                if rc == 0:  # only a flip that zlib too decodes to the same bytes may pass
                    assert same and " ".join(out.split()[:2]) == fnv(data), (label, piece, w, out)
                else:
                    assert rc in (3, 4), (label, piece, w, rc, out)
