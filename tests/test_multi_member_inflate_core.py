"""SEVERAL gzip members (concatenated files, appending writers, BGZF) decoded in pieces the way
sgc_fastq_stream_submit_gzip does it on the device (csrc/inflate_core.h: member_start_at, merge_starts,
members_chain, piece_boundary with a per-piece reach), run serially by sgcount_b200/lib/member_core_test
with its fourth argument set.  Whatever the piece size and however wrong the candidate starts, the result
is the exact bytes of the concatenated members or a decline, never other bytes; damaged input is an error
or a decline."""
import os
import random
import struct
import subprocess
import zlib

import pytest

from test_host_inflate import fnv, member
from test_member_inflate_core import EXE, PIECES, fastq_random_qualities

STRATEGIES = [(6, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_DEFAULT_STRATEGY),
              (6, zlib.Z_FIXED), (0, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_HUFFMAN_ONLY)]


@pytest.fixture(scope="module", autouse=True)
def built():
    if not os.path.exists(EXE):
        import __graft_entry__ as g

        g.build()
    assert os.path.exists(EXE)


def run(path, piece, skew):
    p = subprocess.run([EXE, str(path), str(piece), str(int(skew)), "1"], capture_output=True, text=True, timeout=300)
    return p.returncode, p.stdout.strip()


def cut(data, m, rng):
    at = sorted(rng.randrange(len(data) + 1) for _ in range(m - 1))
    return [data[a:b] for a, b in zip([0] + at, at + [len(data)])]


def raw_member(text, level=6, header=None):
    """a member with a chosen header (default: the plain 10-byte one)"""
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    body = c.compress(text) + c.flush()
    header = header or bytes([0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 0, 3])
    return header + body + struct.pack("<II", zlib.crc32(text), len(text) & 0xFFFFFFFF)


def fname_header(name: bytes):
    return bytes([0x1f, 0x8b, 8, 8, 0, 0, 0, 0, 0, 3]) + name + b"\0"


def bgzf(text, block=60000):
    """BGZF: members of at most 64 KB carrying their size in a 'BC' extra subfield, then the EOF block"""
    out = []
    for i in range(0, len(text), block):
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        body = c.compress(text[i:i + block]) + c.flush()
        size = 18 + len(body) + 8
        out.append(bytes([0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, ord("B"), ord("C"), 2, 0]) + struct.pack("<H", size - 1) +
                   body + struct.pack("<II", zlib.crc32(text[i:i + block]), len(text[i:i + block])))
    out.append(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
    return b"".join(out)


def check(path, blob, data, n_members, may_decline, pieces=PIECES):
    assert b"".join(_members(blob)) == data
    passed = 0
    for piece in pieces:
        for skew in (False, True):
            rc, out = run(path, piece, skew)
            if rc == 3 and may_decline:
                continue
            assert rc == 0, (path.name, piece, skew, rc, out)
            f = out.split()
            assert " ".join(f[:2]) == fnv(data), (path.name, piece, skew)
            assert int(f[5]) == n_members, (path.name, piece, skew, out)
            passed += 1
    return passed


def _members(blob):
    """the text of every member, as gzip -d concatenates it"""
    out = []
    while blob:
        d = zlib.decompressobj(31)
        out.append(d.decompress(blob))
        assert d.eof
        blob = d.unused_data
    return out


@pytest.mark.parametrize("m", [2, 3, 7, 16, 64])
def test_mixed_levels_and_strategies(tmp_path, m):
    rng = random.Random(m)
    data = fastq_random_qualities(1500, seed=m)
    parts = cut(data, m, rng)
    # default strategies only: every member starts a piece and dynamic blocks follow, the chain must hold
    plain = b"".join(member(p, rng.choice([1, 6, 9])) for p in parts)
    (tmp_path / "plain.gz").write_bytes(plain)
    assert check(tmp_path / "plain.gz", plain, data, m, False) == 2 * len(PIECES)
    # stored, fixed-code and Huffman-only members too: long runs without a dynamic block may decline
    mixed = b"".join(member(p, *STRATEGIES[i % len(STRATEGIES)]) for i, p in enumerate(parts))
    (tmp_path / "mixed.gz").write_bytes(mixed)
    check(tmp_path / "mixed.gz", mixed, data, m, True)


def test_empty_and_tiny_members(tmp_path):
    rng = random.Random(5)
    data = fastq_random_qualities(300, seed=5)
    parts = [b""] + cut(data, 40, rng) + [b""]
    parts[10:10] = [b"", b""]
    blob = b"".join(member(p, 6) for p in parts)  # ~40 members, most far smaller than a piece
    (tmp_path / "tiny.gz").write_bytes(blob)
    assert check(tmp_path / "tiny.gz", blob, data, len(parts), False) == 2 * len(PIECES)
    only_empty = member(b"") * 3
    (tmp_path / "empty.gz").write_bytes(only_empty)
    assert check(tmp_path / "empty.gz", only_empty, b"", 3, False) == 2 * len(PIECES)


def test_member_boundary_on_a_nominal_piece_boundary(tmp_path):
    data = fastq_random_qualities(2000, seed=6)
    a, b = data[:len(data) // 3], data[len(data) // 3:]
    first = raw_member(a)
    for piece in (300, 4096, 32768):
        k = (len(first) + 12 + piece - 1) // piece * piece
        for target in (k, k + piece):
            # the second member's DEFLATE stream starts at `target` (its FNAME pads its header) ...
            on_stream = first + raw_member(b, header=fname_header(b"x" * (target - len(first) - 11)))
            # ... or its header does (the first member's FNAME pads the first member)
            on_header = raw_member(a, header=fname_header(b"y" * (target - len(first) - 1))) + raw_member(b)
            assert on_header[target:target + 2] == b"\x1f\x8b"
            for label, blob in (("stream", on_stream), ("header", on_header)):
                (tmp_path / f"{label}.gz").write_bytes(blob)
                assert check(tmp_path / f"{label}.gz", blob, data, 2, False, pieces=[piece]) == 2


def test_header_fields_bgzf_and_gzip_inside_a_stored_block(tmp_path):
    data = fastq_random_qualities(2000, seed=8)
    a, b, c = data[:20000], data[20000:200000], data[200000:]
    extra = bytes([0x1f, 0x8b, 8, 4 | 8 | 16, 0, 0, 0, 0, 0, 3]) + struct.pack("<H", 9) + b"AB\x05\x00extra" + b"r.fq\0" + b"note\0"
    blob = raw_member(a, header=extra) + raw_member(b, header=fname_header(b"reads.fastq")) + raw_member(c, 9)
    (tmp_path / "hdr.gz").write_bytes(blob)
    assert check(tmp_path / "hdr.gz", blob, data, 3, False) == 2 * len(PIECES)
    bg = bgzf(data)
    (tmp_path / "bgzf.gz").write_bytes(bg)
    assert check(tmp_path / "bgzf.gz", bg, data, len(data) // 60000 + 2, False) == 2 * len(PIECES)
    # a whole gzip file as the payload of a stored block: true signatures inside another member
    inner = member(a, 6) + member(c, 1)
    nested = member(b, 6) + member(inner, 0) + member(c, 6)
    (tmp_path / "nested.gz").write_bytes(nested)
    check(tmp_path / "nested.gz", nested, b + inner + c, 3, True)
    nested_small = member(inner, 0) + member(b, 6)  # one stored block of the payload and a dynamic member
    (tmp_path / "nested_small.gz").write_bytes(nested_small)
    check(tmp_path / "nested_small.gz", nested_small, inner + b, 2, True)


def test_damaged_input_is_never_other_bytes(tmp_path):
    rng = random.Random(12)
    data = fastq_random_qualities(1500, seed=12)
    parts = cut(data, 5, rng)
    ms = [member(p, 6) for p in parts]
    blob = b"".join(ms)
    mid = len(ms[0]) + len(ms[1])  # the end of the second member
    cases = {"cut_last_body": blob[:len(blob) - len(ms[-1]) // 2], "cut_last_trailer": blob[:-3], "no_last_trailer": blob[:-8],
             "bad_crc_middle": blob[:mid - 8] + struct.pack("<I", zlib.crc32(parts[1]) ^ 1) + blob[mid - 4:],
             "bad_isize_middle": blob[:mid - 4] + struct.pack("<I", len(parts[1]) + 1) + blob[mid:],
             "trailing_garbage": blob + b"garbage!", "zero_padding": blob + b"\0" * 512,
             "half_a_header": blob + blob[:6]}
    for i in range(16):  # flipped bits anywhere, headers and trailers included
        b = bytearray(blob)
        b[rng.randrange(len(b))] ^= 1 << rng.randrange(8)
        cases[f"flip{i}"] = bytes(b)
    for label, bad in cases.items():
        (tmp_path / "bad.gz").write_bytes(bad)
        try:
            same = b"".join(_members(bad)) == data
        except (zlib.error, AssertionError):
            same = False
        for piece in (300, 4096, 32768):
            for skew in (False, True):
                rc, out = run(tmp_path / "bad.gz", piece, skew)
                if rc == 0:  # only a flip that zlib too decodes to the same bytes may pass
                    assert same and label.startswith("flip"), (label, piece, skew, out)
                    assert " ".join(out.split()[:2]) == fnv(data)
                else:
                    assert rc in (3, 4), (label, piece, skew, rc, out)
