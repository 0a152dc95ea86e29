"""ONE gzip member decoded in pieces (csrc/inflate_core.h: probe_block_start, piece_boundary,
inflate_piece; the device runs them in gzip.cu's member_* kernels), run serially on the host by
sgcount_b200/lib/member_core_test against zlib.  Whatever the piece size and however wrong the
candidate starts, the result is the member's exact bytes or a decline (the device then hands the file
to the host reader), never other bytes; damaged input is an error or a decline."""
import os
import random
import struct
import subprocess
import zlib

import pytest

from test_host_inflate import corpus, fnv, member

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "sgcount_b200", "lib", "member_core_test")
PIECES = [300, 4096, 32768, 131072]


@pytest.fixture(scope="module", autouse=True)
def built():
    if not os.path.exists(EXE):
        import __graft_entry__ as g

        g.build()
    assert os.path.exists(EXE)


def run(path, piece, skew):
    p = subprocess.run([EXE, str(path), str(piece), str(int(skew))], capture_output=True, text=True, timeout=300)
    return p.returncode, p.stdout.strip()


def fastq_random_qualities(n=4000, seed=3):
    rng = random.Random(seed)
    return b"".join(b"@r%d x\n%s\n+\n%s\n" % (i, bytes(rng.choice(b"ACGT") for _ in range(75)),
                                            bytes(33 + rng.randrange(41) for _ in range(75))) for i in range(n))


def texts():
    t = dict(corpus())
    t["fastq_random_q"] = fastq_random_qualities()
    return t


def flushed(data, mode, every=128 << 10, level=6):
    """a pigz-like stream: a sync or full flush every `every` bytes of input"""
    c = zlib.compressobj(level, zlib.DEFLATED, 31)
    out = b"".join(c.compress(data[i:i + every]) + c.flush(mode) for i in range(0, len(data), every))
    return out + c.flush()


def check(path, data, may_decline):
    for piece in PIECES:
        for skew in (False, True):
            rc, out = run(path, piece, skew)
            if rc == 3 and may_decline:
                continue
            assert rc == 0, (path.name, piece, skew, rc, out)
            assert " ".join(out.split()[:2]) == fnv(data), (path.name, piece, skew)


@pytest.mark.parametrize("name", list(texts()))
def test_exact_bytes_or_decline(tmp_path, name):
    data = texts()[name]
    variants = {"l1": (member(data, 1), False), "l6": (member(data, 6), False), "l9": (member(data, 9), False),
                "huffman_only": (member(data, 6, zlib.Z_HUFFMAN_ONLY), False), "rle": (member(data, 6, zlib.Z_RLE), False),
                "mem1": (member(data, 9, memlevel=1), False),
                # no dynamic block to start a piece at: one piece decodes it all, or the stream declines
                "fixed": (member(data, 6, zlib.Z_FIXED), True), "stored": (member(data, 0), True)}
    for vname, (blob, may_decline) in variants.items():
        assert zlib.decompress(blob, 31) == data
        path = tmp_path / f"{name}.{vname}.gz"
        path.write_bytes(blob)
        check(path, data, may_decline)


def test_pigz_like_flushes_and_header_fields(tmp_path):
    data = fastq_random_qualities(6000, seed=9)
    for mode, label in [(zlib.Z_SYNC_FLUSH, "sync"), (zlib.Z_FULL_FLUSH, "full")]:
        blob = flushed(data, mode)
        assert zlib.decompress(blob, 31) == data
        (tmp_path / f"{label}.gz").write_bytes(blob)
        check(tmp_path / f"{label}.gz", data, False)
    # FEXTRA | FNAME in front of the stream
    raw = zlib.compressobj(6, zlib.DEFLATED, -15)
    body = raw.compress(data) + raw.flush()
    header = bytes([0x1f, 0x8b, 8, 4 | 8, 0, 0, 0, 0, 0, 3]) + struct.pack("<H", 9) + b"AB\x05\x00extra" + b"reads.fastq\0"
    blob = header + body + struct.pack("<II", zlib.crc32(data), len(data))
    assert zlib.decompress(blob, 31) == data
    (tmp_path / "hdr.gz").write_bytes(blob)
    check(tmp_path / "hdr.gz", data, False)


def test_damaged_input_is_never_other_bytes(tmp_path):
    data = fastq_random_qualities(3000, seed=4)
    blob = member(data, 6)
    rng = random.Random(11)
    cases = {"cut_body": blob[:len(blob) // 2], "cut_trailer": blob[:-3], "no_trailer": blob[:-8],
             "bad_crc": blob[:-8] + struct.pack("<I", zlib.crc32(data) ^ 1) + blob[-4:],
             "bad_isize": blob[:-4] + struct.pack("<I", len(data) + 1),
             "two_members": blob + member(b"@x\nACGT\n+\nIIII\n"), "trailing_garbage": blob + b"\0" * 5}
    for i in range(12):  # flipped bits anywhere in the DEFLATE stream
        b = bytearray(blob)
        at = rng.randrange(20, len(b) - 8)
        b[at] ^= 1 << rng.randrange(8)
        cases[f"flip{i}"] = bytes(b)
    for label, bad in cases.items():
        (tmp_path / "bad.gz").write_bytes(bad)
        for piece in (300, 4096, 32768):
            for skew in (False, True):
                rc, out = run(tmp_path / "bad.gz", piece, skew)
                try:
                    same = zlib.decompress(bad, 31) == data
                except zlib.error:
                    same = False
                if rc == 0:  # only a flip that zlib too decodes to the same bytes may pass
                    assert same and label.startswith("flip"), (label, piece, skew, out)
                    assert " ".join(out.split()[:2]) == fnv(data)
                else:
                    assert rc in (3, 4), (label, piece, skew, rc, out)
