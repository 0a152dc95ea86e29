"""gzip decoding on DEFLATE streams zlib cannot write (tests/deflate_writer.py): matches that reach the
oldest bytes of the 32 KiB window (distances 32 507 - 32 768, which zlib never emits), dynamic blocks
with one distance code or none (incomplete codes, zlib always sends two), stored blocks of LEN 0 and
65 535, empty blocks and block ends at every bit offset, on realistic FASTQ (literal-heavy, long codes)
and on the corpus texts.  Every decoder must give the exact bytes: the host's whole-member decoder
(fastx_dump inflate), the device decoder's core compiled for the host (inflate_core_test, every output
alignment) and the piece / wave path run serially (member_core_test), which may decline only streams
without dynamic blocks.  Invalid twins (a match one byte too far back for its member) are errors or
declines, never bytes."""
import os
import random
import subprocess
import zlib

import numpy as np
import pytest

import deflate_writer as dw
from helpers import make_library, make_reads, realistic_fastq
from test_host_inflate import DUMP, corpus, fnv
from test_device_inflate_core import EXE as CORE_EXE
from test_member_inflate_core import EXE as MEMBER_EXE


@pytest.fixture(scope="module", autouse=True)
def built():
    if not all(os.path.exists(x) for x in (DUMP, CORE_EXE, MEMBER_EXE)):
        import __graft_entry__ as g

        g.build()
    assert all(os.path.exists(x) for x in (DUMP, CORE_EXE, MEMBER_EXE))


FAR = [d for d in dw.EDGE_DISTS if d > 32506]
NEAR = [d for d in dw.EDGE_DISTS if d < 32506]
MIXED = ("dynamic", "dynamic", "dynamic", "fixed", "stored", "empty")


def fastq(n_reads, seed):
    rng = np.random.default_rng(seed)
    seqs = make_reads(rng, make_library(rng, 200, 20), n_reads, 75, 5)
    return realistic_fastq(rng, seqs)


def stream(text, slots, seed, kinds=MIXED, n_far=60, lengths=tuple(range(3, 19)), sizes=(50, 4000)):
    """a raw DEFLATE stream of `text` with matches planted at every edge distance (n_far of them
    farther than 32 506, and some at exactly 32 768): (text, tokens, body, stats)"""
    rng = random.Random(seed)
    buf = bytearray(text)
    force = dw.plant(buf, rng, slots, [(FAR, lengths, n_far), ([32768], lengths, 8 if n_far else 0), (NEAR, lengths, 40)])
    text = bytes(buf)
    tokens = dw.parse(text, force=force)
    stats = dw.Stats()
    body = dw.deflate(tokens, dw.layout(len(tokens), rng, kinds, sizes), text, stats)
    return text, tokens, body, stats


def dump(path):
    p = subprocess.run([DUMP, str(path), "1", "inflate"], capture_output=True, text=True, timeout=120)
    return p.returncode, p.stdout.strip()


def core(path, align):
    p = subprocess.run([CORE_EXE, str(path), str(1 << 30), str(align)], capture_output=True, text=True, timeout=120)
    return p.returncode, p.stdout.strip()


def member_core(path, piece, skew, members, waves):
    p = subprocess.run([MEMBER_EXE, str(path), str(piece), str(int(skew)), str(int(members)), str(waves)], capture_output=True,
                       text=True, timeout=300)
    return p.returncode, p.stdout.strip()


def members_of(blob):
    out = []
    while blob:
        d = zlib.decompressobj(31)
        out.append(d.decompress(blob))
        assert d.eof
        blob = d.unused_data
    return out


def check_all(path, datas, may_decline=False, pieces=(300, 4096, 32768), waves=(1, 2, 7, 40), members=(0, 1)):
    """every decoder gives the bytes of every member; the piece path may decline only if allowed"""
    text = b"".join(datas)
    assert dump(path) == (0, fnv(text)), path.name
    for align in range(8):
        assert core(path, align) == (0, f"{len(datas)} {fnv(text)}"), (path.name, align)
    passed = 0
    for m in members:
        if not m and len(datas) > 1:
            continue
        for piece in pieces:
            for skew in (False, True):
                for w in waves:
                    rc, out = member_core(path, piece, skew, m, w)
                    if rc == 3 and may_decline:
                        continue
                    assert rc == 0, (path.name, piece, skew, m, w, rc, out)
                    f = out.split()
                    assert " ".join(f[:2]) == fnv(text), (path.name, piece, skew, m, w)
                    if m:
                        assert int(f[5]) == len(datas), (path.name, out)
                    passed += 1
    return passed


def test_writer_round_trips_and_holds_its_edges():
    text, slots = fastq(1500, 1)
    rng = random.Random(2)
    buf = bytearray(text)
    lengths = list(range(3, 19))
    force = dw.plant(buf, rng, slots, [(FAR, lengths, 60), ([32768], [3, 10, 18], 8), (NEAR, lengths, 60)])
    # the corpus's long runs for lengths 256 - 258
    runs = bytearray(corpus()["far"])
    force_runs = dw.plant(runs, rng, [(0, len(runs))], [([1, 2, 17, 256, 32768], [256, 257, 258], 12)])
    for label, t, f, lits in (("fastq", bytes(buf), force, 65535 + 7), ("runs", bytes(runs), force_runs, 0)):
        tokens = dw.parse(t, force=f, literals=lits)
        assert dw.expand(tokens) == t
        got = {(p, ln, d) for p, ln, d in f if p >= lits}
        at = 0
        for tok in tokens:  # every forced match is in the token list where it was planted
            if not isinstance(tok, int):
                got.discard((at, tok[0], tok[1]))
            at += 1 if isinstance(tok, int) else tok[0]
        assert not got, (label, sorted(got)[:5])
        stats = dw.Stats()
        blocks = ([("stored", 65535), ("stored", 0)] if lits else []) + \
            dw.layout(len(tokens) - (65535 if lits else 0), rng, MIXED, (50, 4000))
        body = dw.deflate(tokens, blocks, t, stats)
        assert zlib.decompress(body, -15) == t
        member = dw.gzip_member(body, t, dw.gzip_header(2, extra=b"AB\x02\x00xy", name=b"r.fq", comment=b"c"))
        assert zlib.decompress(member, 31) == t
        d = stats.dists
        assert sum(x > 32506 for x in d) >= (40 if label == "fastq" else 1) and 32768 in d, label
        if label == "fastq":
            assert set(range(1, 18)) | {31, 32, 33, 255, 256, 257} <= set(d)
            assert set(range(3, 19)) <= set(stats.lengths)
            assert {0, 65535} <= set(stats.stored_lens)
            assert stats.lone_dist and stats.no_dist and stats.straddle > 10
            assert {"dynamic", "fixed", "stored", "empty"} <= set(stats.kinds)
            assert {e % 8 for e in stats.end_bits} == set(range(8))
        else:
            assert {256, 257, 258} <= set(stats.lengths)


def test_code_lengths_are_limited_and_complete():
    fib = [1, 1]
    while len(fib) < 40:
        fib.append(fib[-1] + fib[-2])
    for limit, freq in ((15, fib[:30]), (7, fib[:19]), (15, [1] * 286), (7, [5, 0, 0, 1])):
        lengths = dw.code_lengths(freq, limit)
        used = [n for f, n in zip(freq, lengths) if f]
        assert max(used) <= limit and all(used)
        assert sum(2.0 ** -n for n in used) == 1.0
    assert max(dw.code_lengths(fib[:30], 15)) == 15  # the limit binds: Huffman alone would go to 29
    assert dw.code_lengths([0, 0, 9], 15) == [0, 0, 1] and dw.code_lengths([0, 0], 15) == [0, 0]


def test_fastq_far_window_stream(tmp_path):
    """single member, mixed block kinds with dynamic blocks among them: the exact bytes everywhere"""
    text, slots = fastq(1500, 3)
    text, _, body, stats = stream(text, slots, 4)
    assert sum(d > 32506 for d in stats.dists) >= 40 and stats.lone_dist and stats.no_dist
    path = tmp_path / "far.gz"
    path.write_bytes(dw.gzip_member(body, text))
    assert zlib.decompress(path.read_bytes(), 31) == text
    assert check_all(path, [text]) == 48


def test_members_with_an_empty_one_and_header_fields(tmp_path):
    text, slots = fastq(1500, 5)
    cut = [0, len(text) // 3 + 11, len(text) // 3 + 11, 2 * len(text) // 3 - 5, len(text)]
    datas = [text[a:b] for a, b in zip(cut, cut[1:])]
    headers = [dw.gzip_header(), dw.gzip_header(2, name=b"empty.fq"), dw.gzip_header(2, extra=b"AB\x02\x00xy", comment=b"lane 1"),
               dw.gzip_header(name=b"tail.fq")]
    blob = b""
    for i, (d, h) in enumerate(zip(datas, headers)):
        sl = [(a - cut[i], b - cut[i]) for a, b in slots if a >= cut[i] and b <= cut[i + 1]]
        if d:
            d, _, body, _ = stream(d, sl, 10 + i, n_far=20)
            datas[i] = d
        else:
            body = dw.deflate([], [("empty", 0)])
        blob += dw.gzip_member(body, d, h)
    assert members_of(blob) == datas
    path = tmp_path / "members.gz"
    path.write_bytes(blob)
    assert check_all(path, datas, members=(1,)) == 24


@pytest.mark.parametrize("name", list(corpus()))
def test_corpus_texts(tmp_path, name):
    data = corpus()[name]
    if not data:
        body = dw.deflate([], [("empty", 0)])
    else:
        slots = [(0, len(data))]
        data, _, body, _ = stream(data, slots, len(name), n_far=20 if len(data) > 40000 else 0,
                                  lengths=(3, 4, 9, 18, 256, 257, 258), sizes=(20, 3000))
    path = tmp_path / f"{name}.gz"
    path.write_bytes(dw.gzip_member(body, data))
    assert zlib.decompress(path.read_bytes(), 31) == data
    check_all(path, [data], pieces=(300, 4096), waves=(1, 7))


@pytest.mark.parametrize("kind", ["fixed", "stored"])
def test_runs_without_dynamic_blocks_decline_or_give_the_bytes(tmp_path, kind):
    text, slots = fastq(800, 6)
    text, _, body, _ = stream(text, slots, 7, kinds=(kind,), n_far=20)
    path = tmp_path / f"{kind}.gz"
    path.write_bytes(dw.gzip_member(body, text))
    check_all(path, [text], may_decline=True, waves=(1, 7))


def test_invalid_twins_are_errors_or_declines(tmp_path):
    """a match whose distance reaches one byte in front of its member: 32 768 placed one byte too
    early, a short one at the start of the member, and one in a second member that reaches into the
    first.  The trailer holds what a decoder that did not check would make, so only the distance
    check can tell."""
    text, _ = fastq(400, 8)
    cases = {"32768 one byte early": list(text[:32767]) + [(4, 32768)] + list(text[32767:40000]),
             "first match too far": list(text[:100]) + [(3, 101)] + list(text[100:5000]),
             "max distance at position 0": [(258, 32768)] + list(text[:3000])}
    # the first twin's valid form, one byte later, copies the member's first bytes
    ok = list(text[:32768]) + [(4, 32768)] + list(text[32768:40000])
    assert dw.expand(ok)[32768:32772] == text[:4]
    for label, toks in cases.items():
        permissive = dw.expand(toks, before=bytes(32768))
        body = dw.deflate(toks, [("dynamic", len(toks))])
        blob = dw.gzip_member(body, permissive)
        with pytest.raises(zlib.error):
            zlib.decompress(blob, 31)
        check_rejected(tmp_path, label, blob)
    # a second member whose match reaches into the first: the text of the two, as a shared window makes it
    first = text[:20000]
    toks = list(text[20000:20100]) + [(6, 101)] + list(text[20100:30000])
    second = dw.expand(toks, before=first)
    blob = dw.gzip_member(dw.deflate(list(first), [("dynamic", len(first))]), first) + \
        dw.gzip_member(dw.deflate(toks, [("dynamic", len(toks))]), second)
    check_rejected(tmp_path, "into the previous member", blob)
    # its valid twin (the match one byte nearer) decodes everywhere
    toks[100] = (6, 100)
    second = dw.expand(toks, before=first)
    blob = dw.gzip_member(dw.deflate(list(first), [("dynamic", len(first))]), first) + \
        dw.gzip_member(dw.deflate(toks, [("dynamic", len(toks))]), second)
    path = tmp_path / "valid_twin.gz"
    path.write_bytes(blob)
    assert members_of(blob) == [first, second]
    check_all(path, [first, second], pieces=(300, 4096), waves=(1, 7), members=(1,))


def check_rejected(tmp_path, label, blob):
    path = tmp_path / "twin.gz"
    path.write_bytes(blob)
    assert dump(path)[0] == 4, label
    for align in (0, 3):
        assert core(path, align)[0] in (4, 5), label
    for m in (0, 1):
        for piece in (300, 4096):
            for skew in (False, True):
                for w in (1, 7):
                    rc, out = member_core(path, piece, skew, m, w)
                    assert rc in (3, 4), (label, m, piece, skew, w, rc, out)
