"""Plain gzip and BGZF FASTQ with real quality strings, decoded, framed and counted on the device, against
the CPU oracle and the serial reference of the piece path.

The text is what instruments write (helpers.realistic_fastq: Illumina headers of varying length, '+'
lines that repeat the name, Phred+33 qualities drawn per position, some starting with '@' or '+'), so
it inflates from literal-heavy blocks with codes longer than the 7-bit look-ahead, unlike the constant
qualities of the other device tests.  It is compressed by zlib at several levels and strategies, with
pigz-like flushes, as several members, as BGZF, and by tests/deflate_writer.py with matches reaching
the oldest bytes of the window and incomplete distance codes, which zlib never writes.

For every case:
  1. counts, total and matched equal the oracle's over the reads parsed back from the decompressed
     file, and the records finish() reports add up to the file's;
  2. plain gzip: the device declines (ERR_GZIP) exactly when member_core_test, which runs the same
     steps serially, declines the file at the same piece size, skew and members flag; when both
     accept, member_stats() and gzip_members() equal its pieces, chain, absorbed and members;
  3. BGZF is never declined.
The entry points (submit_member, submit_gzip, submit_gzip_split over 1-5 streams), modes and piece /
wave settings are sampled from a fixed seed so that every one of them meets several encodings."""
import gzip
import json
import os
import random
import subprocess
import zlib

import numpy as np
import pytest

import deflate_writer as dw
import sgcount_b200 as sg
from sgcount_b200 import _cabi

from helpers import make_library, make_reads, realistic_fastq
from test_gpu_device_inflate import device_counts
from test_gpu_parity import oracle_count
from test_member_inflate_core import EXE as MEMBER_EXE

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
N_READS = 40_000
ENV_NAMES = ("SGC_MEMBER_PIECE", "SGC_MEMBER_SKEW", "SGC_MEMBER_WAVE_TEXT")
SETTINGS = [{}, {"SGC_MEMBER_PIECE": "4096"}, {"SGC_MEMBER_PIECE": "2000", "SGC_MEMBER_SKEW": "1"},
            {"SGC_MEMBER_WAVE_TEXT": "20000"}, {"SGC_MEMBER_PIECE": "4096", "SGC_MEMBER_WAVE_TEXT": "1"}]
ENTRIES = ["member", "gzip", "split1", "split2", "split3", "split5"]
FAR = [d for d in dw.EDGE_DISTS if d > 32506]


def member(text, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, memlevel=8):
    c = zlib.compressobj(level, zlib.DEFLATED, 31, memlevel, strategy)
    return c.compress(text) + c.flush()


def flushed(text, mode, every=128 << 10):
    """pigz-like: a sync or full flush every 128 KiB of input"""
    c = zlib.compressobj(6, zlib.DEFLATED, 31)
    return b"".join(c.compress(text[i:i + every]) + c.flush(mode) for i in range(0, len(text), every)) + c.flush()


def members(text, m, seed):
    """m members cut at random bytes (records straddle them); with m >= 5 one of them is empty"""
    rng = random.Random(seed)
    at = sorted(rng.randrange(1, len(text)) for _ in range(m - 1))
    if m >= 5:
        at[m // 2] = at[m // 2 - 1]
    return b"".join(member(text[a:b], rng.choice([1, 6, 9])) for a, b in zip([0] + at, at + [len(text)]))


def far_stream(text, slots, seed):
    """the writer's stream: matches at every distance beyond zlib's reach, mixed block kinds"""
    rng = random.Random(seed)
    buf = bytearray(text)
    force = dw.plant(buf, rng, slots, [(FAR, list(range(3, 19)), 400), ([32768], [3, 8, 30], 60)])
    text = bytes(buf)
    tokens = dw.parse(text, force=force)
    body = dw.deflate(tokens, dw.layout(len(tokens), rng, ("dynamic",) * 4 + ("fixed", "stored", "empty"), (100, 20000)), text)
    return dw.gzip_member(body, text)


def bgzf(text, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, block=0xFF00):
    out = []
    for i in range(0, len(text), block):
        c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
        out.append(dw.bgzf_member(c.compress(text[i:i + block]) + c.flush(), text[i:i + block]))
    return b"".join(out) + dw.BGZF_EOF


def writer_bgzf(text, slots, seed, block=0xFF00):
    """the writer's BGZF: blocks of 65 280 bytes, each with matches at distance 32 768 inside it"""
    rng = random.Random(seed)
    buf = bytearray(text)
    dw.plant(buf, rng, slots, [([32768], [3, 10, 40], 3 * len(text) // block), (FAR, [4, 12], len(text) // block)], block=block)
    text = bytes(buf)
    out = []
    for i in range(0, len(text), block):
        part = text[i:i + block]
        tokens = dw.parse(part)
        out.append(dw.bgzf_member(dw.deflate(tokens, dw.layout(len(tokens), rng, ("dynamic", "dynamic", "fixed"), (500, 8000)), part),
                                  part))
    return b"".join(out) + dw.BGZF_EOF


class World:
    def __init__(self, tmp):
        rng = np.random.default_rng(0x5EED)
        self.guides = make_library(rng, 600, 20)
        self.library = sg.Library(self.guides, [b"g%d" % i for i in range(len(self.guides))])
        self.permuter = sg.Permuter.new(self.library)
        self.off = sg.Offset.Forward(5)
        fixed, fslots = realistic_fastq(rng, make_reads(rng, self.guides, N_READS, 75, 5))
        trimmed, tslots = realistic_fastq(rng, make_reads(rng, self.guides, N_READS, 75, 5, variable=True))
        self.tmp = tmp
        # name: (blob, modes); 75 = span mode, 0 = reads of any length
        self.plain = {"l1": (member(fixed, 1), (75, 0)), "l6": (member(fixed, 6), (75, 0)), "l9": (member(fixed, 9), (75, 0)),
                      "filtered": (member(fixed, 6, zlib.Z_FILTERED), (75, 0)),
                      "huffman_only": (member(fixed, 6, zlib.Z_HUFFMAN_ONLY), (75, 0)), "rle": (member(fixed, 6, zlib.Z_RLE), (75, 0)),
                      "memlevel1": (member(fixed, 6, memlevel=1), (75, 0)),
                      "sync_flush": (flushed(fixed, zlib.Z_SYNC_FLUSH), (75, 0)), "full_flush": (flushed(fixed, zlib.Z_FULL_FLUSH), (75,)),
                      "fixed": (member(fixed, 6, zlib.Z_FIXED), (75, 0)), "stored": (member(fixed, 0), (75,)),
                      "far": (far_stream(fixed, fslots, 1), (75, 0)),
                      "members2": (members(fixed, 2, 2), (75, 0)), "members5": (members(fixed, 5, 5), (75,)),
                      "members16": (members(fixed, 16, 16), (75, 0)),
                      "trimmed_l6": (member(trimmed, 6), (0,)), "trimmed_far": (far_stream(trimmed, tslots, 3), (0,)),
                      "trimmed_members5": (members(trimmed, 5, 7), (0,))}
        self.bgzf = {"l6": (bgzf(fixed), (75, 0)), "fixed": (bgzf(fixed, strategy=zlib.Z_FIXED), (75,)),
                     "stored": (bgzf(fixed, 0), (75,)), "writer": (writer_bgzf(fixed, fslots, 4), (75, 0)),
                     "trimmed_l6": (bgzf(trimmed), (0,))}
        self.paths, self.oracles, self.harness = {}, {}, {}

    def path(self, name, blob):
        if name not in self.paths:
            self.paths[name] = self.tmp / f"{name}.gz"
            self.paths[name].write_bytes(blob)
        return self.paths[name]

    def oracle(self, text):
        """(counts, total, matched) of the oracle over the reads parsed back from the text"""
        key = (len(text), zlib.crc32(text))
        if key not in self.oracles:
            lines = text.split(b"\n")
            assert lines[-1] == b"" and len(lines) % 4 == 1
            seqs = lines[1::4]
            _, counts, total, matched = oracle_count(self.guides, seqs, True, self.off)
            self.oracles[key] = (counts, total, matched, len(seqs))
        return self.oracles[key]

    def reference(self, name, blob, piece, skew, members_flag):
        """member_core_test on the file: None (decline) or (pieces, chain, absorbed, members)"""
        key = (name, piece, skew, members_flag)
        if key not in self.harness:
            p = subprocess.run([MEMBER_EXE, str(self.path(name, blob)), str(piece), str(int(skew)), str(members_flag)],
                               capture_output=True, text=True, timeout=600)
            assert p.returncode in (0, 3), (name, piece, skew, p.returncode, p.stdout)
            f = p.stdout.split()
            self.harness[key] = None if p.returncode == 3 else (int(f[2]), int(f[3]), int(f[4]), int(f[5]) if members_flag else 1)
        return self.harness[key]


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    if not os.path.exists(MEMBER_EXE):
        import __graft_entry__ as g

        g.build()
    return World(tmp_path_factory.mktemp("realistic"))


def geometry(read_len, off):
    return sg.span_geometry(20, read_len, off, True) if read_len else (0, 0, off)


def run_plain(w, blob, mode, entry):
    """(records, (counts, total, matched), members, stats) of one device run, or the SgcError"""
    start, length, span_off = geometry(mode, w.off)
    arr = np.frombuffer(blob, dtype=np.uint8)
    n = int(entry[5:]) if entry.startswith("split") else 1
    counters = [sg.Counter(w.library, w.permuter, span_off, True) for _ in range(n)]
    streams = [sg.FastqStream(c, mode, start, length) for c in counters]
    try:
        if entry == "member":
            streams[0].submit_member(arr)
        elif entry == "gzip":
            streams[0].submit_gzip(arr)
        else:
            sg.submit_gzip_split(streams, arr)
        records = sum(s.finish() for s in streams)
    except sg.SgcError as e:
        return e
    stats = {s.member_stats() for s in streams}
    m = {s.gzip_members() for s in streams}
    assert len(stats) == 1 and len(m) == 1, (stats, m)
    sg.reduce_counts(counters, 0)
    return records, counters[0].finish(), m.pop(), stats.pop()


def plan(w):
    """(name, mode, entry, setting) for every plain file: two sampled per file and mode"""
    rng = random.Random(20261022)
    out = []
    for name, (blob, modes) in w.plain.items():
        one = len(members_list(blob)) == 1
        for mode in modes:
            for entry, setting in rng.sample([(e, s) for e in ENTRIES if one or e != "member" for s in range(len(SETTINGS))], 2):
                out.append((name, mode, entry, setting))
    assert {e for _, _, e, _ in out} == set(ENTRIES) and {s for *_, s in out} == set(range(len(SETTINGS)))
    return out


def members_list(blob):
    out = []
    while blob:
        d = zlib.decompressobj(31)
        out.append(d.decompress(blob))
        assert d.eof
        blob = d.unused_data
    return out


def test_plain_gzip_equals_oracle_and_reference(world, monkeypatch):
    w = world
    declined = accepted = 0
    for name, mode, entry, setting in plan(w):
        blob = w.plain[name][0]
        env = SETTINGS[setting]
        for k in ENV_NAMES:
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        label = (name, mode, entry, env)
        piece, skew = int(env.get("SGC_MEMBER_PIECE", 32768)), env.get("SGC_MEMBER_SKEW") == "1"
        ref = w.reference(name, blob, piece, skew, 0 if entry == "member" else 1)
        got = run_plain(w, blob, mode, entry)
        if isinstance(got, sg.SgcError):
            assert got.code == _cabi.ERR_GZIP and ref is None, (label, got.code, str(got), ref)
            declined += 1
            continue
        assert ref is not None, (label, "the device decodes what the reference declines")
        records, (counts, total, matched), m, stats = got
        want_counts, want_total, want_matched, n_records = w.oracle(b"".join(members_list(blob)))
        assert records == n_records == want_total, (label, records, n_records)
        assert np.array_equal(counts, want_counts) and (total, matched) == (want_total, want_matched), label
        assert stats + (m,) == ref, (label, stats, m, ref)
        accepted += 1
    assert accepted > 2 * declined, (accepted, declined)


@pytest.mark.parametrize("name", ["l6", "fixed", "stored", "writer", "trimmed_l6"])
def test_bgzf_equals_oracle_and_is_never_declined(world, monkeypatch, name):
    w = world
    for k in ENV_NAMES:
        monkeypatch.delenv(k, raising=False)
    blob, modes = w.bgzf[name]
    want_counts, want_total, want_matched, n_records = w.oracle(gzip.decompress(blob))
    for mode in modes:
        for wave in (1, 7, 64):
            n, (counts, total, matched) = device_counts(w.library, w.permuter, blob, mode, 20, w.off, wave=wave)
            assert n == n_records == want_total, (name, mode, wave)
            assert np.array_equal(counts, want_counts) and (total, matched) == (want_total, want_matched), (name, mode, wave)
    # through the plain-gzip path (every block a member): as the reference decides
    got = run_plain(w, blob, modes[0], "gzip")
    ref = w.reference("bgzf_" + name, blob, 32768, False, 1)
    if isinstance(got, sg.SgcError):
        assert ref is None, (name, str(got))
    else:
        assert ref is not None and got[3] + (got[2],) == ref and got[0] == n_records, (name, got[2:], ref)
        assert np.array_equal(got[1][0], want_counts)


def run_cli(*args, env=None):
    p = subprocess.run([BIN, *args], capture_output=True, text=True, timeout=900, env={**os.environ, **(env or {})})
    assert p.returncode == 0, p.stderr
    return p


def timing(proc):
    return json.loads([l for l in proc.stderr.splitlines() if l.startswith("{")][-1])


def finished(proc):
    return [l for l in proc.stderr.splitlines() if l.startswith("Finished:")]


def test_cli_takes_realistic_files_to_the_device(world, tmp_path):
    w = world
    lib = tmp_path / "lib.fa"
    lib.write_bytes(b"".join(b">g%d\n%s\n" % (i, g) for i, g in enumerate(w.guides)))
    rng = np.random.default_rng(77)
    text, _ = realistic_fastq(rng, make_reads(rng, w.guides, 200_000, 75, 5))
    cases = [("one.fastq.gz", member(text), {}), ("two.fastq.gz", members(text, 2, 3),
                                                 {"SGC_MULTI_MEMBER_DEVICE": "1", "SGC_MEMBER_LANES": "3"}),
             ("writer_bgzf.fastq.gz", w.bgzf["writer"][0], {})]
    for name, blob, env in cases:
        path = tmp_path / name
        path.write_bytes(blob)
        dev = run_cli("-l", str(lib), "-i", str(path), "-a", "5", "--timing", env=env)
        assert timing(dev)["device_ingest_samples"] == 1, (name, timing(dev))
        host = run_cli("-l", str(lib), "-i", str(path), "-a", "5", "--host-inflate")
        assert dev.stdout == host.stdout and finished(dev) == finished(host), name
