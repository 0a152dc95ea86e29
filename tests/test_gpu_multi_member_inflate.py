"""gzip files of SEVERAL members that are not BGZF (`cat a.gz b.gz`, appending writers) inflated in
speculative pieces across member boundaries, framed and counted on the device (FastqStream.submit_gzip,
csrc/gzip.cu): the counts, totals and record count of the host path however the members cut the text;
BGZF through submit_gzip counts as through submit; irregular input is reported, never miscounted; the
CLI takes a large two-member file to the device unless read shards or --host-inflate are asked for."""
import json
import os
import random
import struct
import subprocess
import zlib

import numpy as np
import pytest

import sgcount_b200 as sg
from sgcount_b200 import _cabi, synth

from helpers import make_library, make_reads
from test_gpu_device_inflate import bgzf, device_counts, fastq_text, host_counts

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
ENV = ("SGC_MEMBER_PIECE", "SGC_MEMBER_SKEW", "SGC_MEMBER_WAVE_TEXT")


def member(text: bytes, level=6) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, 31)
    return c.compress(text) + c.flush()


def members(text: bytes, m: int, seed: int, level=6) -> bytes:
    """m members whose texts are `text` cut at random bytes (records straddle the boundaries)"""
    rng = random.Random(seed)
    at = sorted(rng.randrange(1, len(text)) for _ in range(m - 1))
    return b"".join(member(text[a:b], level) for a, b in zip([0] + at, at + [len(text)]))


def gzip_counts(library, permuter, blob, read_len, k, off, recursion=True):
    if read_len:
        start, length, span_off = sg.span_geometry(k, read_len, off, recursion)
    else:
        start, length, span_off = 0, 0, off
    c = sg.Counter(library, permuter, span_off, recursion)
    stream = sg.FastqStream(c, read_len, start, length)
    stream.submit_gzip(np.frombuffer(blob, dtype=np.uint8))
    n = stream.finish()
    return n, c.finish(), stream.gzip_members(), stream.member_stats()


def setenv(monkeypatch, env):
    for name in ENV:
        monkeypatch.delenv(name, raising=False)
    for name, v in env.items():
        monkeypatch.setenv(name, v)


@pytest.mark.parametrize("reverse,offset,k", [(False, 5, 20), (True, 12, 20)])
def test_gzip_members_equal_host_path(monkeypatch, reverse, offset, k):
    rng = np.random.default_rng(91 + offset)
    guides = make_library(rng, 500, k)
    read_len = 75
    seqs = make_reads(rng, guides, 30_000, read_len, offset, reverse, False, wild=b"J" if reverse else b"N")
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    permuter = sg.Permuter.new(library)
    off = sg.Offset(reverse, offset)
    want = host_counts(library, permuter, seqs, off)
    text = fastq_text(seqs)
    # a middle member that ends just before a newline, and one that ends on a record boundary
    nl = text.index(b"\n", len(text) // 2)
    rec = text.index(b"\n@", len(text) // 3) + 1
    cases = [("1 member", member(text), 1, {}), ("2 members", members(text, 2, 1), 2, {}),
             ("7 members l1 small pieces", members(text, 7, 2, 1), 7, {"SGC_MEMBER_PIECE": "2000"}),
             ("40 members skewed", members(text, 40, 3, 9), 40, {"SGC_MEMBER_PIECE": "3000", "SGC_MEMBER_SKEW": "1"}),
             ("7 members small waves", members(text, 7, 4), 7, {"SGC_MEMBER_PIECE": "4096", "SGC_MEMBER_WAVE_TEXT": "300000"}),
             ("no final newline mid", member(text[:rec]) + member(text[rec:nl]) + member(text[nl:]), 3, {"SGC_MEMBER_PIECE": "5000"}),
             ("empty members", member(b"") + members(text, 3, 5) + member(b""), 5, {})]
    for label, blob, m, env in cases:
        setenv(monkeypatch, env)
        for mode in (read_len, 0):
            n, got, n_members, (pieces, chain, absorbed) = gzip_counts(library, permuter, blob, mode, k, off)
            assert n == len(seqs), (label, mode)
            assert np.array_equal(got[0], want[0]) and got[1:] == want[1:], (label, mode)
            assert n_members == m, (label, n_members)
            assert chain >= m, (label, pieces, chain)
            if "SKEW" in env:
                assert absorbed > 0, (label, pieces, chain, absorbed)


def test_bgzf_through_submit_gzip_counts_as_through_submit(monkeypatch):
    setenv(monkeypatch, {})
    rng = np.random.default_rng(17)
    guides = make_library(rng, 300, 20)
    seqs = make_reads(rng, guides, 20_000, 75, 5)
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    permuter = sg.Permuter.new(library)
    off = sg.Offset.Forward(5)
    blob = bgzf(fastq_text(seqs))
    for mode in (75, 0):
        n_ref, want = device_counts(library, permuter, blob, mode, 20, off)
        n, got, n_members, _ = gzip_counts(library, permuter, blob, mode, 20, off)
        assert n == n_ref == len(seqs)
        assert np.array_equal(got[0], want[0]) and got[1:] == want[1:]
        assert n_members == len(sg.bgzf_blocks(blob)[1])


def test_irregular_input_is_reported_not_miscounted(monkeypatch):
    setenv(monkeypatch, {"SGC_MEMBER_PIECE": "4096"})
    rng = np.random.default_rng(19)
    guides = make_library(rng, 100, 20)
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    permuter = sg.Permuter.new(library)
    seqs = make_reads(rng, guides, 5000, 75, 5)
    off = sg.Offset.Forward(5)

    def fails(blob, codes=(_cabi.ERR_GZIP, _cabi.ERR_FASTQ_FORMAT)):
        with pytest.raises(sg.SgcError) as e:
            gzip_counts(library, permuter, blob, 75, 20, off)
        assert e.value.code in codes, (e.value.code, str(e.value))

    text = fastq_text(seqs)
    ms = [member(text[:100000]), member(text[100000:300000]), member(text[300000:])]
    blob = b"".join(ms)
    mid = len(ms[0]) + len(ms[1])
    odd = list(seqs)
    odd[3777] = odd[3777][:60]
    fails(members(fastq_text(odd), 3, 7), codes=(_cabi.ERR_FASTQ_FORMAT,))  # a read of another length in span mode
    fails(members(b"".join(b">r\n%s\n" % s for s in seqs), 3, 8), codes=(_cabi.ERR_FASTQ_FORMAT,))  # FASTA
    fails(members(text[:-100], 3, 9), codes=(_cabi.ERR_FASTQ_FORMAT,))  # a truncated record
    fails(blob[:mid - 8] + struct.pack("<I", zlib.crc32(text[100000:300000]) ^ 1) + blob[mid - 4:], codes=(_cabi.ERR_GZIP,))
    fails(blob[:mid - 4] + struct.pack("<I", 200001) + blob[mid:], codes=(_cabi.ERR_GZIP,))  # ISIZE
    fails(blob + b"\0" * 64, codes=(_cabi.ERR_GZIP,))  # zero padding
    fails(blob + b"trailing", codes=(_cabi.ERR_GZIP,))
    fails(blob[:-5], codes=(_cabi.ERR_GZIP,))  # a truncated last member
    bad = bytearray(blob)
    bad[len(ms[0]) + len(ms[1]) // 2] ^= 0x10  # a flipped bit inside the middle member
    fails(bytes(bad))
    n, got, n_members, _ = gzip_counts(library, permuter, blob, 75, 20, off)
    want = host_counts(library, permuter, seqs, off)
    assert n == 5000 and n_members == 3 and np.array_equal(got[0], want[0]) and got[1:] == want[1:]


def run(*args):
    p = subprocess.run([BIN, *args], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    return p


def timing(proc):
    return json.loads([l for l in proc.stderr.splitlines() if l.startswith("{")][-1])


def finished(proc):
    return [l for l in proc.stderr.splitlines() if l.startswith("Finished:")]


def test_cli_two_members_on_the_device(tmp_path):
    seed = 0xB2000011
    arr = synth.make_library(seed, 77441, 20)
    lib_path = str(tmp_path / "lib.fa")
    with open(lib_path, "wb") as f:
        f.write(b"".join(b">lib.%d\n%s\n" % (i, arr[i].tobytes()) for i in range(len(arr))))
    sample = synth.Sample(seed, 0, arr, 75, 5, False)
    n = 6_000_000  # ~90 MB of gzip: above the size below which several members stay on the host
    two = str(tmp_path / "two.fastq.gz")
    sample.write_fastq(two, 0, n, reads_per_member=n // 2)
    assert os.path.getsize(two) >= 64 << 20
    dev = run("-l", lib_path, "-i", two, "-a", "5", "--timing")
    t = timing(dev)
    assert t["device_ingest_samples"] == 1 and t["gzip_members"] == 2, t
    host = run("-l", lib_path, "-i", two, "-a", "5", "--timing", "--host-inflate")
    assert timing(host)["device_ingest_samples"] == 0
    assert dev.stdout == host.stdout and finished(dev) == finished(host)
    library = sg.Library([arr[i].tobytes() for i in range(len(arr))], [b"lib.%d" % i for i in range(len(arr))])
    want = sg.Counter(library, sg.Permuter.new(library), sg.Offset.Forward(5))
    want.submit(sg.ReadBatch(sample.fill_host(0, n), n, None, 76, 75))
    counts, total, matched = want.finish()
    rows = {r.split("\t")[0]: int(r.split("\t")[1]) for r in dev.stdout.rstrip("\n").split("\n")[1:]}
    assert rows == {f"lib.{i}": int(c) for i, c in enumerate(counts) if c}
    assert total == n and f"[{matched} / {n}]" in dev.stderr
    shards = run("-l", lib_path, "-i", two, "-a", "5", "--timing", "--read-shards", "2")
    assert timing(shards)["device_ingest_samples"] == 0 and timing(shards)["gzip_members"] == 0
    assert shards.stdout == dev.stdout
