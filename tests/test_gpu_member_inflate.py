"""ONE gzip member that is not BGZF (what gzip and pigz write), inflated in speculative pieces, framed
and counted on the device (FastqStream.submit_member, csrc/gzip.cu member_* kernels): the counts,
totals and record count of the host path whatever the compression level, piece size, wrong candidate
starts and wave size; irregular input reported, never miscounted; the CLI takes single-member files
to the device and leaves multi-member files on the host."""
import gzip
import json
import os
import subprocess
import zlib

import numpy as np
import pytest

import sgcount_b200 as sg
from sgcount_b200 import _cabi, synth

from helpers import make_library, make_reads
from test_gpu_device_inflate import fastq_text, host_counts

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
EXAMPLE = os.path.join(ROOT, "tests", "golden", "example")


def member(text: bytes, level=6) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, 31)
    return c.compress(text) + c.flush()


def member_counts(library, permuter, blob, read_len, k, off, recursion=True):
    if read_len:
        start, length, span_off = sg.span_geometry(k, read_len, off, recursion)
    else:
        start, length, span_off = 0, 0, off
    c = sg.Counter(library, permuter, span_off, recursion)
    stream = sg.FastqStream(c, read_len, start, length)
    stream.submit_member(np.frombuffer(blob, dtype=np.uint8))
    n = stream.finish()
    return n, c.finish(), stream.member_stats()


@pytest.mark.parametrize("reverse,offset,k", [(False, 5, 20), (True, 12, 20), (False, 0, 16), (True, 31, 24)])
def test_member_equals_host_path(monkeypatch, reverse, offset, k):
    rng = np.random.default_rng(71 + offset)
    guides = make_library(rng, 500, k)
    read_len = 75
    seqs = make_reads(rng, guides, 30_000, read_len, offset, reverse, False, wild=b"J" if reverse else b"N")
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    permuter = sg.Permuter.new(library)
    off = sg.Offset(reverse, offset)
    want = host_counts(library, permuter, seqs, off)
    text = fastq_text(seqs)
    cases = [("l6", 6, {}), ("l1 small pieces", 1, {"SGC_MEMBER_PIECE": "2000"}),
             ("l9 skewed", 9, {"SGC_MEMBER_PIECE": "3000", "SGC_MEMBER_SKEW": "1"}),
             ("l6 small waves", 6, {"SGC_MEMBER_PIECE": "4096", "SGC_MEMBER_WAVE_TEXT": "300000"}),
             ("no final newline", 6, {"SGC_MEMBER_PIECE": "5000"})]
    for label, level, env in cases:
        for name in ("SGC_MEMBER_PIECE", "SGC_MEMBER_SKEW", "SGC_MEMBER_WAVE_TEXT"):
            monkeypatch.delenv(name, raising=False)
        for name, v in env.items():
            monkeypatch.setenv(name, v)
        body = text[:-1] if label == "no final newline" else text
        for read_len_mode in (read_len, 0):
            n, got, (pieces, chain, absorbed) = member_counts(library, permuter, member(body, level), read_len_mode, k, off)
            assert n == len(seqs), label
            assert np.array_equal(got[0], want[0]) and got[1:] == want[1:], (label, read_len_mode)
            if "PIECE" in str(env):  # (pieces can only start at true block starts: a few dozen here)
                assert chain > 1, (label, pieces, chain)
            if "SKEW" in env:
                assert absorbed > 0, (label, pieces, chain, absorbed)


def test_irregular_input_is_reported_not_miscounted(monkeypatch):
    monkeypatch.setenv("SGC_MEMBER_PIECE", "4096")
    rng = np.random.default_rng(9)
    guides = make_library(rng, 100, 20)
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    permuter = sg.Permuter.new(library)
    seqs = make_reads(rng, guides, 5000, 75, 5)
    off = sg.Offset.Forward(5)

    def fails(blob, read_len=75, codes=(_cabi.ERR_GZIP, _cabi.ERR_FASTQ_FORMAT)):
        with pytest.raises(sg.SgcError) as e:
            member_counts(library, permuter, blob, read_len, 20, off)
        assert e.value.code in codes
        return e.value

    odd = list(seqs)
    odd[3777] = odd[3777][:60]
    fails(member(fastq_text(odd)), codes=(_cabi.ERR_FASTQ_FORMAT,))  # a read of another length in span mode
    fails(member(b"".join(b">r\n%s\n" % s for s in seqs)), codes=(_cabi.ERR_FASTQ_FORMAT,))  # FASTA
    fails(member(fastq_text(seqs)[:-100]), codes=(_cabi.ERR_FASTQ_FORMAT,))  # a truncated record
    blob = member(fastq_text(seqs))
    fails(blob + member(b"@x\nACGT\n+\nIIII\n"), codes=(_cabi.ERR_GZIP,))  # a second member
    bad = bytearray(blob)
    bad[len(bad) // 2] ^= 0x10  # a flipped bit in a Huffman block
    fails(bytes(bad))
    stored = bytearray(member(fastq_text(seqs), 0))
    stored[len(stored) // 2] ^= 0x01  # in a stored block's bytes: only the CRC-32 sees it
    e = fails(bytes(stored))
    if e.code == _cabi.ERR_GZIP:
        assert "CRC-32" in str(e) or "pieces" in str(e)
    n, got, _ = member_counts(library, permuter, blob, 75, 20, off)
    want = host_counts(library, permuter, seqs, off)
    assert n == 5000 and np.array_equal(got[0], want[0]) and got[1:] == want[1:]


def run(*args):
    p = subprocess.run([BIN, *args], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    return p


def timing(proc):
    return json.loads([l for l in proc.stderr.splitlines() if l.startswith("{")][-1])


def test_cli_golden_fixtures_on_the_device(expected):
    lib = os.path.join(EXAMPLE, "library.fasta.gz")
    for name in ["sequence", "zero.sequence", "diff.sequence", "offset", "offset_clipped"]:
        path = os.path.join(EXAMPLE, name + ".fastq.gz")
        dev = run("-l", lib, "-i", path, "--timing", "-z")
        host = run("-l", lib, "-i", path, "--timing", "-z", "--host-inflate")
        assert timing(dev)["device_ingest_samples"] == 1, (name, timing(dev))
        assert timing(host)["device_ingest_samples"] == 0
        assert dev.stdout == host.stdout, name
        fx = expected["fixtures"][name]
        rows = dev.stdout.rstrip("\n").split("\n")[1:]
        assert [int(r.split("\t")[1]) for r in rows] == list(fx["counts"]), name
        assert f"[{fx['matched_reads']} / {fx['total_reads']}]" in dev.stderr


def test_cli_single_member_synthetic_and_multi_member_routing(tmp_path):
    seed = 0xB2000007
    arr = synth.make_library(seed, 77441, 20)
    lib_path = str(tmp_path / "lib.fa")
    with open(lib_path, "wb") as f:
        f.write(b"".join(b">lib.%d\n%s\n" % (i, arr[i].tobytes()) for i in range(len(arr))))
    sample = synth.Sample(seed, 0, arr, 75, 5, False)
    n = 1_000_000
    one = str(tmp_path / "one.fastq.gz")
    sample.write_fastq(one, 0, n, reads_per_member=n)
    dev = run("-l", lib_path, "-i", one, "-a", "5", "--timing")
    t = timing(dev)
    assert t["device_ingest_samples"] == 1 and t["member_chain"] > 100, t
    # the oracle's table: the host counter over the same reads
    library = sg.Library([arr[i].tobytes() for i in range(len(arr))], [b"lib.%d" % i for i in range(len(arr))])
    want = sg.Counter(library, sg.Permuter.new(library), sg.Offset.Forward(5))
    want.submit(sg.ReadBatch(sample.fill_host(0, n), n, None, 76, 75))
    counts, total, matched = want.finish()
    rows = {r.split("\t")[0]: int(r.split("\t")[1]) for r in dev.stdout.rstrip("\n").split("\n")[1:]}
    assert rows == {f"lib.{i}": int(c) for i, c in enumerate(counts) if c}
    assert total == n and f"[{matched} / {n}]" in dev.stderr
    # several members: the host path, as before
    multi = str(tmp_path / "multi.fastq.gz")
    sample.write_fastq(multi, 0, 200_000, reads_per_member=50_000)
    m = run("-l", lib_path, "-i", multi, "-a", "5", "--timing")
    assert timing(m)["device_ingest_samples"] == 0
    assert "member" in timing(m)["host_ingest_because"]
    assert gzip.decompress(open(multi, "rb").read()).count(b"\n") == 800_000
