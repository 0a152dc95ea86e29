"""One plain gzip FASTQ (one member or several) decoded by SEVERAL streams together
(sg.submit_gzip_split, sgc_fastq_stream_submit_gzip_split in csrc/gzip.cu): waves dealt round robin,
windows relayed through the host, records framed wave after wave.  The summed counters, totals and
finish() records equal the host path's however the waves cut the records; statistics equal the
one-stream call's; damaged input is reported, never miscounted; the CLI with SGC_MEMBER_LANES prints
what --host-inflate prints."""
import ctypes as C
import json
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

import sgcount_b200 as sg
from sgcount_b200 import _cabi, synth

from helpers import make_library, make_reads
from test_gpu_device_inflate import fastq_text, host_counts
from test_gpu_multi_member_inflate import member, members

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
ENV = ("SGC_MEMBER_PIECE", "SGC_MEMBER_SKEW", "SGC_MEMBER_WAVE_TEXT")


def device_count():
    n = C.c_int(0)
    return n.value if _cabi.load().sgc_device_count(C.byref(n)) == _cabi.OK else 0


def setenv(monkeypatch, env):
    for name in ENV:
        monkeypatch.delenv(name, raising=False)
    for name, v in env.items():
        monkeypatch.setenv(name, v)


def geometry(read_len, k, off):
    return sg.span_geometry(k, read_len, off, True) if read_len else (0, 0, off)


def split_counts(libraries, permuters, blob, read_len, k, off, n):
    """n streams, stream i on libraries[i % len]: (records of each stream, summed counts, members, stats)"""
    start, length, span_off = geometry(read_len, k, off)
    counters = [sg.Counter(libraries[i % len(libraries)], permuters[i % len(libraries)], span_off, True) for i in range(n)]
    streams = [sg.FastqStream(c, read_len, start, length) for c in counters]
    sg.submit_gzip_split(streams, np.frombuffer(blob, dtype=np.uint8))
    records = [s.finish() for s in streams]
    members_, stats = [s.gzip_members() for s in streams], [s.member_stats() for s in streams]
    assert len(set(members_)) == 1 and len(set(stats)) == 1, (members_, stats)
    sg.reduce_counts(counters, 0)
    return records, counters[0].finish(), members_[0], stats[0]


def one_stream(library, permuter, blob, read_len, k, off):
    start, length, span_off = geometry(read_len, k, off)
    c = sg.Counter(library, permuter, span_off, True)
    s = sg.FastqStream(c, read_len, start, length)
    s.submit_gzip(np.frombuffer(blob, dtype=np.uint8))
    return s.finish(), s.gzip_members(), s.member_stats()


def setup(seed, n_reads, devices=(0,)):
    rng = np.random.default_rng(seed)
    guides = make_library(rng, 400, 20)
    seqs = make_reads(rng, guides, n_reads, 75, 5)
    libraries = [sg.Library(guides, [b"g%d" % i for i in range(len(guides))], device=d) for d in devices]
    permuters = [sg.Permuter.new(lib) for lib in libraries]
    off = sg.Offset.Forward(5)
    return seqs, libraries, permuters, off, host_counts(libraries[0], permuters[0], seqs, off)


def cases(seqs):
    text = fastq_text(seqs)
    return [("1 member", member(text), 1, {}),
            ("4 members", members(text, 4, 11), 4, {}),
            ("small pieces, tiny waves", members(text, 3, 12, 1), 3, {"SGC_MEMBER_PIECE": "2000", "SGC_MEMBER_WAVE_TEXT": "20000"}),
            ("waves of one piece", member(text), 1, {"SGC_MEMBER_PIECE": "4096", "SGC_MEMBER_WAVE_TEXT": "1"}),
            ("skewed", members(text, 2, 13, 9), 2, {"SGC_MEMBER_PIECE": "3000", "SGC_MEMBER_SKEW": "1"}),
            ("no final newline", member(text[:-1]), 1, {"SGC_MEMBER_PIECE": "5000", "SGC_MEMBER_WAVE_TEXT": "50000"})]


def check_split(monkeypatch, seqs, libraries, permuters, off, want, n_streams):
    for label, blob, m, env in cases(seqs):
        setenv(monkeypatch, env)
        for mode in (75, 0):
            n1, m1, stats1 = one_stream(libraries[0], permuters[0], blob, mode, 20, off)
            for n in n_streams:
                records, got, n_members, stats = split_counts(libraries, permuters, blob, mode, 20, off, n)
                assert sum(records) == n1 == len(seqs), (label, mode, n, records)
                assert np.array_equal(got[0], want[0]) and got[1:] == want[1:], (label, mode, n)
                assert n_members == m1 == m and stats == stats1, (label, mode, n, stats, stats1)


@pytest.mark.parametrize("n", [2, 3, 5])
def test_split_on_one_device_equals_host_path(monkeypatch, n):
    seqs, libraries, permuters, off, want = setup(31 + n, 20_000)
    check_split(monkeypatch, seqs, libraries, permuters, off, want, (n,))


def test_fewer_waves_than_streams(monkeypatch):
    setenv(monkeypatch, {})
    seqs, libraries, permuters, off, want = setup(37, 300)  # one piece: one wave
    blob = member(fastq_text(seqs))
    for mode in (75, 0):
        records, got, n_members, _ = split_counts(libraries, permuters, blob, mode, 20, off, 5)
        assert records[0] == len(seqs) and records[1:] == [0] * 4, records
        assert np.array_equal(got[0], want[0]) and got[1:] == want[1:]
    # waves of ~20 KB over 5 streams: every wave boundary cuts a record, one stream per wave
    setenv(monkeypatch, {"SGC_MEMBER_PIECE": "1000", "SGC_MEMBER_WAVE_TEXT": "20000"})
    seqs, libraries, permuters, off, want = setup(38, 3000)
    text = fastq_text(seqs)
    c = zlib.compressobj(6, zlib.DEFLATED, 31, 1)  # small blocks: pieces of a few KB
    blob = c.compress(text) + c.flush()
    records, got, _, (pieces, chain, _) = split_counts(libraries, permuters, blob, 75, 20, off, 5)
    assert chain > 10 and sum(records) == len(seqs) and min(records) > 0, (chain, records)
    assert np.array_equal(got[0], want[0]) and got[1:] == want[1:]


def test_split_rejects_mismatched_streams(monkeypatch):
    setenv(monkeypatch, {})
    seqs, libraries, permuters, off, _ = setup(41, 500)
    blob = np.frombuffer(member(fastq_text(seqs)), dtype=np.uint8)
    start, length, span_off = sg.span_geometry(20, 75, off, True)
    a, b = sg.Counter(libraries[0], permuters[0], span_off), sg.Counter(libraries[0], permuters[0], span_off)
    with pytest.raises(sg.SgcError) as e:
        sg.submit_gzip_split([sg.FastqStream(a, 75, start, length), sg.FastqStream(b, 0, 0, 0)], blob)
    assert e.value.code == _cabi.ERR_INVALID_ARG
    other = sg.Library(make_library(np.random.default_rng(5), 300, 20), [b"x%d" % i for i in range(300)])
    c = sg.Counter(other, sg.Permuter.new(other), span_off)
    with pytest.raises(sg.SgcError) as e:
        sg.submit_gzip_split([sg.FastqStream(a, 75, start, length), sg.FastqStream(c, 75, start, length)], blob)
    assert e.value.code == _cabi.ERR_INVALID_ARG
    used = sg.FastqStream(a, 75, start, length)
    used.submit_gzip(blob)
    with pytest.raises(sg.SgcError) as e:
        sg.submit_gzip_split([used, sg.FastqStream(b, 75, start, length)], blob)
    assert e.value.code == _cabi.ERR_INVALID_ARG


def test_damaged_input_is_reported_not_miscounted(monkeypatch):
    setenv(monkeypatch, {"SGC_MEMBER_PIECE": "4096", "SGC_MEMBER_WAVE_TEXT": "100000"})
    seqs, libraries, permuters, off, want = setup(43, 5000)
    text = fastq_text(seqs)
    ms = [member(text[:100000]), member(text[100000:300000]), member(text[300000:])]
    blob = b"".join(ms)
    mid = len(ms[0]) + len(ms[1])
    bad = bytearray(blob)
    bad[len(ms[0]) + len(ms[1]) // 2] ^= 0x10
    damaged = {"crc": blob[:mid - 8] + struct.pack("<I", zlib.crc32(text[100000:300000]) ^ 1) + blob[mid - 4:],
               "truncated": blob[:-5], "flipped": bytes(bad), "truncated record": members(text[:-100], 3, 9)}
    start, length, span_off = sg.span_geometry(20, 75, off, True)
    for label, b in damaged.items():
        streams = [sg.FastqStream(sg.Counter(libraries[0], permuters[0], span_off), 75, start, length) for _ in range(3)]
        with pytest.raises(sg.SgcError) as e:
            sg.submit_gzip_split(streams, np.frombuffer(b, dtype=np.uint8))
            for s in streams:
                s.finish()
        assert e.value.code in (_cabi.ERR_GZIP, _cabi.ERR_FASTQ_FORMAT), (label, e.value.code, str(e.value))
    records, got, n_members, _ = split_counts(libraries, permuters, blob, 75, 20, off, 3)
    assert sum(records) == 5000 and n_members == 3 and np.array_equal(got[0], want[0]) and got[1:] == want[1:]


@pytest.mark.skipif(device_count() < 2, reason="needs two devices")
def test_split_over_devices_equals_host_path(monkeypatch):
    n_dev = device_count()
    seqs, libraries, permuters, off, want = setup(47, 20_000, devices=tuple(range(n_dev)))
    check_split(monkeypatch, seqs, libraries, permuters, off, want, (n_dev, 2 * n_dev + 1))


def run(*args, env=None):
    p = subprocess.run([BIN, *args], capture_output=True, text=True, timeout=600, env={**os.environ, **(env or {})})
    assert p.returncode == 0, p.stderr
    return p


def timing(proc):
    return json.loads([l for l in proc.stderr.splitlines() if l.startswith("{")][-1])


def finished(proc):
    return [l for l in proc.stderr.splitlines() if l.startswith("Finished:")]


def test_cli_member_lanes(tmp_path):
    seed = 0xB2000013
    arr = synth.make_library(seed, 20000, 20)
    lib_path = str(tmp_path / "lib.fa")
    with open(lib_path, "wb") as f:
        f.write(b"".join(b">lib.%d\n%s\n" % (i, arr[i].tobytes()) for i in range(len(arr))))
    sample = synth.Sample(seed, 0, arr, 75, 5, False)
    n = 400_000
    for label, per_member, m in (("one", n, 1), ("two", n // 2, 2)):
        path = str(tmp_path / f"{label}.fastq.gz")
        sample.write_fastq(path, 0, n, reads_per_member=per_member)
        # (SGC_MULTI_MEMBER_DEVICE: a two-member file this small would otherwise stay on the host)
        dev = run("-l", lib_path, "-i", path, "-a", "5", "--timing", env={"SGC_MEMBER_LANES": "3", "SGC_MULTI_MEMBER_DEVICE": "1"})
        t = timing(dev)
        assert t["device_ingest_samples"] == 1 and t["member_lanes"] == 3 and t["gzip_members"] == m, t
        host = run("-l", lib_path, "-i", path, "-a", "5", "--host-inflate")
        assert dev.stdout == host.stdout and finished(dev) == finished(host), label
