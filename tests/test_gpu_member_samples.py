"""Several plain-gzip samples side by side on one device.  Through the library: distinct streams of one
device submitting single- and multi-member files from several host threads at once each count exactly
what the host counter counts.  Through the CLI: when every sample is device-bound (BGZF, or a gzip
file the device takes), four samples per device are in flight and the tables and `Finished:` lines equal
--host-inflate's; a device budget below one sample's scratch bound runs the samples one at a time with
the same table; a run with a host-bound sample keeps its worker count."""
import ctypes as C
import json
import os
import subprocess
import threading
import zlib

import numpy as np
import pytest

import sgcount_b200 as sg
from sgcount_b200 import _cabi, synth

from helpers import make_library, make_reads

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
SEED = 0xB2000017
ENV = ("SGC_MEMBER_PIECE", "SGC_MEMBER_SKEW", "SGC_MEMBER_WAVE_TEXT", "SGC_MEMBER_LANES", "SGC_MULTI_MEMBER_DEVICE",
       "SGC_DEVICE_BUDGET", "SGC_DEVICE_SAMPLES_IN_FLIGHT")


def member(text: bytes, level=6) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, 31)
    return c.compress(text) + c.flush()


def fastq(seqs) -> bytes:
    return b"".join(b"@r%d\n%s\n+\n%s\n" % (i, s, b"I" * len(s)) for i, s in enumerate(seqs))


def device_count():
    n = C.c_int(0)
    return n.value if _cabi.load().sgc_device_count(C.byref(n)) == _cabi.OK else 0


@pytest.fixture(autouse=True)
def clean_env(monkeypatch):
    for name in ENV:
        monkeypatch.delenv(name, raising=False)


# ---- the scratch bound (no device needed) ----

def test_scratch_bound_covers_the_buffers(monkeypatch):
    gz = 250 << 20
    span = sg.fastq_stream_scratch_bound(False, gz, 0, 75, 22)
    variable = sg.fastq_stream_scratch_bound(False, gz, 0, 0, 0)
    # the wave's text (4 GiB in span mode, 3 GiB with reads of any length), its 16-bit symbols, the file
    assert span >= (4 << 30) * 3 + gz and variable >= (3 << 30) * 3 + gz, (span, variable)
    assert span < 24 << 30 and variable < 24 << 30
    # a known text, or a small file, bounds the wave
    assert sg.fastq_stream_scratch_bound(False, gz, 1 << 30, 75, 22) < span
    assert sg.fastq_stream_scratch_bound(False, 1 << 20, 0, 75, 22) < span // 3
    # BGZF: waves of the given compressed and inflated size
    b = sg.fastq_stream_scratch_bound(True, 1 << 30, 4 << 30, 75, 22)
    assert (4 << 30) + (1 << 30) <= b < 12 << 30
    monkeypatch.setenv("SGC_MEMBER_WAVE_TEXT", str(64 << 20))
    assert sg.fastq_stream_scratch_bound(False, gz, 0, 75, 22) < 1 << 30
    with pytest.raises(sg.SgcError):
        sg.fastq_stream_scratch_bound(False, gz, 0, 75, 0)


# ---- the library: several streams of one device from several host threads ----

@pytest.mark.gpu
def test_concurrent_member_submits_equal_host_counter():
    rng = np.random.default_rng(SEED)
    guides = make_library(rng, 400, 20)
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    permuter = sg.Permuter.new(library)
    off = sg.Offset.Forward(5)
    free, total = sg.device_memory(0)
    assert 0 < free <= total
    jobs = []  # (reads, blob, read_len, submit_gzip)
    for i in range(4):
        seqs = make_reads(np.random.default_rng(SEED + i), guides, 40_000, 75, 5, variable=(i == 3))
        text = fastq(seqs)
        if i == 2:  # two members, the cut inside a record
            cut = len(text) // 2 + 17
            jobs.append((seqs, member(text[:cut]) + member(text[cut:]), 75, True))
        else:
            jobs.append((seqs, member(text), 0 if i == 3 else 75, False))
    streams, counters = [], []
    for seqs, blob, read_len, _ in jobs:
        start, length, span_off = sg.span_geometry(20, read_len, off, True) if read_len else (0, 0, off)
        c = sg.Counter(library, permuter, span_off, True)
        counters.append(c)
        streams.append(sg.FastqStream(c, read_len, start, length))
    records, errors = [None] * 4, []
    barrier = threading.Barrier(4)

    def run(i):
        try:
            blob = np.frombuffer(jobs[i][1], dtype=np.uint8)
            barrier.wait()
            (streams[i].submit_gzip if jobs[i][3] else streams[i].submit_member)(blob)
            records[i] = streams[i].finish()
        except Exception as e:  # reported below
            errors.append((i, e))

    threads = [threading.Thread(target=run, args=(i,)) for i in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for i, (seqs, _, _, several) in enumerate(jobs):
        c = sg.Counter(library, permuter, off, True)
        c.submit(sg.ReadBatch.from_seqs(seqs))
        want, got = c.finish(), counters[i].finish()
        assert records[i] == len(seqs), (i, records[i])
        assert np.array_equal(got[0], want[0]) and got[1:] == want[1:], i
        assert streams[i].gzip_members() == (2 if several else 1)


# ---- the CLI ----

def run(*args, env=None):
    p = subprocess.run([BIN, *args], capture_output=True, text=True, timeout=900, env={**os.environ, **(env or {})})
    assert p.returncode == 0, p.stderr
    return p


def timing(proc):
    return json.loads([l for l in proc.stderr.splitlines() if l.startswith("{")][-1])


def finished(proc):
    return [l for l in proc.stderr.splitlines() if l.startswith("Finished:")]


@pytest.fixture(scope="module")
def inputs(tmp_path_factory):
    """a library and single-member gzip samples of several seeds: forward and reverse synthetic reads, reads of
    any length, and fixed-length reads with one read of another length deep in the file; BGZF samples; a
    small two-member file"""
    d = tmp_path_factory.mktemp("member_samples")
    arr = synth.make_library(SEED, 5000, 20)
    lib = str(d / "lib.fa")
    with open(lib, "wb") as f:
        f.write(b"".join(b">lib.%d\n%s\n" % (i, arr[i].tobytes()) for i in range(len(arr))))
    guides = [arr[i].tobytes() for i in range(len(arr))]
    n = 300_000
    out = {"lib": lib, "member": [], "bgzf": []}
    for i, reverse in enumerate((False, True, False, True)):
        path = str(d / f"s{i}.fastq.gz")
        synth.Sample(SEED + i, i, arr, 75, 5 + i, reverse).write_fastq(path, 0, n, reads_per_member=n)
        out["member"].append(path)
    seqs = make_reads(np.random.default_rng(SEED + 10), guides, 30_000, 75, 6, variable=True)
    seqs[0] = next(s for s in seqs if len(s) == 75)  # (the first read sets the length the library is checked against)
    path = str(d / "variable.fastq.gz")
    with open(path, "wb") as f:
        f.write(member(fastq(seqs)))
    out["member"].append(path)
    seqs = make_reads(np.random.default_rng(SEED + 11), guides, 30_000, 75, 4)
    seqs[25_000] = seqs[25_000][:60]  # span mode fails there: the sample starts over with reads of any length
    path = str(d / "odd_read.fastq.gz")
    with open(path, "wb") as f:
        f.write(member(fastq(seqs)))
    out["member"].append(path)
    for i in range(2):
        path = str(d / f"b{i}.fastq.gz")
        synth.Sample(SEED + 20 + i, 20 + i, arr, 75, 5, False).write_fastq_bgzf(path, 0, n)
        out["bgzf"].append(path)
    path = str(d / "two_members.fastq.gz")
    synth.Sample(SEED + 30, 30, arr, 75, 5, False).write_fastq(path, 0, 20_000, reads_per_member=10_000)
    out["two_members"] = path
    return out


def against_host(lib, paths, extra=(), env=None):
    dev = run("-l", lib, "-i", *paths, "--timing", *extra, env=env)
    host = run("-l", lib, "-i", *paths, "--host-inflate", *extra)
    assert dev.stdout == host.stdout
    assert finished(dev) == finished(host) and len(finished(dev)) == len(paths)
    return timing(dev)


@pytest.mark.gpu
def test_cli_all_single_member_samples_in_flight(inputs):
    t = against_host(inputs["lib"], inputs["member"])
    assert t["device_ingest_samples"] == 6 and t["gzip_members"] == 6, t
    assert t["sample_workers"] == min(4 * t["gpus"], 6), t
    assert t["device_samples_in_flight"] >= 2, t
    assert t["span_reads"] < t["reads"], t  # the variable-length samples were counted as whole lines


@pytest.mark.gpu
def test_cli_bgzf_and_single_member_side_by_side(inputs):
    paths = [inputs["bgzf"][0], inputs["member"][0], inputs["bgzf"][1], inputs["member"][1]]
    t = against_host(inputs["lib"], paths)
    assert t["device_ingest_samples"] == 4 and t["device_blocks"] > 0 and t["gzip_members"] == 2, t
    assert t["sample_workers"] == 4 and t["device_samples_in_flight"] >= 2, t


@pytest.mark.gpu
def test_cli_budget_below_one_sample_runs_them_one_at_a_time(inputs):
    paths = inputs["member"][:3] + inputs["bgzf"][:1]
    t = against_host(inputs["lib"], paths, env={"SGC_DEVICE_BUDGET": "1"})
    assert t["device_ingest_samples"] == 4 and t["sample_workers"] == 4, t
    assert t["device_samples_in_flight"] == 1, t


@pytest.mark.gpu
def test_cli_host_bound_sample_keeps_the_worker_count(inputs):
    paths = inputs["member"][:3] + [inputs["two_members"]]
    t = against_host(inputs["lib"], paths)
    assert t["device_ingest_samples"] == 3 and "host" in t["host_ingest_because"], t
    assert t["sample_workers"] == max(1, t["gpus"]), t
    t = against_host(inputs["lib"], paths, extra=("-t", "3"))
    assert t["sample_workers"] == 3, t


@pytest.mark.gpu
@pytest.mark.skipif(device_count() < 2, reason="needs two devices")
def test_cli_two_devices_equal_one(inputs):
    paths = inputs["member"][:4]
    one = run("-l", inputs["lib"], "-i", *paths)
    two = run("-l", inputs["lib"], "-i", *paths, "--gpus", "2", "--timing")
    assert two.stdout == one.stdout and finished(two) == finished(one)
    t = timing(two)
    assert t["gpus"] == 2 and t["device_ingest_samples"] == 4 and t["sample_workers"] == 4, t
