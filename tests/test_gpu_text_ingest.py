"""Uncompressed FASTQ framed and counted on the device (FastqStream.submit_text, sgc_fastq_stream_submit_text
in csrc/gzip.cu).  Through the library: span mode and line mode count exactly what the host counter counts,
whether a file comes in one call or in many cut anywhere, over many internal waves (SGC_TEXT_WAVE), from
several streams and threads at once or from an np.memmap; irregular text is declined, never miscounted.
Through the CLI: plain .fastq / .fq samples go to the device by default and print what --host-inflate
prints; FASTA stays on the host; plain, BGZF and gzip samples run side by side; read shards cut the text
at record ends."""
import ctypes as C
import json
import os
import subprocess
import threading

import numpy as np
import pytest

import sgcount_b200 as sg
from sgcount_b200 import _cabi, synth

from helpers import make_library, make_reads, realistic_fastq

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
SEED = 0xB2000019
ENV = ("SGC_TEXT_WAVE", "SGC_DEVICE_BUDGET", "SGC_DEVICE_SAMPLES_IN_FLIGHT", "SGC_MEMBER_WAVE_TEXT")


def fastq(seqs, final_newline=True) -> bytes:
    text = b"".join(b"@r%d\n%s\n+\n%s\n" % (i, s, b"I" * len(s)) for i, s in enumerate(seqs))
    return text if final_newline else text[:-1]


def device_count():
    n = C.c_int(0)
    return n.value if _cabi.load().sgc_device_count(C.byref(n)) == _cabi.OK else 0


@pytest.fixture(autouse=True)
def clean_env(monkeypatch):
    for name in ENV:
        monkeypatch.delenv(name, raising=False)


# ---- the scratch bound (no device needed) ----

def test_text_scratch_bound_covers_two_waves(monkeypatch):
    span = sg.fastq_stream_text_scratch_bound(75, 22)
    line = sg.fastq_stream_text_scratch_bound(0, 0)
    wave = 64 << 20
    # two text buffers of one wave each, plus a span record (24 bytes a 75 bp read) or two line offsets a record
    assert span >= 2 * wave + wave // 81 * 24 and line >= 2 * wave + wave // 6 * 8, (span, line)
    assert span < 2 << 30 and line < 2 << 30
    monkeypatch.setenv("SGC_TEXT_WAVE", str(1 << 20))
    assert sg.fastq_stream_text_scratch_bound(75, 22) < span - wave
    assert sg.fastq_stream_text_scratch_bound(0, 0) < line - wave
    with pytest.raises(sg.SgcError):
        sg.fastq_stream_text_scratch_bound(75, 0)


# ---- the library ----

K = 20


def library_of(seed, devices=(0,)):
    rng = np.random.default_rng(seed)
    guides = make_library(rng, 400, K)
    libraries = [sg.Library(guides, [b"g%d" % i for i in range(len(guides))], device=d) for d in devices]
    return guides, libraries, [sg.Permuter.new(lib) for lib in libraries]


def host_counts(library, permuter, seqs, off):
    c = sg.Counter(library, permuter, off, True)
    c.submit(sg.ReadBatch.from_seqs(seqs))
    return c.finish()


def text_stream(library, permuter, read_len, off):
    """(counter, stream): read_len > 0 span mode, 0 line mode"""
    if read_len:
        start, length, span_off = sg.span_geometry(K, read_len, off, True)
        c = sg.Counter(library, permuter, span_off, True)
        return c, sg.FastqStream(c, read_len, start, length)
    c = sg.Counter(library, permuter, off, True)
    return c, sg.FastqStream(c, 0, 0, 0)


def count_text(library, permuter, text, read_len, off, cuts=None):
    """the text in calls [cuts[i], cuts[i + 1]) on one stream: (records, counts)"""
    c, s = text_stream(library, permuter, read_len, off)
    blob = np.frombuffer(text, dtype=np.uint8)
    cuts = [0, len(text)] if cuts is None else [0, *cuts, len(text)]
    for a, b in zip(cuts[:-1], cuts[1:]):
        s.submit_text(blob[a:b])
    return s.finish(), c.finish()


def same(got, want):
    return np.array_equal(got[0], want[0]) and got[1:] == want[1:]


@pytest.mark.gpu
@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("realistic", [False, True])
def test_one_call_equals_host_counter(reverse, realistic):
    guides, (library,), (permuter,) = library_of(SEED)
    off = sg.Offset.Reverse(6) if reverse else sg.Offset.Forward(6)
    seqs = make_reads(np.random.default_rng(SEED + 1), guides, 60_000, 75, 6, reverse=reverse)
    text = realistic_fastq(np.random.default_rng(SEED + 2), seqs)[0] if realistic else fastq(seqs)
    want = host_counts(library, permuter, seqs, off)
    for read_len in (75, 0):
        records, got = count_text(library, permuter, text, read_len, off)
        assert records == len(seqs) and same(got, want), (read_len, records)


def cut_points(text, seqs):
    """one cut of every kind inside the file, plus seeded random ones and one-byte calls"""
    starts = [0]
    for _ in range(len(seqs)):
        at = starts[-1]
        for _ in range(4):
            at = text.index(b"\n", at) + 1
        starts.append(at)
    r = starts[len(seqs) // 3]
    header_end = text.index(b"\n", r) + 1
    seq_end = text.index(b"\n", header_end)
    plus_end = text.index(b"\n", seq_end + 1) + 1
    fixed = [r + 2,                      # inside a header
             header_end,                 # right after a newline
             header_end + 30,            # inside a sequence
             seq_end + 1,                # between a sequence and its '+' line
             plus_end + 10,              # inside a quality line
             len(text) - 1]              # one byte before the end
    rng = np.random.default_rng(SEED + 3)
    rand = rng.integers(1, len(text) - 1, 40).tolist()
    ones = [x + d for x in rng.integers(1, len(text) - 10, 5).tolist() for d in range(4)]  # three one-byte calls each
    return sorted(set(fixed + rand + ones))


@pytest.mark.gpu
def test_many_calls_and_waves_equal_one(monkeypatch):
    monkeypatch.setenv("SGC_TEXT_WAVE", "65536")
    guides, (library,), (permuter,) = library_of(SEED + 10)
    off = sg.Offset.Forward(5)
    seqs = make_reads(np.random.default_rng(SEED + 11), guides, 40_000, 75, 5)
    want = host_counts(library, permuter, seqs, off)
    for text in (fastq(seqs), realistic_fastq(np.random.default_rng(SEED + 12), seqs)[0]):
        cuts = cut_points(text, seqs)
        for read_len in (75, 0):
            records, got = count_text(library, permuter, text, read_len, off, cuts)
            assert records == len(seqs) and same(got, want), (read_len, records)


@pytest.mark.gpu
def test_endings_and_empty_calls(monkeypatch):
    monkeypatch.setenv("SGC_TEXT_WAVE", "100000")
    guides, (library,), (permuter,) = library_of(SEED + 20)
    off = sg.Offset.Forward(5)
    seqs = make_reads(np.random.default_rng(SEED + 21), guides, 20_000, 75, 5)
    want = host_counts(library, permuter, seqs, off)
    text = fastq(seqs, final_newline=False)
    for read_len in (75, 0):
        c, s = text_stream(library, permuter, read_len, off)
        blob = np.frombuffer(text, dtype=np.uint8)
        s.submit_text(blob[:0])
        s.submit_text(blob[:12345])
        s.submit_text(blob[:0])
        s.submit_text(blob[12345:])
        assert s.finish() == len(seqs) and same(c.finish(), want), read_len
        # a truncated last record: it ends inside its sequence line
        c, s = text_stream(library, permuter, read_len, off)
        last = text.rindex(b"\n@") + 1
        s.submit_text(blob[:text.index(b"\n", last) + 20])
        with pytest.raises(sg.SgcError) as e:
            s.finish()
        assert e.value.code == _cabi.ERR_FASTQ_FORMAT


@pytest.mark.gpu
def test_declines(monkeypatch):
    monkeypatch.setenv("SGC_TEXT_WAVE", "262144")
    guides, (library,), (permuter,) = library_of(SEED + 30)
    off = sg.Offset.Forward(5)
    seqs = make_reads(np.random.default_rng(SEED + 31), guides, 20_000, 75, 5)

    def declined(text, read_len):
        c, s = text_stream(library, permuter, read_len, off)
        with pytest.raises(sg.SgcError) as e:
            s.submit_text(np.frombuffer(text, dtype=np.uint8))
            s.finish()
        assert e.value.code == _cabi.ERR_FASTQ_FORMAT, e.value
        with pytest.raises(sg.SgcError) as e:  # a failed stream refuses the next call
            s.submit_text(np.frombuffer(text[:1000], dtype=np.uint8))
        assert e.value.code == _cabi.ERR_INVALID_ARG

    for read_len in (75, 0):
        declined(b"#" + fastq(seqs)[1:], read_len)  # first byte not '@'
        long_seqs = list(seqs)
        long_seqs[10_000] = b"A" * (600 << 10)  # a record over 64 KiB (and over two waves)
        declined(fastq(long_seqs), read_len)
    odd = list(seqs)
    odd[15_000] = odd[15_000][:60]  # one read of another length deep in the file: span mode declines
    declined(fastq(odd), 75)
    records, got = count_text(library, permuter, fastq(odd), 0, off)
    assert records == len(odd) and same(got, host_counts(library, permuter, odd, off))


def record_cuts(text, parts):
    """offsets that cut `text` into `parts` parts at record ends"""
    out = []
    for i in range(1, parts):
        at = len(text) * i // parts
        while not (text[at - 1:at] == b"\n" and text[at:at + 1] == b"@" and text.count(b"\n", 0, at) % 4 == 0):
            at += 1
        out.append(at)
    return out


def self_contained_parts(libraries, permuters, text, read_len, off, n):
    cuts = [0, *record_cuts(text, n), len(text)]
    blob = np.frombuffer(text, dtype=np.uint8)
    counters, records = [], 0
    for i in range(n):
        c, s = text_stream(libraries[i % len(libraries)], permuters[i % len(libraries)], read_len, off)
        s.submit_text(blob[cuts[i]:cuts[i + 1]], self_contained=True)
        records += s.finish()
        counters.append(c)
    sg.reduce_counts(counters, 0)
    return records, counters[0].finish()


@pytest.mark.gpu
def test_self_contained_parts_on_three_streams(monkeypatch):
    monkeypatch.setenv("SGC_TEXT_WAVE", "300000")
    guides, (library,), (permuter,) = library_of(SEED + 40)
    off = sg.Offset.Forward(5)
    seqs = make_reads(np.random.default_rng(SEED + 41), guides, 30_000, 75, 5)
    want = host_counts(library, permuter, seqs, off)
    text = realistic_fastq(np.random.default_rng(SEED + 42), seqs)[0]
    for read_len in (75, 0):
        records, got = self_contained_parts([library], [permuter], text, read_len, off, 3)
        assert records == len(seqs) and same(got, want), read_len
        # a self-contained call that ends inside a record fails
        c, s = text_stream(library, permuter, read_len, off)
        with pytest.raises(sg.SgcError) as e:
            s.submit_text(np.frombuffer(text[:len(text) // 2 + 7], dtype=np.uint8), self_contained=True)
        assert e.value.code == _cabi.ERR_FASTQ_FORMAT
        # ... and so does one that follows carried bytes
        c, s = text_stream(library, permuter, read_len, off)
        cut = record_cuts(text, 2)[0]
        s.submit_text(np.frombuffer(text[:cut - 5], dtype=np.uint8))
        with pytest.raises(sg.SgcError) as e:
            s.submit_text(np.frombuffer(text[cut:], dtype=np.uint8), self_contained=True)
        assert e.value.code == _cabi.ERR_FASTQ_FORMAT


@pytest.mark.gpu
@pytest.mark.skipif(device_count() < 2, reason="needs two devices")
def test_self_contained_parts_on_two_devices():
    guides, libraries, permuters = library_of(SEED + 50, devices=(0, 1))
    off = sg.Offset.Forward(5)
    seqs = make_reads(np.random.default_rng(SEED + 51), guides, 30_000, 75, 5)
    want = host_counts(libraries[0], permuters[0], seqs, off)
    for read_len in (75, 0):
        records, got = self_contained_parts(libraries, permuters, fastq(seqs), read_len, off, 4)
        assert records == len(seqs) and same(got, want), read_len


@pytest.mark.gpu
def test_concurrent_text_submits_equal_host_counter(monkeypatch):
    monkeypatch.setenv("SGC_TEXT_WAVE", "1000000")
    guides, (library,), (permuter,) = library_of(SEED + 60)
    off = sg.Offset.Forward(5)
    jobs = []
    for i in range(4):
        seqs = make_reads(np.random.default_rng(SEED + 61 + i), guides, 40_000, 75, 5, variable=(i == 3))
        jobs.append((seqs, fastq(seqs), 0 if i == 3 else 75))
    pairs = [text_stream(library, permuter, read_len, off) for _, _, read_len in jobs]
    records, errors = [None] * 4, []
    barrier = threading.Barrier(4)

    def run(i):
        try:
            blob = np.frombuffer(jobs[i][1], dtype=np.uint8)
            barrier.wait()
            pairs[i][1].submit_text(blob)
            records[i] = pairs[i][1].finish()
        except Exception as e:  # reported below
            errors.append((i, e))

    threads = [threading.Thread(target=run, args=(i,)) for i in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for i, (seqs, _, _) in enumerate(jobs):
        assert records[i] == len(seqs) and same(pairs[i][0].finish(), host_counts(library, permuter, seqs, off)), i


@pytest.mark.gpu
def test_memmap_input(tmp_path):
    guides, (library,), (permuter,) = library_of(SEED + 70)
    off = sg.Offset.Forward(5)
    seqs = make_reads(np.random.default_rng(SEED + 71), guides, 50_000, 75, 5)
    path = tmp_path / "reads.fastq"
    path.write_bytes(fastq(seqs))
    want = host_counts(library, permuter, seqs, off)
    for read_len in (75, 0):
        c, s = text_stream(library, permuter, read_len, off)
        s.submit_text(np.memmap(path, dtype=np.uint8, mode="r"))
        assert s.finish() == len(seqs) and same(c.finish(), want), read_len


# ---- the CLI ----

def run(*args, env=None):
    p = subprocess.run([BIN, *args], capture_output=True, text=True, timeout=900, env={**os.environ, **(env or {})})
    assert p.returncode == 0, p.stderr
    return p


def timing(proc):
    return json.loads([l for l in proc.stderr.splitlines() if l.startswith("{")][-1])


def finished(proc):
    return [l for l in proc.stderr.splitlines() if l.startswith("Finished:")]


def oracle_table(lib, paths):
    from oracle import oracle as orc
    recs = orc.Records.from_path(lib)
    olib = orc.Library.from_reader(recs)
    perm = orc.Permuter.new(olib)
    cols = []
    for p in paths:
        reads = orc.Records.from_path(p)
        cols.append(orc.Counter.new(reads, olib, perm, orc.entropy_offset(recs, reads, 5000)).counts_by_index())
    return cols


def table_counts(stdout, n_guides, n_samples):
    """the table's counts by guide index (lib.<i> aliases), zero rows included"""
    out = np.zeros((n_samples, n_guides), dtype=np.uint64)
    for line in stdout.splitlines()[1:]:
        f = line.split("\t")
        out[:, int(f[0].split(".")[1])] = [int(x) for x in f[1:]]
    return out


@pytest.fixture(scope="module")
def inputs(tmp_path_factory):
    """a library; plain samples: fixed length forward and reverse, reads of any length, realistic qualities,
    one odd read deep in the file, no final newline; a FASTA sample; a BGZF and a gzip sample"""
    d = tmp_path_factory.mktemp("text_ingest")
    arr = synth.make_library(SEED, 3000, 20)
    lib = str(d / "lib.fa")
    with open(lib, "wb") as f:
        f.write(b"".join(b">lib.%d\n%s\n" % (i, arr[i].tobytes()) for i in range(len(arr))))
    guides = [arr[i].tobytes() for i in range(len(arr))]
    out = {"lib": lib, "n_guides": len(arr), "plain": []}
    for i, reverse in enumerate((False, True)):
        path = str(d / f"s{i}.fastq")
        synth.Sample(SEED + i, i, arr, 75, 5 + i, reverse).write_fastq(path, 0, 250_000, gz_level=0)
        out["plain"].append(path)
    rng = np.random.default_rng(SEED + 100)
    variable = make_reads(rng, guides, 30_000, 75, 6, variable=True)
    variable[0] = next(s for s in variable if len(s) == 75)  # (the first read sets the length the library is checked against)
    odd = make_reads(rng, guides, 30_000, 75, 4)
    odd[25_000] = odd[25_000][:60]  # span mode fails there: the sample starts over in line mode, on the device
    texts = {"variable.fq": fastq(variable),
             "realistic.fq": realistic_fastq(rng, make_reads(rng, guides, 40_000, 75, 4))[0],
             "odd_read.fastq": fastq(odd),
             "no_newline.fastq": fastq(make_reads(rng, guides, 20_000, 75, 5), final_newline=False)}
    for name, text in texts.items():
        out["plain"].append(str(d / name))
        with open(out["plain"][-1], "wb") as f:
            f.write(text)
    out["fasta"] = str(d / "reads.fa")
    with open(out["fasta"], "wb") as f:
        f.write(b"".join(b">r%d\n%s\n" % (i, s) for i, s in enumerate(make_reads(rng, guides, 10_000, 75, 5))))
    out["bgzf"] = str(d / "b.fastq.gz")
    synth.Sample(SEED + 20, 20, arr, 75, 5, False).write_fastq_bgzf(out["bgzf"], 0, 100_000)
    out["gzip"] = str(d / "m.fastq.gz")
    synth.Sample(SEED + 21, 21, arr, 75, 5, False).write_fastq(out["gzip"], 0, 100_000, reads_per_member=100_000)
    # quality lines that start with '@' everywhere, for read shards (some fall right at a cut)
    seqs = make_reads(np.random.default_rng(SEED + 102), guides, 60_000, 75, 5)
    text = bytearray(fastq(seqs))
    nl = np.flatnonzero(np.frombuffer(bytes(text), dtype=np.uint8) == 10)
    for q in nl[2::4][::3]:
        text[q + 1] = ord("@")
    out["at_quals"] = str(d / "at_quals.fastq")
    with open(out["at_quals"], "wb") as f:
        f.write(bytes(text))
    return out


def against_host(inputs, paths, extra=(), env=None):
    dev = run("-l", inputs["lib"], "-i", *paths, "--timing", *extra, env=env)
    host = run("-l", inputs["lib"], "-i", *paths, "--host-inflate", *extra)
    assert dev.stdout == host.stdout
    assert finished(dev) == finished(host) and len(finished(dev)) == len(paths)
    return dev, timing(dev)


@pytest.mark.gpu
def test_cli_plain_samples_on_the_device_equal_host_and_oracle(inputs):
    paths = inputs["plain"]
    dev, t = against_host(inputs, paths, extra=("-z",))
    assert t["device_ingest_samples"] == len(paths), t
    assert t["device_text_bytes"] == sum(os.path.getsize(p) for p in paths), t
    assert t["span_reads"] < t["reads"], t  # the variable-length and odd-read samples went as whole lines
    got = table_counts(dev.stdout, inputs["n_guides"], len(paths))
    want = oracle_table(inputs["lib"], paths)
    for i in range(len(paths)):
        assert np.array_equal(got[i], np.asarray(want[i], dtype=np.uint64)), paths[i]


@pytest.mark.gpu
def test_cli_whole_lines_and_fasta(inputs):
    _, t = against_host(inputs, inputs["plain"][:2], extra=("--whole-lines",))
    assert t["device_ingest_samples"] == 2 and t["span_reads"] == 0, t
    _, t = against_host(inputs, [inputs["fasta"]])
    assert t["device_ingest_samples"] == 0 and t["host_ingest_because"] == "not FASTQ", t


@pytest.mark.gpu
def test_cli_plain_bgzf_and_gzip_side_by_side(inputs):
    paths = [inputs["plain"][0], inputs["bgzf"], inputs["plain"][1], inputs["gzip"], inputs["plain"][3]]
    dev, t = against_host(inputs, paths)
    assert t["device_ingest_samples"] == 5 and t["device_blocks"] > 0 and t["gzip_members"] == 1, t
    assert t["sample_workers"] == min(4 * t["gpus"], 5), t
    one, t1 = against_host(inputs, paths, env={"SGC_DEVICE_BUDGET": "1"})
    assert one.stdout == dev.stdout
    assert t1["device_ingest_samples"] == 5 and t1["device_samples_in_flight"] == 1, t1


@pytest.mark.gpu
def test_cli_read_shards_cut_at_record_ends(inputs):
    env = {"SGC_TEXT_WAVE": str(200_000)}
    dev, t = against_host(inputs, [inputs["at_quals"]], extra=("--read-shards", "3"), env=env)
    assert t["device_ingest_samples"] == 1 and t["read_shards_per_sample"] == 3, t
    one = run("-l", inputs["lib"], "-i", inputs["at_quals"])
    assert one.stdout == dev.stdout and finished(one) == finished(dev)


@pytest.mark.gpu
@pytest.mark.skipif(device_count() < 2, reason="needs two devices")
def test_cli_two_devices_equal_one(inputs):
    paths = inputs["plain"][:4]
    one = run("-l", inputs["lib"], "-i", *paths)
    two = run("-l", inputs["lib"], "-i", *paths, "--gpus", "2", "--timing")
    assert two.stdout == one.stdout and finished(two) == finished(one)
    t = timing(two)
    assert t["gpus"] == 2 and t["device_ingest_samples"] == 4, t
    shards = run("-l", inputs["lib"], "-i", paths[0], "--gpus", "2", "--read-shards", "2", "--timing",
                 env={"SGC_TEXT_WAVE": str(1 << 20)})
    assert shards.stdout == run("-l", inputs["lib"], "-i", paths[0]).stdout
    assert timing(shards)["device_ingest_samples"] == 1
