"""The unmatched report on the device (sgc_counter_set_unmatched_report, unmatched_collect_kernel in
csrc/count.cu) against its statement (tests/unmatched_oracle.py): the full table and the tallies must be
equal bit for bit on every key family, both orientations and rc_modes, Permuter and exact, recursion on
and off, max_shift 1 and 8, every read layout, span records, the skew plan, launch splitting and the
device ingest; a report that overflows keeps exact counts for what it holds; and the CLI's
--unmatched-report writes the statement's TSV on every ingest path."""
import gzip
import json
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

import sgcount_b200 as sg
from oracle import oracle as orc
from sgcount_b200 import _cabi

import unmatched_oracle as U
from helpers import ACGT, make_library, make_reads

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
SEED = 0x0A3C7
KS = [16, 17, 20, 21, 24, 25, 28, 29, 30]


def sample(rng, guides, n, read_len, offset, reverse=False, variable=False):
    """the class mix of make_reads (members, mismatches, wildcards, shifts, truncated reads, junk), plus
    reads with two Ns and repeats of a few junk windows, so that windows have counts above one"""
    k = len(guides[0])
    seqs = make_reads(rng, guides, n, read_len, offset, reverse=reverse, variable=variable, junk=0.15)
    repeats = [ACGT[rng.integers(0, 4, read_len)].tobytes() for _ in range(12)]
    for i in rng.choice(n, n // 10, replace=False):
        seqs[i] = repeats[rng.integers(len(repeats))][:len(seqs[i])]
    for i in rng.choice(n, n // 20, replace=False):
        row = bytearray(seqs[i])
        for p in rng.integers(offset, offset + k, 2):
            if p < len(row):
                row[p] = ord("N")
        seqs[i] = bytes(row)
    return seqs


def device_report(library, permuter, batch, offset, capacity=1 << 16, max_shift=1, recursion=True,
                  rc_mode=_cabi.RC_BITTRICK, base=0, with_assign=False):
    """(rows, info, (counts, total, matched), assignments or None) of one submit_device, the lines `base`
    bytes into the device buffer"""
    import torch

    lines = np.concatenate([np.zeros(base, np.uint8), batch.lines, np.zeros(64, np.uint8)])
    d_lines = torch.from_numpy(lines).cuda()
    d_off = None if batch.line_off is None else torch.from_numpy(batch.line_off).cuda()
    d_assign = torch.full((max(len(batch), 1),), -7, dtype=torch.int32, device="cuda") if with_assign else None
    c = sg.Counter(library, permuter, offset, recursion, rc_mode, max_shift=max_shift, unmatched_capacity=capacity)
    c.submit_device(d_lines.data_ptr() + base, batch.lines.nbytes, len(batch), batch.stride, batch.read_len,
                    None if d_off is None else d_off.data_ptr(), None if d_assign is None else d_assign.data_ptr())
    result = c.finish()
    rows, info = c.unmatched()
    assert c.launch_info().kernel == (3 if max_shift >= 2 else 1)
    return rows, info, result, None if d_assign is None else d_assign.cpu().numpy()[:len(batch)]


def assert_exact(rows, info, want_rows, want_tally, label=""):
    assert info["overflow"] == 0, label
    assert info["distinct"] == len(want_rows), label
    for key in ("unmatched", "short_reads", "non_acgt"):
        assert info[key] == want_tally[key], (label, key, info, want_tally)
    assert rows == want_rows, (label, rows[:3], want_rows[:3])


def libs_for(guides):
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    return library, sg.Permuter.new(library)


@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("reverse", [False, True])
def test_report_equals_statement(k, reverse):
    rng = np.random.default_rng(SEED + 100 * k + reverse)
    guides = make_library(rng, 300, k)
    library, permuter = libs_for(guides)
    o = 5
    off = sg.Offset(reverse, o)
    fixed = sample(rng, guides, 2500, o + k + 12, o, reverse)
    var = sample(rng, guides, 2500, o + k + 16, o, reverse, variable=True)
    assert min(len(s) for s in var) < o + k  # some reads have no window
    layouts = [("fixed aligned", fixed, sg.ReadBatch.from_seqs(fixed), 0),
               ("fixed unaligned", fixed, sg.ReadBatch.from_seqs(fixed), 3),
               ("variable", var, sg.ReadBatch.from_seqs(var, force_offsets=True), 5)]
    searches = [(1, True), (1, False), (8, True)]
    for rc_mode in (_cabi.RC_BITTRICK, _cabi.RC_KEEP_N):
        for with_perm in (True, False):
            for S, recursion in searches:
                for label, seqs, batch, base in layouts:
                    want_rows, want_tally, assign = U.statement(seqs, guides, with_perm, orc.Offset(reverse, o), rc_mode,
                                                                S, recursion)
                    rows, info, (counts, total, matched), _ = device_report(
                        library, permuter if with_perm else None, batch, off, max_shift=S, recursion=recursion,
                        rc_mode=rc_mode, base=base)
                    what = (label, rc_mode, with_perm, S, recursion)
                    assert total - matched == int((assign < 0).sum()), what
                    assert_exact(rows, info, want_rows, want_tally, what)


@pytest.mark.parametrize("max_shift", [1, 8])
@pytest.mark.parametrize("reverse", [False, True])
def test_span_records_report_like_whole_reads(max_shift, reverse):
    rng = np.random.default_rng(SEED + 7 + 2 * max_shift + reverse)
    for k in (17, 20, 30):
        guides = make_library(rng, 200, k)
        library, permuter = libs_for(guides)
        for o in (0, 4, 11):
            read_len = o + k + 9
            off = sg.Offset(reverse, o)
            seqs = sample(rng, guides, 2000, read_len, o, reverse)
            reader = sg.ReadBatch.from_seqs(seqs)
            spans, span_off = sg.span_batch(reader, k, off, True, max_shift=max_shift)
            whole = device_report(library, permuter, reader, off, max_shift=max_shift)
            part = device_report(library, permuter, spans, span_off, max_shift=max_shift)
            assert whole[0] == part[0] and whole[1] == part[1], (k, o)
            want_rows, want_tally, _ = U.statement(seqs, guides, True, orc.Offset(reverse, o), max_shift=max_shift)
            assert_exact(part[0], part[1], want_rows, want_tally, (k, o))


def test_caller_assignments_serve_as_scratch():
    rng = np.random.default_rng(SEED + 11)
    guides = make_library(rng, 500, 20)
    library, permuter = libs_for(guides)
    seqs = sample(rng, guides, 20_000, 40, 6)
    rows, info, _, assign = device_report(library, permuter, sg.ReadBatch.from_seqs(seqs), sg.Offset.Forward(6),
                                          with_assign=True)
    want_rows, want_tally, want_assign = U.statement(seqs, guides, True, orc.Offset.Forward(6))
    assert np.array_equal(assign, want_assign)
    assert_exact(rows, info, want_rows, want_tally)


@pytest.mark.parametrize("share", [0.1, 0.9])
def test_report_keeps_counts_and_skew_plan(share):
    """one guide on `share` of the reads, automatic plan: counts, total and matched as without the report,
    replicas and hot guides still in use, and the plan's sample reads collected too"""
    import torch

    rng = np.random.default_rng(SEED + int(share * 10))
    guides = make_library(rng, 2000, 20)
    library, permuter = libs_for(guides)
    n = 300_000
    seqs = sample(rng, guides, n, 40, 5)
    hot = rng.random(n) < share
    vec = ACGT[rng.integers(0, 4, 5)].tobytes()
    tail = ACGT[rng.integers(0, 4, 15)].tobytes()
    for i in np.flatnonzero(hot):
        seqs[i] = vec + guides[7] + tail
    batch = sg.ReadBatch.from_seqs(seqs)
    d_lines = torch.from_numpy(np.concatenate([batch.lines, np.zeros(64, np.uint8)])).cuda()
    results = []
    for capacity in (None, 1 << 16):
        c = sg.Counter(library, permuter, sg.Offset.Forward(5), unmatched_capacity=capacity)
        c.submit_device(d_lines.data_ptr(), batch.lines.nbytes, len(batch), batch.stride, batch.read_len)
        results.append(c.finish())
        info = c.launch_info()
        assert info.replicas > 1 and info.hot_guides >= 1, (capacity, info.replicas, info.hot_guides)
    assert np.array_equal(results[0][0], results[1][0]) and results[0][1:] == results[1][1:]
    rows, info = c.unmatched()
    want_rows, want_tally, _ = U.statement(seqs, guides, True, orc.Offset.Forward(5))
    assert_exact(rows, info, want_rows, want_tally)


def test_one_window_on_half_the_reads():
    """an adapter dimer on half the reads next to ~10^5 distinct junk windows: exact counts"""
    rng = np.random.default_rng(SEED + 21)
    guides = make_library(rng, 3000, 20)
    library, permuter = libs_for(guides)
    n = 400_000
    seqs = sample(rng, guides, n, 40, 5)
    dimer = ACGT[rng.integers(0, 4, 40)].tobytes()
    pick = rng.permutation(n)
    for i in pick[:n // 2]:
        seqs[i] = dimer
    for i in pick[n // 2:n // 2 + 100_000]:
        seqs[i] = ACGT[rng.integers(0, 4, 40)].tobytes()
    rows, info, _, _ = device_report(library, permuter, sg.ReadBatch.from_seqs(seqs), sg.Offset.Forward(5),
                                     capacity=1 << 20)
    want_rows, want_tally, _ = U.statement(seqs, guides, True, orc.Offset.Forward(5))
    assert want_rows[0] == (dimer[5:25], n // 2) and len(want_rows) > 90_000
    assert_exact(rows, info, want_rows, want_tally)


def test_overflow_keeps_held_counts_exact():
    rng = np.random.default_rng(SEED + 22)
    guides = make_library(rng, 500, 20)
    library, permuter = libs_for(guides)
    junk = [ACGT[rng.integers(0, 4, 40)].tobytes() for _ in range(3000)]
    seqs = [junk[int(j)] for j in rng.zipf(1.3, 60_000) % len(junk)] + sample(rng, guides, 20_000, 40, 5)
    rows, info, (_, total, matched), _ = device_report(library, permuter, sg.ReadBatch.from_seqs(seqs),
                                                       sg.Offset.Forward(5), capacity=64)
    want_rows, want_tally, _ = U.statement(seqs, guides, True, orc.Offset.Forward(5))
    true = dict(want_rows)
    assert info["overflow"] > 0 and 0 < info["distinct"] <= 64 and len(rows) == info["distinct"]
    for key in ("unmatched", "short_reads", "non_acgt"):
        assert info[key] == want_tally[key]
    assert info["unmatched"] == total - matched
    assert info["unmatched"] == info["short_reads"] + info["non_acgt"] + info["overflow"] + sum(c for _, c in rows)
    for w, c in rows:
        assert true[w] == c, w
    held = {w for w, _ in rows}
    assert all(c <= info["overflow"] for w, c in want_rows if w not in held)
    assert rows == sorted(rows, key=lambda kv: (-kv[1], kv[0]))


def test_launch_splitting(monkeypatch):
    rng = np.random.default_rng(SEED + 23)
    guides = make_library(rng, 400, 20)
    library, permuter = libs_for(guides)
    seqs = sample(rng, guides, 10_000, 50, 6, variable=True)
    batch = sg.ReadBatch.from_seqs(seqs, force_offsets=True)
    for S in (1, 8):
        whole = device_report(library, permuter, batch, sg.Offset.Forward(6), max_shift=S)
        monkeypatch.setenv("SGC_MAX_LAUNCH_TILES", "3")  # 96 reads a launch
        cut = device_report(library, permuter, batch, sg.Offset.Forward(6), max_shift=S, base=1)
        monkeypatch.delenv("SGC_MAX_LAUNCH_TILES")
        assert whole[0] == cut[0] and whole[1] == cut[1]
        assert np.array_equal(whole[2][0], cut[2][0]) and whole[2][1:] == cut[2][1:]


def test_submits_accumulate_and_reset_clears():
    rng = np.random.default_rng(SEED + 24)
    guides = make_library(rng, 400, 20)
    library, permuter = libs_for(guides)
    a, b = sample(rng, guides, 5000, 40, 5), sample(rng, guides, 7000, 40, 5, variable=True)
    c = sg.Counter(library, permuter, sg.Offset.Forward(5), unmatched_capacity=1 << 15)
    c.submit(sg.ReadBatch.from_seqs(a))
    c.submit(sg.ReadBatch.from_seqs(b))
    rows, info = c.unmatched()
    want_rows, want_tally, _ = U.statement(a + b, guides, True, orc.Offset.Forward(5))
    assert_exact(rows, info, want_rows, want_tally)
    assert c.unmatched(5)[0] == want_rows[:5]
    c.reset()
    rows, info = c.unmatched()
    assert rows == [] and info == {"unmatched": 0, "short_reads": 0, "non_acgt": 0, "overflow": 0, "distinct": 0}
    c.submit(sg.ReadBatch.from_seqs(b))
    want_rows, want_tally, _ = U.statement(b, guides, True, orc.Offset.Forward(5))
    assert_exact(*c.unmatched(), want_rows, want_tally)


def test_errors():
    guides = make_library(np.random.default_rng(SEED + 25), 50, 20)
    library, _ = libs_for(guides)
    off = sg.Offset.Forward(2)
    for bad in (0, (1 << 26) + 1):
        with pytest.raises(sg.SgcError) as e:
            sg.Counter(library, None, off, unmatched_capacity=bad)
        assert e.value.code == _cabi.ERR_INVALID_ARG
        with pytest.raises(sg.SgcError):
            sg.unmatched_report_bytes(bad)
    assert sg.unmatched_report_bytes(1 << 22) == (1 << 22) * 16 + (64 << 20) + 5 * 8
    c = sg.Counter(library, None, off)
    with pytest.raises(sg.SgcError):
        c.unmatched()  # no report
    c.submit(sg.ReadBatch.from_seqs([guides[0] + b"ACGT"] * 10))
    with pytest.raises(sg.SgcError) as e:
        c.set_unmatched_report(100)
    assert e.value.code == _cabi.ERR_INVALID_ARG
    for seqs in ([b"ACGTNACGTA", b"ACGTACGTAA"], [b"A" * 31, b"C" * 31]):
        opaque = sg.Library(seqs, [b"a", b"b"])
        assert opaque._exact.info().opaque == 1
        with pytest.raises(sg.SgcError) as e:
            sg.Counter(opaque, None, off, unmatched_capacity=100)
        assert e.value.code == _cabi.ERR_INVALID_ARG


# ---- device ingest ----

def bgzf(text: bytes, block=0xff00) -> bytes:
    out = b""
    for b in [text[i:i + block] for i in range(0, len(text), block)] + [b""]:
        raw = zlib.compressobj(6, zlib.DEFLATED, -15)
        body = raw.compress(b) + raw.flush()
        out += bytes([0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0]) + b"BC" + struct.pack("<HH", 2, 18 + len(body) + 8 - 1) + \
            body + struct.pack("<II", zlib.crc32(b), len(b))
    return out


def fastq(seqs) -> bytes:
    return b"".join(b"@r%d\n%s\n+\n%s\n" % (i, s, b"F" * len(s)) for i, s in enumerate(seqs))


@pytest.mark.parametrize("reverse", [False, True])
def test_device_ingest_equals_statement(reverse):
    rng = np.random.default_rng(SEED + 30 + reverse)
    k, read_len, o = 20, 75, 7
    guides = make_library(rng, 1000, k)
    library, permuter = libs_for(guides)
    off = sg.Offset(reverse, o)
    seqs = sample(rng, guides, 60_000, read_len, o, reverse)
    text = fastq(seqs)
    half = text.index(b"@r30000\n")
    blobs = {"bgzf": bgzf(text), "gzip": gzip.compress(text, 6),
             "members": gzip.compress(text[:half], 6) + gzip.compress(text[half:], 6)}
    want_rows, want_tally, _ = U.statement(seqs, guides, True, orc.Offset(reverse, o))
    for mode in ("span", "lines"):
        for kind in ("text", "bgzf", "gzip", "members"):
            if mode == "span":
                start, length, span_off = sg.span_geometry(k, read_len, off, True)
                c = sg.Counter(library, permuter, span_off, True, unmatched_capacity=1 << 16)
                s = sg.FastqStream(c, read_len, start, length)
            else:
                c = sg.Counter(library, permuter, off, True, unmatched_capacity=1 << 16)
                s = sg.FastqStream(c, 0, 0, 0)
            if kind == "text":
                s.submit_text(np.frombuffer(text, dtype=np.uint8))
            elif kind == "bgzf":
                begin, isize = sg.bgzf_blocks(blobs["bgzf"])
                arr = np.frombuffer(blobs["bgzf"], dtype=np.uint8)
                for a in range(0, len(isize), 40):
                    b = min(len(isize), a + 40)
                    s.submit(arr, begin[a:b + 1], isize[a:b])
            elif kind == "gzip":
                s.submit_member(np.frombuffer(blobs["gzip"], dtype=np.uint8))
            else:
                s.submit_gzip(np.frombuffer(blobs["members"], dtype=np.uint8))
            assert s.finish() == len(seqs)
            assert_exact(*c.unmatched(), want_rows, want_tally, (mode, kind))


# ---- the CLI ----

def run(*args, env=None, ok=True):
    p = subprocess.run([BIN, *args], capture_output=True, text=True, timeout=900, env={**os.environ, **(env or {})})
    if ok:
        assert p.returncode == 0, p.stderr
    return p


def timing(proc):
    return json.loads([l for l in proc.stderr.splitlines() if l.startswith("{")][-1])


def expected_tsv(samples):
    """the statement's TSV: (name, ordered windows, tallies) per sample"""
    out = "Sample\tWindow\tCount\n"
    for name, rows, tally in samples:
        top = rows[:100]
        other = sum(c for _, c in rows[100:])
        out += "".join(f"{name}\t{w.decode()}\t{c}\n" for w, c in top)
        out += f"{name}\t<other>\t{other}\n{name}\t<non-ACGT>\t{tally['non_acgt']}\n{name}\t<short>\t{tally['short_reads']}\n"
    return out


def assert_rows_sum_to_finished(tsv, stderr):
    per = {}
    for line in tsv.splitlines()[1:]:
        name, _, c = line.split("\t")
        per[name] = per.get(name, 0) + int(c)
    for line in stderr.splitlines():
        if line.startswith("Finished: "):
            name = line[len("Finished: "):line.index(";")]
            matched, total = line[line.index("[") + 1:line.index("]")].split(" / ")
            assert per[name] == int(total) - int(matched), line


@pytest.fixture(scope="module")
def inputs(tmp_path_factory):
    """a 20-base library; a fixed-length sample (75 bp) as BGZF, single-member gzip and plain FASTQ, and a
    variable-length one"""
    d = tmp_path_factory.mktemp("unmatched")
    rng = np.random.default_rng(SEED + 40)
    guides = make_library(rng, 3000, 20)
    lib = str(d / "lib.fa")
    with open(lib, "wb") as f:
        f.write(b"".join(b">lib.%d\n%s\n" % (i, g) for i, g in enumerate(guides)))
    fixed = sample(rng, guides, 150_000, 75, 10)
    var = sample(rng, guides, 80_000, 75, 10, variable=True)
    var = [s or b"A" for s in var]  # (no empty sequence lines)
    var[0] = var[0] + b"A" * 75  # the head must hold a full read
    paths = {"bgzf": str(d / "b.fastq.gz"), "gzip": str(d / "m.fastq.gz"), "plain": str(d / "p.fastq"),
             "var": str(d / "v.fastq.gz")}
    text = fastq(fixed)
    with open(paths["bgzf"], "wb") as f:
        f.write(bgzf(text))
    with open(paths["gzip"], "wb") as f:
        f.write(gzip.compress(text, 6))
    with open(paths["plain"], "wb") as f:
        f.write(text)
    with open(paths["var"], "wb") as f:
        f.write(bgzf(fastq(var)))
    opaque = str(d / "opaque.fa")
    with open(opaque, "wb") as f:
        f.write(b">a\nACGTNACGTACGTACGTACG\n>b\nACGTACGTACGTACGTACGA\n")
    return {"lib": lib, "guides": guides, "fixed": fixed, "var": var, "paths": paths, "opaque": opaque, "dir": d}


def statement_for(inputs, key, max_shift=1):
    seqs = inputs["var"] if key == "var" else inputs["fixed"]
    rows, tally, _ = U.statement(seqs, inputs["guides"], True, orc.Offset.Forward(10), max_shift=max_shift)
    return rows, tally


def test_cli_report_equals_statement_on_every_path(inputs, tmp_path):
    keys = ["bgzf", "gzip", "plain", "var"]
    paths = [inputs["paths"][x] for x in keys]
    names = ["b", "m", "p", "v"]
    want = expected_tsv([(n, *statement_for(inputs, key)) for n, key in zip(names, keys)])
    common = ("-l", inputs["lib"], "-a", "10", "-i", *paths)
    dev = run(*common, "--unmatched-report", str(tmp_path / "dev.tsv"), "--timing")
    t = timing(dev)
    assert t["device_ingest_samples"] == 4 and "unmatched_s" in t, t
    host = run(*common, "--unmatched-report", str(tmp_path / "host.tsv"), "--host-inflate")
    dev_tsv, host_tsv = (tmp_path / "dev.tsv").read_text(), (tmp_path / "host.tsv").read_text()
    assert dev_tsv == host_tsv
    assert dev_tsv == want
    assert_rows_sum_to_finished(dev_tsv, dev.stderr)
    # without the flag: the same table, stderr and timing keys
    plain = run(*common)
    assert plain.stdout == dev.stdout and plain.stdout == host.stdout
    assert plain.stderr == run(*common, "--unmatched-report", str(tmp_path / "x.tsv")).stderr
    assert "unmatched_s" not in timing(run(*common, "--timing"))
    # one sample alone
    run("-l", inputs["lib"], "-a", "10", "-i", inputs["paths"]["gzip"], "--unmatched-report", str(tmp_path / "one.tsv"))
    assert (tmp_path / "one.tsv").read_text() == expected_tsv([("m", *statement_for(inputs, "gzip"))])


def test_cli_read_shards_and_max_shift(inputs, tmp_path):
    for kind, name in (("bgzf", "b"), ("plain", "p")):
        base = ("-l", inputs["lib"], "-a", "10", "-i", inputs["paths"][kind])
        p = run(*base, "--read-shards", "3", "--unmatched-report", str(tmp_path / "s.tsv"), env={"SGC_TEXT_WAVE": str(1 << 20)})
        assert (tmp_path / "s.tsv").read_text() == expected_tsv([(name, *statement_for(inputs, kind))])
        assert_rows_sum_to_finished((tmp_path / "s.tsv").read_text(), p.stderr)
        p = run(*base, "--max-shift", "8", "--unmatched-report", str(tmp_path / "m.tsv"))
        assert (tmp_path / "m.tsv").read_text() == expected_tsv([(name, *statement_for(inputs, kind, 8))])
        assert_rows_sum_to_finished((tmp_path / "m.tsv").read_text(), p.stderr)


def test_cli_example_fixtures(example_dir, tmp_path):
    lib = os.path.join(example_dir, "library.fasta.gz")
    paths = [os.path.join(example_dir, f) for f in ("diff.sequence.fastq.gz", "offset_clipped.fastq.gz")]
    for extra in ((), ("--host-inflate",)):
        p = run("-l", lib, "-i", *paths, "-a", "5", "--unmatched-report", str(tmp_path / "ex.tsv"), *extra)
        got = (tmp_path / "ex.tsv").read_text()
        assert got == ("Sample\tWindow\tCount\n"
                       "diff.sequence\tCTAGGGACCACAGCCATTAT\t101\n"
                       "diff.sequence\t<other>\t0\ndiff.sequence\t<non-ACGT>\t0\ndiff.sequence\t<short>\t0\n"
                       "offset_clipped\t<other>\t0\noffset_clipped\t<non-ACGT>\t0\noffset_clipped\t<short>\t1\n"), extra
        assert_rows_sum_to_finished(got, p.stderr)


def test_cli_errors(inputs, tmp_path):
    target = tmp_path / "never.tsv"
    p = run("-l", inputs["opaque"], "-i", inputs["paths"]["plain"], "--unmatched-report", str(target), ok=False)
    assert p.returncode == 1 and "--unmatched-report" in p.stderr and not p.stdout, p.stderr
    p = run("-l", inputs["lib"], "-i", inputs["paths"]["plain"], "--unmatched-report", str(tmp_path / "no" / "dir.tsv"),
            ok=False)
    assert p.returncode == 1 and "cannot create" in p.stderr and not p.stdout, p.stderr
