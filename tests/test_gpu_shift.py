"""Staggered reads on the device: counters with max_shift S >= 2 (sgc_counter_set_max_shift) run the shift
kernel (count_shift_kernel in csrc/count.cu) and must assign every read exactly as the CPU statement of
the rule does, on every read layout, every key family, both orientations, with and without the
Permuter; span records cut with sgc_span_geometry_shift count like whole reads; the skew plan does not
change counts; the device ingest paths (text, BGZF, single-member gzip, span and line mode) dispatch to
it; and the CLI's --max-shift gives the host path's and the oracle's table.  The oracle of S >= 2 is
tests/shift_oracle.py (the rule over the CPU oracle's lookups)."""
import ctypes as C
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

import shift_oracle
from helpers import COMP, make_library, oracle_library

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
SEED = 0x5C1F7
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def staggered(rng, guides, n, read_len, offset, S, reverse=False, variable=False, stagger=True):
    """Reads whose guide sits at offset + d, d drawn from -S-1 .. S+1 (some of them just outside the
    search), in the class mix exact / one mismatch / one N / two mismatches / junk, plus planted ties:
    a one-mismatch hit nearer the offset than an exact hit of another guide, and guides at +d and -d.
    Coordinates are those of the trimmed read; reverse reads are stored reverse-complemented.
    variable: lengths from k - 3 to read_len."""
    k = len(guides[0])
    g = np.frombuffer(b"".join(guides), dtype=np.uint8).reshape(len(guides), k)

    def mutate(w, m):
        w = w.copy()
        for p in rng.choice(k, m, replace=False):
            w[p] = rng.choice([x for x in b"ACGT" if x != w[p]])
        return w

    def put(row, at, w):
        if 0 <= at and at + k <= len(row):
            row[at:at + k] = w

    out = []
    for _ in range(n):
        L = int(rng.integers(max(1, k - 3), read_len + 1)) if variable else read_len
        row = ACGT[rng.integers(0, 4, L)].copy()
        d = int(rng.integers(-S - 1, S + 2)) if stagger else 0
        w = g[rng.integers(len(g))]
        c = rng.random()
        if c < 0.55:
            put(row, offset + d, w)
        elif c < 0.67:
            put(row, offset + d, mutate(w, 1))
        elif c < 0.72:
            w = w.copy()
            w[rng.integers(k)] = ord("N")
            put(row, offset + d, w)
        elif c < 0.76:
            put(row, offset + d, mutate(w, 2))
        elif c < 0.80:
            pass  # junk
        elif c < 0.90:  # one mismatch at +e, exact hit of another guide further out
            e = int(rng.integers(0, S))
            put(row, offset - e - 1, g[rng.integers(len(g))])
            put(row, offset + e + 1, g[rng.integers(len(g))])
            put(row, offset + e, mutate(w, 1))
        else:  # guides at +e and -e
            e = int(rng.integers(1, S + 1))
            put(row, offset - e, g[rng.integers(len(g))])
            put(row, offset + e, w)
        if rng.random() < 0.05:
            row[rng.integers(L)] = ord("N")
        if reverse:
            row = COMP[row[::-1]]
        out.append(row.tobytes())
    return out


def oracle_assign(guides, seqs, with_perm, offset, S, rc_mode=orc.RC_BITTRICK):
    olib, _ = oracle_library(guides)
    operm = orc.Permuter.new(olib) if with_perm else None
    return shift_oracle.count(orc.Records.from_seqs(seqs), olib, operm, orc.Offset(offset.reverse, offset.index),
                              rc_mode=rc_mode, max_shift=S)


def device_assign(library, permuter, batch, offset, S, base=0, rc_mode=_cabi.RC_BITTRICK):
    """per-read assignment + (counts, total, matched) through sgc_counter_submit_device, the lines
    `base` bytes into the device buffer"""
    import torch

    lines = np.concatenate([np.zeros(base, np.uint8), batch.lines, np.zeros(64, np.uint8)])
    d_lines = torch.from_numpy(lines).cuda()
    d_off = None if batch.line_off is None else torch.from_numpy(batch.line_off).cuda()
    d_assign = torch.full((max(len(batch), 1),), -7, dtype=torch.int32, device="cuda")
    c = sg.Counter(library, permuter, offset, True, rc_mode, max_shift=S)
    c.submit_device(d_lines.data_ptr() + base, batch.lines.nbytes, len(batch), batch.stride, batch.read_len,
                    None if d_off is None else d_off.data_ptr(), d_assign.data_ptr())
    counts, total, matched = c.finish()
    assert c.launch_info().kernel == 3
    return d_assign.cpu().numpy()[:len(batch)], counts, total, matched


KS = [5, 16, 17, 20, 21, 24, 25, 28, 29, 30]


@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("S", [2, 8, 16])
@pytest.mark.parametrize("reverse", [False, True])
def test_assignments_equal_oracle(k, S, reverse):
    rng = np.random.default_rng(SEED + 1000 * k + 10 * S + reverse)
    guides = make_library(rng, 300, k)
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    permuter = sg.Permuter.new(library)
    for offset_index in (3, S + 2):
        off = sg.Offset(reverse, offset_index)
        read_len = offset_index + k + S + int(rng.integers(-3, 8))
        fixed = staggered(rng, guides, 3000, read_len, offset_index, S, reverse)
        var = staggered(rng, guides, 3000, read_len + 4, offset_index, S, reverse, variable=True)
        cases = [("fixed aligned", sg.ReadBatch.from_seqs(fixed), 0),
                 ("fixed unaligned", sg.ReadBatch.from_seqs(fixed), 3),
                 ("variable", sg.ReadBatch.from_seqs(var, force_offsets=True), 5)]
        for with_perm in (True, False):
            for label, batch, base in cases:
                seqs = fixed if label.startswith("fixed") else var
                want = oracle_assign(guides, seqs, with_perm, off, S)
                got = device_assign(library, permuter if with_perm else None, batch, off, S, base)
                bad = np.flatnonzero(got[0] != want[0])
                assert bad.size == 0, (label, with_perm, offset_index, bad[:5], seqs[bad[0]], got[0][bad[0]], want[0][bad[0]])
                assert np.array_equal(got[1], want[1]) and got[2:] == want[2:], (label, with_perm)


def test_rc_keep_n_and_host_batches():
    rng = np.random.default_rng(SEED + 7)
    guides = make_library(rng, 500, 20)
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    permuter = sg.Permuter.new(library)
    off = sg.Offset.Reverse(4)
    seqs = staggered(rng, guides, 20_000, 40, 4, 8, reverse=True)
    want = oracle_assign(guides, seqs, True, off, 8, rc_mode=orc.RC_KEEP_N)
    got = device_assign(library, permuter, sg.ReadBatch.from_seqs(seqs), off, 8, rc_mode=_cabi.RC_KEEP_N)
    assert np.array_equal(got[0], want[0])
    # a host batch goes through the chunked copy pipeline, then the same kernel
    c = sg.Counter(library, permuter, off, True, _cabi.RC_KEEP_N, max_shift=8)
    c.submit(sg.ReadBatch.from_seqs(seqs))
    counts, total, matched = c.finish()
    assert np.array_equal(counts, want[1]) and (total, matched) == want[2:]


def test_launches_cut_at_any_size(monkeypatch):
    rng = np.random.default_rng(SEED + 8)
    guides = make_library(rng, 400, 20)
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    permuter = sg.Permuter.new(library)
    off = sg.Offset.Forward(6)
    seqs = staggered(rng, guides, 10_000, 50, 6, 8)
    batch = sg.ReadBatch.from_seqs(seqs)
    whole = device_assign(library, permuter, batch, off, 8)
    monkeypatch.setenv("SGC_MAX_LAUNCH_TILES", "3")  # 96 reads a launch
    cut = device_assign(library, permuter, batch, off, 8, base=1)
    assert np.array_equal(whole[0], cut[0]) and np.array_equal(whole[1], cut[1]) and whole[2:] == cut[2:]


@pytest.mark.parametrize("reverse", [False, True])
def test_shift_span_records_count_like_whole_reads(reverse):
    rng = np.random.default_rng(SEED + 9 + reverse)
    for k in (5, 20, 30):
        guides = make_library(rng, 200, k)
        library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
        permuter = sg.Permuter.new(library)
        for S in (2, 8, 16):
            for offset_index in (0, 3, S, S + 5):
                for read_len in (offset_index + k - 2, offset_index + k + S // 2, offset_index + k + S + 9):
                    off = sg.Offset(reverse, offset_index)
                    try:
                        sg.span_geometry(k, read_len, off, True, S)
                    except sg.SgcError:
                        assert read_len < k or offset_index + k > read_len + S
                        continue
                    seqs = staggered(rng, guides, 500, read_len, offset_index, S, reverse)
                    reader = sg.ReadBatch.from_seqs(seqs)
                    spans, span_off = sg.span_batch(reader, k, off, True, max_shift=S)
                    whole = sg.Counter(library, permuter, off, True, max_shift=S)
                    whole.submit(reader)
                    part = sg.Counter(library, permuter, span_off, True, max_shift=S)
                    part.submit(spans)
                    w, p = whole.finish(), part.finish()
                    assert np.array_equal(w[0], p[0]) and w[1:] == p[1:], (k, S, offset_index, read_len)


def test_skew_plan_does_not_change_counts():
    """10 % of the reads on one guide: the plan counts into replicas and registers; counts must not move"""
    import torch

    rng = np.random.default_rng(SEED + 11)
    guides = make_library(rng, 2000, 20)
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    permuter = sg.Permuter.new(library)
    off = sg.Offset.Forward(5)
    hot = [guides[7]] * 10 + guides[:90]
    seqs = staggered(rng, hot, 300_000, 40, 5, 8)
    batch = sg.ReadBatch.from_seqs(seqs)
    d_lines = torch.from_numpy(np.concatenate([batch.lines, np.zeros(64, np.uint8)])).cuda()
    results = []
    for replicas in (0, 1):
        c = sg.Counter(library, permuter, off, True, max_shift=8)
        c.set_replicas(replicas)
        c.submit_device(d_lines.data_ptr(), batch.lines.nbytes, len(batch), batch.stride, batch.read_len)
        results.append(c.finish())
        info = c.launch_info()
        assert info.kernel == 3
        if replicas == 0:
            assert info.replicas > 1 and info.hot_guides >= 1, (info.replicas, info.hot_guides)
    assert np.array_equal(results[0][0], results[1][0]) and results[0][1:] == results[1][1:]
    want = oracle_assign(guides, seqs, True, off, 8)
    assert np.array_equal(results[0][0], want[1]) and results[0][1:] == want[2:]


def test_set_max_shift_errors():
    guides = make_library(np.random.default_rng(SEED + 12), 50, 20)
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    off = sg.Offset.Forward(2)
    for bad in (0, 17):
        with pytest.raises(sg.SgcError) as e:
            sg.Counter(library, None, off, True, max_shift=bad)
        assert e.value.code == _cabi.ERR_INVALID_ARG
    with pytest.raises(sg.SgcError) as e:
        sg.Counter(library, None, off, False, max_shift=2)  # -p
    assert e.value.code == _cabi.ERR_INVALID_ARG
    sg.Counter(library, None, off, False, max_shift=1)  # S = 1 is today's counter, with or without recursion
    c = sg.Counter(library, None, off, True)
    c.submit(sg.ReadBatch.from_seqs([guides[0] + b"ACGT"] * 10))
    with pytest.raises(sg.SgcError) as e:
        c.set_max_shift(4)
    assert e.value.code == _cabi.ERR_INVALID_ARG
    # byte-keyed libraries: a non-ACGT byte, or guides longer than 30 bases
    for seqs in ([b"ACGTNACGTA", b"ACGTACGTAA"], [b"A" * 31, b"C" * 31]):
        opaque = sg.Library(seqs, [b"a", b"b"])
        assert opaque._exact.info().opaque == 1
        sg.Counter(opaque, None, off, True, max_shift=1)
        with pytest.raises(sg.SgcError) as e:
            sg.Counter(opaque, None, off, True, max_shift=3)
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
def test_streams_dispatch_to_the_shift_kernel(reverse):
    rng = np.random.default_rng(SEED + 13 + reverse)
    k, S, read_len, offset_index = 20, 8, 75, 7
    guides = make_library(rng, 1000, k)
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    permuter = sg.Permuter.new(library)
    off = sg.Offset(reverse, offset_index)
    seqs = staggered(rng, guides, 80_000, read_len, offset_index, S, reverse)
    text = fastq(seqs)
    host = sg.Counter(library, permuter, off, True, max_shift=S)
    host.submit(sg.ReadBatch.from_seqs(seqs))
    want = host.finish()
    oracle = oracle_assign(guides, seqs, True, off, S)
    assert np.array_equal(want[0], oracle[1]) and want[1:] == oracle[2:]
    bz, gz = bgzf(text), gzip.compress(text, 6)
    for mode in ("span", "lines"):
        for kind in ("text", "bgzf", "gzip"):
            if mode == "span":
                start, length, span_off = sg.span_geometry(k, read_len, off, True, S)
                c = sg.Counter(library, permuter, span_off, True, max_shift=S)
                s = sg.FastqStream(c, read_len, start, length)
            else:
                c = sg.Counter(library, permuter, off, True, max_shift=S)
                s = sg.FastqStream(c, 0, 0, 0)
            if kind == "text":
                s.submit_text(np.frombuffer(text, dtype=np.uint8))
            elif kind == "bgzf":
                begin, isize = sg.bgzf_blocks(bz)
                arr = np.frombuffer(bz, dtype=np.uint8)
                for a in range(0, len(isize), 40):
                    b = min(len(isize), a + 40)
                    s.submit(arr, begin[a:b + 1], isize[a:b])
            else:
                s.submit_member(np.frombuffer(gz, dtype=np.uint8))
            assert s.finish() == len(seqs)
            got = c.finish()
            assert c.launch_info().kernel == 3, (mode, kind)
            assert np.array_equal(got[0], want[0]) and got[1:] == want[1:], (mode, kind)


# ---- the CLI ----

def run(*args, env=None, ok=True):
    p = subprocess.run([BIN, *args], capture_output=True, text=True, timeout=900, env={**os.environ, **(env or {})})
    if ok:
        assert p.returncode == 0, p.stderr
    return p


def timing(proc):
    return json.loads([l for l in proc.stderr.splitlines() if l.startswith("{")][-1])


def table_counts(stdout, n_guides, n_samples):
    out = np.zeros((n_samples, n_guides), dtype=np.uint64)
    for line in stdout.splitlines()[1:]:
        f = line.split("\t")
        out[:, int(f[0].split(".")[1])] = [int(x) for x in f[1:]]
    return out


@pytest.fixture(scope="module")
def inputs(tmp_path_factory):
    """a 20-base library; one staggered sample (0-8 random bases before the vector, reads of 75 bp) as
    BGZF, as single-member gzip and as plain FASTQ"""
    d = tmp_path_factory.mktemp("shift")
    rng = np.random.default_rng(SEED + 20)
    guides = make_library(rng, 3000, 20)
    lib = str(d / "lib.fa")
    with open(lib, "wb") as f:
        f.write(b"".join(b">lib.%d\n%s\n" % (i, g) for i, g in enumerate(guides)))
    seqs = staggered(rng, guides, 150_000, 75, 10, 8)
    text = fastq(seqs)
    paths = {"bgzf": str(d / "b.fastq.gz"), "gzip": str(d / "m.fastq.gz"), "plain": str(d / "p.fastq")}
    with open(paths["bgzf"], "wb") as f:
        f.write(bgzf(text))
    with open(paths["gzip"], "wb") as f:
        f.write(gzip.compress(text, 6))
    with open(paths["plain"], "wb") as f:
        f.write(text)
    opaque = str(d / "opaque.fa")
    with open(opaque, "wb") as f:
        f.write(b">a\nACGTNACGTACGTACGTACG\n>b\nACGTACGTACGTACGTACGA\n")
    return {"lib": lib, "guides": guides, "seqs": seqs, "paths": paths, "opaque": opaque}


def test_cli_max_shift_equals_host_and_oracle(inputs):
    paths = [inputs["paths"][x] for x in ("bgzf", "gzip", "plain")]
    common = ("-l", inputs["lib"], "-a", "10", "-z", "--max-shift", "8")
    dev = run(*common, "-i", *paths, "--timing")
    t = timing(dev)
    assert t["device_ingest_samples"] == 3 and t["max_shift"] == 8, t
    host = run(*common, "-i", *paths, "--host-inflate")
    assert dev.stdout == host.stdout
    lines = run(*common, "-i", *paths, "--host-inflate", "--whole-lines")
    assert lines.stdout == host.stdout
    got = table_counts(dev.stdout, len(inputs["guides"]), 3)
    want = oracle_assign(inputs["guides"], inputs["seqs"], True, sg.Offset.Forward(10), 8)[1]
    for i in range(3):
        assert np.array_equal(got[i], want), paths[i]
    # the staggered sample needs the search: the reference's +-1 finds far fewer reads
    plain = table_counts(run("-l", inputs["lib"], "-a", "10", "-z", "-i", paths[2]).stdout, len(inputs["guides"]), 1)
    assert plain.sum() < 0.6 * got[2].sum()


def test_cli_max_shift_one_is_no_flag(inputs):
    paths = [inputs["paths"]["bgzf"], inputs["paths"]["plain"]]
    a = run("-l", inputs["lib"], "-i", *paths)
    b = run("-l", inputs["lib"], "-i", *paths, "--max-shift", "1")
    assert a.stdout == b.stdout and a.stderr == b.stderr
    ta = timing(run("-l", inputs["lib"], "-i", *paths, "--timing"))
    assert "max_shift" not in ta


def test_cli_read_shards(inputs):
    for kind in ("bgzf", "plain"):
        common = ("-l", inputs["lib"], "-a", "10", "--max-shift", "8", "-i", inputs["paths"][kind])
        one = run(*common)
        two = run(*common, "--read-shards", "2", env={"SGC_TEXT_WAVE": str(1 << 20)})
        assert one.stdout == two.stdout, kind


def test_cli_errors(inputs):
    base = ("-l", inputs["lib"], "-i", inputs["paths"]["plain"])
    for extra in (("-p", "--max-shift", "2"), ("--max-shift", "0"), ("--max-shift", "17")):
        p = run(*base, *extra, ok=False)
        assert p.returncode == 1 and "max-shift" in p.stderr, (extra, p.stderr)
    p = run("-l", inputs["opaque"], "-i", inputs["paths"]["plain"], "--max-shift", "2", ok=False)
    assert p.returncode == 1 and "max-shift" in p.stderr, p.stderr
    assert run("-l", inputs["opaque"], "-i", inputs["paths"]["plain"], "--max-shift", "1").returncode == 0
