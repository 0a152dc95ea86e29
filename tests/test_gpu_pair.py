"""Dual-guide constructs on the device (sgc_pair_counter, csrc/pair.cu) against the pair rule
(tests/pair_oracle.py) and against standalone counters: construct counts, the five class tallies, the
full recombinant report and both mates' marginal results must be equal bit for bit on key-family
boundaries (unequal mate lengths and a byte-keyed library included), every orientation pair and rc_mode,
Permuter and exact, recursion on and off, max_shift 1 and 8, mixed read layouts and span records, dense
and sparse construct lists, a dominant construct, launch splitting, a batch above 2^24 pairs, host and
device submits, accumulation, reset, report overflow and every error case."""
import numpy as np
import pytest

import sgcount_b200 as sg
from oracle import oracle as orc
from sgcount_b200 import _cabi

import pair_oracle as PO
from helpers import ACGT, make_library, make_reads

pytestmark = pytest.mark.gpu

SEED = 0x9A12


def libs_for(guides):
    library = sg.Library(guides, [b"g%d" % i for i in range(len(guides))])
    return library, sg.Permuter.new(library)


def mate_reads(rng, guides, picks, read_len, offset, reverse=False, variable=False):
    """read i carries guides[picks[i]] in make_reads' class mix (mismatches, Ns, shifts, truncation, junk);
    picks[i] < 0: a read of random bases"""
    out = [None] * len(picks)
    for g in np.unique(picks):
        idx = np.flatnonzero(picks == g)
        if g < 0:
            reads = [ACGT[rng.integers(0, 4, read_len)].tobytes() for _ in idx]
        else:
            reads = make_reads(rng, [guides[g]], len(idx), read_len, offset, reverse=reverse, variable=variable,
                               junk=0.05)
        for i, r in zip(idx, reads):
            out[i] = r
    return out


def construct_picks(rng, pairs, n, n1, n2, listed=0.7, missing=0.05):
    """intended guides per pair: a listed construct (lognormal weights), else two independent guides, and a
    few mates with no guide at all"""
    w = rng.lognormal(0.0, 1.0, len(pairs))
    j = rng.choice(len(pairs), n, p=w / w.sum())
    p = np.asarray(pairs)
    g1, g2 = p[j, 0].copy(), p[j, 1].copy()
    other = rng.random(n) >= listed
    g1[other] = rng.integers(0, n1, int(other.sum()))
    g2[other] = rng.integers(0, n2, int(other.sum()))
    g1[rng.random(n) < missing] = -1
    g2[rng.random(n) < missing] = -1
    return g1, g2


class Mate:
    """one mate's library and counter settings"""

    def __init__(self, guides, offset, with_perm=True, rc_mode=_cabi.RC_BITTRICK, max_shift=1, recursion=True):
        self.guides = guides
        self.library, self.permuter = libs_for(guides)
        self.offset = offset
        self.with_perm = with_perm
        self.rc_mode = rc_mode
        self.max_shift = max_shift
        self.recursion = recursion

    def counter(self, offset=None):
        return sg.Counter(self.library, self.permuter if self.with_perm else None, offset or self.offset, self.recursion,
                          self.rc_mode, max_shift=self.max_shift)

    def assignments(self, seqs):
        return PO.mate_assignments(seqs, self.guides, self.with_perm, orc.Offset(self.offset.reverse, self.offset.index),
                                   self.rc_mode, self.max_shift, self.recursion)


def standalone(mate, batch, offset=None):
    c = mate.counter(offset)
    c.submit(batch)
    counts, total, matched = c.finish()
    return counts.copy(), total, matched


def run_pair(m1, m2, batch1, batch2, pairs, capacity=1 << 16, off1=None, off2=None):
    c1, c2 = m1.counter(off1), m2.counter(off2)
    pc = sg.PairCounter(c1, c2, pairs, capacity)
    pc.submit(batch1, batch2)
    counts, info = pc.finish()
    rows = pc.recombinants() if capacity else None
    return counts, info, rows, c1.finish(), c2.finish(), (pc, c1, c2)


def check_against_statement(m1, m2, seqs1, seqs2, pairs, got, label=""):
    counts, info, rows, r1, r2, _ = got
    a1, a2 = m1.assignments(seqs1), m2.assignments(seqs2)
    want_counts, want, rec = PO.classify(a1, a2, pairs)
    assert np.array_equal(counts, want_counts), label
    for key in ("total",) + PO.CLASSES:
        assert info[key] == want[key], (label, key, info, want)
    assert info["overflow"] == 0 and info["distinct"] == len(rec), label
    if rows is not None:
        assert rows == PO.ordered(rec), label
    # the mates' own results: marginal counts, total = pairs, mate 1 matched = listed + recombined + first_only
    for r, a, m in ((r1, a1, m1), (r2, a2, m2)):
        assert np.array_equal(r[0], np.bincount(a[a >= 0], minlength=len(m.guides)).astype(np.uint64)), label
        assert r[1] == len(a) and r[2] == int((a >= 0).sum()), label
    assert r1[2] == want["listed"] + want["recombined"] + want["first_only"], label


def sparse_pairs(rng, n1, n2, n):
    """a 1:1 list plus one guide of each library shared by many constructs"""
    pairs = {(i % n1, (7 * i + 3) % n2) for i in range(n)}
    pairs |= {(0, j) for j in range(0, n2, 2)} | {(i, 1) for i in range(0, n1, 3)}
    return sorted(pairs)


@pytest.mark.parametrize("k1,k2", [(16, 30), (20, 20), (19, 21), (17, 25), (29, 16)])
@pytest.mark.parametrize("rev1,rev2", [(False, False), (False, True), (True, False), (True, True)])
def test_pairs_equal_statement(k1, k2, rev1, rev2):
    rng = np.random.default_rng(SEED + 100 * k1 + k2 + 7 * rev1 + 3 * rev2)
    g1, g2 = make_library(rng, 120, k1), make_library(rng, 90, k2)
    pairs = sparse_pairs(rng, len(g1), len(g2), 150)
    n = 3000
    p1, p2 = construct_picks(rng, pairs, n, len(g1), len(g2))
    o1, o2 = 4, 7
    seqs1 = mate_reads(rng, g1, p1, o1 + k1 + 10, o1, rev1)
    seqs2 = mate_reads(rng, g2, p2, o2 + k2 + 6, o2, rev2)
    b1, b2 = sg.ReadBatch.from_seqs(seqs1), sg.ReadBatch.from_seqs(seqs2)
    for rc_mode in (_cabi.RC_BITTRICK, _cabi.RC_KEEP_N):
        for with_perm in (True, False):
            m1 = Mate(g1, sg.Offset(rev1, o1), with_perm, rc_mode)
            m2 = Mate(g2, sg.Offset(rev2, o2), not with_perm, rc_mode)
            got = run_pair(m1, m2, b1, b2, pairs)
            check_against_statement(m1, m2, seqs1, seqs2, pairs, got, (rc_mode, with_perm))
            for mine, (m, b) in ((got[3], (m1, b1)), (got[4], (m2, b2))):
                alone = standalone(m, b)
                assert np.array_equal(mine[0], alone[0]) and mine[1:] == alone[1:], (rc_mode, with_perm)


def test_byte_keyed_library():
    """mate 2's library holds an N: its counter takes the byte-keyed kernel"""
    rng = np.random.default_rng(SEED + 1)
    g1, g2 = make_library(rng, 80, 20), make_library(rng, 60, 20)
    g2[5] = g2[5][:9] + b"N" + g2[5][10:]
    pairs = sparse_pairs(rng, len(g1), len(g2), 100)
    p1, p2 = construct_picks(rng, pairs, 4000, len(g1), len(g2))
    seqs1 = mate_reads(rng, g1, p1, 36, 5)
    seqs2 = mate_reads(rng, g2, p2, 40, 3, reverse=True, variable=True)
    m1, m2 = Mate(g1, sg.Offset.Forward(5)), Mate(g2, sg.Offset.Reverse(3))
    assert m2.library._exact.info().opaque == 1
    b1, b2 = sg.ReadBatch.from_seqs(seqs1), sg.ReadBatch.from_seqs(seqs2, force_offsets=True)
    got = run_pair(m1, m2, b1, b2, pairs)
    check_against_statement(m1, m2, seqs1, seqs2, pairs, got)
    assert got[5][2].launch_info().kernel == 2


@pytest.mark.parametrize("search1,search2", [((1, True), (1, False)), ((8, True), (1, True)), ((1, False), (8, True)),
                                             ((8, True), (8, True))])
def test_search_options(search1, search2):
    rng = np.random.default_rng(SEED + 10 * search1[0] + search2[0] + 2 * search1[1] + search2[1])
    g1, g2 = make_library(rng, 200, 20), make_library(rng, 200, 20)
    pairs = sparse_pairs(rng, 200, 200, 300)
    p1, p2 = construct_picks(rng, pairs, 4000, 200, 200)
    seqs1, seqs2 = mate_reads(rng, g1, p1, 42, 9), mate_reads(rng, g2, p2, 42, 9, reverse=True)
    b1, b2 = sg.ReadBatch.from_seqs(seqs1), sg.ReadBatch.from_seqs(seqs2)
    for with_perm in (True, False):
        m1 = Mate(g1, sg.Offset.Forward(9), with_perm, max_shift=search1[0], recursion=search1[1])
        m2 = Mate(g2, sg.Offset.Reverse(9), with_perm, max_shift=search2[0], recursion=search2[1])
        check_against_statement(m1, m2, seqs1, seqs2, pairs, run_pair(m1, m2, b1, b2, pairs), with_perm)


def test_mixed_layouts_and_span_records():
    """mate 1 fixed stride on an unaligned device base or as span records, mate 2 variable length or
    whole lines: every combination gives what whole lines give"""
    import torch

    rng = np.random.default_rng(SEED + 2)
    g1, g2 = make_library(rng, 150, 20), make_library(rng, 150, 18)
    pairs = sparse_pairs(rng, 150, 150, 200)
    p1, p2 = construct_picks(rng, pairs, 5000, 150, 150)
    o1, o2 = 6, 4
    seqs1 = mate_reads(rng, g1, p1, 50, o1)
    seqs2 = mate_reads(rng, g2, p2, 40, o2, reverse=True)
    var2 = mate_reads(rng, g2, p2, 40, o2, reverse=True, variable=True)
    for S in (1, 8):
        m1 = Mate(g1, sg.Offset.Forward(o1), max_shift=S)
        m2 = Mate(g2, sg.Offset.Reverse(o2), max_shift=S)
        whole1, whole2 = sg.ReadBatch.from_seqs(seqs1), sg.ReadBatch.from_seqs(seqs2)
        want = run_pair(m1, m2, whole1, whole2, pairs)
        check_against_statement(m1, m2, seqs1, seqs2, pairs, want, S)
        span1, soff1 = sg.span_batch(whole1, 20, m1.offset, True, max_shift=S)
        span2, soff2 = sg.span_batch(whole2, 18, m2.offset, True, max_shift=S)
        for b1, b2, off1, off2 in ((span1, whole2, soff1, None), (whole1, span2, None, soff2), (span1, span2, soff1, soff2)):
            got = run_pair(m1, m2, b1, b2, pairs, off1=off1, off2=off2)
            assert np.array_equal(got[0], want[0]) and got[1] == want[1] and got[2] == want[2], S
        # variable-length mate 2 on the host; unaligned fixed-stride mate 1 on the device
        vb2 = sg.ReadBatch.from_seqs(var2, force_offsets=True)
        check_against_statement(m1, m2, seqs1, var2, pairs, run_pair(m1, m2, whole1, vb2, pairs), ("var", S))
        base = 3
        d1 = torch.from_numpy(np.concatenate([np.zeros(base, np.uint8), whole1.lines, np.zeros(64, np.uint8)])).cuda()
        d2 = torch.from_numpy(np.concatenate([vb2.lines, np.zeros(64, np.uint8)])).cuda()
        d2off = torch.from_numpy(vb2.line_off).cuda()
        c1, c2 = m1.counter(), m2.counter()
        pc = sg.PairCounter(c1, c2, pairs, 1 << 16)
        pc.submit_device(len(seqs1), d1.data_ptr() + base, whole1.lines.nbytes, d2.data_ptr(), vb2.lines.nbytes,
                         stride1=whole1.stride, read_len1=whole1.read_len, d_line_off2=d2off.data_ptr())
        counts, info = pc.finish()
        got = (counts, info, pc.recombinants(), c1.finish(), c2.finish(), None)
        check_against_statement(m1, m2, seqs1, var2, pairs, got, ("device", S))


@pytest.mark.parametrize("kind", ["all_by_all", "sparse"])
def test_dense_and_sparse_lists(kind):
    rng = np.random.default_rng(SEED + (kind == "sparse"))
    n1 = n2 = 300
    g1, g2 = make_library(rng, n1, 20), make_library(rng, n2, 20)
    if kind == "all_by_all":
        pairs = [(i, j) for i in range(n1) for j in range(n2)]
    else:
        pairs = sparse_pairs(rng, n1, n2, 300)
    p1, p2 = construct_picks(rng, pairs, 20_000, n1, n2)
    seqs1, seqs2 = mate_reads(rng, g1, p1, 40, 5), mate_reads(rng, g2, p2, 40, 5)
    m1, m2 = Mate(g1, sg.Offset.Forward(5)), Mate(g2, sg.Offset.Forward(5))
    got = run_pair(m1, m2, sg.ReadBatch.from_seqs(seqs1), sg.ReadBatch.from_seqs(seqs2), pairs)
    check_against_statement(m1, m2, seqs1, seqs2, pairs, got, kind)
    if kind == "all_by_all":
        assert got[1]["recombined"] == 0


def test_dominant_construct_keeps_the_skew_plan():
    """90 % of 300 000 pairs on one construct: the mates' counters make their skew plan (replicas, hot
    guides) and every count is still exact"""
    rng = np.random.default_rng(SEED + 3)
    g1, g2 = make_library(rng, 500, 20), make_library(rng, 500, 20)
    pairs = sparse_pairs(rng, 500, 500, 600)
    n = 300_000
    n_rest = n // 10
    p1, p2 = construct_picks(rng, pairs, n_rest, 500, 500)
    rest1, rest2 = mate_reads(rng, g1, p1, 40, 5), mate_reads(rng, g2, p2, 40, 5)
    top = pairs[17]
    r1 = b"ACGTA" + g1[top[0]] + b"TTGCAGGATCCAATGC"[:15]
    r2 = b"CCATG" + g2[top[1]] + b"GATTACAGATTACAG"
    order = rng.permutation(n)
    seqs1 = [r1] * (n - n_rest) + rest1
    seqs2 = [r2] * (n - n_rest) + rest2
    seqs1 = [seqs1[i] for i in order]
    seqs2 = [seqs2[i] for i in order]
    m1, m2 = Mate(g1, sg.Offset.Forward(5)), Mate(g2, sg.Offset.Forward(5))
    got = run_pair(m1, m2, sg.ReadBatch.from_seqs(seqs1), sg.ReadBatch.from_seqs(seqs2), pairs)
    check_against_statement(m1, m2, seqs1, seqs2, pairs, got)
    assert got[0][17] >= n - n_rest
    for c in got[5][1:]:
        li = c.launch_info()
        assert li.kernel == 1 and li.replicas > 1 and li.hot_guides >= 1


def test_launch_splitting(monkeypatch):
    rng = np.random.default_rng(SEED + 4)
    g1, g2 = make_library(rng, 100, 20), make_library(rng, 100, 24)
    pairs = sparse_pairs(rng, 100, 100, 100)
    p1, p2 = construct_picks(rng, pairs, 9000, 100, 100)
    seqs1, seqs2 = mate_reads(rng, g1, p1, 40, 5), mate_reads(rng, g2, p2, 41, 2, variable=True)
    b1, b2 = sg.ReadBatch.from_seqs(seqs1), sg.ReadBatch.from_seqs(seqs2, force_offsets=True)
    for S in (1, 8):
        m1, m2 = Mate(g1, sg.Offset.Forward(5), max_shift=S), Mate(g2, sg.Offset.Forward(2))
        whole = run_pair(m1, m2, b1, b2, pairs)
        monkeypatch.setenv("SGC_MAX_LAUNCH_TILES", "37")
        split = run_pair(m1, m2, b1, b2, pairs)
        monkeypatch.delenv("SGC_MAX_LAUNCH_TILES")
        assert split[5][1].launch_info().launches_total > whole[5][1].launch_info().launches_total
        check_against_statement(m1, m2, seqs1, seqs2, pairs, split, S)
        assert np.array_equal(whole[0], split[0]) and whole[1] == split[1] and whole[2] == split[2], S


def test_batch_above_2_24_pairs():
    """one device batch of 2^24 + 4099 pairs: a block of pairs repeated; counts scale exactly"""
    import torch

    rng = np.random.default_rng(SEED + 5)
    g1, g2 = make_library(rng, 200, 20), make_library(rng, 200, 20)
    pairs = sparse_pairs(rng, 200, 200, 300)
    block = 8192
    p1, p2 = construct_picks(rng, pairs, block, 200, 200)
    seqs1, seqs2 = mate_reads(rng, g1, p1, 36, 5), mate_reads(rng, g2, p2, 44, 7, reverse=True)
    b1, b2 = sg.ReadBatch.from_seqs(seqs1), sg.ReadBatch.from_seqs(seqs2)
    n = (1 << 24) + 4099
    reps, rest = divmod(n, block)
    m1, m2 = Mate(g1, sg.Offset.Forward(5)), Mate(g2, sg.Offset.Reverse(7))
    d1 = torch.from_numpy(b1.lines.copy()).cuda().repeat(reps + 1)
    d2 = torch.from_numpy(b2.lines.copy()).cuda().repeat(reps + 1)
    c1, c2 = m1.counter(), m2.counter()
    pc = sg.PairCounter(c1, c2, pairs, 1 << 16)
    pc.submit_device(n, d1.data_ptr(), n * b1.stride, d2.data_ptr(), n * b2.stride, stride1=b1.stride,
                     read_len1=b1.read_len, stride2=b2.stride, read_len2=b2.read_len)
    counts, info = pc.finish()
    a1, a2 = m1.assignments(seqs1), m2.assignments(seqs2)
    wc, wt, wr = PO.classify(a1, a2, pairs)
    pc_, pt, pr = PO.classify(a1[:rest], a2[:rest], pairs)
    assert np.array_equal(counts, wc * reps + pc_)
    for key in ("total",) + PO.CLASSES:
        assert info[key] == wt[key] * reps + pt[key], key
    want_rec = {key: v * reps + pr.get(key, 0) for key, v in wr.items()}
    assert pc.recombinants() == PO.ordered(PO.Tally(want_rec))
    t1 = c1.finish()
    assert t1[1] == n and t1[2] == int((a1 >= 0).sum()) * reps + int((a1[:rest] >= 0).sum())


def test_host_and_device_submit_accumulate_and_reset():
    import torch

    rng = np.random.default_rng(SEED + 6)
    g1, g2 = make_library(rng, 100, 20), make_library(rng, 100, 20)
    pairs = sparse_pairs(rng, 100, 100, 150)
    p1, p2 = construct_picks(rng, pairs, 6000, 100, 100)
    seqs1, seqs2 = mate_reads(rng, g1, p1, 40, 5), mate_reads(rng, g2, p2, 40, 5)
    b1, b2 = sg.ReadBatch.from_seqs(seqs1), sg.ReadBatch.from_seqs(seqs2, force_offsets=True)
    m1, m2 = Mate(g1, sg.Offset.Forward(5)), Mate(g2, sg.Offset.Forward(5))
    c1, c2 = m1.counter(), m2.counter()
    pc = sg.PairCounter(c1, c2, pairs, 1 << 16)
    pc.submit(b1, b2)
    pc.wait_copies()
    host = pc.finish()
    d1 = torch.from_numpy(b1.lines.copy()).cuda()
    d2 = torch.from_numpy(b2.lines.copy()).cuda()
    d2off = torch.from_numpy(b2.line_off).cuda()
    pc.submit_device(len(seqs1), d1.data_ptr(), b1.lines.nbytes, d2.data_ptr(), b2.lines.nbytes, stride1=b1.stride,
                     read_len1=b1.read_len, d_line_off2=d2off.data_ptr())
    both = pc.finish()
    assert np.array_equal(both[0], 2 * host[0])
    for key in ("total",) + PO.CLASSES + ("distinct",):
        assert both[1][key] == (host[1][key] if key == "distinct" else 2 * host[1][key]), key
    assert c1.finish()[1] == 2 * len(seqs1) and c2.finish()[1] == 2 * len(seqs2)
    pc.reset()
    counts, info = pc.finish()
    assert not counts.any() and not any(info.values()) and pc.recombinants() == []
    assert c1.finish()[1] == 0 and c2.finish()[1] == 0 and not c2.finish()[0].any()
    pc.submit(b1, b2)
    got = pc.finish()
    assert np.array_equal(got[0], host[0]) and got[1] == host[1]
    check_against_statement(m1, m2, seqs1, seqs2, pairs, (*got, pc.recombinants(), c1.finish(), c2.finish(), None))


def test_recombinant_overflow_keeps_held_counts_exact():
    rng = np.random.default_rng(SEED + 7)
    g1, g2 = make_library(rng, 100, 20), make_library(rng, 100, 20)
    pairs = [(i, i) for i in range(100)]
    p1, p2 = construct_picks(rng, pairs, 20_000, 100, 100, listed=0.3)
    seqs1, seqs2 = mate_reads(rng, g1, p1, 40, 5), mate_reads(rng, g2, p2, 40, 5)
    m1, m2 = Mate(g1, sg.Offset.Forward(5)), Mate(g2, sg.Offset.Forward(5))
    counts, info, rows, _, _, _ = run_pair(m1, m2, sg.ReadBatch.from_seqs(seqs1), sg.ReadBatch.from_seqs(seqs2), pairs,
                                           capacity=64)
    _, want, rec = PO.classify(m1.assignments(seqs1), m2.assignments(seqs2), pairs)
    assert len(rec) > 64 and info["overflow"] > 0
    assert info["distinct"] == len(rows) <= 64
    assert info["recombined"] == want["recombined"] == info["overflow"] + sum(n for _, _, n in rows)
    for a, b, n in rows:
        assert rec[(a, b)] == n
    assert rows == sorted(rows, key=lambda r: (-r[2], r[0], r[1]))


def test_errors():
    rng = np.random.default_rng(SEED + 8)
    g1, g2 = make_library(rng, 10, 20), make_library(rng, 12, 20)
    m1, m2 = Mate(g1, sg.Offset.Forward(0)), Mate(g2, sg.Offset.Forward(0))
    pairs = [(0, 0), (1, 2)]

    def refused(code, *args, **kw):
        with pytest.raises(sg.SgcError) as e:
            sg.PairCounter(*args, **kw)
        assert e.value.code == code, e.value

    c1, c2 = m1.counter(), m2.counter()
    refused(_cabi.ERR_INVALID_ARG, c1, c1, pairs)
    refused(_cabi.ERR_INVALID_ARG, c1, c2, [])
    refused(_cabi.ERR_INVALID_ARG, c1, c2, [(10, 0)])
    refused(_cabi.ERR_INVALID_ARG, c1, c2, [(0, 12)])
    refused(_cabi.ERR_INVALID_ARG, c1, c2, [(0, -1)])
    refused(_cabi.ERR_INVALID_ARG, c1, c2, pairs, (1 << 26) + 1)
    refused(_cabi.ERR_DUPLICATE_SEQUENCE, c1, c2, [(0, 0), (1, 2), (3, 4), (1, 2)])
    reported = sg.Counter(m1.library, m1.permuter, m1.offset, unmatched_capacity=16)
    refused(_cabi.ERR_INVALID_ARG, reported, c2, pairs)
    refused(_cabi.ERR_INVALID_ARG, c1, reported, pairs)
    counted = m2.counter()
    counted.submit(sg.ReadBatch.from_seqs([g2[0] + b"ACGT"]))
    refused(_cabi.ERR_INVALID_ARG, c1, counted, pairs)
    pc = sg.PairCounter(c1, c2, pairs)  # no report
    with pytest.raises(sg.SgcError) as e:
        pc.recombinants()
    assert e.value.code == _cabi.ERR_INVALID_ARG
    one, two = sg.ReadBatch.from_seqs([g1[0]]), sg.ReadBatch.from_seqs([g2[0], g2[1]])
    with pytest.raises(sg.SgcError):
        pc.submit(one, two)
    # a fixed-stride batch that does not fit its bytes
    with pytest.raises(sg.SgcError) as e:
        _cabi.check(_cabi.load().sgc_pair_counter_submit(pc._ptr, one.lines.ctypes.data, 3, None, one.stride, one.read_len, two.lines.ctypes.data,
                             two.lines.nbytes, None, two.stride, two.read_len, 1))
    assert e.value.code == _cabi.ERR_INVALID_ARG
    pc.submit(sg.ReadBatch.from_seqs([g1[1]]), sg.ReadBatch.from_seqs([g2[2]]))
    counts, info = pc.finish()
    assert counts.tolist() == [0, 1] and info["listed"] == 1 == info["total"]
    import ctypes as C

    dev = C.c_int()
    _cabi.check(_cabi.load().sgc_device_count(C.byref(dev)))
    if dev.value >= 2:
        other = sg.Library(g2, [b"x%d" % i for i in range(len(g2))], device=1)
        refused(_cabi.ERR_INVALID_ARG, m1.counter(), sg.Counter(other, None, m2.offset), pairs)


def test_launch_cut_changed_between_create_and_submit(monkeypatch):
    """the assignment scratch has a fixed size, so chunks sized under another SGC_MAX_LAUNCH_TILES than the one
    at create still fit it"""
    rng = np.random.default_rng(SEED + 9)
    g1, g2 = make_library(rng, 100, 20), make_library(rng, 100, 20)
    pairs = sparse_pairs(rng, 100, 100, 100)
    p1, p2 = construct_picks(rng, pairs, 9000, 100, 100)
    seqs1, seqs2 = mate_reads(rng, g1, p1, 40, 5), mate_reads(rng, g2, p2, 40, 5)
    b1, b2 = sg.ReadBatch.from_seqs(seqs1), sg.ReadBatch.from_seqs(seqs2)
    m1, m2 = Mate(g1, sg.Offset.Forward(5)), Mate(g2, sg.Offset.Forward(5))
    for at_create, at_submit in (("37", None), (None, "37")):
        c1, c2 = m1.counter(), m2.counter()
        if at_create:
            monkeypatch.setenv("SGC_MAX_LAUNCH_TILES", at_create)
        pc = sg.PairCounter(c1, c2, pairs, 1 << 16)
        monkeypatch.delenv("SGC_MAX_LAUNCH_TILES", raising=False)
        if at_submit:
            monkeypatch.setenv("SGC_MAX_LAUNCH_TILES", at_submit)
        pc.submit(b1, b2)
        monkeypatch.delenv("SGC_MAX_LAUNCH_TILES", raising=False)
        counts, info = pc.finish()
        got = (counts, info, pc.recombinants(), c1.finish(), c2.finish(), None)
        check_against_statement(m1, m2, seqs1, seqs2, pairs, got, (at_create, at_submit))
