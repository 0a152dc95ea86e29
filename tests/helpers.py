"""Shared test helpers: a small numpy generator of sgcount-shaped inputs (SURVEY.md §8d shapes,
scaled down) and oracle/CUDA adapters.  Test infrastructure only."""
import numpy as np

from oracle import oracle as orc

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
COMP = np.zeros(256, dtype=np.uint8)
COMP[:] = np.arange(256)
for a, b in zip(b"ACGT", b"TGCA"):
    COMP[a] = b


def make_library(rng, n, k, plant=0.01):
    """n unique k-mers with the position-dependent G skew of SURVEY.md §8d; a fraction
    `plant` of them are Hamming-1 and another `plant` Hamming-2 neighbours of earlier guides
    (forces ambiguous variants)."""
    seen, out = set(), []
    pg = 0.55 - 0.30 * np.arange(k) / max(k - 1, 1)
    while len(out) < n:
        u = rng.random(k)
        other = rng.integers(0, 3, k)
        s = np.where(u < pg, ord("G"), np.frombuffer(b"ACT", dtype=np.uint8)[other]).astype(np.uint8)
        r = rng.random()
        if out and r < 2 * plant:
            s = np.frombuffer(out[rng.integers(len(out))], dtype=np.uint8).copy()
            for p in rng.choice(k, 1 if r < plant else 2, replace=False):
                s[p] = rng.choice([c for c in b"ACGT" if c != s[p]])
        b = s.tobytes()
        if b not in seen:
            seen.add(b)
            out.append(b)
    return out


def make_reads(rng, guides, n_reads, read_len, offset, reverse=False, variable=False, junk=0.03, wild=b"N"):
    """Reads in the §8d class mix: exact, 1 substitution, 1 wildcard, 2 substitutions, +1/-1
    shift, truncated, random.  Returns a list of bytes."""
    k = len(guides[0])
    g = np.frombuffer(b"".join(guides), dtype=np.uint8).reshape(len(guides), k)
    weights = rng.lognormal(0.0, 1.0, len(guides))
    pick = rng.choice(len(guides), n_reads, p=weights / weights.sum())
    prefix = ACGT[rng.integers(0, 4, offset + 1)]
    suffix = ACGT[rng.integers(0, 4, read_len + 8)]
    reads = np.empty((n_reads, read_len), dtype=np.uint8)
    cls = rng.random(n_reads)
    lens = np.full(n_reads, read_len)
    for i in range(n_reads):
        w = g[pick[i]].copy()
        c = cls[i]
        shift = 0
        if c < 0.70:
            pass
        elif c < 0.80:
            p = rng.integers(k)
            w[p] = rng.choice([x for x in b"ACGT" if x != w[p]])
        elif c < 0.84:
            w[rng.integers(k)] = wild[0]
        elif c < 0.87:
            for p in rng.choice(k, 2, replace=False):
                w[p] = rng.choice([x for x in b"ACGT" if x != w[p]])
        elif c < 0.90:
            shift = 1
        elif c < 0.93:
            shift = -1
        elif c < 0.95:
            lens[i] = rng.integers(0, offset + k + 2)  # truncated around the window end
        elif c < 0.95 + junk:
            w = ACGT[rng.integers(0, 4, k)]
        elif c < 0.99:
            w[rng.integers(k)] = rng.choice(list(b"acgtJXN"))
        o = offset + shift
        row = np.concatenate([prefix[:max(o, 0)], w, suffix])[:read_len]
        if o < 0:
            row = np.concatenate([w[1:], suffix])[:read_len]
        reads[i] = row
    out = []
    for i in range(n_reads):
        r = reads[i, :lens[i]] if variable or lens[i] == read_len else reads[i]
        if not variable:
            r = reads[i]
        if reverse:
            r = COMP[r[::-1]]
        out.append(r.tobytes())
    return out


def realistic_fastq(rng, seqs):
    """FASTQ text as an Illumina instrument writes it, around the sequences `seqs`: headers
    '@A00123:45:HXXXXDSXX:1:1101:<x>:<y> 1:N:0:<index>' of varying length, a '+' line that repeats
    the name on some records, and Phred+33 qualities over '#'..'J' drawn per position, some of them
    starting with '@' (Q31) or '+' (Q10), which a framer must not take for a record or separator
    line.  Such text inflates from literal-heavy DEFLATE with long codes, unlike constant qualities.
    Returns the text and the (begin, end) of every quality line."""
    n = len(seqs)
    width = max(len(s) for s in seqs) if n else 0
    qual = rng.integers(ord("#"), ord("J") + 1, size=(n, max(width, 1)), dtype=np.uint8)
    first = rng.random(n)
    qual[first < 0.05, 0] = ord("@")
    qual[(first >= 0.05) & (first < 0.08), 0] = ord("+")
    xs, ys = rng.integers(1000, 10 ** rng.integers(4, 6, n)), rng.integers(1000, 10 ** rng.integers(4, 6, n))
    lanes, tiles = rng.integers(1, 5, n), rng.integers(1101, 2679, n)
    index = ACGT[rng.integers(0, 4, (n, 16))]
    dual = rng.random(n) < 0.5
    repeat = rng.random(n) < 0.2
    parts, slots, at = [], [], 0
    for i, s in enumerate(seqs):
        name = b"A00123:45:HXXXXDSXX:%d:%d:%d:%d" % (lanes[i], tiles[i], xs[i], ys[i])
        idx = index[i].tobytes() if dual[i] else index[i, :8].tobytes()
        rec = b"@%s 1:N:0:%s\n%s\n+%s\n" % (name, idx, s, name if repeat[i] else b"")
        q = qual[i, :len(s)].tobytes()
        slots.append((at + len(rec), at + len(rec) + len(q)))
        parts.append(rec + q + b"\n")
        at += len(parts[-1])
    return b"".join(parts), slots


def oracle_library(guides, aliases=None):
    aliases = aliases or [b"g%d" % i for i in range(len(guides))]
    recs = orc.Records.from_bytes(b"".join(b">" + a + b"\n" + s + b"\n" for a, s in zip(aliases, guides)))
    return orc.Library.from_reader(recs), recs
