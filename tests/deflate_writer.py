"""A token-level DEFLATE writer (RFC 1951) with gzip (RFC 1952) and BGZF framing, for tests only.

zlib's encoder, which writes every other compressed input of the suite, never emits a distance above
32 506 (its MAX_DIST is 32 768 - 262) and always sends at least two distance codes.  Other encoders
(libdeflate, which bgzip uses when built with it, ISA-L igzip, zopfli, 7-Zip) do both, so a decoder
must take the whole 32 KiB window and the incomplete distance codes RFC 1951 allows.  This writer
makes such streams from an explicit token list:

  tokens   a list of literals (int 0..255) and matches ((length, distance) tuples); `parse` makes one
           from a text with a greedy LZ77 parse over the full window, `plant` puts edge matches into a
           text for it to find;
  blocks   a list of (kind, n_tokens), kind in "dynamic", "fixed", "stored", "empty"; see `deflate`.

It is written for clarity over speed, but parses and writes ~1 MB of text in a few seconds.
"""
import bisect
import heapq
import struct
import zlib

WINDOW = 32768
MAX_MATCH = 258

# RFC 1951 3.2.5: (symbol, extra bits, base) of every length and distance
_LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
_LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
_DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
              6145, 8193, 12289, 16385, 24577]
_DIST_EXTRA = [0, 0, 0, 0] + [e for e in range(1, 14) for _ in (0, 1)]
_CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]


def _table(bases, extras, top):
    sym = [0] * (top + 1)
    for s, (b, e) in enumerate(zip(bases, extras)):
        for v in range(b, min(b + (1 << e), top + 1)):
            sym[v] = s
    return sym


_LEN_SYM = _table(_LEN_BASE, _LEN_EXTRA, MAX_MATCH)
_LEN_SYM[258] = 28  # 258 has a code of its own (symbol 285), not 284 with extra bits 31
_DIST_SYM = _table(_DIST_BASE, _DIST_EXTRA, WINDOW)


class BitWriter:
    """LSB-first bits, as DEFLATE packs them"""

    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def bits(self, v, n):
        self.acc |= v << self.n
        self.n += n
        if self.n >= 64:
            k = self.n // 8
            self.out += (self.acc & ((1 << (8 * k)) - 1)).to_bytes(k, "little")
            self.acc >>= 8 * k
            self.n -= 8 * k


    def align(self):
        self.bits(0, -self.n % 8)

    def bit_pos(self):
        return 8 * len(self.out) + self.n

    def getvalue(self):
        k = (self.n + 7) // 8
        return bytes(self.out) + self.acc.to_bytes(k, "little")


def code_lengths(freq, limit):
    """Huffman code lengths of at most `limit` bits for the symbols of nonzero frequency.  One used
    symbol gets one code of length 1 (an incomplete code); otherwise the code is complete."""
    used = [s for s, f in enumerate(freq) if f]
    lengths = [0] * len(freq)
    if len(used) == 1:
        lengths[used[0]] = 1
        return lengths
    if not used:
        return lengths
    heap = [(freq[s], s, [s]) for s in used]
    heapq.heapify(heap)
    tie = len(freq)
    while len(heap) > 1:
        fa, _, a = heapq.heappop(heap)
        fb, _, b = heapq.heappop(heap)
        for s in a + b:
            lengths[s] += 1
        heapq.heappush(heap, (fa + fb, tie, a + b))
        tie += 1
    if max(lengths) > limit:
        # clamp, then restore the Kraft sum: lengthen the longest codes below the limit while the code
        # is over-subscribed, shorten the longest ones while it is incomplete
        for s in used:
            lengths[s] = min(lengths[s], limit)
        kraft = sum(1 << (limit - lengths[s]) for s in used)
        by_rarity = sorted(used, key=lambda s: freq[s])
        while kraft > 1 << limit:
            s = max((x for x in by_rarity if lengths[x] < limit), key=lambda x: lengths[x])
            lengths[s] += 1
            kraft -= 1 << (limit - lengths[s])
        while kraft < 1 << limit:
            s = max((x for x in reversed(by_rarity) if lengths[x] > 1 and (1 << (limit - lengths[x])) <= (1 << limit) - kraft), key=lambda x: lengths[x])
            kraft += 1 << (limit - lengths[s])
            lengths[s] -= 1
    assert sum(1 << (limit - lengths[s]) for s in used) == 1 << limit
    return lengths


def canonical_codes(lengths):
    """RFC 1951 3.2.2: the code of every symbol from the code lengths, bit-reversed (a Huffman code goes
    out most significant bit first, the bit writer sends the least significant first)"""
    count = [0] * 16
    for n in lengths:
        count[n] += 1
    count[0] = 0
    code, nxt = 0, [0] * 16
    for b in range(1, 16):
        code = (code + count[b - 1]) << 1
        nxt[b] = code
    codes = [0] * len(lengths)
    for s, n in enumerate(lengths):
        if n:
            codes[s] = int(format(nxt[n], f"0{n}b")[::-1], 2)
            nxt[n] += 1
    return codes


FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 30


def _rle_lengths(lengths):
    """the code-length alphabet's symbols (sym, extra value, extra bits) for a run of code lengths"""
    out, i = [], 0
    while i < len(lengths):
        v = lengths[i]
        run = 1
        while i + run < len(lengths) and lengths[i + run] == v:
            run += 1
        if v == 0 and run >= 3:
            r = min(run, 138)
            out.append((18, r - 11, 7) if r >= 11 else (17, r - 3, 3))
            i += r
            continue
        out.append((v, 0, 0))
        i += 1
        run -= 1
        while run >= 3:
            r = min(run, 6)
            out.append((16, r - 3, 2))
            i += r
            run -= r
    return out


class Stats:
    """what a stream holds: the tests check that the edges they ask for are really there"""

    def __init__(self):
        self.dists = []          # distance of every match
        self.lengths = []        # length of every match
        self.kinds = []          # kind of every block
        self.end_bits = []       # bit offset (in the DEFLATE stream) where every block ends
        self.lone_dist = 0       # dynamic blocks with one distance code
        self.no_dist = 0         # dynamic blocks with no distance code
        self.straddle = 0        # matches whose source runs across an earlier block end
        self.stored_lens = []    # LEN of every stored block


def _write_block(bw, kind, toks, last, stats, text_at, out_pos, block_starts):
    """one block of tokens; text_at(i, n): n bytes of the text at i (for stored blocks)"""
    bw.bits(int(last), 1)
    if kind == "stored":
        n = sum(1 if isinstance(t, int) else t[0] for t in toks)
        assert n <= 0xFFFF
        bw.bits(0, 2)
        bw.align()
        bw.bits(n, 16)
        bw.bits(n ^ 0xFFFF, 16)
        for b in text_at(out_pos, n):
            bw.bits(b, 8)
        stats.stored_lens.append(n)
        return
    lit_f, dist_f = [0] * 286, [0] * 30
    lit_f[256] = 1
    for t in toks:
        if isinstance(t, int):
            lit_f[t] += 1
        else:
            lit_f[257 + _LEN_SYM[t[0]]] += 1
            dist_f[_DIST_SYM[t[1]]] += 1
    if kind == "fixed":
        bw.bits(1, 2)
        ll, dl = FIXED_LIT, FIXED_DIST
    else:
        bw.bits(2, 2)
        if sum(1 for f in lit_f if f) == 1:  # the end-of-block code alone: complete it with literal 0
            lit_f[0] = 1
        ll = code_lengths(lit_f, 15)
        dl = code_lengths(dist_f, 15)  # one code of length 1, or none at all, when at most one distance is used
        used_d = sum(1 for f in dist_f if f)
        stats.lone_dist += used_d == 1
        stats.no_dist += used_d == 0
        nl = max(257, max(s for s in range(286) if ll[s]) + 1)
        nd = max(1, max((s for s in range(30) if dl[s]), default=0) + 1)
        rle = _rle_lengths(ll[:nl] + dl[:nd])
        cl_f = [0] * 19
        for s, _, _ in rle:
            cl_f[s] += 1
        if sum(1 for f in cl_f if f) == 1:  # the code-length code must be complete
            cl_f[0 if rle[0][0] else 1] += 1
        cl = code_lengths(cl_f, 7)
        ncl = max(4, max(i for i in range(19) if cl[_CL_ORDER[i]]) + 1)
        bw.bits(nl - 257, 5)
        bw.bits(nd - 1, 5)
        bw.bits(ncl - 4, 4)
        for i in range(ncl):
            bw.bits(cl[_CL_ORDER[i]], 3)
        clc = canonical_codes(cl)
        for s, v, n in rle:
            bw.bits(clc[s], cl[s])
            if n:
                bw.bits(v, n)
    lc, dc = canonical_codes(ll), canonical_codes(dl)
    pos = out_pos
    for t in toks:
        if isinstance(t, int):
            bw.bits(lc[t], ll[t])
            pos += 1
            continue
        length, dist = t
        s = _LEN_SYM[length]
        bw.bits(lc[257 + s], ll[257 + s])
        if _LEN_EXTRA[s]:
            bw.bits(length - _LEN_BASE[s], _LEN_EXTRA[s])
        d = _DIST_SYM[dist]
        bw.bits(dc[d], dl[d])
        if _DIST_EXTRA[d]:
            bw.bits(dist - _DIST_BASE[d], _DIST_EXTRA[d])
        stats.dists.append(dist)
        stats.lengths.append(length)
        src = pos - dist
        if any(src < b < src + length for b in block_starts[-8:]):
            stats.straddle += 1
        pos += length
    bw.bits(lc[256], ll[256])


def deflate(tokens, blocks, text=None, stats=None):
    """Raw DEFLATE of `tokens` cut into `blocks` [(kind, n_tokens)], which must cover the tokens.
    Kinds: "dynamic" (code lengths from the block's own frequencies, at most 15 bits, 7 for the
    code-length code), "fixed", "stored" (its tokens are sent as their bytes, so `text` is needed;
    more than 65 535 bytes become several stored blocks), "empty" (a dynamic block of the end-of-block
    code alone; n_tokens must be 0).  The last block is marked final."""
    assert sum(n for _, n in blocks) == len(tokens)
    stats = stats if stats is not None else Stats()
    if any(k == "stored" for k, _ in blocks) and text is None:
        text = expand(tokens)
    bw = BitWriter()
    at, out_pos, block_starts = 0, 0, []
    for bi, (kind, n) in enumerate(blocks):
        toks = tokens[at:at + n]
        parts = [(kind, toks)]
        if kind == "stored":  # LEN is 16 bits
            parts, cur, size = [], [], 0
            for t in toks:
                w = 1 if isinstance(t, int) else t[0]
                if size + w > 0xFFFF:
                    parts.append(("stored", cur))
                    cur, size = [], 0
                cur.append(t)
                size += w
            parts.append(("stored", cur))
        elif kind == "empty":
            assert n == 0
            parts = [("dynamic", [])]
        for pi, (k, ts) in enumerate(parts):
            last = bi == len(blocks) - 1 and pi == len(parts) - 1
            block_starts.append(out_pos)
            _write_block(bw, k, ts, last, stats, lambda i, m: text[i:i + m], out_pos, block_starts)
            out_pos += sum(1 if isinstance(t, int) else t[0] for t in ts)
            stats.kinds.append(kind)
            stats.end_bits.append(bw.bit_pos())
        at += n
    return bw.getvalue()


def expand(tokens, before=None):
    """the text of a token list, byte by byte (an independent check of the writer); ValueError for a
    match reaching in front of the text, unless `before` gives the bytes a decoder that does not
    check would find there"""
    out = bytearray(before or b"")
    for t in tokens:
        if isinstance(t, int):
            out.append(t)
            continue
        length, dist = t
        if not (3 <= length <= MAX_MATCH and 1 <= dist <= WINDOW) or dist > len(out):
            raise ValueError(f"bad match {t} at {len(out)}")
        for _ in range(length):
            out.append(out[-dist])
    return bytes(out[len(before or b""):])


def gzip_header(flags=0, extra=b"", name=b"", comment=b""):
    """an RFC 1952 header; flags: FHCRC 2, FEXTRA 4, FNAME 8, FCOMMENT 16 (FEXTRA, FNAME, FCOMMENT are
    set by their fields)"""
    flg = (flags & 2) | (4 if extra else 0) | (8 if name else 0) | (16 if comment else 0)
    h = bytes([0x1F, 0x8B, 8, flg, 0, 0, 0, 0, 0, 3])
    if extra:
        h += struct.pack("<H", len(extra)) + extra
    if name:
        h += name + b"\0"
    if comment:
        h += comment + b"\0"
    if flg & 2:
        h += struct.pack("<H", zlib.crc32(h) & 0xFFFF)
    return h


def gzip_member(body, text, header=None):
    """a gzip member around the raw DEFLATE `body` of `text` (CRC-32 and ISIZE of `text`)"""
    return (header or gzip_header()) + body + struct.pack("<II", zlib.crc32(text), len(text) & 0xFFFFFFFF)


BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf_member(body, text):
    """one BGZF block: a gzip member whose 'BC' extra subfield holds its size - 1"""
    assert len(text) <= 0x10000
    size = 18 + len(body) + 8
    assert size <= 0x10000
    head = bytes([0x1F, 0x8B, 8, 4, 0, 0, 0, 0, 0, 0xFF, 6, 0]) + b"BC" + struct.pack("<HH", 2, size - 1)
    return head + body + struct.pack("<II", zlib.crc32(text), len(text))


# ---- the parser ---------------------------------------------------------------------------------

def _match_len(t, a, b, limit):
    """the longest L <= limit with t[a:a+L] == t[b:b+L] (a < b; the source may overlap the target)"""
    if t[a:a + 3] != t[b:b + 3]:
        return 0
    lo, hi = 3, limit
    while lo < hi:
        mid = (lo + hi + 1) // 2
        if t[a:a + mid] == t[b:b + mid]:
            lo = mid
        else:
            hi = mid - 1
    return lo


def parse(text, force=(), chain=8, literals=0):
    """Greedy LZ77 over the full 32 768-byte window: at every position the longest match a 3-byte hash
    chain (at most `chain` steps) finds, the farthest among equally long ones, or a literal.
    `force`: (position, length, distance) matches the parse must emit exactly (the text must hold
    them, as `plant` makes it); a match in front of one is shortened so that the forced one starts on
    time.  The first `literals` bytes are sent as literals (for stored blocks of an exact size)."""
    t = bytes(text)
    n = len(t)
    forced = dict((p, (ln, d)) for p, ln, d in force)
    marks = sorted(forced)
    mi = 0
    head, prev = {}, [-1] * n
    out = []
    i = 0
    inserted = 0

    def insert_to(j):
        nonlocal inserted
        while inserted < j and inserted + 3 <= n:
            k = t[inserted:inserted + 3]
            prev[inserted] = head.get(k, -1)
            head[k] = inserted
            inserted += 1
        inserted = max(inserted, j)

    while i < n:
        while mi < len(marks) and marks[mi] < i:
            mi += 1
        nxt = marks[mi] if mi < len(marks) else n + MAX_MATCH
        if i < literals:
            out.append(t[i])
            i += 1
            continue
        if i in forced:
            ln, d = forced[i]
            assert t[i - d:i - d + ln] == t[i:i + ln], (i, ln, d)
            out.append((ln, d))
            insert_to(i + ln)
            i += ln
            continue
        limit = min(MAX_MATCH, n - i, nxt - i)
        best, best_d = 0, 0
        if limit >= 3:
            insert_to(i)
            c, steps = head.get(t[i:i + 3], -1), 0
            while c >= 0 and i - c <= WINDOW and steps < chain:
                m = _match_len(t, c, i, limit)
                if m >= best and m >= 3:  # the chain runs from near to far: the farthest of equal length wins
                    best, best_d = m, i - c
                c = prev[c]
                steps += 1
        if best >= 3:
            out.append((best, best_d))
            insert_to(i + best)
            i += best
        else:
            out.append(t[i])
            i += 1
    return out


EDGE_DISTS = list(range(1, 18)) + [31, 32, 33, 255, 256, 257] + list(range(32506, 32769))
EDGE_LENS = list(range(3, 19)) + [256, 257, 258]


def plant(text, rng, slots, specs, block=None):
    """Copies matches into `text` (a bytearray): for every (dists, lengths, count) of `specs`, `count`
    of them with a distance from `dists` and a length from `lengths`.  Source and target lie inside
    one of `slots`, a list of (begin, end) ranges that may be overwritten (the quality lines of a FASTQ
    text, or the whole text); with `block`, inside one `block`-byte piece of the text too (a BGZF
    block).  No target overlaps another match's source or target, so every planted match still holds
    at the end.  Returns the planted (position, length, distance), sorted."""
    begins = [a for a, _ in slots]
    busy = bytearray(len(text))  # 1: a source, 2: a target
    out = []
    for dists, lengths, count in specs:
        placed, tries = 0, 0
        while placed < count and tries < 200 * count:
            tries += 1
            d, ln = rng.choice(dists), rng.choice(lengths)
            a, b = slots[rng.randrange(len(slots))]
            if b - a < ln:
                continue
            p = rng.randrange(a, b - ln + 1)
            src = p - d
            k = bisect.bisect_right(begins, src) - 1
            if src < 0 or k < 0 or src + min(ln, d) > slots[k][1] or (d < ln and slots[k] != (a, b)):
                continue
            if block and src // block != (p + ln - 1) // block:
                continue
            if busy[p:p + ln].count(0) != ln or 2 in busy[src:min(src + ln, p)]:
                continue
            for j in range(ln):  # (d < ln: the copy reads what it writes, a run of period d)
                text[p + j] = text[p + j - d]
            busy[src:min(src + ln, p)] = b"\1" * (min(src + ln, p) - src)
            busy[p:p + ln] = b"\2" * ln
            out.append((p, ln, d))
            placed += 1
    return sorted(out)


def layout(n_tokens, rng, kinds=("dynamic",), sizes=(200, 20000), tiny=0.2):
    """blocks of random kind (from `kinds`) and random size covering n_tokens tokens; a share `tiny` of
    them hold 1-4 tokens (at most one distance: a lone distance code, or none)"""
    blocks, left = [], n_tokens
    while left:
        k = rng.choice(kinds)
        if k == "empty":
            blocks.append((k, 0))
            continue
        n = min(left, rng.randint(1, 4) if rng.random() < tiny else rng.randint(*sizes))
        blocks.append((k, n))
        left -= n
    return blocks
