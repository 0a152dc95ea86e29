// inflate_core.h — one gzip member (RFC 1952 framing, RFC 1951 DEFLATE), decoded by ONE sequential
// context: a thread of the device kernel in gzip.cu, or the host (the same source compiles with
// g++ for tests/test_device_inflate_core.py, which checks it against zlib on every block kind).
//
// Written from the RFCs for this use: many small members (BGZF blocks, the blocked gzip that
// sequencers and bgzip write) decoded side by side, one thread each, so the state per stream must
// be small.  Huffman codes are kept in canonical form — count of codes per length + symbols in code
// order, 640 bytes for the literal/length alphabet — and decoded through a 7-bit look-ahead table
// (covers every code of up to 7 bits: the bases and quality characters of a FASTQ) with the
// bit-serial canonical walk behind it for longer codes.  The tables live wherever the `Tables`
// policy puts them: plain arrays on the host, bank-interleaved shared memory on the device.
#pragma once

#include <stddef.h>
#include <stdint.h>

#ifdef __CUDACC__
#define SGC_HD __host__ __device__ __forceinline__
#define SGC_HD_COLD __host__ __device__ __noinline__  // block headers: kept out of the symbol loop's code
#else
#define SGC_HD inline
#define SGC_HD_COLD inline
#endif

namespace sgc {
namespace inflate {

enum Status : int {
  kOk = 0,
  kBadHeader = 1,      // not a gzip member (magic, method, reserved flags)
  kTruncated = 2,      // input ended inside the member
  kBadBlock = 3,       // reserved block type, stored-length check, bad code lengths
  kBadCode = 4,        // a bit pattern that is no code, or an invalid length / distance symbol
  kBadDistance = 5,    // a match reaching before the start of the member's output
  kOutputFull = 6,     // more output than the caller's capacity
  kNoEnd = 7,          // a piece of a member: no block end where the next piece starts (see inflate_piece)
};

constexpr int kMaxBits = 15;
// Width of the look-ahead tables (literal/length, distance); overridable for A/B builds.  Measured on the
// device (profiles/r2_inflate_tables_ab.txt): the tables share the SM with the L1 the decoders read their
// input, their matches and their symbol lists through, and 7 + 5 bits (24.5 KB per 64 threads) beat 8 + 6
// (45 KB) by a third and 9 + 6 by a factor of two.
#ifndef SGC_INFLATE_FAST_BITS
#define SGC_INFLATE_FAST_BITS 7
#endif
#ifndef SGC_INFLATE_DIST_FAST_BITS
#define SGC_INFLATE_DIST_FAST_BITS 5
#endif
constexpr int kLitLenSyms = 288, kDistSyms = 32, kFastBits = SGC_INFLATE_FAST_BITS, kDistFastBits = SGC_INFLATE_DIST_FAST_BITS;

// A `Tables` type is a HANDLE, passed by value: a pointer or two to wherever the tables live.
// (The decoder's state must stay in registers; an object whose address is handed to the
// out-of-line header parser would be pinned to memory for the whole loop.)
// Plain-array tables (host, and the reference point for the device layout).
struct PlainTableStorage {
  uint16_t lcount[kMaxBits + 1], lsym[kLitLenSyms];
  uint16_t dcount[kMaxBits + 1], dsym[kDistSyms];
  uint16_t lfast[1 << kFastBits];  // (symbol << 4) | code length, 0 = longer than kFastBits
  uint16_t dfast[1 << kDistFastBits];
};
struct PlainTables {
  PlainTableStorage* s;
  SGC_HD uint16_t get_lcount(int i) const { return s->lcount[i]; }
  SGC_HD void set_lcount(int i, uint16_t v) const { s->lcount[i] = v; }
  SGC_HD uint16_t get_lsym(int i) const { return s->lsym[i]; }
  SGC_HD void set_lsym(int i, uint16_t v) const { s->lsym[i] = v; }
  SGC_HD uint16_t get_dcount(int i) const { return s->dcount[i]; }
  SGC_HD void set_dcount(int i, uint16_t v) const { s->dcount[i] = v; }
  SGC_HD uint16_t get_dsym(int i) const { return s->dsym[i]; }
  SGC_HD void set_dsym(int i, uint16_t v) const { s->dsym[i] = v; }
  SGC_HD uint16_t get_lfast(int i) const { return s->lfast[i]; }
  SGC_HD void set_lfast(int i, uint16_t v) const { s->lfast[i] = v; }
  SGC_HD uint16_t get_dfast(int i) const { return s->dfast[i]; }
  SGC_HD void set_dfast(int i, uint16_t v) const { s->dfast[i] = v; }
};

// LSB-first bit reader over a byte range, refilled 32 bits at a time from a register queue that
// is itself filled with ALIGNED 16-byte loads one block ahead: the load of block i + 1 is issued
// when the decoder starts on block i, four refills before its first word is needed, so the
// latency of the input stream never sits on the decode chain.  Up to 15 bytes before `in` and
// 47 bytes after in + len may be touched; bits past the range read as zero, and `overrun` says
// that the decoder asked for bits beyond it.
struct Block16 {
  uint32_t w[4];
};
SGC_HD Block16 load_block16(const uint8_t* p) {
  Block16 b;
#ifdef __CUDA_ARCH__
  const uint4 v = *reinterpret_cast<const uint4*>(p);
  b.w[0] = v.x;
  b.w[1] = v.y;
  b.w[2] = v.z;
  b.w[3] = v.w;
#else
  __builtin_memcpy(b.w, p, 16);
#endif
  return b;
}

struct BitReader {
  const uint8_t* ahead;   // the block after `pre`
  Block16 blk, pre;       // the block being consumed, and the next one (already loaded)
  uint32_t wi;            // next word of blk
  size_t len;             // bytes of the range
  size_t next;            // byte offset (from `in`) of the next word; may be negative mod 2^64 at first
  uint64_t buf;
  int cnt;
  bool overrun;
  SGC_HD void init(const uint8_t* in, size_t n, size_t at) {
    const uintptr_t a = (uintptr_t)(in + at);
    const uint8_t* b0 = reinterpret_cast<const uint8_t*>(a & ~(uintptr_t)15);
    const uint32_t lead = (uint32_t)(a & 3u);
    len = n;
    wi = (uint32_t)(a & 15u) >> 2;
    next = at - lead;  // offset of the word that holds the position (wraps when it starts before `in`)
    blk = load_block16(b0);
    pre = load_block16(b0 + 16);
    ahead = b0 + 32;
    overrun = false;
    // first word: drop the bytes in front of the position
    const uint32_t w = load_word();
    buf = (uint64_t)(w >> (8 * lead));
    cnt = 32 - 8 * (int)lead;
  }
  SGC_HD uint32_t load_word() {
    uint32_t w = wi == 0 ? blk.w[0] : (wi == 1 ? blk.w[1] : (wi == 2 ? blk.w[2] : blk.w[3]));
    // bytes of this word that lie inside [0, len) keep their value, the others read as zero
    const size_t off = next;  // may be "negative" for the very first word only
    if ((ptrdiff_t)off < (ptrdiff_t)len) {
      const ptrdiff_t over = (ptrdiff_t)off + 4 - (ptrdiff_t)len;  // bytes of the word past the range
      if (over > 0) w &= over >= 4 ? 0u : (0xFFFFFFFFu >> (8 * (int)over));
    } else {
      w = 0;
      if ((ptrdiff_t)off >= (ptrdiff_t)len + 8) overrun = true;  // more than the slack a decoder may look ahead
    }
    next += 4;
    if (++wi == 4) {
      wi = 0;
      blk = pre;
      // never a load that reaches 48 bytes or more past the range (the caller guarantees 47)
      if ((ptrdiff_t)(next + 16) < (ptrdiff_t)len + 32) pre = load_block16(ahead);
      ahead += 16;
    }
    return w;
  }
  SGC_HD void refill() {  // more than 32 valid bits afterwards
    if (cnt <= 32) {
      buf |= (uint64_t)load_word() << cnt;
      cnt += 32;
    }
  }
  SGC_HD uint32_t peek(int n) const { return (uint32_t)(buf & ((1ull << n) - 1)); }
  SGC_HD void drop(int n) {
    buf >>= n;
    cnt -= n;
  }
  SGC_HD uint32_t take(int n) {  // n <= 32, after a refill
    const uint32_t v = peek(n);
    drop(n);
    return v;
  }
  // bytes of input consumed so far, counting whole bytes still in the buffer as unread
  SGC_HD size_t consumed() const { return next - (size_t)(cnt >> 3); }
  SGC_HD void align_to_byte() { drop(cnt & 7); }
  // the same reader started at bit `bit` of the range, and the bit it has reached
  SGC_HD void init_bit(const uint8_t* in, size_t n, uint64_t bit) {
    init(in, n, (size_t)(bit >> 3));
    drop((int)(bit & 7));  // (init leaves at least 8 bits in the buffer)
  }
  SGC_HD uint64_t bit_pos() const { return (uint64_t)next * 8 - (uint64_t)cnt; }
};

// Output of one member, written in ALIGNED 64-bit words: the bytes of the word in progress collect
// in a register and go out with one store when it is full.  (Byte stores made the first version
// of the device decoder a stream of one-byte memory transactions: 5 G L2 sector accesses and
// 6.7 GB of DRAM fill reads for 2.8 GB of text.)  The member's first and last word are shared with
// its neighbours in the text, which other threads write: their bytes go out one by one.
// Reads of earlier output (matches) see the unflushed bytes through the same object.  The words
// holding out[0] and out[cap - 1] must be readable.
SGC_HD uint64_t load_u64(const void* p) {
#ifdef __CUDA_ARCH__
  return *static_cast<const uint64_t*>(p);
#else
  uint64_t v;
  __builtin_memcpy(&v, p, 8);
  return v;
#endif
}
SGC_HD void store_u64(void* p, uint64_t v) {
#ifdef __CUDA_ARCH__
  *static_cast<uint64_t*>(p) = v;
#else
  __builtin_memcpy(p, &v, 8);
#endif
}

struct OutWriter {
  uint8_t* base;
  size_t cap, op;
  uint64_t acc;      // bytes [first, k) of the current aligned word, byte i at bits 8i
  uint32_t k;        // position of the next byte in that word
  uint32_t first;    // 0, or where the member starts inside its first word
  SGC_HD void init(uint8_t* out, size_t n) {
    base = out;
    cap = n;
    op = 0;
    acc = 0;
    k = first = (uint32_t)((uintptr_t)out & 7u);
  }
  SGC_HD uint8_t* word_ptr() const { return reinterpret_cast<uint8_t*>(((uintptr_t)base + op - k)); }  // aligned
  SGC_HD void flush_word() {  // k == 8
    uint8_t* w = reinterpret_cast<uint8_t*>((uintptr_t)base + op - 8);
    if (first == 0) {
      store_u64(w, acc);
    } else {
      for (uint32_t i = first; i < 8; ++i) w[i] = (uint8_t)(acc >> (8 * i));
      first = 0;
    }
    acc = 0;
    k = 0;
  }
  SGC_HD void put(uint8_t b) {
    acc |= (uint64_t)b << (8 * k);
    ++k;
    ++op;
    if (k == 8) flush_word();
  }
  // n <= 8 bytes at once (the low n bytes of v, low byte first)
  SGC_HD void put_n(uint64_t v, uint32_t n) {
    if (n < 8) v &= (1ull << (8 * n)) - 1;
    if (first != 0) {  // still in the member's first word, shared with its neighbour
      for (uint32_t i = 0; i < n; ++i) put((uint8_t)(v >> (8 * i)));
      return;
    }
    uint8_t* w = word_ptr();
    acc |= v << (8 * k);  // k < 8
    const uint32_t nk = k + n;
    if (nk >= 8) {
      store_u64(w, acc);
      acc = k ? v >> (8 * (8 - k)) : 0;
      k = nk - 8;
    } else {
      k = nk;
    }
    op += n;
  }
  SGC_HD void finish() {  // the last, partial word
    uint8_t* w = word_ptr();
    for (uint32_t i = first; i < k; ++i) w[i] = (uint8_t)(acc >> (8 * i));
    first = k;  // nothing left to write
  }
  // Eight bytes of the output starting at byte j <= op - 1, flushed or not: memory where the
  // words have gone out, the register for the word in progress.  Bytes at or beyond `op` are
  // unspecified (a caller copying a short period masks them off).
  SGC_HD uint64_t get8(size_t j) const {
    const uintptr_t a = (uintptr_t)base + j, cur = (uintptr_t)base + op - k;  // cur: the word in progress
    if (a >= cur) return acc >> (8 * (uint32_t)(a - cur));
    const uint8_t* w = reinterpret_cast<const uint8_t*>(a & ~(uintptr_t)7);
    const uint32_t sh = 8 * (uint32_t)(a & 7);
    uint64_t v = load_u64(w) >> sh;
    if (sh && (uintptr_t)w + 8 < cur) v |= load_u64(w + 8) << (64 - sh);
    const uintptr_t d = cur - a;  // bytes of the result that come from memory: the rest from the register
    if (d < 8) v = (v & ((1ull << (8 * d)) - 1)) | (acc << (8 * d));
    return v;
  }
};

// Canonical code of one alphabet from its code lengths: counts per length and symbols in code
// order.  Returns false for an over-subscribed set, or an incomplete one that is not the single
// code RFC 1951 allows for a one-symbol distance alphabet.
template <typename SetCount, typename SetSym>
SGC_HD bool build_canonical(const uint8_t* lengths, int n, SetCount set_count, SetSym set_sym, uint16_t* count_out,
                            bool must_be_complete = false) {
  uint16_t count[kMaxBits + 1];
  for (int i = 0; i <= kMaxBits; ++i) count[i] = 0;
  for (int i = 0; i < n; ++i) ++count[lengths[i]];
  int left = 1;  // codes still available at the current length
  for (int l = 1; l <= kMaxBits; ++l) {
    left <<= 1;
    left -= count[l];
    if (left < 0) return false;  // over-subscribed
  }
  uint16_t offs[kMaxBits + 1];
  offs[1] = 0;
  for (int l = 1; l < kMaxBits; ++l) offs[l + 1] = (uint16_t)(offs[l] + count[l]);
  for (int i = 0; i < n; ++i)
    if (lengths[i]) set_sym(offs[lengths[i]]++, (uint16_t)i);
  for (int l = 0; l <= kMaxBits; ++l) {
    set_count(l, count[l]);
    count_out[l] = count[l];
  }
  // incomplete: legal only for a literal/length or distance alphabet whose codes all have length 1
  // (a lone distance code — or none: a block of literals only), as zlib decides it
  if (left == 0) return true;
  if (must_be_complete) return false;
  for (int l = 2; l <= kMaxBits; ++l)
    if (count[l]) return false;
  return true;
}

// Bit-serial canonical decode: the code is read most significant bit first; at each length the
// codes are consecutive, so "code - first < count" decides membership (RFC 1951 3.2.2).
template <typename GetCount, typename GetSym>
SGC_HD int decode_slow(BitReader& br, GetCount get_count, GetSym get_sym) {
  int code = 0, first = 0, index = 0;
  uint64_t bits = br.buf;
  for (int l = 1; l <= kMaxBits; ++l) {
    code |= (int)(bits & 1);
    bits >>= 1;
    const int cnt = get_count(l);
    if (code - first < cnt) {
      br.drop(l);
      return get_sym(index + (code - first));
    }
    index += cnt;
    first = (first + cnt) << 1;
    code <<= 1;
  }
  return -1;
}

// RFC 1951 3.2.5 as arithmetic (no tables to place in device memory): base value and number of
// extra bits of length symbol c (257 + c) and of distance symbol d.
SGC_HD uint32_t len_extra_bits(int c) { return c < 8 || c == 28 ? 0u : (uint32_t)(c >> 2) - 1u; }
SGC_HD uint32_t len_base(int c) { return c < 8 ? (uint32_t)c + 3u : (c == 28 ? 258u : ((4u | ((uint32_t)c & 3u)) << len_extra_bits(c)) + 3u); }
SGC_HD uint32_t dist_extra_bits(int d) { return d < 4 ? 0u : (uint32_t)(d >> 1) - 1u; }
SGC_HD uint32_t dist_base(int d) { return d < 4 ? (uint32_t)d + 1u : ((2u | ((uint32_t)d & 1u)) << dist_extra_bits(d)) + 1u; }
// order in which the code-length code's own lengths are sent (RFC 1951 3.2.7)
SGC_HD int cl_order(int i) { return "\x10\x11\x12\x00\x08\x07\x09\x06\x0a\x05\x0b\x04\x0c\x03\x0d\x02\x0e\x01\x0f"[i]; }

template <typename GetSym, typename SetFast>
SGC_HD void fill_lookahead(const uint16_t* count, int bits, GetSym get_sym, SetFast set_fast) {
  for (int i = 0; i < (1 << bits); ++i) set_fast(i, 0);
  int code = 0, index = 0;
  for (int l = 1; l <= bits; ++l) {
    for (int j = 0; j < count[l]; ++j, ++code, ++index) {
      // the code's bits arrive most significant first: reverse them into stream order
      uint32_t r = 0;
      for (int b = 0; b < l; ++b) r |= ((uint32_t)(code >> b) & 1u) << (l - 1 - b);
      const uint16_t entry = (uint16_t)((get_sym(index) << 4) | l);
      for (uint32_t i = r; i < (1u << bits); i += 1u << l) set_fast((int)i, entry);
    }
    code <<= 1;
  }
}

// Tables of one block from the two length arrays; also fills the look-ahead tables.
template <typename Tables>
SGC_HD bool install_codes(Tables t, const uint8_t* ll, int nl, const uint8_t* dl, int nd) {
  uint16_t lc[kMaxBits + 1], dc[kMaxBits + 1];
  if (!build_canonical(ll, nl, [&](int i, uint16_t v) { t.set_lcount(i, v); }, [&](int i, uint16_t v) { t.set_lsym(i, v); }, lc))
    return false;
  if (!build_canonical(dl, nd, [&](int i, uint16_t v) { t.set_dcount(i, v); }, [&](int i, uint16_t v) { t.set_dsym(i, v); }, dc))
    return false;
  if (lc[0] == nl) return false;  // no literal/length code at all: not even end-of-block
  // look-ahead tables: walk the codes of up to `bits` bits in canonical order
  fill_lookahead(lc, kFastBits, [&](int i) { return t.get_lsym(i); }, [&](int i, uint16_t v) { t.set_lfast(i, v); });
  fill_lookahead(dc, kDistFastBits, [&](int i) { return t.get_dsym(i); }, [&](int i, uint16_t v) { t.set_dfast(i, v); });
  return true;
}

// The code tables of a fixed (type 1) or dynamic (type 2) block, read from the block header.
// (`br` is the caller's COPY of its reader: see gunzip_member.)
template <typename Tables>
SGC_HD_COLD int read_codes(BitReader& br, Tables t, uint32_t type) {
  uint8_t lengths[kLitLenSyms + kDistSyms];
  int nl, nd;
  if (type == 1) {  // fixed code
    nl = 288;
    nd = 32;  // 30 and 31 complete the 5-bit code and are errors if they occur
    for (int i = 0; i < 144; ++i) lengths[i] = 8;
    for (int i = 144; i < 256; ++i) lengths[i] = 9;
    for (int i = 256; i < 280; ++i) lengths[i] = 7;
    for (int i = 280; i < 288; ++i) lengths[i] = 8;
    for (int i = 0; i < 32; ++i) lengths[288 + i] = 5;
  } else {  // dynamic code: the code-length code first
    br.refill();
    nl = (int)br.take(5) + 257;
    nd = (int)br.take(5) + 1;
    const int nc = (int)br.take(4) + 4;
    if (nl > 286 || nd > 30) return br.overrun ? kTruncated : kBadBlock;
    uint8_t cl[19];
    for (int i = 0; i < 19; ++i) cl[i] = 0;
    for (int i = 0; i < nc; ++i) {
      br.refill();
      cl[cl_order(i)] = (uint8_t)br.take(3);
    }
    // the code-length alphabet is tiny: its canonical form lives in registers / local arrays
    uint16_t ccount[kMaxBits + 1], csym[19], dummy[kMaxBits + 1];
    if (!build_canonical(cl, 19, [&](int i, uint16_t v) { ccount[i] = v; }, [&](int i, uint16_t v) { csym[i] = v; }, dummy, true))
      return kBadBlock;
    int i = 0;
    while (i < nl + nd) {
      br.refill();
      const int s = decode_slow(br, [&](int l) { return (int)ccount[l]; }, [&](int k) { return (int)csym[k]; });
      if (s < 0) return br.overrun ? kTruncated : kBadCode;
      if (s < 16) {
        lengths[i++] = (uint8_t)s;
      } else {
        uint8_t prev = 0;
        int rep;
        if (s == 16) {
          if (i == 0) return kBadBlock;
          prev = lengths[i - 1];
          rep = 3 + (int)br.take(2);
        } else if (s == 17) {
          rep = 3 + (int)br.take(3);
        } else {
          rep = 11 + (int)br.take(7);
        }
        if (i + rep > nl + nd) return kBadBlock;
        while (rep--) lengths[i++] = prev;
      }
    }
    if (lengths[256] == 0) return kBadBlock;  // no end-of-block code
    // the tables below want the distance lengths at a fixed place
    if (nl != 288)
      for (int j = nd - 1; j >= 0; --j) lengths[288 + j] = lengths[nl + j];
  }
  return install_codes(t, lengths, nl, lengths + 288, nd) ? kOk : kBadBlock;
}

// One gzip member at in[0 .. in_len).  On kOk: *consumed = bytes of the member including its
// 8-byte trailer, *produced = bytes written to out, *crc32 / *isize = the trailer's fields.
//
// Written as ONE loop over a small state machine — block header, one symbol, eight bytes of a
// pending match, eight bytes of a stored block — instead of nested loops: the threads of a warp
// decode different members, and with a single loop head they reconverge every iteration, each
// doing one step of whatever state it is in, instead of drifting apart for good.  A long match
// (a quality line is one 75-byte match) is copied in steps, so no lane waits for another's copy.
template <typename Tables>
SGC_HD int gunzip_member(const uint8_t* in, size_t in_len, uint8_t* out, size_t out_cap, Tables t, size_t* consumed,
                         size_t* produced, uint32_t* crc32, uint32_t* isize) {
  // ---- RFC 1952 header
  if (in_len < 18) return in_len < 4 || (in[0] == 0x1f && in[1] == 0x8b) ? kTruncated : kBadHeader;
  if (in[0] != 0x1f || in[1] != 0x8b || in[2] != 8 || (in[3] & 0xE0)) return kBadHeader;
  const uint8_t flg = in[3];
  size_t pos = 10;
  if (flg & 4) {  // FEXTRA (BGZF keeps its block size here)
    if (pos + 2 > in_len) return kTruncated;
    pos += 2 + ((size_t)in[pos] | ((size_t)in[pos + 1] << 8));
  }
  for (int field = 0; field < 2; ++field)  // FNAME, FCOMMENT: zero-terminated
    if (flg & (field ? 16 : 8)) {
      while (pos < in_len && in[pos]) ++pos;
      ++pos;
    }
  if (flg & 2) pos += 2;  // FHCRC
  if (pos >= in_len) return kTruncated;

  // ---- RFC 1951 blocks
  enum { kHeader, kSymbol, kCopy, kStored, kDone };
  BitReader br;
  br.init(in, in_len, pos);
  OutWriter ow;
  ow.init(out, out_cap);
  int state = kHeader, rc = kOk;
  uint32_t last = 0;
  uint32_t run = 0;      // bytes of the pending match / stored block still to copy
  uint32_t dist = 0;     // distance of the pending match
  uint64_t pattern = 0;  // dist < 8: the next eight bytes of the repetition, lowest byte first
  uint32_t phase = 0;    //           and 8 mod dist
  size_t stored_at = 0;  // input position of the stored bytes
  while (state != kDone) {
    if (state == kSymbol) {
      br.refill();
      int sym;
      const uint16_t e = t.get_lfast((int)br.peek(kFastBits));
      if (e) {
        br.drop(e & 15);
        sym = e >> 4;
      } else {
        sym = decode_slow(br, [&](int l) { return (int)t.get_lcount(l); }, [&](int k) { return (int)t.get_lsym(k); });
      }
      if (sym < 0 || sym > 285) {
        rc = br.overrun ? kTruncated : kBadCode;
        state = kDone;
      } else if (sym < 256) {
        if (ow.op >= out_cap) {
          rc = kOutputFull;
          state = kDone;
        } else {
          ow.put((uint8_t)sym);
          // literals come in runs (a sequence line): if the next code is a short literal too, take
          // it in the same step (at least 17 bits are left after the first code)
          const uint16_t e2 = t.get_lfast((int)br.peek(kFastBits));
          if (e2 && (e2 >> 4) < 256 && ow.op < out_cap) {
            br.drop(e2 & 15);
            ow.put((uint8_t)(e2 >> 4));
          }
        }
      } else if (sym == 256) {
        if (br.overrun) {
          rc = kTruncated;
          state = kDone;
        } else {
          state = last ? kDone : kHeader;
        }
      } else {
        sym -= 257;
        run = len_base(sym) + br.take((int)len_extra_bits(sym));
        br.refill();
        int ds;
        const uint16_t de = t.get_dfast((int)br.peek(kDistFastBits));
        if (de) {
          br.drop(de & 15);
          ds = de >> 4;
        } else {
          ds = decode_slow(br, [&](int l) { return (int)t.get_dcount(l); }, [&](int k) { return (int)t.get_dsym(k); });
        }
        if (ds < 0 || ds >= 30) {
          rc = br.overrun ? kTruncated : kBadCode;
          state = kDone;
        } else {
          dist = dist_base(ds) + br.take((int)dist_extra_bits(ds));
          if (dist > ow.op) {
            rc = kBadDistance;
            state = kDone;
          } else if (ow.op + run > out_cap) {
            rc = kOutputFull;
            state = kDone;
          } else {
            if (dist < 8) {  // a short period: keep eight bytes of the repetition in a register
              pattern = ow.get8(ow.op - dist) & ((1ull << (8 * dist)) - 1);
              for (uint32_t sh = 8 * dist; sh < 64; sh *= 2) pattern |= pattern << sh;
              phase = 8 % dist;  // how far eight bytes advance the period
            }
            state = kCopy;
          }
        }
      }
    } else if (state == kCopy) {
      const uint32_t n = run < 8 ? run : 8;
      if (dist >= 8) {
        ow.put_n(ow.get8(ow.op - dist), n);  // the source ends before this step's first byte
      } else {
        // a short period: `pattern` holds the next eight bytes of the repetition; eight bytes on,
        // the repetition is 8 mod dist bytes further into its period
        ow.put_n(pattern, n);
        if (phase) pattern = (pattern >> (8 * phase)) | (pattern << (8 * (dist - phase)));
      }
      run -= n;
      if (run == 0) state = kSymbol;
    } else if (state == kStored) {
      const uint32_t n = run < 8 ? run : 8;
      for (uint32_t i = 0; i < 8; ++i)
        if (i < n) ow.put(in[stored_at + i]);
      stored_at += n;
      run -= n;
      if (run == 0) {
        br.init(in, in_len, stored_at);
        state = last ? kDone : kHeader;
      }
    } else {  // kHeader
      br.refill();
      last = br.take(1);
      const uint32_t type = br.take(2);
      if (type == 0) {  // stored
        br.align_to_byte();
        br.refill();
        const uint32_t n = br.take(16);
        br.refill();
        const uint32_t nn = br.take(16);
        stored_at = br.consumed();  // the buffer holds whole bytes only
        if ((n ^ nn) != 0xFFFFu) {
          rc = br.overrun ? kTruncated : kBadBlock;
          state = kDone;
        } else if (stored_at + n > in_len) {
          rc = kTruncated;
          state = kDone;
        } else if (ow.op + n > out_cap) {
          rc = kOutputFull;
          state = kDone;
        } else if (n == 0) {
          br.init(in, in_len, stored_at);
          state = last ? kDone : kHeader;
        } else {
          run = n;
          state = kStored;
        }
      } else if (type == 3) {
        rc = br.overrun ? kTruncated : kBadBlock;
        state = kDone;
      } else {
        // through a copy: only the copy's address leaves this function, `br` itself stays in registers
        BitReader header_reader = br;
        rc = read_codes(header_reader, t, type);
        br = header_reader;
        state = rc == kOk ? kSymbol : kDone;
      }
    }
  }
  ow.finish();
  if (rc != kOk) return rc;
  // ---- trailer
  br.align_to_byte();
  const size_t at = br.consumed();
  if (at + 8 > in_len) return kTruncated;
  *crc32 = (uint32_t)in[at] | ((uint32_t)in[at + 1] << 8) | ((uint32_t)in[at + 2] << 16) | ((uint32_t)in[at + 3] << 24);
  *isize = (uint32_t)in[at + 4] | ((uint32_t)in[at + 5] << 8) | ((uint32_t)in[at + 6] << 16) | ((uint32_t)in[at + 7] << 24);
  *consumed = at + 8;
  *produced = ow.op;
  return kOk;
}

// ---- gzip members in pieces --------------------------------------------------------------------
// A gzip file, one member (what gzip and pigz write) or several concatenated (`cat a.gz b.gz`,
// appending writers, BGZF), is one text; it is decoded in parallel by speculation (gzip.cu member_*
// kernels; host/member_core_test.cpp runs the same steps serially):
//   1. near every C-th byte, the first bit where a dynamic-Huffman block header parses and a short
//      trial decode behind it succeeds (probe_block_start) is a candidate piece start; so is the bit
//      after every gzip header that is listed (member_start_at), flagged as a member start (its first
//      block may be of any kind, so it is not probed);
//   2. every piece is decoded without output up to the first block end at or beyond the next
//      candidate (piece_boundary); ending exactly on one links the two, overshooting absorbs it.  A
//      piece that starts a member may copy from nothing in front of it;
//   3. the links followed from the first member's first block give the true block boundaries; from a
//      member's last block the chain steps over its trailer and the next header to exactly the
//      candidate that follows them (members_chain).  A false signature costs one piece that fails or
//      is never linked;
//   4. each piece on that chain is decoded into 16-bit symbols: 0-255 bytes, 256 + i byte i of the
//      32 KiB window in front of the piece, still unknown (MarkSink);
//   5. the text is cut into waves, and each wave's windows are relayed piece after piece ("waves: the
//      window relay" below), then everything else is resolved in parallel.
// A single member is the case where no gzip header inside the file is listed: the first trailer must
// then end the file, and a file of several members is declined.
// These functions are written for that use, separately from gunzip_member, whose symbol loop is the
// BGZF decoder's hot path and stays as it is.
constexpr uint32_t kWindow = 32768;
constexpr uint32_t kPieceFinal = 0xFFFFFFFFu;  // `next` of a piece that ends with the member's last block
constexpr int kProbeTrial = 64;                // symbols a candidate block start must decode
constexpr uint32_t kMaxAbsorb = 8;             // candidates a piece may run past before it gives up

// The RFC 1952 header (FEXTRA, FNAME, FCOMMENT, FHCRC): kOk and *pos = where the DEFLATE stream starts.
SGC_HD int gzip_header(const uint8_t* in, size_t in_len, size_t* pos_out) {
  if (in_len < 18) return in_len < 4 || (in[0] == 0x1f && in[1] == 0x8b) ? kTruncated : kBadHeader;
  if (in[0] != 0x1f || in[1] != 0x8b || in[2] != 8 || (in[3] & 0xE0)) return kBadHeader;
  const uint8_t flg = in[3];
  size_t pos = 10;
  if (flg & 4) {
    if (pos + 2 > in_len) return kTruncated;
    pos += 2 + ((size_t)in[pos] | ((size_t)in[pos + 1] << 8));
  }
  for (int field = 0; field < 2; ++field)
    if (flg & (field ? 16 : 8)) {
      while (pos < in_len && in[pos]) ++pos;
      ++pos;
    }
  if (flg & 2) pos += 2;
  if (pos >= in_len) return kTruncated;
  *pos_out = pos;
  return kOk;
}

// one literal/length or distance symbol (-1: no code)
template <typename Tables>
SGC_HD int decode_litlen(BitReader& br, Tables t) {
  br.refill();
  const uint16_t e = t.get_lfast((int)br.peek(kFastBits));
  if (e) {
    br.drop(e & 15);
    return e >> 4;
  }
  return decode_slow(br, [&](int l) { return (int)t.get_lcount(l); }, [&](int k) { return (int)t.get_lsym(k); });
}
template <typename Tables>
SGC_HD int decode_dist(BitReader& br, Tables t) {
  br.refill();
  const uint16_t e = t.get_dfast((int)br.peek(kDistFastBits));
  if (e) {
    br.drop(e & 15);
    return e >> 4;
  }
  return decode_slow(br, [&](int l) { return (int)t.get_dcount(l); }, [&](int k) { return (int)t.get_dsym(k); });
}

// Where a piece's output goes.  `reach`: how far before the piece's first byte a match may copy
// from (0 for the member's first piece; a match reaching further is kBadDistance).
struct CountSink {  // nothing: only the length
  uint64_t op, reach;
  SGC_HD int literal(uint32_t) {
    ++op;
    return kOk;
  }
  SGC_HD int match(uint32_t len, uint32_t dist) {
    if (dist > op + reach) return kBadDistance;
    op += len;
    return kOk;
  }
  SGC_HD int stored(const uint8_t*, uint32_t n) {
    op += n;
    return kOk;
  }
};
struct MarkSink {  // 16-bit symbols: a byte, or 256 + i for byte i of the window in front of the piece
  uint16_t* out;
  uint64_t op, cap, reach;
  SGC_HD int literal(uint32_t b) {
    if (op >= cap) return kOutputFull;
    out[op++] = (uint16_t)b;
    return kOk;
  }
  SGC_HD int match(uint32_t len, uint32_t dist) {
    if (dist > op + reach) return kBadDistance;
    if (op + len > cap) return kOutputFull;
    for (uint32_t i = 0; i < len; ++i, ++op) {
      // a source before the piece is a window marker; a source that is a marker copies the marker
      const int64_t s = (int64_t)op - (int64_t)dist;
      out[op] = s >= 0 ? out[s] : (uint16_t)(256 + (int64_t)kWindow + s);
    }
    return kOk;
  }
  SGC_HD int stored(const uint8_t* p, uint32_t n) {
    if (op + n > cap) return kOutputFull;
    for (uint32_t i = 0; i < n; ++i) out[op++] = p[i];
    return kOk;
  }
};

// Decodes blocks of the DEFLATE stream in[0 .. in_len) from bit `start` (a block header) until the
// end of the member's last block or a block end `stop(end_bit)` accepts; *end_bit, *final_block say
// which.  A reader position beyond `limit_bit` is kNoEnd.  Reads stay inside the BitReader's range
// and slack (garbage input included); the sink is the only thing written.
template <typename Tables, typename Sink, typename Stop>
SGC_HD int inflate_piece(const uint8_t* in, size_t in_len, uint64_t start, uint64_t limit_bit, Tables t, Sink& out, Stop stop,
                         uint64_t* end_bit, bool* final_block) {
  if (start >= (uint64_t)in_len * 8) return kTruncated;
  BitReader br;
  br.init_bit(in, in_len, start);
  for (;;) {
    br.refill();
    const uint32_t last = br.take(1);
    const uint32_t type = br.take(2);
    if (type == 0) {
      br.align_to_byte();
      br.refill();
      const uint32_t n = br.take(16);
      br.refill();
      const uint32_t nn = br.take(16);
      const size_t at = br.consumed();
      if ((n ^ nn) != 0xFFFFu) return br.overrun ? kTruncated : kBadBlock;
      if (at + n > in_len) return kTruncated;
      if ((uint64_t)(at + n) * 8 > limit_bit) return kNoEnd;
      if (int rc = out.stored(in + at, n)) return rc;
      br.init(in, in_len, at + n);
    } else if (type == 3) {
      return br.overrun ? kTruncated : kBadBlock;
    } else {
      BitReader header_reader = br;  // (a copy, as in gunzip_member: `br` stays in registers)
      const int rc = read_codes(header_reader, t, type);
      br = header_reader;
      if (rc != kOk) return rc;
      for (;;) {
        if (br.bit_pos() > limit_bit) return kNoEnd;
        int sym = decode_litlen(br, t);
        if (sym < 0 || sym > 285) return br.overrun ? kTruncated : kBadCode;
        if (sym == 256) break;
        if (sym < 256) {
          if (int rc = out.literal((uint32_t)sym)) return rc;
          continue;
        }
        sym -= 257;
        const uint32_t len = len_base(sym) + br.take((int)len_extra_bits(sym));
        const int ds = decode_dist(br, t);
        if (ds < 0 || ds >= 30) return br.overrun ? kTruncated : kBadCode;
        const uint32_t dist = dist_base(ds) + br.take((int)dist_extra_bits(ds));
        if (int rc = out.match(len, dist)) return rc;
      }
    }
    if (br.overrun) return kTruncated;
    const uint64_t e = br.bit_pos();
    if (e > limit_bit) return kNoEnd;
    if (last || stop(e)) {
      *end_bit = e;
      *final_block = last != 0;
      return kOk;
    }
  }
}

// Does a dynamic-Huffman block that is not the member's last start at bit `bit`?  Its header must
// parse (read_codes: HLIT, HDIST <= 29, a complete code-length code, lengths that form valid codes
// with an end-of-block code) and `trial` symbols after it, or up to its end, must decode.
template <typename Tables>
SGC_HD bool probe_block_start(const uint8_t* in, size_t in_len, uint64_t bit, Tables t, int trial) {
  BitReader br;
  br.init_bit(in, in_len, bit);
  br.refill();
  if (br.peek(3) != 4u) return false;  // BFINAL = 0, BTYPE = 10
  if ((br.peek(8) >> 3) > 29u || (br.peek(13) >> 8) > 29u) return false;
  br.drop(3);
  if (read_codes(br, t, 2) != kOk || br.overrun) return false;
  for (int i = 0; i < trial; ++i) {
    int sym = decode_litlen(br, t);
    if (sym < 0 || sym > 285) return false;
    if (sym == 256) break;
    if (sym > 256) {
      br.take((int)len_extra_bits(sym - 257));
      const int ds = decode_dist(br, t);
      if (ds < 0 || ds >= 30) return false;
      br.take((int)dist_extra_bits(ds));
    }
  }
  return !br.overrun;
}

// Step 2 for piece j of `n` whose candidate starts (bits, increasing) are starts[0 .. n): decodes it
// without output to the first block end at or beyond starts[j + 1].  kOk: *next = the piece that
// starts exactly there (j + 1, or up to j + 1 + max_absorb when candidates in between were false or
// skipped), or kPieceFinal when the member's last block ended first; *end_bit and *out_len describe
// the piece.  Anything else means the piece does not lie on the chain.
// `reach`: how far before the piece a match may copy from; 0 for a piece that starts a member.
template <typename Tables>
SGC_HD int piece_boundary(const uint8_t* in, size_t in_len, const uint64_t* starts, uint32_t n, uint32_t j,
                          uint32_t max_absorb, Tables t, uint32_t* next, uint64_t* end_bit, uint64_t* out_len, uint64_t reach) {
  CountSink sink{0, reach};
  const uint32_t last_ok = j + 1 + max_absorb < n ? j + 1 + max_absorb : n - 1;
  const uint64_t limit = j + 1 + max_absorb < n ? starts[j + 1 + max_absorb] : (uint64_t)in_len * 8;
  uint32_t m = j + 1;
  auto stop = [&](uint64_t e) {
    while (m < n && starts[m] < e) ++m;
    return m < n && starts[m] == e;
  };
  bool fin = false;
  const int rc = inflate_piece(in, in_len, starts[j], limit, t, sink, stop, end_bit, &fin);
  if (rc != kOk) return rc;
  if (!fin && m > last_ok) return kNoEnd;
  *next = fin ? kPieceFinal : m;
  *out_len = sink.op;
  return kOk;
}

// what step 2 learns about a piece (piece_boundary)
struct PieceMeta {
  uint64_t end_bit, out_len;
  uint32_t next;
  int32_t status;
};

// Does a gzip member header start at byte `pos`?  true and *bit = the first bit of its DEFLATE stream.
SGC_HD bool member_start_at(const uint8_t* in, size_t in_len, size_t pos, uint64_t* bit) {
  if (pos + 4 > in_len || in[pos] != 0x1f || in[pos + 1] != 0x8b || in[pos + 2] != 8 || (in[pos + 3] & 0xE0)) return false;
  size_t h = 0;
  if (gzip_header(in + pos, in_len - pos, &h) != kOk) return false;
  *bit = (uint64_t)(pos + h) * 8;
  return true;
}

SGC_HD uint32_t le32(const uint8_t* p) {
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

// Step 1 (host): the block-start candidates probe[0 .. np) and the member starts member[0 .. nm), each
// sorted, into one sorted starts[] without duplicates; is_member[i] = 1 where a member starts (that
// flag wins over a block-start candidate at the same bit).  Returns the number of starts.
inline uint32_t merge_starts(const uint64_t* probe, uint32_t np, const uint64_t* member, uint32_t nm, uint64_t* starts,
                             uint8_t* is_member) {
  uint32_t i = 0, k = 0, n = 0;
  while (i < np || k < nm) {
    const bool m = k < nm && (i >= np || member[k] <= probe[i]);
    const uint64_t v = m ? member[k++] : probe[i++];
    if (n && starts[n - 1] == v) {
      is_member[n - 1] |= (uint8_t)m;
    } else {
      starts[n] = v;
      is_member[n++] = (uint8_t)m;
    }
  }
  return n;
}

// A member's trailer (RFC 1952): where it starts, the CRC-32 and ISIZE it holds.
struct MemberTrailer {
  uint64_t at;
  uint32_t crc, isize;
};

// Step 3 (host): from piece 0 (the first member's start) along the links of meta[]; where a piece ends
// a member's last block, the member's 8-byte trailer follows at the next byte, and unless it ends the
// input, a gzip header and the member-start candidate right behind it.  Fills chain[], member_of[]
// (the member of each chain piece) and trailers[] (one per member, *n_members of them); returns the
// chain's length, or 0 (decline) when a link is missing, a piece on the way failed, or anything but a
// whole member follows a trailer (zero padding included).
inline uint32_t members_chain(const uint8_t* in, size_t in_len, const uint64_t* starts, const uint8_t* is_member,
                              const PieceMeta* meta, uint32_t n, uint32_t* chain, uint32_t* member_of, MemberTrailer* trailers,
                              uint32_t* n_members, uint64_t* absorbed) {
  uint32_t len = 0, j = 0, m = 0;
  *absorbed = 0;
  *n_members = 0;
  if (n == 0 || !is_member[0]) return 0;
  for (;;) {
    if (j >= n || meta[j].status != kOk) return 0;
    chain[len] = j;
    member_of[len++] = m;
    if (meta[j].next != kPieceFinal) {
      *absorbed += meta[j].next - j - 1;
      j = meta[j].next;
      continue;
    }
    const uint64_t at = (meta[j].end_bit + 7) / 8;
    if (at + 8 > in_len) return 0;
    trailers[m++] = MemberTrailer{at, le32(in + at), le32(in + at + 4)};
    if (at + 8 == in_len) {
      *n_members = m;
      return len;
    }
    uint64_t bit = 0;
    if (!member_start_at(in, in_len, (size_t)(at + 8), &bit)) return 0;
    uint32_t lo = j + 1, hi = n;  // the first start at or beyond `bit`
    while (lo < hi) {
      const uint32_t mid = lo + (hi - lo) / 2;
      if (starts[mid] < bit) lo = mid + 1;
      else hi = mid;
    }
    if (lo >= n || starts[lo] != bit || !is_member[lo]) return 0;
    j = lo;
  }
}

// ---- waves: the window relay --------------------------------------------------------------------
// The chain's text is cut into waves k = 0, 1, ..., which one stream decodes one after another or
// several streams at once (sgc_fastq_stream_submit_gzip_split; one stream is its n = 1 case;
// member_core_test with <waves>).  Wave k's first pieces refer, through their markers, to W_k, the
// 32 KiB of text in front of the wave, which earlier waves make.  So that no wave waits for another
// while it decodes:
//   a. the last 32 KiB (or all) of every piece, piece after piece, are relayed in place
//      (relay_symbol): a marker that names a byte of the wave takes the symbol already relayed
//      there, one that names a byte in front of the wave becomes 256 + j, byte j of W_k;
//   b. F_k, the wave's last 32 KiB as such symbols (wave_front), composes the next window:
//      W_0 is zeros and W_{k+1} = compose_window(F_k, W_k), one wave after another;
//   c. with W_k known every relayed symbol settles (settle_symbol), all pieces side by side.
// A symbol of a piece that did not decode may be anything: the window index is masked so that it
// stays inside the window (that wave is reported as bad).
SGC_HD uint16_t relay_symbol(uint16_t s, uint64_t piece_off, const uint16_t* wave_sym) {
  if (s < 256) return s;
  const int64_t g = (int64_t)piece_off - (int64_t)kWindow + (int64_t)((s - 256) & (kWindow - 1));
  return g >= 0 ? wave_sym[g] : (uint16_t)(256 + (int64_t)kWindow + g);
}
SGC_HD uint8_t settle_symbol(uint16_t s, const uint8_t* window) {
  return s < 256 ? (uint8_t)s : window[(s - 256) & (kWindow - 1)];
}
// F_k of a wave of n_text bytes: the caller put its last min(n_text, kWindow) relayed symbols at the
// end of f[kWindow]; in front of them, when the wave is shorter than the window, the bytes in front
// of the wave: f[j] names byte n_text + j of W_k.
SGC_HD void wave_front(uint16_t* f, uint64_t n_text) {
  for (uint64_t j = 0; j + n_text < kWindow; ++j) f[j] = (uint16_t)(256 + n_text + j);
}
SGC_HD void compose_window(const uint16_t* f, const uint8_t* w_in, uint8_t* w_out) {
  for (uint32_t j = 0; j < kWindow; ++j) w_out[j] = settle_symbol(f[j], w_in);
}

}  // namespace inflate
}  // namespace sgc

// ---- CRC-32 (RFC 1952 8.) of a member's output, computed by 32 cooperating lanes -------------------
// Lane l takes one contiguous piece of the bytes, runs the table-driven CRC over it, and the
// pieces are joined with crc(A || B) = x^(8 |B|) * crc(A) + crc(B) (polynomial arithmetic modulo
// the CRC polynomial; the identity zlib's crc32_combine uses).  All pieces but the first have the
// same length, so every level of the join tree multiplies by one power of x^(8 c).
namespace sgc {
namespace inflate {

constexpr uint32_t kCrcPoly = 0xEDB88320u;  // reflected

// entry i of the byte table
SGC_HD uint32_t crc_table_entry(uint32_t i) {
  uint32_t c = i;
  for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ kCrcPoly : c >> 1;
  return c;
}

// a(x) * b(x) mod p(x), reflected representation (bit 31 = x^0)
SGC_HD uint32_t crc_multmodp(uint32_t a, uint32_t b) {
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1)) == 0) break;
    }
    m >>= 1;
    b = (b & 1) ? (b >> 1) ^ kCrcPoly : b >> 1;
  }
  return p;
}

// x^(8 n) mod p(x)
SGC_HD uint32_t crc_x8n(uint64_t n) {
  uint32_t p = 1u << 31;          // x^0
  uint32_t sq = 1u << (31 - 8);   // x^8
  while (n) {
    if (n & 1) p = crc_multmodp(sq, p);
    sq = crc_multmodp(sq, sq);
    n >>= 1;
  }
  return p;
}

// CRC-32 of A || B from crc(A), crc(B) and |B|
SGC_HD uint32_t crc_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b) { return crc_multmodp(crc_x8n(len_b), crc_a) ^ crc_b; }

// standard CRC-32 of bytes [0, n) given a 256-entry table accessor
template <typename Table>
SGC_HD uint32_t crc_bytes(const uint8_t* p, size_t n, Table table) {
  uint32_t c = 0xFFFFFFFFu;
  for (size_t i = 0; i < n; ++i) c = table((c ^ p[i]) & 0xFFu) ^ (c >> 8);
  return c ^ 0xFFFFFFFFu;
}

// how n bytes are cut into 32 pieces: pieces 1..31 have `c` bytes, piece 0 the rest (possibly none)
SGC_HD size_t crc_piece_len(size_t n) { return n / 32; }

}  // namespace inflate
}  // namespace sgc
