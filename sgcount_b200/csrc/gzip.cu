// gzip.cu — FASTQ straight from BGZF blocks: inflate, record framing and counting on the device.
//
// The reference reads its samples through fxread::initialize_reader (count.rs:24): gzip inflate and
// line splitting on one host thread per sample.  The C++ host spreads that over its cores
// (host/fastx.cpp), which is where it stops: ~0.2 core-seconds per million reads whatever the GPU
// does.  Blocked gzip — BGZF, what bgzip and sequencers write: independent members of at most
// 64 KB, each announcing its size in a 'BC' extra field — needs no host core at all:
//
//   inflate_blocks_kernel   ONE THREAD per block runs the sequential DEFLATE decoder of
//                           inflate_core.h (canonical Huffman, 7- and 5-bit look-ahead tables in
//                           bank-interleaved shared memory, the rest of the code tables in local
//                           memory), writing its text where the prefix sum of the blocks' ISIZE
//                           fields puts it.  Tens of thousands of blocks are in flight, so the
//                           serial bit-by-bit dependency of one stream does not matter.
//   newline_count_kernel    newlines per 4 KB chunk of the contiguous text           } record
//   (exclusive scan)        line number of every chunk's first newline               } framing:
//   span_extract_kernel     every line 4r+1 is the sequence of record r: its guide   } FASTQ is
//                           window span (sgc_span_geometry) goes to span record r    } 4 lines
//   count_stream_kernel     the ordinary count of fixed-stride span records (count.cu).
//
// BGZF cuts blocks anywhere, so a wave of blocks ends inside a record: the bytes after the last
// complete record are carried in front of the next wave's text.  Only fixed-length 4-line FASTQ
// takes this path (the head of the sample, which the host reads for the offset detector, says so);
// anything irregular is reported and the caller counts the sample through the host path instead.
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <condition_variable>
#include <cstddef>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "inflate_core.h"
#include "internal.h"

namespace sgc {
namespace {

constexpr int kInflateThreads = 64;
constexpr uint32_t kHeadroom = 1u << 16;  // room in front of a wave's text for the carried bytes
constexpr uint32_t kChunk = 4096;         // bytes per newline-count chunk
constexpr uint32_t kChunkThreads = 256;   // 16 bytes per thread

// look-ahead tables and per-length code counts in shared memory, one column per thread: element e
// of thread t at [e * T + t]; the symbol lists stay in local memory (one access per long code).
// The handle is two pointers, passed by value (inflate_core.h).
struct DeviceSymbols {
  uint16_t lsym[inflate::kLitLenSyms], dsym[inflate::kDistSyms];
};
struct DeviceTables {
  uint16_t* col;
  DeviceSymbols* syms;
  static constexpr int kCounts = (1 << inflate::kFastBits) + (1 << inflate::kDistFastBits);
  __host__ __device__ __forceinline__ uint16_t get_lcount(int i) const { return col[(kCounts + i) * kInflateThreads]; }
  __host__ __device__ __forceinline__ void set_lcount(int i, uint16_t v) const { col[(kCounts + i) * kInflateThreads] = v; }
  __host__ __device__ __forceinline__ uint16_t get_lsym(int i) const { return syms->lsym[i]; }
  __host__ __device__ __forceinline__ void set_lsym(int i, uint16_t v) const { syms->lsym[i] = v; }
  __host__ __device__ __forceinline__ uint16_t get_dcount(int i) const { return col[(kCounts + 16 + i) * kInflateThreads]; }
  __host__ __device__ __forceinline__ void set_dcount(int i, uint16_t v) const { col[(kCounts + 16 + i) * kInflateThreads] = v; }
  __host__ __device__ __forceinline__ uint16_t get_dsym(int i) const { return syms->dsym[i]; }
  __host__ __device__ __forceinline__ void set_dsym(int i, uint16_t v) const { syms->dsym[i] = v; }
  __host__ __device__ __forceinline__ uint16_t get_lfast(int i) const { return col[i * kInflateThreads]; }
  __host__ __device__ __forceinline__ void set_lfast(int i, uint16_t v) const { col[i * kInflateThreads] = v; }
  __host__ __device__ __forceinline__ uint16_t get_dfast(int i) const { return col[((1 << inflate::kFastBits) + i) * kInflateThreads]; }
  __host__ __device__ __forceinline__ void set_dfast(int i, uint16_t v) const { col[((1 << inflate::kFastBits) + i) * kInflateThreads] = v; }
};
constexpr size_t kInflateSmem = (DeviceTables::kCounts + 32) * kInflateThreads * sizeof(uint16_t);

// what the kernels of a stream hand from wave to wave, and back to the host
struct StreamState {
  unsigned int bad_block;       // first block (index within its wave) that did not decode, or 0xFFFFFFFF
  int bad_status;               // its inflate::Status; 100: size / length disagreement; 101: CRC-32 mismatch
  unsigned int format_error;    // 1 irregular read length, 2 not FASTQ framing, 4 a record longer than the headroom
  unsigned int tail;            // bytes carried in front of the next wave
  unsigned int next_tail;
  unsigned int head_skip;       // bytes at the start of this wave's text that belong to the previous wave
  unsigned int self_contained;  // the caller cut this wave at record boundaries: nothing may be left over
  unsigned long long lines;     // newlines of the current wave's region
  unsigned long long records;   // records of the current wave
  unsigned long long records_total;
};

__global__ void __launch_bounds__(kInflateThreads) inflate_blocks_kernel(const uint8_t* __restrict__ gz,
                                                                        const uint64_t* __restrict__ begin,
                                                                        const uint64_t* __restrict__ out_off, uint32_t n,
                                                                        uint8_t* __restrict__ text, StreamState* st) {
  extern __shared__ uint16_t sm[];
  const uint32_t m = blockIdx.x * kInflateThreads + threadIdx.x;
  if (m >= n) return;
  DeviceSymbols symbols;
  const DeviceTables t{sm + threadIdx.x, &symbols};
  const uint64_t base = begin[0];
  const uint8_t* in = gz + (begin[m] - base);
  const size_t in_len = (size_t)(begin[m + 1] - begin[m]);
  uint8_t* out = text + out_off[m];
  const size_t cap = (size_t)(out_off[m + 1] - out_off[m]);
  size_t consumed = 0, produced = 0;
  uint32_t crc = 0, isize = 0;
  int rc = inflate::gunzip_member(in, in_len, out, cap, t, &consumed, &produced, &crc, &isize);
  if (rc == inflate::kOk && (consumed != in_len || produced != cap || isize != (uint32_t)cap)) rc = 100;
  if (rc != inflate::kOk) {
    const unsigned int prev = atomicMin(&st->bad_block, m);
    if (m < prev) st->bad_status = rc;  // (benign race between two bad blocks: either status will do)
  }
}

// CRC-32 of d[0 .. len) by the 32 lanes of a warp (the same d and len in every lane): 32 pieces joined
// as inflate_core.h describes, the result in lane 0.  `table`: the byte table, in shared memory.
__device__ __forceinline__ uint32_t warp_crc32(const uint8_t* d, size_t len, const uint32_t* table) {
  const uint32_t lane = threadIdx.x & 31;
  const size_t c = inflate::crc_piece_len(len), first = len - 31 * c;
  const size_t at = lane == 0 ? 0 : first + (lane - 1) * c;
  uint32_t crc = inflate::crc_bytes(d + at, lane == 0 ? first : c, [&](uint32_t i) { return table[i]; });
  uint32_t p = inflate::crc_x8n(c);  // the same in every lane
#pragma unroll
  for (int s = 1; s < 32; s *= 2) {
    const uint32_t other = __shfl_down_sync(0xffffffffu, crc, s);
    if ((lane & (2 * s - 1)) == 0) crc = inflate::crc_multmodp(p, crc) ^ other;
    p = inflate::crc_multmodp(p, p);
  }
  return crc;
}

// CRC-32 of every block's text against the trailer of its member (RFC 1952; flate2 checks it for
// the reference): one warp per block.
constexpr int kCrcWarps = 8;
__global__ void __launch_bounds__(kCrcWarps * 32) crc_blocks_kernel(const uint8_t* __restrict__ gz,
                                                                   const uint64_t* __restrict__ begin,
                                                                   const uint64_t* __restrict__ out_off, uint32_t n,
                                                                   const uint8_t* __restrict__ text, StreamState* st) {
  __shared__ uint32_t table[256];
  table[threadIdx.x] = inflate::crc_table_entry(threadIdx.x);
  __syncthreads();
  const uint32_t m = blockIdx.x * kCrcWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (m >= n) return;
  const uint32_t crc = warp_crc32(text + out_off[m], (size_t)(out_off[m + 1] - out_off[m]), table);
  if (lane == 0) {
    const uint8_t* t = gz + (begin[m + 1] - begin[0]) - 8;
    const uint32_t stored = (uint32_t)t[0] | ((uint32_t)t[1] << 8) | ((uint32_t)t[2] << 16) | ((uint32_t)t[3] << 24);
    if (crc != stored) {
      const unsigned int prev = atomicMin(&st->bad_block, m);
      if (m < prev) st->bad_status = 101;
    }
  }
}

// bytes [lo, hi) of the text are the current region: the carried tail, then this wave's text
__device__ __forceinline__ void region_of(const StreamState* st, uint64_t n_text, uint64_t* lo, uint64_t* hi) {
  *lo = kHeadroom - st->tail + st->head_skip;
  *hi = (uint64_t)kHeadroom + n_text;
}

__device__ __forceinline__ uint32_t newline_mask16(const uint8_t* __restrict__ text, uint64_t at, uint64_t lo, uint64_t hi) {
  // 16 bytes at `at` (16-byte aligned); bit j set iff byte at + j is a newline inside [lo, hi)
  const uint4 v = *reinterpret_cast<const uint4*>(text + at);
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  uint32_t mask = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t x = w[i] ^ 0x0A0A0A0Au;                                 // zero byte where a newline is
    const uint32_t z = ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u;  // bit 7 of every zero byte
    mask |= (((z >> 7) & 1u) | ((z >> 14) & 2u) | ((z >> 21) & 4u) | ((z >> 28) & 8u)) << (4 * i);
  }
  if (at < lo) mask &= lo - at >= 16 ? 0u : ~0u << (uint32_t)(lo - at);
  if (at + 16 > hi) mask &= hi <= at ? 0u : (1u << (uint32_t)(hi - at)) - 1u;
  return mask;
}

__global__ void __launch_bounds__(kChunkThreads) newline_count_kernel(const uint8_t* __restrict__ text, uint64_t n_text,
                                                                     const StreamState* st, uint32_t* __restrict__ counts) {
  uint64_t lo, hi;
  region_of(st, n_text, &lo, &hi);
  const uint64_t at = (uint64_t)blockIdx.x * kChunk + threadIdx.x * 16;
  uint32_t c = at < hi && at + 16 > lo ? __popc(newline_mask16(text, at, lo, hi)) : 0u;
  c = __reduce_add_sync(0xffffffffu, c);
  __shared__ uint32_t warp_sums[kChunkThreads / 32];
  if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t s = 0;
    for (uint32_t i = 0; i < kChunkThreads / 32; ++i) s += warp_sums[i];
    counts[blockIdx.x] = s;
  }
}

// counts[n_chunks] (set to 0 by the caller) scans to the number of lines of the region
__global__ void wave_totals_kernel(const uint32_t* __restrict__ first_line, uint32_t n_chunks, StreamState* st) {
  st->lines = first_line[n_chunks];
  st->records = st->lines / 4;
  st->next_tail = 0;  // set by span_extract_kernel when a last complete record exists
}

__global__ void __launch_bounds__(kChunkThreads) span_extract_kernel(const uint8_t* __restrict__ text, uint64_t n_text,
                                                                    StreamState* st, const uint32_t* __restrict__ first_line,
                                                                    uint32_t read_len, uint32_t span_start, uint32_t span_len,
                                                                    uint32_t span_stride, uint8_t* __restrict__ spans,
                                                                    uint32_t* __restrict__ seq_start, uint32_t* __restrict__ seq_end) {
  uint64_t lo, hi;
  region_of(st, n_text, &lo, &hi);
  const uint64_t lines = st->lines, records = st->records;
  const uint64_t at = (uint64_t)blockIdx.x * kChunk + threadIdx.x * 16;
  uint32_t mask = at < hi && at + 16 > lo ? newline_mask16(text, at, lo, hi) : 0u;
  // line number of this thread's first newline: chunk base + newlines of the threads before it
  const uint32_t mine = __popc(mask);
  uint32_t inc = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t v = __shfl_up_sync(0xffffffffu, inc, d);
    if ((threadIdx.x & 31) >= (uint32_t)d) inc += v;
  }
  __shared__ uint32_t warp_sums[kChunkThreads / 32];
  if ((threadIdx.x & 31) == 31) warp_sums[threadIdx.x >> 5] = inc;
  __syncthreads();
  uint32_t before = first_line[blockIdx.x] + inc - mine;
  for (uint32_t w = 0; w < (threadIdx.x >> 5); ++w) before += warp_sums[w];
  if (blockIdx.x == 0 && threadIdx.x == 0 && hi > lo && text[lo] != '@') atomicOr(&st->format_error, 2u);
  uint64_t line = before;
  while (mask) {
    const uint32_t j = __ffs((int)mask) - 1;
    mask &= mask - 1;
    const uint64_t p = at + j;  // a newline: the end of line `line` of the region
    const uint64_t r = line >> 2;
    if (read_len == 0 && r < records) {
      // reads of any length: the sequence line stays where it is, [seq_start[r], seq_end[r]) of the text
      if ((line & 3) == 0) {
        seq_start[r] = (uint32_t)(p + 1);
      } else if ((line & 3) == 1) {
        seq_end[r] = (uint32_t)p;
        if (text[p + 1] != '+') atomicOr(&st->format_error, 2u);  // (p + 1 < hi: the record is complete)
      } else if ((line & 3) == 3 && p + 1 < hi && text[p + 1] != '@') {
        atomicOr(&st->format_error, 2u);
      }
    } else if ((line & 3) == 0 && r < records) {
      // the header of record r ends here; its sequence is the next read_len bytes, then "\n+"
      const uint64_t s = p + 1;
      if (s + read_len + 1 >= hi || text[s + read_len] != '\n' || text[s + read_len + 1] != '+') {
        atomicOr(&st->format_error, 1u);
      } else {
        uint8_t* dst = spans + r * span_stride;
        for (uint32_t b = 0; b < span_len; ++b) dst[b] = text[s + span_start + b];
      }
    }
    if ((line & 3) == 3 && r + 1 == records) {
      st->next_tail = (unsigned int)(hi - (p + 1));  // what follows the last complete record
    }
    ++line;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && records == 0) {
    // no complete record in the region: all of it is carried on (it must fit the headroom)
    if (hi - lo > kHeadroom) atomicOr(&st->format_error, 4u);
    st->next_tail = (unsigned int)min((uint64_t)kHeadroom, hi - lo);
  }
  (void)lines;
}

// the bytes after the last complete record, parked in `tail_buf`, then put in front of the next
// wave's text (two steps: source and destination may overlap when a wave is tiny)
__global__ void tail_save_kernel(const uint8_t* __restrict__ text, uint64_t n_text, StreamState* st, uint8_t* __restrict__ tail_buf) {
  const uint64_t hi = (uint64_t)kHeadroom + n_text;
  const uint32_t tail = st->next_tail;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < tail; i += gridDim.x * blockDim.x) tail_buf[i] = text[hi - tail + i];
}
__global__ void wave_begin_kernel(StreamState* st, unsigned int head_skip, unsigned int self_contained) {
  st->head_skip = head_skip;
  st->self_contained = self_contained;
}
__global__ void wave_commit_kernel(StreamState* st) {
  if (st->self_contained && st->next_tail) atomicOr(&st->format_error, 8u);  // the cut was not a record boundary
  st->tail = st->next_tail;
  st->head_skip = 0;
  st->records_total += st->records;
}
__global__ void tail_restore_kernel(uint8_t* __restrict__ text, const StreamState* st, const uint8_t* __restrict__ tail_buf) {
  const uint32_t tail = st->tail;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < tail; i += gridDim.x * blockDim.x)
    text[kHeadroom - tail + i] = tail_buf[i];
}

// ---- gzip members (not BGZF) decoded in pieces: the steps of inflate_core.h "gzip members in pieces" ----
// Candidate piece starts: one warp per nominal boundary c_j = j * piece bytes (j >= 1), its lanes probing
// consecutive bit offsets; the first that passes wins (or ~0: none before c_{j+1}).
__global__ void __launch_bounds__(kInflateThreads) member_find_kernel(const uint8_t* __restrict__ gz, uint64_t n_gz,
                                                                     uint64_t piece, uint32_t n_bounds, uint64_t* __restrict__ cand) {
  extern __shared__ uint16_t sm[];
  const uint32_t j = 1 + blockIdx.x * (kInflateThreads / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (j >= n_bounds) return;  // (whole warps)
  DeviceSymbols symbols;
  const DeviceTables t{sm + threadIdx.x, &symbols};
  const uint64_t lo = j * piece * 8, hi = min((uint64_t)(j + 1) * piece, n_gz) * 8;
  uint64_t found = ~0ull;
  for (uint64_t base = lo; base < hi; base += 32) {
    const uint64_t bit = base + lane;
    const bool ok = bit < hi && inflate::probe_block_start(gz, (size_t)n_gz, bit, t, inflate::kProbeTrial);
    const uint32_t votes = __ballot_sync(0xffffffffu, ok);
    if (votes) {
      found = base + (uint64_t)(__ffs((int)votes) - 1);
      break;
    }
  }
  if (lane == 0) cand[j] = found;
}

// is_member[j]: piece j starts a gzip member, so none of its matches may reach in front of it
__global__ void __launch_bounds__(kInflateThreads) member_boundary_kernel(const uint8_t* __restrict__ gz, uint64_t n_gz,
                                                                         const uint64_t* __restrict__ starts,
                                                                         const uint8_t* __restrict__ is_member, uint32_t n,
                                                                         inflate::PieceMeta* __restrict__ meta) {
  extern __shared__ uint16_t sm[];
  const uint32_t j = blockIdx.x * kInflateThreads + threadIdx.x;
  if (j >= n) return;
  DeviceSymbols symbols;
  const DeviceTables t{sm + threadIdx.x, &symbols};
  inflate::PieceMeta m{0, 0, 0, 0};
  m.status = inflate::piece_boundary(gz, (size_t)n_gz, starts, n, j, inflate::kMaxAbsorb, t, &m.next, &m.end_bit, &m.out_len,
                                     is_member[j] ? 0u : inflate::kWindow);
  meta[j] = m;
}

// Member-start candidates of several members: one thread per 4 KiB of input finds every gzip header in
// it (inflate::member_start_at) and appends the bit its DEFLATE stream starts at to heads[] (unordered;
// heads[cap], as a 64-bit counter, ends up holding the number found, which may exceed cap).
constexpr uint32_t kSignatureBytes = 4096;
__global__ void __launch_bounds__(256) member_signature_kernel(const uint8_t* __restrict__ gz, uint64_t n_gz,
                                                              uint64_t* __restrict__ heads, uint64_t cap) {
  const uint64_t lo = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * kSignatureBytes;
  if (lo >= n_gz) return;
  const uint64_t hi = min(lo + kSignatureBytes, n_gz);
  unsigned long long* found = reinterpret_cast<unsigned long long*>(heads + cap);
  for (uint64_t at = lo; at < hi; at += 16) {  // (the buffer has 64 bytes of slack behind the input)
    const uint4 v = *reinterpret_cast<const uint4*>(gz + at);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t x = w[i] ^ 0x1F1F1F1Fu;                                  // zero byte where a 0x1f is
      uint32_t z = ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u;  // bit 7 of every zero byte
      while (z) {
        const uint64_t pos = at + 4 * i + ((__ffs((int)z) - 1) >> 3);
        z &= z - 1;
        uint64_t bit = 0;
        if (pos < hi && inflate::member_start_at(gz, (size_t)n_gz, (size_t)pos, &bit)) {
          const unsigned long long k = atomicAdd(found, 1ull);
          if (k < cap) heads[k] = bit;
        }
      }
    }
  }
}

// a piece of the chain in the current wave: where its bits start and end, where its text goes
// (offset within the wave's text) and how far before its start a match may reach
struct WavePiece {
  uint64_t start_bit, end_bit, off, reach;
};
__global__ void __launch_bounds__(kInflateThreads) member_decode_kernel(const uint8_t* __restrict__ gz, uint64_t n_gz,
                                                                       const WavePiece* __restrict__ wp, uint32_t n,
                                                                       uint16_t* __restrict__ sym, StreamState* st) {
  extern __shared__ uint16_t sm[];
  const uint32_t i = blockIdx.x * kInflateThreads + threadIdx.x;
  if (i >= n) return;
  DeviceSymbols symbols;
  const DeviceTables t{sm + threadIdx.x, &symbols};
  const WavePiece p = wp[i];
  const uint64_t len = wp[i + 1].off - p.off;
  inflate::MarkSink sink{sym + p.off, 0, len, p.reach};
  uint64_t e = 0;
  bool fin = false;
  int rc = inflate::inflate_piece(gz, (size_t)n_gz, p.start_bit, p.end_bit, t, sink, [&](uint64_t b) { return b >= p.end_bit; },
                                  &e, &fin);
  if (rc == inflate::kOk && (e != p.end_bit || sink.op != len)) rc = 100;
  if (rc != inflate::kOk) {
    const unsigned int prev = atomicMin(&st->bad_block, i);
    if (i < prev) st->bad_status = rc;
  }
}

// byte x of the wave's text from its symbol: a marker names a byte of the 32 KiB in front of the
// piece, which is either earlier text of this wave or the end of the previous waves (`window`)
__device__ __forceinline__ uint8_t member_resolve(uint16_t s, uint64_t piece_off, const uint8_t* text, const uint8_t* window) {
  if (s < 256) return (uint8_t)s;
  const int64_t g = (int64_t)piece_off - (int64_t)inflate::kWindow + (int64_t)(s - 256);
  return g >= 0 ? text[g] : window[inflate::kWindow + g];
}

// everything else, every piece side by side (its window is resolved)
__global__ void __launch_bounds__(256) member_resolve_kernel(const uint16_t* __restrict__ sym, const WavePiece* __restrict__ wp,
                                                            uint8_t* text, const uint8_t* __restrict__ window) {
  const uint64_t a = wp[blockIdx.x].off, b = wp[blockIdx.x + 1].off;
  if (b - a <= inflate::kWindow) return;
  const uint64_t end = b - inflate::kWindow;
  for (uint64_t x = a + threadIdx.x; x < end; x += blockDim.x) text[x] = member_resolve(sym[x], a, text, window);
}

// CRC-32 of every piece's text, one warp each (joined on the host across pieces and waves)
__global__ void __launch_bounds__(kCrcWarps * 32) member_crc_kernel(const WavePiece* __restrict__ wp, uint32_t n,
                                                                   const uint8_t* __restrict__ text, uint32_t* __restrict__ crc_out) {
  __shared__ uint32_t table[256];
  table[threadIdx.x] = inflate::crc_table_entry(threadIdx.x);
  __syncthreads();
  const uint32_t i = blockIdx.x * kCrcWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= n) return;
  const uint32_t crc = warp_crc32(text + wp[i].off, (size_t)(wp[i + 1].off - wp[i].off), table);
  if (lane == 0) crc_out[i] = crc;
}

// Step 5 of inflate_core.h, the window relay ("waves: the window relay"), in place on the symbols of the
// last 32 KiB (or all) of every piece, piece after piece: a marker that names a byte of this wave takes
// the symbol relayed there, one that names a byte in front of the wave becomes a marker of the wave's
// entering window.  It needs nothing from another wave.  The only sequential step: one block, 32
// symbols a thread.
constexpr int kWindowThreads = 1024;
__global__ void __launch_bounds__(kWindowThreads) member_window_sym_kernel(uint16_t* sym, const WavePiece* __restrict__ wp,
                                                                          uint32_t n) {
  for (uint32_t i = 0; i < n; ++i) {
    const uint64_t a = wp[i].off, b = wp[i + 1].off;
    const uint64_t lo = b - a > inflate::kWindow ? b - inflate::kWindow : a;
    const uint64_t x0 = lo + (uint64_t)threadIdx.x * 32;
    uint16_t v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = x0 + k < b ? inflate::relay_symbol(sym[x0 + k], a, sym) : 0;
#pragma unroll
    for (int k = 0; k < 32; ++k)
      if (x0 + k < b) sym[x0 + k] = v[k];
    __syncthreads();  // (the next piece reads these symbols)
  }
}

// with the entering window known: the relayed last 32 KiB (or all) of every piece, side by side
__global__ void __launch_bounds__(256) member_settle_kernel(const uint16_t* __restrict__ sym, const WavePiece* __restrict__ wp,
                                                           uint8_t* __restrict__ text, const uint8_t* __restrict__ window) {
  const uint64_t a = wp[blockIdx.x].off, b = wp[blockIdx.x + 1].off;
  const uint64_t lo = b - a > inflate::kWindow ? b - inflate::kWindow : a;
  for (uint64_t x = lo + threadIdx.x; x < b; x += blockDim.x) text[x] = inflate::settle_symbol(sym[x], window);
}

// Device scratch of the ingest streams comes from one memory pool per device whose unused memory stays
// cached, through the stream-ordered allocator.  cudaFree waits for ALL work on the device and cudaMalloc
// queues up behind it: with several samples in flight on one device (the CLI runs four) every sample that
// finished — a dozen buffers to release — stalled the others' next allocation until their kernels had
// drained, and the samples ran one after the other.  cudaFreeAsync is ordered on the stream only.
struct ScratchPools {
  std::mutex mu;
  std::map<int, cudaMemPool_t> pool;  // NULL: the device has no memory pools (cudaMalloc / cudaFree instead)
};
cudaMemPool_t scratch_pool(int device) {
  static ScratchPools pools;
  std::lock_guard<std::mutex> lk(pools.mu);
  auto it = pools.pool.find(device);
  if (it != pools.pool.end()) return it->second;
  cudaMemPool_t pool = nullptr;
  int supported = 0;
  if (cudaDeviceGetAttribute(&supported, cudaDevAttrMemoryPoolsSupported, device) == cudaSuccess && supported) {
    cudaMemPoolProps props{};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = device;
    if (cudaMemPoolCreate(&pool, &props) == cudaSuccess) {
      uint64_t keep = 8ull << 30;  // up to 8 GiB of freed memory stay with the pool for the next wave / sample
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    } else {
      pool = nullptr;
      cudaGetLastError();
    }
  }
  pools.pool[device] = pool;
  return pool;
}
int scratch_alloc(void** p, size_t bytes, cudaMemPool_t pool, cudaStream_t stream) {
  if (pool)
    SGC_CUDA_TRY(cudaMallocFromPoolAsync(p, bytes, pool, stream));
  else
    SGC_CUDA_TRY(cudaMalloc(p, bytes));
  return SGC_OK;
}
void scratch_free(void* p, cudaMemPool_t pool, cudaStream_t stream) {
  if (!p) return;
  if (pool)
    cudaFreeAsync(p, stream);
  else
    cudaFree(p);
}

template <typename T>
int grow(T** p, size_t* cap, size_t need, cudaMemPool_t pool, cudaStream_t stream) {
  if (need <= *cap) return SGC_OK;
  scratch_free(*p, pool, stream);  // (stream order: the kernels that still read it come first)
  *p = nullptr;
  *cap = 0;
  const size_t want = need + need / 4;
  int rc = scratch_alloc(reinterpret_cast<void**>(p), want * sizeof(T), pool, stream);
  if (rc) return rc;
  *cap = want;
  return SGC_OK;
}

}  // namespace
}  // namespace sgc

using namespace sgc;

struct sgc_fastq_stream {
  sgc_counter* counter = nullptr;  // NULL once released (its counter was destroyed first)
  int device = 0;
  uint32_t read_len = 0, span_start = 0, span_len = 0, span_stride = 0;
  cudaStream_t stream = nullptr;
  cudaMemPool_t pool = nullptr;  // scratch_pool(device)
  StreamState* d_state = nullptr;
  uint8_t *d_gz = nullptr, *d_text = nullptr, *d_spans = nullptr, *d_tail = nullptr;
  uint32_t *d_seq_start = nullptr, *d_seq_end = nullptr;  // variable-length mode
  size_t seq_cap_a = 0, seq_cap_b = 0;
  uint64_t *d_begin = nullptr, *d_outoff = nullptr;
  uint32_t *d_counts = nullptr, *d_first = nullptr, *d_sums = nullptr;
  size_t gz_cap = 0, text_cap = 0, spans_cap = 0, begin_cap = 0, outoff_cap = 0, counts_cap = 0, first_cap = 0, sums_cap = 0;
  std::vector<uint64_t> h_begin, h_outoff;
  uint64_t blocks_total = 0, records_total = 0;
  bool failed = false;
  // plain gzip in pieces (sgc_fastq_stream_submit_member, _submit_gzip, _submit_gzip_split)
  uint16_t* d_sym = nullptr;
  uint8_t* d_window = nullptr;  // W_k, the 32 KiB in front of the current wave
  uint64_t* d_cand = nullptr;
  inflate::PieceMeta* d_meta = nullptr;
  WavePiece* d_wave = nullptr;
  uint32_t* d_crc = nullptr;
  size_t sym_cap = 0, cand_cap = 0, meta_cap = 0, wave_cap = 0, crc_cap = 0;
  uint64_t member_pieces = 0, member_chain = 0, member_absorbed = 0;
  bool member_submitted = false;
  // gzip headers inside the file as member starts (all but sgc_fastq_stream_submit_member)
  uint64_t* d_heads = nullptr;  // member-start candidates, then their count
  uint8_t* d_is_member = nullptr;
  size_t heads_cap = 0, is_member_cap = 0;
  uint64_t gzip_members = 0;
};

namespace {

int stream_error(sgc_fastq_stream* s, const StreamState& st, uint64_t first_block) {
  s->failed = true;
  char buf[200];
  if (st.bad_block != 0xFFFFFFFFu) {
    if (st.bad_status == 101)
      snprintf(buf, sizeof buf, "gzip block %llu: CRC-32 of the inflated bytes differs from the member's trailer",
               (unsigned long long)(first_block + st.bad_block));
    else
      snprintf(buf, sizeof buf, "gzip block %llu did not inflate on the device (status %d)",
               (unsigned long long)(first_block + st.bad_block), st.bad_status);
    return set_error(SGC_ERR_GZIP, buf);
  }
  snprintf(buf, sizeof buf, "not fixed-length 4-line FASTQ (%s)",
           (st.format_error & 2) ? "a record does not start with '@'"
                                 : ((st.format_error & 4) ? "a record longer than 64 KB"
                                                          : ((st.format_error & 8) ? "a wave was not cut at a record boundary"
                                                                                   : "a read of another length, or a line that is not '+'")));
  return set_error(SGC_ERR_FASTQ_FORMAT, buf);
}

// frames and counts the region made of the carried tail and n_text fresh bytes at d_text + kHeadroom
int frame_and_count(sgc_fastq_stream* s, uint64_t n_text, uint64_t first_block) {
  const uint32_t n_chunks = (uint32_t)(((uint64_t)kHeadroom + n_text + kChunk - 1) / kChunk);
  int rc = grow(&s->d_counts, &s->counts_cap, (size_t)n_chunks + 1, s->pool, s->stream);
  if (rc == SGC_OK) rc = grow(&s->d_first, &s->first_cap, (size_t)n_chunks + 1, s->pool, s->stream);
  if (rc == SGC_OK) rc = grow(&s->d_sums, &s->sums_cap, (size_t)n_chunks / 2048 + 2, s->pool, s->stream);
  if (rc) return rc;
  // the carried bytes go in front of the fresh text (they are kept in d_tail: d_text may have moved)
  tail_restore_kernel<<<8, 256, 0, s->stream>>>(s->d_text, s->d_state, s->d_tail);
  SGC_CUDA_TRY(cudaMemsetAsync(s->d_counts + n_chunks, 0, sizeof(uint32_t), s->stream));
  newline_count_kernel<<<n_chunks, kChunkThreads, 0, s->stream>>>(s->d_text, n_text, s->d_state, s->d_counts);
  rc = exclusive_scan_u32(s->d_counts, n_chunks + 1, s->d_first, s->d_sums, s->stream);
  if (rc) return rc;
  wave_totals_kernel<<<1, 1, 0, s->stream>>>(s->d_first, n_chunks, s->d_state);
  // how many records the region holds decides the size of the span / offset buffers
  StreamState pre;
  SGC_CUDA_TRY(cudaMemcpyAsync(&pre, s->d_state, sizeof pre, cudaMemcpyDeviceToHost, s->stream));
  SGC_CUDA_TRY(cudaStreamSynchronize(s->stream));
  if (pre.bad_block != 0xFFFFFFFFu) return stream_error(s, pre, first_block);
  const size_t max_records = (size_t)pre.records + 1;
  if (s->read_len) {
    rc = grow(&s->d_spans, &s->spans_cap, max_records * s->span_stride + 256, s->pool, s->stream);
  } else {
    rc = grow(&s->d_seq_start, &s->seq_cap_a, max_records, s->pool, s->stream);
    if (rc == SGC_OK) rc = grow(&s->d_seq_end, &s->seq_cap_b, max_records, s->pool, s->stream);
  }
  if (rc) return rc;
  span_extract_kernel<<<n_chunks, kChunkThreads, 0, s->stream>>>(s->d_text, n_text, s->d_state, s->d_first, s->read_len,
                                                                 s->span_start, s->span_len, s->span_stride, s->d_spans,
                                                                 s->d_seq_start, s->d_seq_end);
  tail_save_kernel<<<8, 256, 0, s->stream>>>(s->d_text, n_text, s->d_state, s->d_tail);
  wave_commit_kernel<<<1, 1, 0, s->stream>>>(s->d_state);
  SGC_CUDA_TRY(cudaGetLastError());
  StreamState st;
  SGC_CUDA_TRY(cudaMemcpyAsync(&st, s->d_state, sizeof st, cudaMemcpyDeviceToHost, s->stream));
  SGC_CUDA_TRY(cudaStreamSynchronize(s->stream));
  if (st.bad_block != 0xFFFFFFFFu || st.format_error) return stream_error(s, st, first_block);
  if (st.records) {
    if (s->read_len)
      rc = sgc_counter_submit_device(s->counter, s->d_spans, st.records * s->span_stride + 64, nullptr, s->span_stride,
                                     s->span_len, st.records, nullptr);
    else  // the sequence lines in place, through the line kernel
      rc = count_gathered_lines(s->counter, s->d_text, (uint64_t)kHeadroom + n_text, s->d_seq_start, s->d_seq_end, st.records);
    if (rc) return rc;
  }
  s->records_total = st.records_total;
  return SGC_OK;
}

// ---- gzip members in pieces: the host side of sgc_fastq_stream_submit_member / _submit_gzip / _submit_gzip_split ----
// Nominal piece size: 32 KiB of compressed input (more pieces than larger ones would give keep more
// threads busy; each piece is a serial decode).  SGC_MEMBER_PIECE overrides it and SGC_MEMBER_SKEW=1
// moves every other candidate start one bit on (tests: many pieces on small files, absorbed pieces);
// SGC_MEMBER_WAVE_TEXT bounds the text of a wave (tests: many waves).
struct MemberParams {
  uint64_t piece, wave_text;
  bool skew;
};
MemberParams member_params(uint32_t read_len) {
  MemberParams p{32u << 10, read_len ? (4ull << 30) : (3ull << 30), false};
  if (const char* e = getenv("SGC_MEMBER_PIECE"); e && atoll(e) >= 64) p.piece = (uint64_t)atoll(e);
  const char* skew_env = getenv("SGC_MEMBER_SKEW");
  p.skew = skew_env && atoi(skew_env) != 0;
  if (const char* e = getenv("SGC_MEMBER_WAVE_TEXT"); e && atoll(e) > 0) p.wave_text = std::min<uint64_t>(p.wave_text, (uint64_t)atoll(e));
  return p;
}

// the caller counts the file on the host instead
int member_decline(sgc_fastq_stream* s, const char* why) {
  s->failed = true;
  char buf[240];
  snprintf(buf, sizeof buf, "gzip file not decoded on the device: %s", why);
  return set_error(SGC_ERR_GZIP, buf);
}

constexpr const char* kTooManyHeaders = "more gzip headers than one per 256 bytes";

// step 1 on the host: the candidates near the nominal boundaries, cand[1 .. n_bounds) (~0: none), after
// the first member's first block, merged with the member starts heads[] (sorted here)
void merge_candidates(const MemberParams& p, size_t header, const std::vector<uint64_t>& cand, uint32_t n_bounds,
                      std::vector<uint64_t>& heads, std::vector<uint64_t>& starts, std::vector<uint8_t>& is_member) {
  std::vector<uint64_t> probe{(uint64_t)header * 8};
  for (uint32_t j = 1; j < n_bounds; ++j) {
    if (cand[j] == ~0ull) continue;
    const uint64_t c = cand[j] + (p.skew && (probe.size() & 1) ? 1 : 0);
    if (c > probe.back()) probe.push_back(c);
  }
  std::sort(heads.begin(), heads.end());
  starts.resize(probe.size() + heads.size());
  is_member.resize(starts.size());
  starts.resize(inflate::merge_starts(probe.data(), (uint32_t)probe.size(), heads.data(), (uint32_t)heads.size(), starts.data(),
                                      is_member.data()));
  is_member.resize(starts.size());
  is_member[0] = 1;  // (the first member's start, found by both scans)
}

// step 3: the chain of pieces, the member of each, the trailers
struct MemberChain {
  std::vector<uint32_t> chain, member_of;
  std::vector<inflate::MemberTrailer> trailers;
  uint32_t n_chain = 0, n_members = 0;
  uint64_t absorbed = 0;
};
// nullptr, or why the file is declined
const char* follow_chain(const uint8_t* gz, uint64_t n_bytes, const std::vector<uint64_t>& starts, const std::vector<uint8_t>& is_member,
                         const std::vector<inflate::PieceMeta>& meta, MemberChain& c) {
  const uint32_t n = (uint32_t)starts.size();
  c.chain.resize(n);
  c.member_of.resize(n);
  c.trailers.resize(n);
  c.n_chain = inflate::members_chain(gz, (size_t)n_bytes, starts.data(), is_member.data(), meta.data(), n, c.chain.data(),
                                     c.member_of.data(), c.trailers.data(), &c.n_members, &c.absorbed);
  if (c.n_chain == 0) return "the blocks could not be followed from piece to piece to a trailer that ends the file";
  std::vector<uint64_t> text(c.n_members, 0);
  for (uint32_t i = 0; i < c.n_chain; ++i) text[c.member_of[i]] += meta[c.chain[i]].out_len;
  for (uint32_t m = 0; m < c.n_members; ++m)
    if (c.trailers[m].isize != (uint32_t)text[m]) return "ISIZE of a member differs from the length of its text";
  return nullptr;
}

// Runs fn(i) for every stream i on a thread of its own, with the stream's device current, and joins
// them all.  Returns the first failure by stream index, its message set on the calling thread.
template <typename Fn>
int on_each_stream(sgc_fastq_stream* const* ss, uint32_t n, Fn fn) {
  std::vector<int> rc(n, SGC_OK);
  std::vector<std::string> msg(n);
  std::vector<std::thread> threads;
  threads.reserve(n);
  for (uint32_t i = 0; i < n; ++i)
    threads.emplace_back([&, i] {
      DeviceGuard guard(ss[i]->device);
      rc[i] = fn(i);
      if (rc[i]) msg[i] = sgc_last_error();
    });
  for (auto& t : threads) t.join();
  for (uint32_t i = 0; i < n; ++i)
    if (rc[i]) return set_error(rc[i], msg[i]);
  return SGC_OK;
}

// where part i of n_items cut into `parts` starts: equal parts, rounded up to a multiple of `grain`
uint64_t part_begin(uint64_t n_items, uint32_t parts, uint32_t i, uint64_t grain) {
  const uint64_t per = (n_items + parts - 1) / parts;
  return std::min(n_items, (per + grain - 1) / grain * grain * i);
}

int fail_all(sgc_fastq_stream* const* ss, uint32_t n, int rc) {
  for (uint32_t i = 0; i < n; ++i) ss[i]->failed = true;
  return rc;
}

// 1-2. the compressed bytes to every stream's device; candidate piece starts near every nominal boundary
// (the first member's first block is piece 0) and, with `find_headers`, at every gzip header; every
// piece to its first block end at or beyond the next candidate.  Each kernel runs over one contiguous
// part per stream, given shifted pointers: member_find_kernel's boundary 1 is boundary j0, its bits
// count from byte (j0 - 1) * piece; member_signature_kernel starts at byte b0 (whole blocks of it per
// part); member_boundary_kernel's piece 0 is piece c0 (so `next` counts from c0).
int find_pieces(sgc_fastq_stream* const* ss, uint32_t ns, const uint8_t* gz, uint64_t n_bytes, size_t header, const MemberParams& p,
                bool find_headers, std::vector<uint64_t>& starts, std::vector<uint8_t>& is_member,
                std::vector<inflate::PieceMeta>& meta) {
  const uint32_t n_bounds = (uint32_t)((n_bytes + p.piece - 1) / p.piece);
  // member-start candidates: up to one per 256 bytes of input (fewer, larger members go to the host)
  const uint64_t heads_cap = find_headers ? n_bytes / 256 + 4096 : 0;
  constexpr uint32_t kWarps = kInflateThreads / 32;
  constexpr uint64_t kSignatureSpan = 256ull * kSignatureBytes;  // the input of one block of member_signature_kernel
  std::vector<uint64_t> cand((size_t)n_bounds + 1, ~0ull), found(ns, 0);
  std::vector<std::vector<uint64_t>> heads(ns);
  int rc = on_each_stream(ss, ns, [&](uint32_t i) {
    sgc_fastq_stream* s = ss[i];
    int rc = grow(&s->d_gz, &s->gz_cap, (size_t)n_bytes + 64, s->pool, s->stream);  // (the reader's slack)
    if (rc == SGC_OK) rc = grow(&s->d_cand, &s->cand_cap, (size_t)n_bounds + 1, s->pool, s->stream);
    if (rc == SGC_OK && find_headers) rc = grow(&s->d_heads, &s->heads_cap, (size_t)heads_cap + 1, s->pool, s->stream);
    if (rc) return rc;
    SGC_CUDA_TRY(cudaMemcpyAsync(s->d_gz, gz, n_bytes, cudaMemcpyHostToDevice, s->stream));
    const uint64_t j0 = 1 + part_begin(n_bounds - 1, ns, i, kWarps), j1 = 1 + part_begin(n_bounds - 1, ns, i + 1, kWarps);
    const uint64_t shift = (j0 - 1) * p.piece;
    if (j1 > j0)
      member_find_kernel<<<(unsigned)((j1 - j0 + kWarps - 1) / kWarps), kInflateThreads, kInflateSmem, s->stream>>>(
          s->d_gz + shift, n_bytes - shift, p.piece, (uint32_t)(j1 - j0 + 1), s->d_cand + (j0 - 1));
    const uint64_t b0 = part_begin(n_bytes, ns, i, kSignatureSpan), b1 = part_begin(n_bytes, ns, i + 1, kSignatureSpan);
    if (find_headers) {
      SGC_CUDA_TRY(cudaMemsetAsync(s->d_heads + heads_cap, 0, sizeof(uint64_t), s->stream));
      if (b1 > b0)
        member_signature_kernel<<<(unsigned)((b1 - b0 + kSignatureSpan - 1) / kSignatureSpan), 256, 0, s->stream>>>(
            s->d_gz + b0, n_bytes - b0, s->d_heads, heads_cap);
      SGC_CUDA_TRY(cudaMemcpyAsync(&found[i], s->d_heads + heads_cap, sizeof(uint64_t), cudaMemcpyDeviceToHost, s->stream));
    }
    SGC_CUDA_TRY(cudaGetLastError());
    if (j1 > j0) SGC_CUDA_TRY(cudaMemcpyAsync(cand.data() + j0, s->d_cand + j0, (j1 - j0) * 8, cudaMemcpyDeviceToHost, s->stream));
    SGC_CUDA_TRY(cudaStreamSynchronize(s->stream));
    for (uint64_t j = j0; j < j1; ++j)
      if (cand[j] != ~0ull) cand[j] += shift * 8;
    heads[i].resize(std::min(found[i], heads_cap));
    if (!heads[i].empty()) {
      SGC_CUDA_TRY(cudaMemcpyAsync(heads[i].data(), s->d_heads, heads[i].size() * 8, cudaMemcpyDeviceToHost, s->stream));
      SGC_CUDA_TRY(cudaStreamSynchronize(s->stream));
    }
    for (uint64_t& h : heads[i]) h += b0 * 8;
    return SGC_OK;
  });
  if (rc) return rc;
  uint64_t n_heads = 0;
  for (uint32_t i = 0; i < ns; ++i) n_heads += found[i];
  if (n_heads > heads_cap) return member_decline(ss[0], kTooManyHeaders);
  std::vector<uint64_t> all_heads;
  all_heads.reserve(n_heads);
  for (auto& h : heads) all_heads.insert(all_heads.end(), h.begin(), h.end());
  merge_candidates(p, header, cand, n_bounds, all_heads, starts, is_member);

  const uint32_t n = (uint32_t)starts.size();
  meta.resize(n);
  return on_each_stream(ss, ns, [&](uint32_t i) {
    sgc_fastq_stream* s = ss[i];
    const uint32_t c0 = (uint32_t)part_begin(n, ns, i, kInflateThreads), c1 = (uint32_t)part_begin(n, ns, i + 1, kInflateThreads);
    if (c1 <= c0) return SGC_OK;
    int rc = grow(&s->d_meta, &s->meta_cap, (size_t)n, s->pool, s->stream);
    if (rc == SGC_OK) rc = grow(&s->d_cand, &s->cand_cap, (size_t)n, s->pool, s->stream);
    if (rc == SGC_OK) rc = grow(&s->d_is_member, &s->is_member_cap, (size_t)n, s->pool, s->stream);
    if (rc) return rc;
    SGC_CUDA_TRY(cudaMemcpyAsync(s->d_cand, starts.data(), n * 8ull, cudaMemcpyHostToDevice, s->stream));
    SGC_CUDA_TRY(cudaMemcpyAsync(s->d_is_member, is_member.data(), n, cudaMemcpyHostToDevice, s->stream));
    member_boundary_kernel<<<(c1 - c0 + kInflateThreads - 1) / kInflateThreads, kInflateThreads, kInflateSmem, s->stream>>>(
        s->d_gz, n_bytes, s->d_cand + c0, s->d_is_member + c0, n - c0, s->d_meta + c0);
    SGC_CUDA_TRY(cudaGetLastError());
    SGC_CUDA_TRY(cudaMemcpyAsync(meta.data() + c0, s->d_meta + c0, (c1 - c0) * sizeof(inflate::PieceMeta), cudaMemcpyDeviceToHost,
                                 s->stream));
    SGC_CUDA_TRY(cudaStreamSynchronize(s->stream));
    for (uint32_t j = c0; j < c1; ++j)
      if (meta[j].status == inflate::kOk && meta[j].next != inflate::kPieceFinal) meta[j].next += c0;
    return SGC_OK;
  });
}

// a wave of the chain: pieces [a, b), their text and where it goes
struct Wave {
  uint32_t a, b;
  uint64_t text;
  std::vector<WavePiece> wp;
};

// What the streams of one call hand each other (one stream: itself, from wave to wave): the entering
// window of every wave, composed on the host as the waves in front publish F_k, and the bytes after the
// last complete record of the wave framed last (framing goes wave after wave).
struct WindowRelay {
  std::mutex mu;
  std::condition_variable cv;
  bool stop = false;                         // a stream failed: the others give up
  std::vector<std::vector<uint16_t>> front;  // F_k, empty until wave k published it
  std::vector<std::vector<uint8_t>> window;  // W_k, known for k < composed
  uint32_t composed = 1;
  uint32_t framed = 0;  // waves framed and counted
  std::vector<uint8_t> tail;
};

// 4-7 for the waves k = i, i + ns, ... dealt to stream i; crc[x] (x: chain position) the CRC-32 of piece x.
// Returns SGC_OK without finishing when another stream failed (relay.stop; the caller sets it on a failure).
int stream_waves(sgc_fastq_stream* s, uint32_t i, uint32_t ns, uint64_t n_bytes, const std::vector<Wave>& waves, WindowRelay& relay,
                 std::vector<uint32_t>& crc) {
  const uint32_t n_waves = (uint32_t)waves.size();
  auto wait_for = [&](auto ready) {  // false: another stream failed
    std::unique_lock<std::mutex> lk(relay.mu);
    relay.cv.wait(lk, [&] { return relay.stop || ready(); });
    return !relay.stop;
  };
  const size_t tail_at = offsetof(StreamState, tail);
  int rc = SGC_OK;
  if (!s->d_window && (rc = scratch_alloc(reinterpret_cast<void**>(&s->d_window), inflate::kWindow, s->pool, s->stream))) return rc;
  for (uint32_t k = i; k < n_waves; k += ns) {
    const Wave& w = waves[k];
    const uint32_t nw = w.b - w.a;
    rc = grow(&s->d_wave, &s->wave_cap, (size_t)nw + 1, s->pool, s->stream);
    if (rc == SGC_OK) rc = grow(&s->d_sym, &s->sym_cap, (size_t)w.text + 1, s->pool, s->stream);
    if (rc == SGC_OK) rc = grow(&s->d_text, &s->text_cap, (size_t)kHeadroom + w.text + 64, s->pool, s->stream);
    if (rc == SGC_OK) rc = grow(&s->d_crc, &s->crc_cap, (size_t)nw, s->pool, s->stream);
    if (rc) return rc;
    SGC_CUDA_TRY(cudaMemcpyAsync(s->d_wave, w.wp.data(), w.wp.size() * sizeof(WavePiece), cudaMemcpyHostToDevice, s->stream));
    // symbols, relayed windows, F_k
    member_decode_kernel<<<(nw + kInflateThreads - 1) / kInflateThreads, kInflateThreads, kInflateSmem, s->stream>>>(
        s->d_gz, n_bytes, s->d_wave, nw, s->d_sym, s->d_state);
    member_window_sym_kernel<<<1, kWindowThreads, 0, s->stream>>>(s->d_sym, s->d_wave, nw);
    SGC_CUDA_TRY(cudaGetLastError());
    std::vector<uint16_t> f(inflate::kWindow);
    const uint64_t m = std::min<uint64_t>(w.text, inflate::kWindow);
    StreamState st;
    SGC_CUDA_TRY(cudaMemcpyAsync(f.data() + (inflate::kWindow - m), s->d_sym + (w.text - m), m * 2, cudaMemcpyDeviceToHost, s->stream));
    SGC_CUDA_TRY(cudaMemcpyAsync(&st, s->d_state, sizeof st, cudaMemcpyDeviceToHost, s->stream));
    SGC_CUDA_TRY(cudaStreamSynchronize(s->stream));
    if (st.bad_block != 0xFFFFFFFFu) return stream_error(s, st, w.a);
    inflate::wave_front(f.data(), w.text);
    {
      std::lock_guard<std::mutex> lk(relay.mu);
      relay.front[k] = std::move(f);
      for (; relay.composed < n_waves && !relay.front[relay.composed - 1].empty(); ++relay.composed)
        inflate::compose_window(relay.front[relay.composed - 1].data(), relay.window[relay.composed - 1].data(),
                                relay.window[relay.composed].data());
      relay.cv.notify_all();
    }
    // the text, once W_k is known
    if (!wait_for([&] { return relay.composed > k; })) return SGC_OK;
    SGC_CUDA_TRY(cudaMemcpyAsync(s->d_window, relay.window[k].data(), inflate::kWindow, cudaMemcpyHostToDevice, s->stream));
    uint8_t* text = s->d_text + kHeadroom;
    member_settle_kernel<<<nw, 256, 0, s->stream>>>(s->d_sym, s->d_wave, text, s->d_window);
    member_resolve_kernel<<<nw, 256, 0, s->stream>>>(s->d_sym, s->d_wave, text, s->d_window);
    member_crc_kernel<<<(nw + kCrcWarps - 1) / kCrcWarps, kCrcWarps * 32, 0, s->stream>>>(s->d_wave, nw, text, s->d_crc);
    SGC_CUDA_TRY(cudaGetLastError());
    // framing, behind the wave in front: its carried bytes come first
    if (!wait_for([&] { return relay.framed == k; })) return SGC_OK;
    const uint32_t carried = (uint32_t)relay.tail.size();
    if (carried) SGC_CUDA_TRY(cudaMemcpyAsync(s->d_tail, relay.tail.data(), carried, cudaMemcpyHostToDevice, s->stream));
    SGC_CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<uint8_t*>(s->d_state) + tail_at, &carried, 4, cudaMemcpyHostToDevice, s->stream));
    wave_begin_kernel<<<1, 1, 0, s->stream>>>(s->d_state, 0, 0);
    if ((rc = frame_and_count(s, w.text, w.a))) return rc;  // (synchronises)
    SGC_CUDA_TRY(cudaMemcpyAsync(crc.data() + w.a, s->d_crc, nw * 4ull, cudaMemcpyDeviceToHost, s->stream));
    SGC_CUDA_TRY(cudaMemcpyAsync(&st, s->d_state, sizeof st, cudaMemcpyDeviceToHost, s->stream));
    SGC_CUDA_TRY(cudaStreamSynchronize(s->stream));
    std::vector<uint8_t> tail;
    if (k + 1 < n_waves) {  // the wave's tail goes on to the next wave's stream (the last wave's stays: finish() counts it)
      tail.resize(st.tail);
      const uint32_t zero = 0;
      if (st.tail) SGC_CUDA_TRY(cudaMemcpyAsync(tail.data(), s->d_tail, st.tail, cudaMemcpyDeviceToHost, s->stream));
      SGC_CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<uint8_t*>(s->d_state) + tail_at, &zero, 4, cudaMemcpyHostToDevice, s->stream));
      SGC_CUDA_TRY(cudaStreamSynchronize(s->stream));
    }
    std::lock_guard<std::mutex> lk(relay.mu);
    relay.tail = std::move(tail);
    relay.framed = k + 1;
    relay.cv.notify_all();
  }
  return SGC_OK;
}

// One gzip file decoded by the ns streams ss[] together: sgc_fastq_stream_submit_gzip_split, and with one
// stream sgc_fastq_stream_submit_gzip and sgc_fastq_stream_submit_member (`find_headers` false: no gzip
// header inside the file is a candidate, so the chain must end at the first trailer).
int submit_plain_gzip(sgc_fastq_stream* const* ss, uint32_t ns, const uint8_t* gz, uint64_t n_bytes, bool find_headers) {
  if (!ss || !gz || ns == 0) return set_error(SGC_ERR_INVALID_ARG, "NULL argument or no stream");
  for (uint32_t i = 0; i < ns; ++i)
    if (!ss[i]) return set_error(SGC_ERR_INVALID_ARG, "NULL stream");
  for (uint32_t i = 0; i < ns; ++i) {
    const sgc_fastq_stream* s = ss[i];
    if (s->failed || !s->counter) return set_error(SGC_ERR_INVALID_ARG, "a stream has failed or its counter is gone");
    if (s->member_submitted || s->blocks_total) return set_error(SGC_ERR_INVALID_ARG, "a gzip file goes to fresh streams, once");
    for (uint32_t j = 0; j < i; ++j)
      if (ss[j] == s) return set_error(SGC_ERR_INVALID_ARG, "a stream is given twice");
    const sgc_fastq_stream* s0 = ss[0];
    if (s->read_len != s0->read_len || s->span_start != s0->span_start || s->span_len != s0->span_len)
      return set_error(SGC_ERR_INVALID_ARG, "the streams differ in read length or span");
    const sgc_library *l = s->counter->lib, *l0 = s0->counter->lib;
    if (l->n != l0->n || l->k != l0->k || l->with_perm != l0->with_perm)
      return set_error(SGC_ERR_INVALID_ARG, "the streams' counters come from different libraries");
  }
  for (uint32_t i = 0; i < ns; ++i) ss[i]->member_submitted = true;
  size_t header = 0;
  if (inflate::gzip_header(gz, (size_t)n_bytes, &header) != inflate::kOk)
    return fail_all(ss, ns, member_decline(ss[0], "not a gzip member"));
  const MemberParams params = member_params(ss[0]->read_len);

  // 1-2. candidate starts near every nominal boundary (and at every gzip header), the boundary pass
  std::vector<uint64_t> starts;
  std::vector<uint8_t> is_member;
  std::vector<inflate::PieceMeta> meta;
  int rc = find_pieces(ss, ns, gz, n_bytes, header, params, find_headers, starts, is_member, meta);
  if (rc) return fail_all(ss, ns, rc);

  // 3. the chain from the first block, over every trailer and header to the last trailer, which must end the file
  MemberChain c;
  if (const char* why = follow_chain(gz, n_bytes, starts, is_member, meta, c)) return fail_all(ss, ns, member_decline(ss[0], why));

  // 4-7. waves of about min(wave_text, text / streams), dealt round robin
  uint64_t total = 0;
  for (uint32_t i = 0; i < c.n_chain; ++i) total += meta[c.chain[i]].out_len;
  const uint64_t cap = std::min(params.wave_text, std::max<uint64_t>(1, (total + ns - 1) / ns));
  std::vector<Wave> waves;
  uint64_t done = 0, member_begin = 0;
  for (uint32_t a = 0; a < c.n_chain;) {
    Wave w{a, a, 0, {}};
    while (w.b < c.n_chain && (w.b == a || w.text + meta[c.chain[w.b]].out_len <= cap)) w.text += meta[c.chain[w.b++]].out_len;
    if (ss[0]->read_len == 0 && w.text >= (1ull << 32) - 2 * kHeadroom)
      return fail_all(ss, ns, member_decline(ss[0], "a piece inflates to 4 GiB or more"));
    uint64_t off = 0;
    for (uint32_t x = a; x < w.b; ++x) {
      if (x > 0 && c.member_of[x] != c.member_of[x - 1]) member_begin = done + off;
      const uint64_t reach = done + off - member_begin;
      w.wp.push_back(WavePiece{starts[c.chain[x]], meta[c.chain[x]].end_bit, off, std::min<uint64_t>(reach, inflate::kWindow)});
      off += meta[c.chain[x]].out_len;
    }
    w.wp.push_back(WavePiece{0, 0, w.text, 0});
    done += w.text;
    a = w.b;
    waves.push_back(std::move(w));
  }
  WindowRelay relay;
  relay.front.resize(waves.size());
  relay.window.assign(waves.size(), std::vector<uint8_t>(inflate::kWindow, 0));  // W_0: zeros
  std::vector<uint32_t> piece_crc(c.n_chain, 0);
  rc = on_each_stream(ss, ns, [&](uint32_t i) {
    const int rc = stream_waves(ss[i], i, ns, n_bytes, waves, relay, piece_crc);
    if (rc) {
      std::lock_guard<std::mutex> lk(relay.mu);
      relay.stop = true;
      relay.cv.notify_all();
    }
    return rc;
  });
  if (rc) return fail_all(ss, ns, rc);
  std::vector<uint32_t> crc(c.n_members, 0);
  for (const Wave& w : waves)
    for (uint32_t x = w.a; x < w.b; ++x) {
      uint32_t& m = crc[c.member_of[x]];
      m = inflate::crc_combine(m, piece_crc[x], w.wp[x - w.a + 1].off - w.wp[x - w.a].off);
    }
  for (uint32_t m = 0; m < c.n_members; ++m)
    if (crc[m] != c.trailers[m].crc) {
      char buf[160];
      snprintf(buf, sizeof buf, "gzip member %u: CRC-32 of the inflated bytes differs from the member's trailer", m);
      return fail_all(ss, ns, set_error(SGC_ERR_GZIP, buf));
    }
  for (uint32_t i = 0; i < ns; ++i) {
    ss[i]->member_pieces = starts.size();
    ss[i]->member_chain = c.n_chain;
    ss[i]->member_absorbed = c.absorbed;
    ss[i]->gzip_members = c.n_members;
  }
  return SGC_OK;
}

}  // namespace

// Frees the device side and detaches the stream from its counter; the handle itself stays valid.
void sgc::fastq_stream_release(sgc_fastq_stream* s) {
  if (!s || !s->counter) return;
  DeviceGuard guard(s->device);
  cudaStreamSynchronize(s->stream);
  auto& list = s->counter->fastq_streams;
  list.erase(std::remove(list.begin(), list.end(), s), list.end());
  s->counter = nullptr;
  s->failed = true;  // nothing more can be submitted
  for (void* p : {(void*)s->d_state, (void*)s->d_gz, (void*)s->d_text, (void*)s->d_spans, (void*)s->d_tail, (void*)s->d_seq_start,
                  (void*)s->d_seq_end, (void*)s->d_begin, (void*)s->d_outoff, (void*)s->d_counts, (void*)s->d_first, (void*)s->d_sums,
                  (void*)s->d_sym, (void*)s->d_window, (void*)s->d_cand, (void*)s->d_meta,
                  (void*)s->d_wave, (void*)s->d_crc, (void*)s->d_heads, (void*)s->d_is_member})
    scratch_free(p, s->pool, s->stream);
}

extern "C" {

int sgc_fastq_stream_create(sgc_counter* counter, uint32_t read_len, uint32_t span_start, uint32_t span_len,
                            sgc_fastq_stream** out) {
  if (!counter || !out) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  if (read_len != 0 && (span_len == 0 || (uint64_t)span_start + span_len > read_len || read_len + 4u > kHeadroom))
    return set_error(SGC_ERR_INVALID_ARG, "the span does not fit the read");
  DeviceGuard guard(counter->lib->device);
  sgc_fastq_stream* s = new sgc_fastq_stream();
  s->counter = counter;
  s->device = counter->lib->device;
  s->read_len = read_len;
  s->span_start = span_start;
  s->span_len = span_len;
  s->span_stride = (span_len + 7u) & ~7u;
  s->device = counter->lib->device;
  s->stream = counter->stream;  // one stream: the count of a wave follows its framing
  s->pool = scratch_pool(s->device);
  struct Cleanup {
    sgc_fastq_stream* s;
    ~Cleanup() {
      if (s) sgc_fastq_stream_destroy(s);
    }
  } cleanup{s};
  if (int rc = scratch_alloc(reinterpret_cast<void**>(&s->d_state), sizeof(StreamState), s->pool, s->stream)) return rc;
  if (int rc = scratch_alloc(reinterpret_cast<void**>(&s->d_tail), kHeadroom, s->pool, s->stream)) return rc;
  StreamState st0{};
  st0.bad_block = 0xFFFFFFFFu;
  SGC_CUDA_TRY(cudaMemcpyAsync(s->d_state, &st0, sizeof st0, cudaMemcpyHostToDevice, s->stream));
  SGC_CUDA_TRY(cudaStreamSynchronize(s->stream));
  // (every create sets the same kInflateSmem, so streams created on several threads at once cannot
  // lower the opt-in under each other's launches, as count.cu's ensure_smem_optin guards against)
  SGC_CUDA_TRY(cudaFuncSetAttribute(inflate_blocks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kInflateSmem));
  SGC_CUDA_TRY(cudaFuncSetAttribute(member_find_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kInflateSmem));
  SGC_CUDA_TRY(cudaFuncSetAttribute(member_boundary_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kInflateSmem));
  SGC_CUDA_TRY(cudaFuncSetAttribute(member_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kInflateSmem));
  counter->fastq_streams.push_back(s);
  cleanup.s = nullptr;
  *out = s;
  return SGC_OK;
}

void sgc_fastq_stream_destroy(sgc_fastq_stream* s) {
  if (!s) return;
  sgc::fastq_stream_release(s);
  delete s;
}

int sgc_fastq_stream_submit(sgc_fastq_stream* s, const uint8_t* gz, const uint64_t* block_begin, const uint32_t* block_isize,
                            uint32_t n_blocks) {
  return sgc_fastq_stream_submit_range(s, gz, block_begin, block_isize, n_blocks, 0, 0, 0);
}

int sgc_fastq_stream_submit_range(sgc_fastq_stream* s, const uint8_t* gz, const uint64_t* block_begin,
                                  const uint32_t* block_isize, uint32_t n_blocks, uint32_t head_skip, uint32_t tail_skip,
                                  int self_contained) {
  if (!s || !gz || !block_begin || !block_isize) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  if (s->failed || !s->counter) return set_error(SGC_ERR_INVALID_ARG, "the stream has failed or its counter is gone");
  if (n_blocks == 0) return SGC_OK;
  DeviceGuard guard(s->device);
  // where every block's text goes: the prefix sum of the ISIZE fields
  s->h_outoff.resize((size_t)n_blocks + 1);
  uint64_t n_text = 0;
  for (uint32_t i = 0; i < n_blocks; ++i) {
    if (block_begin[i + 1] <= block_begin[i]) return set_error(SGC_ERR_INVALID_ARG, "block offsets must increase");
    s->h_outoff[i] = kHeadroom + n_text;
    n_text += block_isize[i];
  }
  s->h_outoff[n_blocks] = kHeadroom + n_text;
  if (n_text >= (64ull << 30)) return set_error(SGC_ERR_BATCH_TOO_LARGE, "a wave of blocks must inflate to less than 64 GiB");
  if (s->read_len == 0 && n_text >= (1ull << 32) - 2 * kHeadroom)
    return set_error(SGC_ERR_BATCH_TOO_LARGE, "in variable-length mode a wave of blocks must inflate to less than 4 GiB");
  const uint64_t gz_bytes = block_begin[n_blocks] - block_begin[0];
  int rc = grow(&s->d_gz, &s->gz_cap, (size_t)gz_bytes + 64, s->pool, s->stream);  // the decoder prefetches up to 47 bytes past a block
  if (rc == SGC_OK) rc = grow(&s->d_text, &s->text_cap, (size_t)kHeadroom + n_text + 64, s->pool, s->stream);
  if (rc == SGC_OK) rc = grow(&s->d_begin, &s->begin_cap, (size_t)n_blocks + 1, s->pool, s->stream);
  if (rc == SGC_OK) rc = grow(&s->d_outoff, &s->outoff_cap, (size_t)n_blocks + 1, s->pool, s->stream);
  if (rc) return rc;
  SGC_CUDA_TRY(cudaMemcpyAsync(s->d_gz, gz + block_begin[0], gz_bytes, cudaMemcpyHostToDevice, s->stream));
  SGC_CUDA_TRY(cudaMemcpyAsync(s->d_begin, block_begin, ((size_t)n_blocks + 1) * 8, cudaMemcpyHostToDevice, s->stream));
  SGC_CUDA_TRY(cudaMemcpyAsync(s->d_outoff, s->h_outoff.data(), ((size_t)n_blocks + 1) * 8, cudaMemcpyHostToDevice, s->stream));
  inflate_blocks_kernel<<<(n_blocks + kInflateThreads - 1) / kInflateThreads, kInflateThreads, kInflateSmem, s->stream>>>(
      s->d_gz, s->d_begin, s->d_outoff, n_blocks, s->d_text, s->d_state);
  crc_blocks_kernel<<<(n_blocks + kCrcWarps - 1) / kCrcWarps, kCrcWarps * 32, 0, s->stream>>>(s->d_gz, s->d_begin, s->d_outoff,
                                                                                           n_blocks, s->d_text, s->d_state);
  SGC_CUDA_TRY(cudaGetLastError());
  if ((uint64_t)head_skip + tail_skip > n_text) return set_error(SGC_ERR_INVALID_ARG, "the skips exceed the wave's text");
  wave_begin_kernel<<<1, 1, 0, s->stream>>>(s->d_state, head_skip, self_contained ? 1u : 0u);
  rc = frame_and_count(s, n_text - tail_skip, s->blocks_total);
  if (rc) return rc;
  s->blocks_total += n_blocks;
  return SGC_OK;
}

int sgc_fastq_stream_finish(sgc_fastq_stream* s, uint64_t* n_records) {
  if (!s) return set_error(SGC_ERR_INVALID_ARG, "stream is NULL");
  if (s->failed || !s->counter) return set_error(SGC_ERR_INVALID_ARG, "the stream has failed or its counter is gone");
  DeviceGuard guard(s->device);
  StreamState st;
  SGC_CUDA_TRY(cudaMemcpyAsync(&st, s->d_state, sizeof st, cudaMemcpyDeviceToHost, s->stream));
  SGC_CUDA_TRY(cudaStreamSynchronize(s->stream));
  if (st.tail) {
    // the file does not end in a newline: the last line still counts (as the host reader has it)
    if (!s->d_text) return set_error(SGC_ERR_INVALID_ARG, "no text");
    SGC_CUDA_TRY(cudaMemsetAsync(s->d_text + kHeadroom, '\n', 1, s->stream));
    int rc = frame_and_count(s, 1, s->blocks_total);
    if (rc) return rc;
    SGC_CUDA_TRY(cudaMemcpyAsync(&st, s->d_state, sizeof st, cudaMemcpyDeviceToHost, s->stream));
    SGC_CUDA_TRY(cudaStreamSynchronize(s->stream));
    if (st.tail) {
      s->failed = true;
      return set_error(SGC_ERR_FASTQ_FORMAT, "truncated FASTQ record at the end of the input");
    }
  }
  if (n_records) *n_records = s->records_total;
  return SGC_OK;
}

int sgc_fastq_stream_submit_member(sgc_fastq_stream* s, const uint8_t* gz, uint64_t n_bytes) { return submit_plain_gzip(&s, 1, gz, n_bytes, false); }

int sgc_fastq_stream_submit_gzip(sgc_fastq_stream* s, const uint8_t* gz, uint64_t n_bytes) { return submit_plain_gzip(&s, 1, gz, n_bytes, true); }

int sgc_fastq_stream_submit_gzip_split(sgc_fastq_stream* const* streams, uint32_t n_streams, const uint8_t* gz, uint64_t n_bytes) {
  return submit_plain_gzip(streams, n_streams, gz, n_bytes, true);
}

// Every buffer a stream keeps is sized by `grow` (need + need / 4 when it grows), so none ever holds
// more than 1.25 times the most the stream needed of it; the needs follow from the wave's text.
int sgc_fastq_stream_scratch_bound(int bgzf, uint64_t gz_bytes, uint64_t text_bytes, uint32_t read_len, uint32_t span_len,
                                   uint64_t* bytes) {
  if (!bytes) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  if (read_len != 0 && (span_len == 0 || span_len > read_len)) return set_error(SGC_ERR_INVALID_ARG, "the span does not fit the read");
  auto grown = [](uint64_t need) { return need + need / 4; };
  const MemberParams p = member_params(read_len);
  // the text of one wave: a member wave stops before it passes p.wave_text, and DEFLATE inflates no byte
  // to more than 1032
  const uint64_t text = bgzf ? text_bytes : std::min(text_bytes ? text_bytes : gz_bytes * 1032, p.wave_text);
  const uint64_t region = kHeadroom + text;  // with the bytes carried in front of it
  const uint64_t chunks = region / kChunk + 2;
  uint64_t b = sizeof(StreamState) + kHeadroom;                             // d_state, d_tail
  b += grown(region + 64);                                                  // d_text
  b += 2 * grown((chunks + 1) * 4) + grown((chunks / 2048 + 2) * 4);        // d_counts, d_first, d_sums
  const uint64_t records = region / ((uint64_t)read_len + 6) + 2;           // a record takes its read and 6 more bytes
  b += read_len ? grown(records * ((span_len + 7u) & ~7u) + 256) : 2 * grown(records * 4);  // d_spans / d_seq_start, d_seq_end
  if (bgzf) {
    const uint64_t blocks = gz_bytes / 28 + 2;  // a BGZF block takes 28 bytes at least
    b += grown(gz_bytes + 64) + 2 * grown(blocks * 8);  // d_gz, d_begin, d_outoff
  } else {
    const uint64_t heads = gz_bytes / 256 + 4096 + 1;
    const uint64_t pieces = (gz_bytes + p.piece - 1) / p.piece + 1 + heads;  // candidates near the boundaries and behind headers
    b += grown(gz_bytes + 64) + grown(pieces * 8) + grown(heads * 8);                      // d_gz, d_cand, d_heads
    b += grown(pieces * sizeof(inflate::PieceMeta)) + grown(pieces);                       // d_meta, d_is_member
    b += grown((text + 1) * 2) + grown((pieces + 1) * sizeof(WavePiece)) + grown(pieces * 4);  // d_sym, d_wave, d_crc
    b += inflate::kWindow;                                                                 // d_window
  }
  // the pool's rounding of some twenty buffers, and the counter's skew replicas (at most 64 MB)
  *bytes = b + (128ull << 20);
  return SGC_OK;
}

int sgc_fastq_stream_gzip_members(const sgc_fastq_stream* s, uint64_t* members) {
  if (!s || !members) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  *members = s->gzip_members;
  return SGC_OK;
}

int sgc_fastq_stream_member_stats(const sgc_fastq_stream* s, uint64_t* pieces, uint64_t* chain, uint64_t* absorbed) {
  if (!s || !pieces || !chain || !absorbed) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  *pieces = s->member_pieces;
  *chain = s->member_chain;
  *absorbed = s->member_absorbed;
  return SGC_OK;
}

}  // extern "C"
