// count.cu — the per-read match-and-count loop (kernel K3) and the sgc_counter entry points.
//
// Replaces /root/reference/src/counter.rs:36-236 (Counter::new/count/assign/bounds/trim_*).
//
//   count_stream_kernel  : fixed-stride sequence lines.  Persistent warps stream tiles of 32
//                          reads HBM -> shared memory with 1-D bulk async copies (TMA engine,
//                          cp.async.bulk + mbarrier complete_tx) through a warp-private
//                          multi-stage ring.  Each lane lifts the words that cover its read's
//                          guide window out of shared memory, the stage goes straight back to
//                          the copy engine, and everything else runs from registers:
//                            fast path  window -> interleaved 2-bit key + ASCII validity ->
//                                       ONE 32-byte front-table bucket -> RED.64 on the guide;
//                            slow path  reads the fast path cannot settle (a mismatch, an N,
//                                       a shifted guide, junk; 10-20 %) are parked in a
//                                       warp-private shared-memory queue as (span words, read,
//                                       position).  32 at a time, with every lane busy, each
//                                       parked read tries ONE position of Counter::assign
//                                       against the seed index and, if that misses, goes back
//                                       on the queue for the next position.
//   count_lines_kernel   : any layout (variable-length lines via u32 offsets, unaligned
//                          buffers, tile remainders); one thread per read, the span lifted from
//                          global memory with 64-bit loads, same window arithmetic and tables.
//   count_shift_kernel   : staggered reads (max_shift S >= 2): the line kernel's layouts, every
//                          position offset + d, |d| <= S, through the parked queue.
//   unmatched_collect_kernel : the unmatched report (sgc_counter_set_unmatched_report): after a line or
//                          shift launch, the windows at the offset of the reads it left unmatched,
//                          tallied in an open-addressing table.
// Per-guide counts are 64-bit atomics in the L2-resident state vector; matched reads are
// accumulated in registers and flushed once per warp.
#include <algorithm>
#include <cstdlib>
#include <mutex>
#include <set>
#include <utility>
#include <vector>

#include "internal.h"

namespace sgc {
namespace {

// Geometry of the streaming kernel: every read has the same length, so it is the same for every
// read of a launch.  It is worked out on the host and travels as a kernel parameter, so that the
// kernel reads its fields straight from the constant bank instead of re-deriving them per tile.
// Positions are in STORED coordinates: for a reverse read the oriented window [o, o+k) is the
// stored window [n-o-k, n-o), Plus (o+1) is one byte EARLIER and Minus one byte later.
struct StreamGeom {
  int k, n, o;
  uint32_t with_perm;
  int win_src;             // stored position of the Centered window
  int lead;                // 1 if the span starts one byte before the Centered window
  uint32_t shift_bits[3];  // where the Centered / Plus / Minus window starts in the span, in bits
  uint32_t try_plus, try_minus;  // the position exists (its trim succeeds) and recursion is on
  int n_words;             // words holding the k window bytes
  uint32_t last_mask;
  uint32_t wild_byte;      // the stored byte the lookup sees as 'N'
};

inline StreamGeom make_geom(uint32_t k, uint32_t read_len, int offset, bool with_perm, bool reverse, bool recursion,
                            int rc_mode) {
  StreamGeom g;
  g.k = (int)k;
  g.n = (int)read_len;
  g.o = offset;
  g.with_perm = with_perm;
  // Plus is tried after a Centered miss if its trim succeeds; Minus after a Plus miss if
  // offset >= 1 (a failed trim returns, counter.rs:105-108: no Plus means no Minus either)
  g.try_plus = recursion && g.o + 1 + g.k <= g.n;
  g.try_minus = g.try_plus && g.o >= 1;
  g.win_src = reverse ? g.n - g.o - g.k : g.o;
  const int d_plus = reverse ? -1 : 1;  // stored displacement of the Plus window
  const bool before = (g.try_plus && d_plus < 0) || (g.try_minus && d_plus > 0);
  g.lead = before ? 1 : 0;
  g.shift_bits[0] = 8u * (uint32_t)g.lead;
  g.shift_bits[1] = 8u * (uint32_t)(g.lead + d_plus);
  g.shift_bits[2] = 8u * (uint32_t)(g.lead - d_plus);
  g.n_words = (g.k + 3) >> 2;
  g.last_mask = (g.k & 3) ? ((1u << (8 * (g.k & 3))) - 1) : ~0u;
  // under the fxread bit trick a reverse-complemented 'J' reads as 'N' (and 'N' as 'J')
  g.wild_byte = (reverse && rc_mode == SGC_RC_BITTRICK) ? (uint32_t)'J' : (uint32_t)'N';
  return g;
}

constexpr int kHotGuides = 4;

struct CountParams {
  LibView lib;
  const uint8_t* lines;
  const uint8_t* lines_end;  // lines + n_bytes: no load starts at or past it
  const uint32_t* line_off;  // NULL => fixed stride
  const uint32_t* line_end;  // with line_off: read r is lines[line_off[r] .. line_end[r]) — lines scattered in a
                             // larger text (the device ingest's variable-length mode); NULL => line_off[r + 1] - 1
  uint64_t n_reads;
  uint64_t first_read;       // index of the first read this launch handles
  uint32_t stride, read_len;
  int offset;
  uint8_t with_perm, reverse, recursion, rc_mode;
  unsigned long long* state;  // counts[n_guides], total, matched
  unsigned long long* rep;    // n_rep replicas of counts[n_guides] (see count_hit)
  uint32_t n_rep;             // power of two
  uint32_t n_guides;
  int32_t hot[kHotGuides];    // MODE 4: guides counted in registers (-2 = unused slot), see count_hit
  uint32_t off_base;          // line_off values are relative to lines - off_base (chunks of a host batch)
  int32_t* assign_out;
  uint32_t debug;  // SGC_DEBUG bit mask (tuning build only): 1 no count atomics, 2 no table probe, 4 no slow path
  uint32_t zero;   // always 0, and unknown to the compiler: see the buffer hand-back in step A
  StreamGeom geom; // streaming kernel only
};

// MODE 0: production (no per-read output, no tuning switches); 1: also writes the per-read
// assignment; 2: tuning build (-DSGC_TUNING) that honours SGC_DEBUG as well; 3: production with
// count replicas; 4: replicas + the sample's hot guides counted in registers.
struct HotCounts {
  uint32_t c[kHotGuides];
};

template <int MODE>
__device__ __forceinline__ void flush_matched(const CountParams& p, uint32_t matched, const HotCounts& hot) {
  matched = __reduce_add_sync(0xffffffffu, matched);
  if ((threadIdx.x & 31) == 0 && matched) atomicAdd(p.state + p.n_guides + 1, (unsigned long long)matched);
  if (MODE == 4) {
#pragma unroll
    for (int j = 0; j < kHotGuides; ++j) {
      const uint32_t h = __reduce_add_sync(0xffffffffu, hot.c[j]);
      if ((threadIdx.x & 31) == 0 && h) atomicAdd(p.state + p.hot[j], (unsigned long long)h);
    }
  }
  // total_reads counts every record this launch walked (counter.rs:223-226)
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(p.state + p.n_guides, (unsigned long long)p.n_reads);
}

// Count update (counter.rs:232-235): one RED.64 per matched read, fire and forget, resolved in L2.
//
// Skewed screens.  The reference's fold costs the same whatever the abundances are; here, when
// one guide carries a large share of the reads, its atomics serialise on ONE L2 address (about
// 1.4 G same-address REDs per second): measured on 50 M device-resident reads (tools/hot.py),
// 1 % of the reads on one guide cost +42 %, 10 % made the plain kernel 6.5x slower, 90 % 41x.
// Warp-level remedies were measured and rejected for the per-read path: grouping lanes with
// MATCH.ANY costs 20 % of the kernel on ordinary data, and even a one-entry register cache of the
// warp's hot guide found by vote + popcount costs 9 %, because any warp-collective forces the lanes
// to reconverge between the table probe and the RED.  Two things are nearly free per read:
//   replicas (MODE 3)  warp w counts into copy (w mod R) of the count vector; fold_replicas_kernel
//                      adds the copies into the state vector after the count kernel (R = 16: +2.5 %
//                      on ordinary data, 1.15 ms instead of 5.1 ms at 10 % skew);
//   hot guides (MODE 4) up to four guide indices known BEFORE the launch are compared per lane and
//                      counted in a register each (no vote: the lane just skips its RED), flushed
//                      once per warp.
// Which of them a counter uses is decided from a sample of its first batch (plan_skew below), so
// the caller does nothing; sgc_counter_set_replicas overrides the decision.
template <int MODE>
__device__ __forceinline__ void count_hit(const CountParams& p, unsigned long long* my_counts, int32_t hit,
                                          uint32_t& matched, HotCounts& hot) {
  if (hit >= 0) {
    ++matched;
    if (MODE == 4) {
      bool is_hot = false;
#pragma unroll
      for (int j = 0; j < kHotGuides; ++j) {
        const bool h = hit == p.hot[j];
        hot.c[j] += h;
        is_hot |= h;
      }
      if (!is_hot) atomicAdd(my_counts + hit, 1ull);
    } else {
      // without replicas the base is the kernel parameter itself (a uniform register)
      if (MODE != 2 || !(p.debug & 1u)) atomicAdd((MODE == 3 ? my_counts : p.state) + hit, 1ull);
    }
  }
}

// state[i] += sum over the replicas, which are left zero for the next launch
__global__ void fold_replicas_kernel(unsigned long long* __restrict__ state, unsigned long long* __restrict__ rep,
                                     uint32_t n, uint32_t n_rep) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long sum = 0;
  for (uint32_t r = 0; r < n_rep; ++r) {
    const unsigned long long v = rep[(size_t)r * n + i];
    if (v) {
      sum += v;
      rep[(size_t)r * n + i] = 0;
    }
  }
  if (sum) state[i] += sum;
}

// ------------------------------------------------------------------------------------------
// streaming kernel: warp-private rings
//
// Every warp owns a ring of kStages shared-memory buffers of ONE warp tile (32 reads =
// 32*stride bytes, always a multiple of 16) and one mbarrier per buffer; lane 0 keeps the
// ring full with 1-D bulk async copies, so warps never synchronise with each other and each
// SM keeps (warps x (kStages-1)) tiles in flight.
// ------------------------------------------------------------------------------------------
constexpr int kWarpReads = 32;
constexpr int kMaxStages = 4;
// How a ring buffer goes back to the copy engine (see step A of count_stream_kernel):
//   0  the refill's byte count depends on a warp vote over the words every lane loaded;
//   1  the documented producer/consumer form: every lane arrives on a per-buffer "empty"
//      mbarrier after its loads, the elected lane waits on it before it issues the copy.
#ifndef SGC_HANDBACK_MBAR
#define SGC_HANDBACK_MBAR 0
#endif
constexpr int kQueueCap = 64;  // <= 31 parked + 32 new
constexpr uint32_t kReadIdxBits = 30;  // queue word: position << 30 | read index

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// The ring is addressed with 32-bit shared-space addresses kept in registers: generic pointers
// would have the compiler rebuild the shared window base for every tile.
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
// 1-D bulk async copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::
          "r"(dst),
      "l"(src), "r"(bytes), "r"(bar), "l"(policy)
      : "memory");
}
// One lane of the (converged) warp.  With `elect.sync` ptxas knows that a single thread runs the
// guarded code and issues the bulk copy once from uniform registers; `lane == 0` made it wrap the
// copy in a loop over the active lanes with a broadcast of every operand.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
  return pred != 0;
}
template <int OFFSET>
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFFSET) : "memory");
  return v;
}
// W[I..N) = consecutive shared-memory words from `addr`
template <int I, int N>
struct LoadWords {
  static __device__ __forceinline__ void run(uint32_t addr, uint32_t* W) {
    W[I] = lds_u32<4 * I>(addr);
    LoadWords<I + 1, N>::run(addr, W);
  }
};
template <int N>
struct LoadWords<N, N> {
  static __device__ __forceinline__ void run(uint32_t, uint32_t*) {}
};

// bit 7 of every non-zero byte of x
__device__ __forceinline__ uint32_t nonzero_byte_flags(uint32_t x) {
  return (((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u;
}

// XOR of a word of four sequence bytes against the ASCII its 2-bit codes stand for
// (A 41, C 43, G 47: 41 | code << 1;  T 54: the same ^ 11): zero iff all four are A/C/G/T.
__device__ __forceinline__ uint32_t ascii_residue(uint32_t w) {
  const uint32_t is_t = (w >> 2) & ~(w >> 1) & 0x01010101u;  // code 2
  return ((w & 0xF9F9F9F9u) ^ (is_t * 0x11u)) ^ 0x41414141u;
}

// The k window bytes, given as NW window-aligned words, as interleaved key + residues.
// Returns the OR of the residues (zero iff every window byte is A/C/G/T).
template <int NW, bool WIDE>
__device__ __forceinline__ uint32_t pack_window(const uint32_t (&w)[NW], int n_words, uint32_t last_mask, Key& key,
                                                uint32_t (&x)[NW]) {
  uint32_t lo = 0, hi = 0, any = 0;
#pragma unroll
  for (int i = 0; i < NW; ++i) {
    x[i] = ascii_residue(w[i]);
    uint32_t c = (w[i] >> 1) & 0x03030303u;
    if (NW >= 5) {  // k >= 17: NW = ceil(k / 4), every word is in use and only the last can hold bytes past the window
      if (i == NW - 1) {
        x[i] &= last_mask;
        c &= last_mask;
      }
    } else {
      const uint32_t mk = i < n_words - 1 ? ~0u : (i == n_words - 1 ? last_mask : 0u);
      x[i] &= mk;
      c &= mk;
    }
    any |= x[i];
    if (i < 4)
      lo += c << (2 * i);
    else
      hi += c << (2 * (i - 4));
  }
  if (!WIDE) hi = (hi * 0x01041040u) >> 24;
  key = Key{lo, hi};
  return any;
}

// Parked reads: NW + 1 span words (the bytes from one before the Centered window on, so the
// entry does not depend on the lane that parked it) and position << 30 | read index.
template <int NW>
struct WarpQueueT {
  uint32_t w[NW + 1][kQueueCap];
  uint32_t tag[kQueueCap];
};

// One position of Counter::assign (counter.rs:111-117) for one parked read: the window that
// starts `shift` bits into the span S.
template <int NW, bool WIDE>
__device__ __forceinline__ int32_t try_position(const LibView& v, const IndexView& ix, const StreamGeom& g,
                                                const uint32_t (&S)[NW + 1], uint32_t shift, uint64_t policy,
                                                uint32_t debug = 0) {
  uint32_t w[NW], x[NW];
#pragma unroll
  for (int i = 0; i < NW; ++i) w[i] = __funnelshift_r(S[i], S[i + 1], shift);  // shift <= 16
  Key key;
  const uint32_t any = pack_window<NW, WIDE>(w, g.n_words, g.last_mask, key, x);
  if (debug & 8u) return (key.lo == 0x12345678u && any == 77u) ? 0 : kMiss;  // tuning: pack only, no lookups
  // Bytes outside A,C,G,T: the window still matches if there is exactly one and it is the
  // wildcard -> its parents (SURVEY.md A.3).  Both kinds of window go through ONE lookup so
  // that the lanes of a pass issue their directory loads together.
  int nbad = 0;
  uint32_t bad_word = 0, bad_flags = 0, bad_w = 0;
#pragma unroll
  for (int i = 0; i < NW; ++i) {
    const uint32_t f = nonzero_byte_flags(x[i]);
    nbad += __popc(f);
    if (f) {
      bad_word = (uint32_t)i;
      bad_flags = f;
      bad_w = w[i];
    }
  }
  const uint32_t byte = ((uint32_t)(__ffs((int)bad_flags) - 8) >> 3) & 3u;  // flags sit at bit 7 of their byte
  const bool wild = g.with_perm && nbad == 1 && ((bad_w >> (8 * byte)) & 0xFFu) == g.wild_byte;
  // stored base position; the keys of the reverse index are in stored order too
  const uint32_t pos = wild ? 4 * bad_word + byte : 0u;
  Key hole{0u, 0u};
  if (wild) {
    hole = base_field(pos, WIDE);
    key.lo &= ~hole.lo;
    key.hi &= ~hole.hi;
  }
  // NW = 5 and the wide kernels only ever see k >= 17: the index's parts are the fixed ones
  constexpr bool kFixedParts = NW == 5 || WIDE;
  static_assert(kFixedPartsMinK <= 17, "k = 17..30 must use the fixed parts");
  return lookup_token<WIDE, kFixedParts>(v, ix, g.with_perm, key, hole,
                                         wild ? part_of_base_t<kFixedParts>(v.parts, pos) : -1, any == 0 || wild,
                                         nullptr, policy);
}

// ------------------------------------------------------------------------------------------
// line kernel: any layout (variable-length lines through u32 offsets, unaligned buffers, tile
// remainders of the streaming kernel).  The same arithmetic as the streaming kernel with a
// PER-READ geometry: a warp takes 32 consecutive reads, every lane lifts the NW + 1 span words of
// its read straight from global memory with 64-bit loads at the read's own alignment (consecutive
// lanes hold consecutive reads, so a warp touches each 32-byte sector of its lines at most once
// and DRAM traffic stays below the algorithmic bytes), the Centered window goes through the
// front table, and what that does not settle is parked in a warp-private shared-memory queue and
// drained 32 reads at a time through the seed index, exactly like the streaming kernel's slow
// path; a parked entry carries its read's geometry (lead byte, Plus / Minus exist) in its tag.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t ldg_stream_u64(const uint64_t* p, uint64_t policy) {
  uint64_t v;
  // L1 allocation stays on: the NL loads of a lane fall into one or two sectors
  asm volatile("ld.global.nc.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(policy));
  return v;
}

// tag of a parked read of the line kernel
constexpr uint32_t kLineIdxBits = 27;  // at most 2^27 reads per launch
constexpr uint32_t kLineLead = 1u << 27, kLinePlus = 1u << 28, kLineMinus = 1u << 29;
constexpr int kLineWarps = 8;

template <int NW, bool WIDE>
__global__ void __launch_bounds__(kLineWarps * 32) count_lines_kernel(CountParams p) {
  __shared__ WarpQueueT<NW> queues[kLineWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WarpQueueT<NW>* q = &queues[warp];
  uint32_t matched = 0;
  HotCounts hot{};
  const uint64_t table_policy = l2_evict_last_policy();
  const uint64_t line_policy = l2_evict_first_policy();
  const int k = (int)p.lib.k;
  const StreamGeom& g = p.geom;  // n_words, last_mask, with_perm, wild_byte: the same for every read
  const IndexView& ix = p.reverse ? p.lib.rev : p.lib.fwd;
  const uint32_t gwarp = blockIdx.x * kLineWarps + warp, gwarps = gridDim.x * kLineWarps;
  unsigned long long* my_counts = p.rep + (size_t)(gwarp & (p.n_rep - 1)) * p.n_guides;
  const int d_plus = p.reverse ? -1 : 1;  // stored displacement of the Plus window
  constexpr int NL = (4 * NW + 11 + 7) / 8;  // 64-bit loads that cover NW + 2 words at any alignment
  static_assert(2 * NL >= NW + 3, "span words");
  uint32_t qn = 0;  // parked reads (warp-uniform)

  auto settle = [&](int32_t hit, uint32_t ridx) {
    if (p.assign_out) p.assign_out[p.first_read + ridx] = hit;
    count_hit<4>(p, my_counts, hit, matched, hot);
  };
  auto drain = [&](bool all) {
    while (qn >= 32 || (all && qn > 0)) {
      const uint32_t cnt = qn < 32 ? qn : 32;
      qn -= cnt;
      int next = -1;
      uint32_t S[NW + 1], tag = 0;
      if ((uint32_t)lane < cnt) {
        const uint32_t e = qn + lane;
#pragma unroll
        for (int i = 0; i < NW + 1; ++i) S[i] = q->w[i][e];
        tag = q->tag[e];
        const uint32_t pos = tag >> 30, ridx = tag & ((1u << kLineIdxBits) - 1);
        const int lead = (tag & kLineLead) ? 1 : 0;
        const uint32_t shift = 8u * (uint32_t)(pos == 0 ? lead : (pos == 1 ? lead + d_plus : lead - d_plus));
        const int32_t hit = try_position<NW, WIDE>(p.lib, ix, g, S, shift, table_policy);
        if (hit == kMiss) next = pos == 0 ? ((tag & kLinePlus) ? 1 : -1) : (pos == 1 && (tag & kLineMinus) ? 2 : -1);
        if (next < 0) settle(hit, ridx);
      }
      __syncwarp();
      const uint32_t pm = __ballot_sync(0xffffffffu, next >= 0);
      if (pm) {
        if (next >= 0) {
          const uint32_t e = qn + __popc(pm & ((1u << lane) - 1));
#pragma unroll
          for (int i = 0; i < NW + 1; ++i) q->w[i][e] = S[i];
          q->tag[e] = ((uint32_t)next << 30) | (tag & 0x3FFFFFFFu);
        }
        qn += __popc(pm);
      }
      __syncwarp();
    }
  };

  const uint64_t n_tiles = (p.n_reads + 31) / 32;
  for (uint64_t t = gwarp; t < n_tiles; t += gwarps) {
    const uint64_t i = t * 32 + lane;  // read of this lane, relative to the launch
    int park = -1;                     // position to resume at, or -1 when the read is settled
    uint32_t S[NW + 1] = {}, flags = 0;
    if (i < p.n_reads) {
      const uint64_t r = p.first_read + i;
      uint64_t start;
      int n;
      if (p.line_end) {
        start = p.line_off[r];
        n = (int)(p.line_end[r] - p.line_off[r]);
      } else if (p.line_off) {
        const uint32_t a = p.line_off[r], b = p.line_off[r + 1];
        start = a - p.off_base;
        n = (int)(b - a) - 1;
      } else {
        start = r * p.stride;
        n = (int)p.read_len;
      }
      // Centered/Null: offset; Plus: offset+1; Minus: offset-1 (counter.rs:164-174).  A failed trim
      // RETURNS (counter.rs:105-108,175-176): no Centered window, no match; no Plus, no Minus either.
      if (p.offset + k > n) {
        settle(kMiss, (uint32_t)i);
      } else {
        const bool try_plus = p.recursion && p.offset + 1 + k <= n;
        const bool try_minus = try_plus && p.offset >= 1;
        const int win_src = p.reverse ? n - p.offset - k : p.offset;  // stored coordinates (see StreamGeom)
        const int lead = ((try_plus && d_plus < 0) || (try_minus && d_plus > 0)) ? 1 : 0;
        flags = (lead ? kLineLead : 0u) | (try_plus ? kLinePlus : 0u) | (try_minus ? kLineMinus : 0u);
        const uint8_t* sb = p.lines + start + win_src - lead;  // first span byte
        const uint64_t* a8 = reinterpret_cast<const uint64_t*>((uintptr_t)sb & ~(uintptr_t)7);
        uint32_t R[2 * NL];
#pragma unroll
        for (int j = 0; j < NL; ++j) {
          // never a load that starts at or past the end of the buffer (bytes past the read only
          // ever reach masked-off positions of a window)
          const uint64_t v =
              reinterpret_cast<const uint8_t*>(a8 + j) < p.lines_end ? ldg_stream_u64(a8 + j, line_policy) : 0ull;
          R[2 * j] = (uint32_t)v;
          R[2 * j + 1] = (uint32_t)(v >> 32);
        }
        const uint32_t sh = (uint32_t)((uintptr_t)sb & 7u);
        const bool odd = (sh & 4u) != 0;
        const uint32_t bits = (sh & 3u) * 8u;
#pragma unroll
        for (int j = 0; j < NW + 1; ++j) {
          const uint32_t w0 = odd ? R[j + 1] : R[j], w1 = odd ? R[j + 2] : R[j + 1];
          S[j] = __funnelshift_r(w0, w1, bits);
        }
        // Centered window: front table first (one sector decides ~80 % of the reads)
        uint32_t w[NW], x[NW];
#pragma unroll
        for (int j = 0; j < NW; ++j) w[j] = __funnelshift_r(S[j], S[j + 1], 8u * (uint32_t)lead);
        Key key;
        const uint32_t any = pack_window<NW, WIDE>(w, g.n_words, g.last_mask, key, x);
        park = 0;
        if (any == 0) {
          uint64_t b[4];
          load_bucket(ix.front + (size_t)(front_hash(key.lo, key.hi) >> p.lib.front_shift) * 4, b, table_policy);
          bool found, flagged;
          int32_t idx;
          if (!WIDE) {
            uint32_t sel = 0;
#pragma unroll
            for (int j = 3; j >= 0; --j)
              if ((uint32_t)b[j] == key.lo) sel = (uint32_t)(b[j] >> 32);
            const uint32_t want = key.hi | (uint32_t)(kFrontOccupied >> 32);
            found = ((sel ^ want) & (0xFFu | (uint32_t)(kFrontOccupied >> 32))) == 0;
            idx = (int32_t)(sel >> (kFrontIdxShift - 32));
            flagged = (b[0] & kFrontFlag) != 0;
          } else {
            const uint64_t probe = ((uint64_t)key.hi << 32) | key.lo;
            const bool m0 = b[0] == probe && (b[1] & kFrontOccupied), m1 = b[2] == probe && (b[3] & kFrontOccupied);
            found = m0 || m1;
            idx = (int32_t)((m0 ? b[1] : b[3]) >> kFrontIdxShift);
            flagged = (b[1] & kFrontFlag) != 0;
          }
          if (found) {
            park = -1;
            settle(idx, (uint32_t)i);
          } else if (!flagged && !g.with_perm) {
            // not a member and no Permuter: Centered is decided, go on with Plus if there is one
            park = try_plus ? 1 : -1;
            if (park < 0) settle(kMiss, (uint32_t)i);
          }
        } else if (!g.with_perm) {
          // a byte outside A,C,G,T and no Permuter: Centered is decided
          park = try_plus ? 1 : -1;
          if (park < 0) settle(kMiss, (uint32_t)i);
        }
      }
    }
    const uint32_t pm = __ballot_sync(0xffffffffu, park >= 0);
    if (pm) {
      if (park >= 0) {
        const uint32_t e = qn + __popc(pm & ((1u << lane) - 1));
#pragma unroll
        for (int j = 0; j < NW + 1; ++j) q->w[j][e] = S[j];
        q->tag[e] = ((uint32_t)park << 30) | flags | (uint32_t)i;
      }
      qn += __popc(pm);
      __syncwarp();
    }
    drain(false);
  }
  drain(true);
  flush_matched<4>(p, matched, hot);
}

// ------------------------------------------------------------------------------------------
// shift kernel: staggered reads (sgc_counter_set_max_shift, S = 2..16).  The windows at
// offset + d, d = 0, +1, -1, ..., +S, -S in the coordinates of the read the reference trims (the
// reverse complement of the whole read in Reverse), the first that yields a guide wins, and a
// window that does not fit the read is skipped.  Any layout, like the line kernel: a warp takes
// 32 consecutive reads, every lane works out its read's positions from the read's length, lifts
// the span that holds them (k + 2S bytes at most) with 64-bit loads and parks it; the warp-private
// queue is drained 32 reads at a time, each trying ONE position through the seed index
// (try_position) and going back on the queue for its next position after a miss.  A position is
// the NW + 1 parked words around it and a bit shift.
// ------------------------------------------------------------------------------------------
constexpr int kMaxShift = 16;
constexpr uint32_t kShiftIdxBits = 26;  // tag: position index (0 .. 2S) << 26 | read index

template <int NW>
struct ShiftQueueT {
  // span words: k + 2S <= 4 NW + 32 bytes; a window starts at most 2S bytes into the span and its
  // NW + 1 words go up to word 8 + NW
  uint32_t w[NW + 9][kQueueCap];
  uint32_t tag[kQueueCap];
  uint32_t range[kQueueCap];  // the read's positions: (dlo + S) | (dhi + S) << 8
};

// displacement of position index j (0, +1, -1, +2, -2, ...)
__device__ __forceinline__ int shift_of(int j) { return (j & 1) ? (j + 1) >> 1 : -(j >> 1); }

template <int NW, bool WIDE>
__global__ void __launch_bounds__(kLineWarps * 32) count_shift_kernel(CountParams p, int max_shift) {
  constexpr int SW = NW + 9;
  __shared__ ShiftQueueT<NW> queues[kLineWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  ShiftQueueT<NW>* q = &queues[warp];
  uint32_t matched = 0;
  HotCounts hot{};
  const uint64_t table_policy = l2_evict_last_policy();
  const uint64_t line_policy = l2_evict_first_policy();
  const int k = (int)p.lib.k, S = max_shift, n_pos = 2 * max_shift + 1;
  const StreamGeom& g = p.geom;  // n_words, last_mask, with_perm, wild_byte: the same for every read
  const IndexView& ix = p.reverse ? p.lib.rev : p.lib.fwd;
  const uint32_t gwarp = blockIdx.x * kLineWarps + warp, gwarps = gridDim.x * kLineWarps;
  unsigned long long* my_counts = p.rep + (size_t)(gwarp & (p.n_rep - 1)) * p.n_guides;
  constexpr int NL = (4 * SW + 7 + 7) / 8;  // 64-bit loads that cover SW words at any alignment
  static_assert(2 * NL >= SW + 2, "span words");
  constexpr uint32_t kIdxMask = (1u << kShiftIdxBits) - 1;
  uint32_t qn = 0;  // parked reads (warp-uniform)

  auto settle = [&](int32_t hit, uint32_t ridx) {
    if (p.assign_out) p.assign_out[p.first_read + ridx] = hit;
    count_hit<4>(p, my_counts, hit, matched, hot);
  };
  // the position index after j whose window fits the read, or n_pos
  auto next_position = [&](int j, int dlo, int dhi) {
    for (++j; j < n_pos; ++j) {
      const int d = shift_of(j);
      if (d >= dlo && d <= dhi) break;
    }
    return j;
  };
  auto drain = [&](bool all) {
    while (qn >= 32 || (all && qn > 0)) {
      const uint32_t cnt = qn < 32 ? qn : 32;
      qn -= cnt;
      int next = -1;
      uint32_t U[SW], tag = 0, range = 0;
      if ((uint32_t)lane < cnt) {
        const uint32_t e = qn + lane;
        tag = q->tag[e];
        range = q->range[e];
        const int j = (int)(tag >> kShiftIdxBits);
        const int dlo = (int)(range & 0xFFu) - S, dhi = (int)(range >> 8) - S, d = shift_of(j);
        const int b = p.reverse ? dhi - d : d - dlo;  // first window byte in the span (stored order)
        uint32_t T[NW + 1];
#pragma unroll
        for (int i = 0; i < NW + 1; ++i) T[i] = q->w[(b >> 2) + i][e];
        const int32_t hit = try_position<NW, WIDE>(p.lib, ix, g, T, 8u * (uint32_t)(b & 3), table_policy);
        if (hit == kMiss) {
          next = next_position(j, dlo, dhi);
          if (next >= n_pos) next = -1;
        }
        if (next < 0) {
          settle(hit, tag & kIdxMask);
        } else {
#pragma unroll
          for (int i = 0; i < SW; ++i) U[i] = q->w[i][e];
        }
      }
      __syncwarp();  // every lane has read its entry before any slot is overwritten
      const uint32_t pm = __ballot_sync(0xffffffffu, next >= 0);
      if (pm) {
        if (next >= 0) {
          const uint32_t e = qn + __popc(pm & ((1u << lane) - 1));
#pragma unroll
          for (int i = 0; i < SW; ++i) q->w[i][e] = U[i];
          q->tag[e] = ((uint32_t)next << kShiftIdxBits) | (tag & kIdxMask);
          q->range[e] = range;
        }
        qn += __popc(pm);
      }
      __syncwarp();
    }
  };

  const uint64_t n_tiles = (p.n_reads + 31) / 32;
  for (uint64_t t = gwarp; t < n_tiles; t += gwarps) {
    const uint64_t i = t * 32 + lane;  // read of this lane, relative to the launch
    int park = -1;                     // first position index whose window fits, or -1
    uint32_t span[SW] = {}, range = 0;
    if (i < p.n_reads) {
      const uint64_t r = p.first_read + i;
      uint64_t start;
      int n;
      if (p.line_end) {
        start = p.line_off[r];
        n = (int)(p.line_end[r] - p.line_off[r]);
      } else if (p.line_off) {
        const uint32_t a = p.line_off[r], b = p.line_off[r + 1];
        start = a - p.off_base;
        n = (int)(b - a) - 1;
      } else {
        start = r * p.stride;
        n = (int)p.read_len;
      }
      // the displacements whose window fits: [dlo, dhi], possibly empty
      const int dlo = p.offset < S ? -p.offset : -S;
      const int dhi = min(S, n - k - p.offset);
      if (dlo <= dhi) {
        park = dhi >= 0 ? 0 : next_position(0, dlo, dhi);
        range = (uint32_t)(dlo + S) | ((uint32_t)(dhi + S) << 8);
        const int span_bytes = k + dhi - dlo;
        const int first = p.reverse ? n - p.offset - dhi - k : p.offset + dlo;  // stored coordinates
        const uint8_t* sb = p.lines + start + first;
        const uint64_t* a8 = reinterpret_cast<const uint64_t*>((uintptr_t)sb & ~(uintptr_t)7);
        const uint32_t sh = (uint32_t)((uintptr_t)sb & 7u);
        const int need = ((int)sh + span_bytes + 4 + 7) >> 3;  // loads that reach one word past the span
        uint32_t R[2 * NL];
#pragma unroll
        for (int j = 0; j < NL; ++j) {
          // never a load that starts at or past the end of the buffer (bytes past the read only
          // ever reach masked-off positions of a window)
          const uint64_t v = j < need && reinterpret_cast<const uint8_t*>(a8 + j) < p.lines_end
                                 ? ldg_stream_u64(a8 + j, line_policy)
                                 : 0ull;
          R[2 * j] = (uint32_t)v;
          R[2 * j + 1] = (uint32_t)(v >> 32);
        }
        const bool odd = (sh & 4u) != 0;
        const uint32_t bits = (sh & 3u) * 8u;
#pragma unroll
        for (int j = 0; j < SW; ++j) {
          const uint32_t w0 = odd ? R[j + 1] : R[j], w1 = odd ? R[j + 2] : R[j + 1];
          span[j] = __funnelshift_r(w0, w1, bits);
        }
      } else {
        settle(kMiss, (uint32_t)i);  // no window fits the read
      }
    }
    const uint32_t pm = __ballot_sync(0xffffffffu, park >= 0);
    if (pm) {
      if (park >= 0) {
        const uint32_t e = qn + __popc(pm & ((1u << lane) - 1));
#pragma unroll
        for (int j = 0; j < SW; ++j) q->w[j][e] = span[j];
        q->tag[e] = ((uint32_t)park << kShiftIdxBits) | (uint32_t)i;
        q->range[e] = range;
      }
      qn += __popc(pm);
      __syncwarp();
    }
    drain(false);
  }
  drain(true);
  flush_matched<4>(p, matched, hot);
}

// ------------------------------------------------------------------------------------------
// unmatched report (sgc_counter_set_unmatched_report): after a count launch of the line or shift
// kernel, the reads it left unmatched (assignment -1) are tallied by their window at the offset,
// trimmed[o, o + k) in library orientation, into an open-addressing table of {key, count} slots.
// A key is the window packed 2-bit, first base in the highest bits (A 0, C 1, G 2, T 3), so keys of
// one k sort like the window bytes; the empty key is all ones (no window has bits 60..63 set).
// A slot is claimed once and never freed: a window that is in the table has every one of its reads
// counted there, and one that found its probe range full is refused for good (tally[3], overflow).
// ------------------------------------------------------------------------------------------
constexpr unsigned long long kEmptyKey = ~0ull;
constexpr int kUnmatchedProbes = 128;  // linear probes before a window is refused
constexpr int kUnmatchedWarps = 8;
enum { kTallyUnmatched, kTallyShort, kTallyNonAcgt, kTallyOverflow, kTallyCompacted, kTallyWords };

__global__ void unmatched_clear_kernel(ulonglong2* __restrict__ table, uint64_t capacity) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < capacity; i += (uint64_t)gridDim.x * blockDim.x)
    table[i] = make_ulonglong2(kEmptyKey, 0ull);
}

// One warp per 32 consecutive reads of the launch p (the read layouts of the line kernel); the
// assignment of read i of the launch is p.assign_out[p.first_read + i].
__global__ void __launch_bounds__(kUnmatchedWarps * 32)
    unmatched_collect_kernel(CountParams p, ulonglong2* __restrict__ table, uint64_t capacity,
                             unsigned long long* __restrict__ tally) {
  const int lane = threadIdx.x & 31;
  const uint32_t gwarp = blockIdx.x * kUnmatchedWarps + (threadIdx.x >> 5), gwarps = gridDim.x * kUnmatchedWarps;
  const int k = (int)p.lib.k, o = p.offset;
  const uint64_t line_policy = l2_evict_first_policy();
  const int probes = capacity < (uint64_t)kUnmatchedProbes ? (int)capacity : kUnmatchedProbes;
  uint32_t n_unmatched = 0, n_short = 0, n_bad = 0, n_over = 0;
  const uint64_t n_tiles = (p.n_reads + 31) / 32;
  for (uint64_t t = gwarp; t < n_tiles; t += gwarps) {
    const uint64_t i = t * 32 + lane;
    bool have_key = false;
    unsigned long long key = 0;
    if (i < p.n_reads && p.assign_out[p.first_read + i] < 0) {
      ++n_unmatched;
      const uint64_t r = p.first_read + i;
      uint64_t start;
      int n;
      if (p.line_end) {
        start = p.line_off[r];
        n = (int)(p.line_end[r] - p.line_off[r]);
      } else if (p.line_off) {
        const uint32_t a = p.line_off[r], b = p.line_off[r + 1];
        start = a - p.off_base;
        n = (int)(b - a) - 1;
      } else {
        start = r * p.stride;
        n = (int)p.read_len;
      }
      if (o + k > n) {
        ++n_short;  // the Centered trim fails: no window
      } else {
        // the stored window: [o, o + k) forward, [n - o - k, n - o) reversed and complemented
        const uint8_t* sb = p.lines + start + (p.reverse ? n - o - k : o);
        const uint64_t* a8 = reinterpret_cast<const uint64_t*>((uintptr_t)sb & ~(uintptr_t)7);
        const uint32_t sh = (uint32_t)((uintptr_t)sb & 7u);
        const int need = ((int)sh + k + 7) >> 3;
        uint64_t R[5];
#pragma unroll
        for (int j = 0; j < 5; ++j)
          R[j] = j < need && reinterpret_cast<const uint8_t*>(a8 + j) < p.lines_end ? ldg_stream_u64(a8 + j, line_policy) : 0ull;
        uint64_t W[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) W[j] = sh ? (R[j] >> (8 * sh)) | (R[j + 1] << (64 - 8 * sh)) : R[j];
        // stored bytes in order, codes A 0 C 1 G 2 T 3; complement and reversal come after (a byte
        // outside A, C, G, T stays outside under either rc_mode, and A, C, G, T complement alike)
        bool bad = false;
#pragma unroll
        for (int j = 0; j < (int)kMaxK; ++j) {
          if (j < k) {
            const uint32_t b = (uint32_t)(W[j >> 3] >> (8 * (j & 7))) & 0xFFu;
            bad |= b != 'A' && b != 'C' && b != 'G' && b != 'T';
            key = (key << 2) | (unsigned long long)((b == 'C') + 2 * (b == 'G') + 3 * (b == 'T'));
          }
        }
        if (bad) {
          ++n_bad;
        } else {
          if (p.reverse) {  // reverse the 2-bit groups, complement every base
            key = __brevll(key);
            key = ((key >> 1) & 0x5555555555555555ull) | ((key & 0x5555555555555555ull) << 1);
            key = (key >> (64 - 2 * k)) ^ ((1ull << (2 * k)) - 1);
          }
          have_key = true;
        }
      }
    }
    // one table update per distinct window of the warp: a window that holds most of the reads
    // costs one atomic per warp, not one per read
    const uint32_t want = __ballot_sync(0xffffffffu, have_key);
    const uint32_t group = have_key ? __match_any_sync(want, key) : 0u;
    if (have_key && lane == __ffs((int)group) - 1) {
      const unsigned long long cnt = (unsigned long long)__popc(group);
      uint64_t slot = __umul64hi(key * 0x9E3779B97F4A7C15ull, capacity);
      bool done = false;
      for (int q = 0; q < probes && !done; ++q) {
        unsigned long long* kp = &table[slot].x;
        unsigned long long cur = __ldcg(kp);
        if (cur == kEmptyKey) cur = atomicCAS(kp, kEmptyKey, key);
        if (cur == kEmptyKey || cur == key) {
          atomicAdd(&table[slot].y, cnt);
          done = true;
        }
        slot = slot + 1 == capacity ? 0 : slot + 1;
      }
      if (!done) n_over += (uint32_t)cnt;
    }
  }
  n_unmatched = __reduce_add_sync(0xffffffffu, n_unmatched);
  n_short = __reduce_add_sync(0xffffffffu, n_short);
  n_bad = __reduce_add_sync(0xffffffffu, n_bad);
  n_over = __reduce_add_sync(0xffffffffu, n_over);
  if (lane == 0) {
    if (n_unmatched) atomicAdd(tally + kTallyUnmatched, (unsigned long long)n_unmatched);
    if (n_short) atomicAdd(tally + kTallyShort, (unsigned long long)n_short);
    if (n_bad) atomicAdd(tally + kTallyNonAcgt, (unsigned long long)n_bad);
    if (n_over) atomicAdd(tally + kTallyOverflow, (unsigned long long)n_over);
  }
}

// The occupied slots of table[0, n) to out[0, ...), in any order; tally[kTallyCompacted] counts them
// (zero before the launch).
__global__ void unmatched_compact_kernel(const ulonglong2* __restrict__ table, uint64_t n, ulonglong2* __restrict__ out,
                                         unsigned long long* __restrict__ tally) {
  const int lane = threadIdx.x & 31;
  for (uint64_t base = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) & ~31ull; base < n;
       base += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t i = base + lane;
    const ulonglong2 s = i < n ? table[i] : make_ulonglong2(kEmptyKey, 0ull);
    const bool full = s.x != kEmptyKey;
    const uint32_t m = __ballot_sync(0xffffffffu, full);
    unsigned long long at = 0;
    if (lane == 0 && m) at = atomicAdd(tally + kTallyCompacted, (unsigned long long)__popc(m));
    at = __shfl_sync(0xffffffffu, at, 0);
    if (full) out[at + __popc(m & ((1u << lane) - 1))] = s;
  }
}

// NW = words that hold the k window bytes: 4 (k <= 16, the number of words in use is read from the
// geometry), or exactly ceil(k / 4) = 5 (k = 17..20, the common guide lengths), 6, 7 or 8.
template <int NW, bool WIDE, int MODE>
__global__ void __launch_bounds__(384, 2) count_stream_kernel(const CountParams p, uint32_t n_wtiles, int n_stages,
                                                              uint32_t stage_bytes) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int lane = threadIdx.x & 31;
  // read from lane 0 so that the compiler knows the warp index — and the ring addresses, tile
  // indices and source pointers derived from it — to be warp-uniform: they then live in uniform
  // registers and the bulk copy is issued without a lane-by-lane broadcast loop
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int warps_per_cta = blockDim.x >> 5;
  // shared layout: [warp][stage] tile buffers | [warp][stage] mbarriers | [warp] queues
  uint8_t* my_tiles = smem + (size_t)warp * n_stages * stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)warps_per_cta * n_stages * stage_bytes);
  uint64_t* my_bar = bars + warp * (2 * kMaxStages);  // [0, kMaxStages) full, [kMaxStages, 2 kMaxStages) empty
  WarpQueueT<NW>* q = reinterpret_cast<WarpQueueT<NW>*>(bars + warps_per_cta * (2 * kMaxStages)) + warp;

  const uint32_t tile_bytes = kWarpReads * p.stride;  // multiple of 16
  const uint32_t gwarp = blockIdx.x * warps_per_cta + warp;
  const uint32_t gwarps = gridDim.x * warps_per_cta;
  const uint64_t src_step = (uint64_t)gwarps * tile_bytes;
  const uint8_t* next_src = p.lines + (uint64_t)gwarp * tile_bytes;  // source of the next tile to request

  const uint32_t tiles_sm = smem_u32(my_tiles), bars_sm = smem_u32(my_bar);
  const uint64_t policy = l2_evict_first_policy();
  uint32_t requested = gwarp;  // tile index of the next request (n_wtiles + gwarps < 2^32); every lane keeps it
  if (lane == 0) {
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(&my_bar[s], 1);
      mbar_init(&my_bar[kMaxStages + s], 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncwarp();
  for (int s = 0; s < n_stages; ++s) {
    if (requested < n_wtiles) {
      if (elect_one()) {
        mbar_expect_tx(bars_sm + 8u * (uint32_t)s, tile_bytes);
        bulk_load(tiles_sm + (uint32_t)s * stage_bytes, next_src, tile_bytes, bars_sm + 8u * (uint32_t)s, policy);
      }
      requested += gwarps;
      next_src += src_step;
    }
  }

  // every read has the same length n, so the geometry is uniform; the host sends reads whose
  // Centered window does not fit (every one of them fails its first trim) to the generic kernel
  const StreamGeom& g = p.geom;
  const uint32_t sbyte = (uint32_t)lane * p.stride + (uint32_t)(g.win_src - g.lead);  // first span byte
  const uint32_t lane_off = sbyte & ~3u;  // byte offset of this lane's first span word in a tile
  const uint32_t off_bits = (sbyte & 3u) * 8;
  const uint32_t win_bits = off_bits + g.shift_bits[0];  // 0..32: where the Centered window starts in W
  const IndexView& ix = p.reverse ? p.lib.rev : p.lib.fwd;
  const uint64_t* __restrict__ front = ix.front;
  const uint32_t front_shift = p.lib.front_shift;
  const uint64_t table_policy = l2_evict_last_policy();
  const uint32_t debug = MODE == 2 ? p.debug : 0u;
  // what a read needs after its Centered window is not a library member
  const bool centered_again = g.with_perm;  // the one-mismatch lookup of the same window
  const bool any_next = centered_again || g.try_plus;

  uint32_t matched = 0;
  HotCounts hot{};
  unsigned long long* my_counts = p.rep + (size_t)(gwarp & (p.n_rep - 1)) * p.n_guides;
  uint32_t qn = 0;  // parked reads (warp-uniform)
  int s = 0;
  uint32_t parity = 0;
  uint32_t cur_tile = tiles_sm, cur_bar = bars_sm;  // stage s of the ring

  // A tile is handled in two steps one loop iteration apart, so that the front-table sector of
  // tile j+1 travels from L2 while tile j's parked reads are drained and tile j+2 is lifted:
  //   step A  wait for the tile, lift the span, hand the buffer back, pack the Centered window;
  //           carried to step B: span words, key, validity
  //   fetch   the front bucket of that window (issued right after step B of the tile before)
  //   step B  compare the bucket, count or park
  struct Pending {
    uint32_t S[NW + 1];  // span words from one byte before the Centered window (lane independent)
    Key key;
    uint32_t any;  // non-zero: some window byte is not A/C/G/T
  };
  // The front bucket of the tile step B handles next, in flight.  ONE register set: step B
  // consumes it and the load for the following tile is issued right behind, so it flies through
  // the drain and the next step A.  (Carrying it inside Pending made the `current = next` copy at
  // the loop tail wait for a load that had just been issued.)
  uint64_t bucket[4];
  auto fetch_bucket = [&](const Pending& pd) {
    if (pd.any == 0 && !(MODE == 2 && (debug & 2u)))
      load_bucket(front + (size_t)(front_hash(pd.key.lo, pd.key.hi) >> front_shift) * 4, bucket, table_policy);
  };
  // a read is settled: its assignment (tests), its guide's counter
  auto settle = [&](int32_t hit, uint32_t ridx) {
    if ((MODE == 1 || MODE == 2) && p.assign_out) p.assign_out[ridx] = hit;
    count_hit<MODE>(p, my_counts, hit, matched, hot);
  };
  auto step_a = [&](Pending& pd) {
    mbar_wait(cur_bar, parity);
    uint32_t W[NW + 2];
    LoadWords<0, NW + 2>::run(cur_tile + lane_off, W);
    // The buffer may be refilled once every lane's loads have RETURNED (the refill is an
    // async-proxy write, the loads are generic-proxy reads: nothing orders them by itself).  The
    // byte count of the refill is made to DEPEND on a warp vote over a value computed from all
    // the loaded words (`& p.zero` keeps it what it was): the copy cannot be issued, in program
    // order or after any rescheduling by ptxas, before the data is in registers.  No CTA-wide
    // membar per tile.
#if SGC_HANDBACK_MBAR
    // consumer release / producer acquire on the buffer's "empty" barrier: the arrive is ordered
    // after this lane's loads, the copy is issued after all 32 arrivals have been observed
    if (requested < n_wtiles) {
      mbar_arrive(cur_bar + 8u * kMaxStages);
      if (elect_one()) {
        mbar_wait(cur_bar + 8u * kMaxStages, parity);
        mbar_expect_tx(cur_bar, tile_bytes);
        bulk_load(cur_tile, next_src, tile_bytes, cur_bar, policy);
      }
      requested += gwarps;
      next_src += src_step;
    }
#else
    uint32_t allw = W[0];
#pragma unroll
    for (int i = 1; i < NW + 2; ++i) allw &= W[i];
    const uint32_t arrived = __ballot_sync(0xffffffffu, allw != 0) & p.zero;
    if (requested < n_wtiles) {
      if (elect_one()) {
        mbar_expect_tx(cur_bar, tile_bytes + arrived);
        bulk_load(cur_tile, next_src, tile_bytes + arrived, cur_bar, policy);
      }
      requested += gwarps;
      next_src += src_step;
    }
#endif
    cur_tile += stage_bytes;
    cur_bar += 8;
    if (++s == n_stages) {
      s = 0;
      parity ^= 1u;
      cur_tile = tiles_sm;
      cur_bar = bars_sm;
    }
#pragma unroll
    for (int i = 0; i < NW + 1; ++i) pd.S[i] = __funnelshift_r(W[i], W[i + 1], off_bits);
    uint32_t w[NW], x[NW];
#pragma unroll
    for (int i = 0; i < NW; ++i) w[i] = __funnelshift_r(pd.S[i], pd.S[i + 1], g.shift_bits[0]);
    pd.any = pack_window<NW, WIDE>(w, g.n_words, g.last_mask, pd.key, x);
  };
  auto step_b = [&](const Pending& pd, uint32_t read_idx) {
    // park = position to resume at (0 Centered, 1 Plus), or -1 when the read is settled
    int park = 0;
    if (pd.any == 0) {
      bool found, flagged;
      int32_t hit;
      if (MODE == 2 && (debug & 2u)) {
        found = true;
        flagged = false;
        hit = (int32_t)((pd.key.lo ^ pd.key.hi) % p.n_guides);
      } else {
        const uint64_t(&b)[4] = bucket;
        if (!WIDE) {
          // the slot whose lo word matches (the build keeps them distinct within a bucket)
          uint32_t sel = 0;
#pragma unroll
          for (int j = 3; j >= 0; --j)
            if ((uint32_t)b[j] == pd.key.lo) sel = (uint32_t)(b[j] >> 32);
          const uint32_t want = pd.key.hi | (uint32_t)(kFrontOccupied >> 32);
          found = ((sel ^ want) & (0xFFu | (uint32_t)(kFrontOccupied >> 32))) == 0;
          hit = (int32_t)(sel >> (kFrontIdxShift - 32));
          flagged = (b[0] & kFrontFlag) != 0;
        } else {
          const uint64_t probe = ((uint64_t)pd.key.hi << 32) | pd.key.lo;
          const bool m0 = b[0] == probe && (b[1] & kFrontOccupied), m1 = b[2] == probe && (b[3] & kFrontOccupied);
          found = m0 || m1;
          hit = (int32_t)((m0 ? b[1] : b[3]) >> kFrontIdxShift);
          flagged = (b[1] & kFrontFlag) != 0;
        }
      }
      if (found) {
        park = -1;
        settle(hit, read_idx);
      } else if (!flagged && !centered_again) {
        // not a member and no Permuter: Centered is decided, go on with Plus if there is one
        park = g.try_plus ? 1 : -1;
        if (park < 0) settle(kMiss, read_idx);
      }
    } else if (!any_next) {
      park = -1;  // a bad byte, no Permuter, no recursion
      settle(kMiss, read_idx);
    }
    if (MODE == 2 && (debug & 4u)) park = -1;
    const uint32_t pm = __ballot_sync(0xffffffffu, park >= 0);
    if (pm) {
      if (park >= 0) {
        const uint32_t e = qn + __popc(pm & ((1u << lane) - 1));
#pragma unroll
        for (int i = 0; i < NW + 1; ++i) q->w[i][e] = pd.S[i];
        q->tag[e] = ((uint32_t)park << kReadIdxBits) | read_idx;
      }
      qn += __popc(pm);
      __syncwarp();
    }
  };
  // Drain: 32 parked reads try one position each; a miss goes back on the queue for its next
  // position.  Between tiles the queue is brought below 32 so a whole tile can park; once the
  // tiles are done it is emptied.
  auto drain = [&](bool all) {
    while (qn >= 32 || (all && qn > 0)) {
      const uint32_t cnt = qn < 32 ? qn : 32;
      qn -= cnt;
      int next = -1;  // position to retry at, or -1
      uint32_t S[NW + 1], tag = 0;
      if ((uint32_t)lane < cnt) {
        const uint32_t e = qn + lane;
#pragma unroll
        for (int i = 0; i < NW + 1; ++i) S[i] = q->w[i][e];
        tag = q->tag[e];
        const uint32_t pos = tag >> kReadIdxBits, ridx = tag & ((1u << kReadIdxBits) - 1);
        const uint32_t shift = pos == 0 ? g.shift_bits[0] : (pos == 1 ? g.shift_bits[1] : g.shift_bits[2]);
        const int32_t hit = try_position<NW, WIDE>(p.lib, ix, g, S, shift, table_policy, debug);
        if (hit == kMiss) next = pos == 0 ? (g.try_plus ? 1 : -1) : (pos == 1 && g.try_minus ? 2 : -1);
        if (next < 0) settle(hit, ridx);
      }
      __syncwarp();  // every lane has read its entry before any slot is overwritten
      const uint32_t pm = __ballot_sync(0xffffffffu, next >= 0);
      if (pm) {
        if (next >= 0) {
          const uint32_t e = qn + __popc(pm & ((1u << lane) - 1));
#pragma unroll
          for (int i = 0; i < NW + 1; ++i) q->w[i][e] = S[i];
          q->tag[e] = ((uint32_t)next << kReadIdxBits) | (tag & ((1u << kReadIdxBits) - 1));
        }
        qn += __popc(pm);
      }
      __syncwarp();
    }
  };

  uint32_t read_idx = gwarp * kWarpReads + lane;
  const uint32_t read_step = gwarps * kWarpReads;
  uint32_t t = gwarp;
  Pending cur;
  bool have_cur = t < n_wtiles;
  if (have_cur) {
    step_a(cur);
    fetch_bucket(cur);
  }
  while (have_cur) {
    Pending nxt;
    const bool have_nxt = t + gwarps < n_wtiles;
    if (have_nxt) step_a(nxt);
    step_b(cur, read_idx);
    if (have_nxt) fetch_bucket(nxt);
    drain(false);
    cur = nxt;
    have_cur = have_nxt;
    t += gwarps;
    read_idx += read_step;
  }
  drain(true);
  flush_matched<MODE>(p, matched, hot);
}

}  // namespace
}  // namespace sgc

// ------------------------------------------------------------------------------------------
// skew plan: which guides (if any) carry a large share of a sample's reads
// ------------------------------------------------------------------------------------------
namespace sgc {
namespace {

struct TopGuides {
  unsigned long long packed[kHotGuides];  // count << 32 | guide index, descending
  unsigned long long total;               // reads counted so far
};

// One block: the kHotGuides largest entries of counts[0..n).  Every thread keeps its own sorted
// short list over a strided slice; lane 0 of every warp merges its warp's lists, thread 0 the
// warps' (two short serial merges instead of one long one).
__device__ __forceinline__ void top_insert(unsigned long long (&top)[kHotGuides], unsigned long long v) {
#pragma unroll
  for (int j = 0; j < kHotGuides; ++j)
    if (v > top[j]) {
      const unsigned long long t = top[j];
      top[j] = v;
      v = t;
    }
}
__global__ void __launch_bounds__(1024) top_guides_kernel(const unsigned long long* __restrict__ counts, uint32_t n,
                                                         TopGuides* out) {
  __shared__ unsigned long long cand[1024 * kHotGuides];
  __shared__ unsigned long long warp_top[32 * kHotGuides];
  unsigned long long best[kHotGuides] = {};
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
    const unsigned long long v = counts[i];
    if (v) top_insert(best, (v << 32) | i);
  }
#pragma unroll
  for (int j = 0; j < kHotGuides; ++j) cand[threadIdx.x * kHotGuides + j] = best[j];
  __syncthreads();
  const uint32_t warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  if ((threadIdx.x & 31) == 0) {
    unsigned long long top[kHotGuides] = {};
    for (uint32_t c = 0; c < 32 * kHotGuides; ++c) top_insert(top, cand[warp * 32 * kHotGuides + c]);
#pragma unroll
    for (int j = 0; j < kHotGuides; ++j) warp_top[warp * kHotGuides + j] = top[j];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long top[kHotGuides] = {};
    for (uint32_t c = 0; c < n_warps * kHotGuides; ++c) top_insert(top, warp_top[c]);
    for (int j = 0; j < kHotGuides; ++j) out->packed[j] = top[j];
    out->total = counts[n];
  }
}

}  // namespace
}  // namespace sgc

// ------------------------------------------------------------------------------------------
// sgc_counter
// ------------------------------------------------------------------------------------------
using namespace sgc;

namespace {

constexpr size_t kChunkBytes = 64ull << 20;
constexpr uint64_t kChunkAlignReads = 256;  // chunk starts stay 16-byte aligned for any stride
constexpr uint64_t kSkewSampleReads = 65536;   // reads of the first batch the skew plan looks at
constexpr uint64_t kSkewMinBatch = 4 * kSkewSampleReads;  // smaller first batches are not worth a plan
constexpr uint64_t kUnmatchedLaunchReads = kAssignScratchReads;  // reads per launch with the unmatched report (its scratch)
constexpr uint64_t kUnmatchedMaxCapacity = 1ull << 26;

// Tuning switches (SGC_DEBUG, SGC_WARPS, SGC_CTAS, SGC_STAGES, SGC_CARVEOUT, SGC_REPLICAS) exist only
// in the tuning build (make tuning: -DSGC_TUNING -> libsgcount_cuda_tuning.so); the production
// library never reads them.  SGC_MAX_LAUNCH_TILES is the one variable both builds honour: it only
// changes how a batch is cut into launches (the tests use it to exercise the launch splitting
// without 2^30 reads), never what is counted.
#ifdef SGC_TUNING
int env_int(const char* name, int fallback) {
  const char* v = getenv(name);
  return v && *v ? atoi(v) : fallback;
}
#else
constexpr int env_int(const char*, int fallback) { return fallback; }
#endif
long long env_ll(const char* name, long long fallback) {
  const char* v = getenv(name);
  return v && *v ? atoll(v) : fallback;
}

CountParams make_params(const sgc_counter* c, const uint8_t* d_lines, const uint32_t* d_off, uint32_t stride,
                        uint32_t read_len, int32_t* d_assign) {
  CountParams p{};
  p.lib = c->lib->view();
  p.lines = d_lines;
  p.line_off = d_off;
  p.stride = stride;
  p.read_len = read_len;
  p.offset = (int)c->offset;
  p.with_perm = c->lib->with_perm;
  p.reverse = c->is_reverse != 0;
  p.recursion = c->recursion != 0;
  p.rc_mode = (uint8_t)c->rc_mode;
  p.state = c->d_state;
  p.rep = c->n_rep > 1 ? c->d_rep : c->d_state;
  p.n_rep = c->n_rep;
  p.n_guides = c->lib->n;
  for (int j = 0; j < kHotGuides; ++j) p.hot[j] = c->hot[j];
  p.assign_out = d_assign;
  p.debug = (uint32_t)env_int("SGC_DEBUG", 0);
  p.geom = make_geom(c->lib->k, read_len, (int)c->offset, c->lib->with_perm, c->is_reverse != 0, c->recursion != 0,
                     c->rc_mode);
  return p;
}

struct StreamConfig {
  int warps = 0, stages = 0, ctas_per_sm = 0;
};
size_t stream_smem_bytes(const StreamConfig& c, uint32_t stage_bytes, size_t queue_bytes) {
  return (size_t)c.warps * ((size_t)c.stages * stage_bytes + 2 * kMaxStages * sizeof(uint64_t) + queue_bytes);
}
// How many warps per CTA and CTAs per SM.  Two things were measured to matter (DESIGN.md): the
// number of resident warps, and the L1 that the shared-memory carve-out leaves for the scattered
// table loads — the carve-out comes in steps, and the step that leaves 28 KB costs 15 % where
// the ones that leave 60 KB or more cost 1 % or nothing.  Every (warps, CTAs) pair that fits is
// scored as resident warps x that factor; 2 ring buffers per warp (a third is worth less than
// the L1 it takes).  SGC_WARPS / SGC_STAGES / SGC_CTAS pin the choice (tuning build only).
StreamConfig pick_stream_config(uint32_t stage_bytes, size_t queue_bytes) {
  const size_t sm_budget = 227 * 1024;
  const int pin_warps = env_int("SGC_WARPS", 0), pin_ctas = env_int("SGC_CTAS", 0);
  const int stages = std::max(2, std::min(env_int("SGC_STAGES", 2), kMaxStages));
  StreamConfig best{};
  double best_score = 0;
  for (int ctas = 2; ctas >= 1; --ctas) {
    if (pin_ctas && ctas != pin_ctas) continue;
    for (int warps = 12; warps >= 1; --warps) {
      if (pin_warps >= 1 && pin_warps <= 12 && warps != pin_warps) continue;
      const StreamConfig c{warps, stages, ctas};
      const size_t total = (stream_smem_bytes(c, stage_bytes, queue_bytes) + 1024) * ctas;
      if (total > sm_budget) continue;
      // carve-out steps of sm_100: ... 132, 164, 196, 228 KB out of 256 KB
      const double l1_factor = total <= 164 * 1024 ? 1.0 : (total <= 196 * 1024 ? 0.99 : 0.85);
      const double score = warps * ctas * l1_factor;
      if (score > best_score) {
        best_score = score;
        best = c;
      }
    }
  }
  return best;
}

// The opt-in shared-memory limit of a kernel is a per-device, process-wide attribute: it is
// raised ONCE per (device, kernel) to the most any launch can ask for, never per launch — two
// counters with different read lengths on two host threads would otherwise lower it under each
// other between the set and the launch.
constexpr int kMaxOptinSmem = 227 * 1024;
int ensure_smem_optin(int device, const void* kernel) {
  static std::mutex mu;
  static std::set<std::pair<int, const void*>> done;
  std::lock_guard<std::mutex> lk(mu);
  if (done.count({device, kernel})) return SGC_OK;
  SGC_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxOptinSmem));
  done.insert({device, kernel});
  return SGC_OK;
}

using StreamKernel = void (*)(const CountParams, uint32_t, int, uint32_t);
#ifdef SGC_TUNING
#define SGC_TUNING_KERNEL(NW, WIDE) count_stream_kernel<NW, WIDE, 2>
#else
#define SGC_TUNING_KERNEL(NW, WIDE) nullptr
#endif
#define SGC_FAMILY(NW, WIDE)                                                                               \
  {                                                                                                        \
    count_stream_kernel<NW, WIDE, 0>, count_stream_kernel<NW, WIDE, 1>, SGC_TUNING_KERNEL(NW, WIDE),       \
        count_stream_kernel<NW, WIDE, 3>, count_stream_kernel<NW, WIDE, 4>                                 \
  }
const StreamKernel kStreamKernels[5][5] = {SGC_FAMILY(4, false), SGC_FAMILY(5, false), SGC_FAMILY(6, true),
                                           SGC_FAMILY(7, true), SGC_FAMILY(8, true)};

// Enqueue the kernels for one device-resident batch.
// Reads [first, n_reads) of the batch.
int launch_count(sgc_counter* c, const uint8_t* d_lines, uint64_t n_bytes, const uint32_t* d_off, uint32_t off_base,
                 uint32_t stride, uint32_t read_len, uint64_t first, uint64_t n_reads, int32_t* d_assign,
                 cudaStream_t stream) {
  if (n_reads <= first) return SGC_OK;
  if (c->lib->opaque) {  // byte-keyed library (opaque.cu): one simple kernel, whatever the layout
    c->last.kernel = 2;
    c->last.block = 256;
    c->last.replicas = 1;
    c->last.hot_guides = 0;
    c->last.launches_total += 1;
    return opaque_count(c, d_lines, d_off, off_base, stride, read_len, first, n_reads, d_assign ? d_assign : c->pair_assign,
                        stream, &c->last.grid);
  }
  CountParams p = make_params(c, d_lines, d_off, stride, read_len, d_assign);
  p.off_base = off_base;
  p.lines_end = d_lines + n_bytes;
  p.line_end = c->gather_end;  // set only by count_gathered_lines
  uint64_t done = first;
  const uint64_t launches_before = c->last.launches_total;
  c->last = sgc_launch_info{};
  c->last.launches_total = launches_before;
  c->last.kernel = 1;
  c->last.replicas = c->n_rep;
  for (int j = 0; j < kHotGuides; ++j) c->last.hot_guides += c->hot[j] >= 0;
  // staggered reads (max_shift >= 2) take the shift kernel whatever the layout
  const bool shifted = c->max_shift >= 2;
  // streaming kernel: fixed stride, 16-byte aligned base, whole warp tiles, < 2^32 reads per
  // launch, and a Centered window that fits (otherwise every read fails its first trim)
  const uint32_t tile_bytes = kWarpReads * stride;
  const uint32_t stage_bytes = (tile_bytes + 48 + 15) & ~15u;  // +48: span words may run past the tile
  // a counter with the unmatched report, or one mate of a pair counter, counts through the line or shift
  // kernel, which write assignments
  const bool report = c->um_capacity != 0;
  const bool to_scratch = report || c->pair_assign;
  const bool stageable = !shifted && !to_scratch && d_off == nullptr && ((uintptr_t)d_lines & 15u) == 0 && stride >= read_len &&
                         (uint64_t)c->offset + c->lib->k <= read_len;
  // kernel family by the words that hold the k window bytes: narrow keys 4 (k <= 16) or 5
  // (k = 17..20, the common guide lengths); wide keys 6 (k = 21..24), 7 (k = 25..28) or 8 (k = 29, 30)
  const int family = c->lib->k <= 16 ? 0 : (int)((c->lib->k + 3) / 4) - 4;
  static const size_t family_queue_bytes[5] = {sizeof(WarpQueueT<4>), sizeof(WarpQueueT<5>), sizeof(WarpQueueT<6>),
                                               sizeof(WarpQueueT<7>), sizeof(WarpQueueT<8>)};
  const size_t queue_bytes = family_queue_bytes[family];
  StreamConfig cfg = stageable ? pick_stream_config(stage_bytes, queue_bytes) : StreamConfig{};
  // whole tiles only, and never a bulk copy that would run past n_bytes; one launch handles at
  // most 2^30 reads (the queue words keep a 30-bit read index)
  const bool first_aligned = ((first * stride) & 15u) == 0;
  uint64_t tiles_left = stageable && cfg.stages && first_aligned
                            ? std::min((n_reads - first) / kWarpReads, (n_bytes - first * stride) / tile_bytes)
                            : 0;
  uint64_t max_tiles = (1ull << kReadIdxBits) / kWarpReads - 65536;
  if (const long long cap = env_ll("SGC_MAX_LAUNCH_TILES", 0); cap > 0) max_tiles = std::min<uint64_t>(max_tiles, cap);
  const bool any_hot = c->last.hot_guides > 0;
  while (tiles_left > 0) {
    const uint64_t n_wtiles = std::min(tiles_left, max_tiles);
    // replicas and hot guides are production features: with a per-read output or tuning switches
    // the counts go straight to the state vector
    int mode = d_assign ? 1 : (any_hot ? 4 : (c->n_rep > 1 ? 3 : 0));
    if (p.debug) mode = 2;
    StreamKernel kernel = kStreamKernels[family][mode];
    const size_t smem = stream_smem_bytes(cfg, stage_bytes, queue_bytes);
    int rc = ensure_smem_optin(c->lib->device, (const void*)kernel);
    if (rc) return rc;
#ifdef SGC_TUNING
    if (const int carve = env_int("SGC_CARVEOUT", -1); carve >= 0)  // shared-memory share of the L1, percent
      SGC_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
#endif
    uint64_t grid = (uint64_t)c->lib->sm_count * cfg.ctas_per_sm;  // persistent: every CTA resident
    const uint64_t ctas_needed = (n_wtiles + cfg.warps - 1) / cfg.warps;
    if (grid > ctas_needed) grid = ctas_needed;
    CountParams q = p;  // this launch's slice: read indices are relative to it
    q.lines = d_lines + done * stride;
    q.assign_out = d_assign ? d_assign + done : nullptr;
    q.n_reads = n_wtiles * kWarpReads;
    q.first_read = 0;
    if (mode == 1 || mode == 2) {  // counts go straight to the state vector
      q.rep = q.state;
      q.n_rep = 1;
    }
    kernel<<<(unsigned)grid, cfg.warps * 32, smem, stream>>>(q, (uint32_t)n_wtiles, cfg.stages, stage_bytes);
    SGC_CUDA_TRY(cudaGetLastError());
    done += n_wtiles * kWarpReads;
    tiles_left -= n_wtiles;
    c->last.grid = (uint32_t)grid;
    c->last.block = cfg.warps * 32;
    c->last.smem_bytes = (uint32_t)smem;
    c->last.kernel = 0;
    c->last.launches_total += 1;
  }
  const bool lines_only = done == first;
  // the shift kernel's queue tags keep a 26-bit read index; SGC_MAX_LAUNCH_TILES cuts its launches too
  uint64_t shift_launch_reads = 1ull << kShiftIdxBits;
  if (const long long cap = env_ll("SGC_MAX_LAUNCH_TILES", 0); cap > 0)
    shift_launch_reads = std::min<uint64_t>(shift_launch_reads, (uint64_t)cap * kWarpReads);
  // with the unmatched report a launch's assignments go to the counter's scratch of kUnmatchedLaunchReads
  const uint64_t report_launch_reads = assign_scratch_reads();
  if (shifted) c->last.kernel = 3;
  while (done < n_reads) {  // what the streaming kernel did not take; at most 2^27 reads per launch
    p.first_read = done;
    p.n_reads = std::min<uint64_t>(n_reads - done, to_scratch ? report_launch_reads
                                                              : (shifted ? shift_launch_reads : 1ull << kLineIdxBits));
    CountParams q = p;
    // a pair counter's batch is one chunk of its scratch: read r's assignment goes to pair_assign[r]
    if (c->pair_assign && !d_assign) q.assign_out = c->pair_assign;
    if (report && !d_assign) {  // the launch's reads start at index 0 of the scratch
      q.first_read = 0;
      if (q.line_off) {
        q.line_off += done;
        if (q.line_end) q.line_end += done;
      } else {
        q.lines += done * stride;
      }
      q.assign_out = c->d_um_assign;
    }
    uint64_t blocks = (p.n_reads + 32 * kLineWarps - 1) / (32 * kLineWarps);
    const uint64_t cap = (uint64_t)c->lib->sm_count * 8;
    if (blocks > cap) blocks = cap;
    using LineKernel = void (*)(CountParams);
    static const LineKernel line_kernels[5] = {count_lines_kernel<4, false>, count_lines_kernel<5, false>,
                                               count_lines_kernel<6, true>, count_lines_kernel<7, true>,
                                               count_lines_kernel<8, true>};
    using ShiftKernel = void (*)(CountParams, int);
    static const ShiftKernel shift_kernels[5] = {count_shift_kernel<4, false>, count_shift_kernel<5, false>,
                                                 count_shift_kernel<6, true>, count_shift_kernel<7, true>,
                                                 count_shift_kernel<8, true>};
    if (shifted)
      shift_kernels[family]<<<(unsigned)blocks, 32 * kLineWarps, 0, stream>>>(q, (int)c->max_shift);
    else
      line_kernels[family]<<<(unsigned)blocks, 32 * kLineWarps, 0, stream>>>(q);
    SGC_CUDA_TRY(cudaGetLastError());
    if (report) {
      uint64_t collect_blocks = (q.n_reads + 32 * kUnmatchedWarps - 1) / (32 * kUnmatchedWarps);
      collect_blocks = std::min<uint64_t>(collect_blocks, (uint64_t)c->lib->sm_count * 8);
      unmatched_collect_kernel<<<(unsigned)collect_blocks, 32 * kUnmatchedWarps, 0, stream>>>(
          q, static_cast<ulonglong2*>(c->d_um_table), c->um_capacity, c->d_um_tally);
      SGC_CUDA_TRY(cudaGetLastError());
      c->last.launches_total += 1;
    }
    if (lines_only) {
      c->last.grid = (uint32_t)blocks;
      c->last.block = 32 * kLineWarps;
    }
    c->last.launches_total += 1;
    done += p.n_reads;
  }
  if (c->n_rep > 1) {
    fold_replicas_kernel<<<(c->lib->n + 255) / 256, 256, 0, stream>>>(c->d_state, c->d_rep, c->lib->n, c->n_rep);
    SGC_CUDA_TRY(cudaGetLastError());
    c->last.launches_total += 1;
  }
  return SGC_OK;
}

// stream: the stream the counter's kernels run on (a pair counter runs both mates on the first mate's)
int alloc_replicas(sgc_counter* c, uint32_t replicas, cudaStream_t stream) {
  // a power of two, at most 64 copies and 64 MB
  uint32_t n_rep = 1;
  while (n_rep * 2 <= replicas && n_rep < 64 && (size_t)n_rep * 2 * c->lib->n * sizeof(uint64_t) <= (64u << 20))
    n_rep *= 2;
  if (n_rep == c->n_rep) return SGC_OK;
  SGC_CUDA_TRY(cudaStreamSynchronize(stream));  // the replicas are zero between launches
  cudaFree(c->d_rep);
  c->d_rep = nullptr;
  c->n_rep = 1;
  if (n_rep > 1) {
    SGC_CUDA_TRY(cudaMalloc(&c->d_rep, (size_t)n_rep * c->lib->n * sizeof(uint64_t)));
    SGC_CUDA_TRY(cudaMemsetAsync(c->d_rep, 0, (size_t)n_rep * c->lib->n * sizeof(uint64_t), stream));
    c->n_rep = n_rep;
  }
  return SGC_OK;
}

// Skew plan of a counter, made once, on its first large batch: the first kSkewSampleReads reads
// are counted (into the state vector, like any others), the four largest counters are read
// back, and
//   top share >= 1/256  -> the rest of the sample is counted into 16 replicas (or as many as
//                          64 MB hold);
//   every guide with a share >= 1 % is counted in registers (count_hit, MODE 4).
// Costs one extra launch boundary and one stream synchronisation per counter (= per sample or
// sample shard).  The counts do not depend on the plan.  Returns the reads already counted.
int plan_skew(sgc_counter* c, const uint8_t* d_lines, uint64_t n_bytes, const uint32_t* d_off, uint32_t off_base,
              uint32_t stride, uint32_t read_len, uint64_t n_reads, cudaStream_t stream, uint64_t* counted) {
  c->skew_planned = true;
  const uint64_t sample = std::min<uint64_t>(n_reads, kSkewSampleReads);
  if (!c->d_top) SGC_CUDA_TRY(cudaMalloc(&c->d_top, sizeof(TopGuides)));
  int rc = launch_count(c, d_lines, n_bytes, d_off, off_base, stride, read_len, 0, sample, nullptr, stream);
  if (rc) return rc;
  *counted = sample;
  top_guides_kernel<<<1, 1024, 0, stream>>>(c->d_state, c->lib->n, static_cast<TopGuides*>(c->d_top));
  SGC_CUDA_TRY(cudaGetLastError());
  TopGuides top;
  SGC_CUDA_TRY(cudaMemcpyAsync(&top, c->d_top, sizeof top, cudaMemcpyDeviceToHost, stream));
  SGC_CUDA_TRY(cudaStreamSynchronize(stream));
  // shares among everything this counter has seen so far (earlier small batches included)
  const uint64_t seen = std::max<uint64_t>(top.total, 1), top_count = top.packed[0] >> 32;
  if (top_count * 256 < seen) return SGC_OK;  // no guide stands out
  rc = alloc_replicas(c, 16, stream);
  if (rc) return rc;
  int n_hot = 0;
  for (int j = 0; j < kHotGuides; ++j)
    if ((top.packed[j] >> 32) * 100 >= seen) c->hot[n_hot++] = (int32_t)(uint32_t)top.packed[j];
  return SGC_OK;
}

// launch_count preceded, for the counter's first large batch, by the skew plan
int count_batch(sgc_counter* c, const uint8_t* d_lines, uint64_t n_bytes, const uint32_t* d_off, uint32_t off_base,
                uint32_t stride, uint32_t read_len, uint64_t n_reads, int32_t* d_assign, cudaStream_t stream) {
  uint64_t counted = 0;
  c->submitted = true;
  if (c->auto_skew && !c->skew_planned && !d_assign && n_reads >= kSkewMinBatch && !c->lib->opaque) {
    int rc = plan_skew(c, d_lines, n_bytes, d_off, off_base, stride, read_len, n_reads, stream, &counted);
    if (rc) return rc;
  }
  return launch_count(c, d_lines, n_bytes, d_off, off_base, stride, read_len, counted, n_reads, d_assign, stream);
}

}  // namespace

// Reads scattered in a device-resident text: read r is d_text[d_start[r] .. d_end[r]) (gzip.cu: the
// sequence lines of FASTQ records in place, no packing).  Counted by the line kernel.
int sgc::count_gathered_lines(sgc_counter* c, const uint8_t* d_text, uint64_t n_bytes, const uint32_t* d_start,
                              const uint32_t* d_end, uint64_t n_reads) {
  if (n_reads == 0) return SGC_OK;
  DeviceGuard guard(c->device);
  c->gather_end = d_end;
  const int rc = count_batch(c, d_text, n_bytes, d_start, 0, 0, 0, n_reads, nullptr, c->stream);
  c->gather_end = nullptr;
  return rc;
}

int sgc::check_batch(const sgc_counter* c, const uint8_t* lines, uint64_t n_bytes, const uint32_t* line_off,
                uint32_t stride, uint32_t read_len, uint64_t n_reads) {
  if (!c) return set_error(SGC_ERR_INVALID_ARG, "counter is NULL");
  if (n_reads == 0) return SGC_OK;
  if (!lines) return set_error(SGC_ERR_INVALID_ARG, "lines is NULL");
  if (line_off) {
    if (n_bytes >= (1ull << 32)) return set_error(SGC_ERR_BATCH_TOO_LARGE, "variable-length batch must stay below 4 GiB");
  } else {
    if (stride == 0 || read_len > stride) return set_error(SGC_ERR_INVALID_ARG, "need 0 < read_len <= stride");
    if ((n_reads - 1) * (uint64_t)stride + read_len > n_bytes)
      return set_error(SGC_ERR_INVALID_ARG, "fixed-stride batch does not fit n_bytes");
  }
  return SGC_OK;
}

uint64_t sgc::assign_scratch_reads() {
  uint64_t n = kUnmatchedLaunchReads;
  if (const long long cap = env_ll("SGC_MAX_LAUNCH_TILES", 0); cap > 0) n = std::min<uint64_t>(n, (uint64_t)cap * kWarpReads);
  return n;
}

int sgc::count_into_scratch(sgc_counter* c, const uint8_t* d_lines, uint64_t n_bytes, const uint32_t* d_off, uint32_t off_base,
                            uint32_t stride, uint32_t read_len, uint64_t n_reads, int32_t* d_assign, cudaStream_t stream) {
  if (n_reads == 0) return SGC_OK;
  if (n_reads > kAssignScratchReads) return set_error(SGC_ERR_INVALID_ARG, "batch larger than the assignment scratch");
  c->pair_assign = d_assign;
  const int rc = count_batch(c, d_lines, n_bytes, d_off, off_base, stride, read_len, n_reads, nullptr, stream);
  c->pair_assign = nullptr;
  return rc;
}

int sgc::ensure_staging(sgc_counter* c) {
  if (c->copy_stream) return SGC_OK;
  SGC_CUDA_TRY(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    SGC_CUDA_TRY(cudaEventCreateWithFlags(&c->copy_done[i], cudaEventDisableTiming));
    SGC_CUDA_TRY(cudaEventCreateWithFlags(&c->kernel_done[i], cudaEventDisableTiming));
  }
  return SGC_OK;
}

// chunk geometry: whole tiles of reads, about kChunkBytes each
uint64_t sgc::host_chunk_end(const uint32_t* line_off, uint32_t stride, uint64_t r0, uint64_t n_reads) {
  if (line_off) {
    // advance until the chunk holds about kChunkBytes
    uint64_t lo = r0, hi = n_reads;
    const uint64_t limit = (uint64_t)line_off[r0] + kChunkBytes;
    while (lo < hi) {  // last r with line_off[r] <= limit
      uint64_t mid = (lo + hi + 1) / 2;
      if (line_off[mid] <= limit) lo = mid; else hi = mid - 1;
    }
    return lo > r0 ? lo : r0 + 1;
  }
  const uint64_t per = std::max<uint64_t>(kChunkAlignReads, (kChunkBytes / stride) / kChunkAlignReads * kChunkAlignReads);
  return std::min(n_reads, r0 + per);
}

int sgc::stage_host_chunk(sgc_counter* c, cudaStream_t stream, const uint8_t* lines, uint64_t n_bytes, const uint32_t* line_off,
                          uint32_t stride, uint64_t r0, uint64_t r1, HostChunk* out) {
  const int b = (int)(c->chunks_submitted & 1);
  const uint64_t byte0 = line_off ? line_off[r0] : r0 * stride;
  const uint64_t byte1 = line_off ? line_off[r1] : std::min<uint64_t>(n_bytes, r1 * stride);
  const size_t bytes = byte1 - byte0;
  // (re)size this staging buffer; +64 so bulk copies of the last tile stay inside the allocation
  if (bytes + 64 > c->stage_cap) {
    SGC_CUDA_TRY(cudaStreamSynchronize(stream));
    SGC_CUDA_TRY(cudaStreamSynchronize(c->copy_stream));
    size_t cap = std::max<size_t>(bytes + 64, std::min<size_t>(kChunkBytes + (1 << 20), n_bytes + 64));
    for (int i = 0; i < 2; ++i) {
      cudaFree(c->d_stage[i]);
      c->d_stage[i] = nullptr;
      SGC_CUDA_TRY(cudaMalloc(&c->d_stage[i], cap));
    }
    c->stage_cap = cap;
  }
  const size_t n_off = line_off ? (r1 - r0 + 1) : 0;
  if (n_off > c->stage_off_cap) {
    SGC_CUDA_TRY(cudaStreamSynchronize(stream));
    SGC_CUDA_TRY(cudaStreamSynchronize(c->copy_stream));
    size_t cap = n_off * 2;
    for (int i = 0; i < 2; ++i) {
      cudaFree(c->d_stage_off[i]);
      c->d_stage_off[i] = nullptr;
      SGC_CUDA_TRY(cudaMalloc(&c->d_stage_off[i], cap * sizeof(uint32_t)));
    }
    c->stage_off_cap = cap;
  }
  // copy stream: wait until the kernel that last read this buffer is done, then copy
  if (c->chunks_submitted >= 2) SGC_CUDA_TRY(cudaStreamWaitEvent(c->copy_stream, c->kernel_done[b], 0));
  SGC_CUDA_TRY(cudaMemcpyAsync(c->d_stage[b], lines + byte0, bytes, cudaMemcpyHostToDevice, c->copy_stream));
  if (line_off)
    SGC_CUDA_TRY(cudaMemcpyAsync(c->d_stage_off[b], line_off + r0, n_off * sizeof(uint32_t), cudaMemcpyHostToDevice,
                                 c->copy_stream));
  SGC_CUDA_TRY(cudaEventRecord(c->copy_done[b], c->copy_stream));
  SGC_CUDA_TRY(cudaStreamWaitEvent(stream, c->copy_done[b], 0));
  out->d_lines = c->d_stage[b];
  out->d_off = line_off ? c->d_stage_off[b] : nullptr;
  out->bytes = bytes;
  out->off_base = (uint32_t)(line_off ? byte0 : 0);
  out->buf = b;
  return SGC_OK;
}

int sgc::end_host_chunk(sgc_counter* c, cudaStream_t stream, const HostChunk& ch) {
  SGC_CUDA_TRY(cudaEventRecord(c->kernel_done[ch.buf], stream));
  c->chunks_submitted += 1;
  return SGC_OK;
}

// ticket of a submit call's copies (sgc_counter_wait_copies)
int sgc::push_copy_ticket(sgc_counter* c) {
  cudaEvent_t ticket = nullptr;
  if (!c->free_tickets.empty()) {
    ticket = c->free_tickets.back();
    c->free_tickets.pop_back();
  } else {
    SGC_CUDA_TRY(cudaEventCreateWithFlags(&ticket, cudaEventDisableTiming));
  }
  c->copy_tickets.push_back(ticket);
  SGC_CUDA_TRY(cudaEventRecord(ticket, c->copy_stream));
  return SGC_OK;
}

namespace {

// an empty unmatched report
int clear_unmatched(sgc_counter* c) {
  const uint64_t blocks = std::min<uint64_t>((c->um_capacity + 255) / 256, (uint64_t)c->lib->sm_count * 8);
  unmatched_clear_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(static_cast<ulonglong2*>(c->d_um_table), c->um_capacity);
  SGC_CUDA_TRY(cudaGetLastError());
  SGC_CUDA_TRY(cudaMemsetAsync(c->d_um_tally, 0, kTallyWords * sizeof(uint64_t), c->stream));
  return SGC_OK;
}

}  // namespace

extern "C" {

int sgc_span_geometry(uint32_t k, uint32_t read_len, int is_reverse, uint32_t offset, int position_recursion,
                      uint32_t* span_start, uint32_t* span_len, uint32_t* span_offset) {
  if (!span_start || !span_len || !span_offset) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  if (k == 0 || (uint64_t)offset + k > read_len)
    return set_error(SGC_ERR_INVALID_ARG, "the Centered window does not fit the read");
  // the same three facts the kernels derive (make_geom): does Plus exist, does Minus exist, and
  // which of them lies before the Centered window in the stored read
  const StreamGeom g = make_geom(k, read_len, (int)offset, true, is_reverse != 0, position_recursion != 0, SGC_RC_BITTRICK);
  const uint32_t before = is_reverse ? g.try_plus : g.try_minus, after = is_reverse ? g.try_minus : g.try_plus;
  *span_start = (uint32_t)g.win_src - before;
  *span_len = before + k + after;
  *span_offset = is_reverse ? after : before;  // Offset index of the span records
  return SGC_OK;
}

int sgc_span_geometry_shift(uint32_t k, uint32_t read_len, int is_reverse, uint32_t offset, uint32_t max_shift,
                            uint32_t* span_start, uint32_t* span_len, uint32_t* span_offset) {
  if (max_shift < 1 || max_shift > (uint32_t)kMaxShift) return set_error(SGC_ERR_INVALID_ARG, "max_shift must be 1..16");
  if (max_shift == 1)
    return sgc_span_geometry(k, read_len, is_reverse, offset, 1, span_start, span_len, span_offset);
  if (!span_start || !span_len || !span_offset) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  // [lo, hi) in the coordinates of the trimmed read: every window offset + d, |d| <= S, that fits
  const int64_t o = offset, lo = std::max<int64_t>(0, o - max_shift),
                hi = std::min<int64_t>(read_len, o + (int64_t)k + max_shift);
  if (k == 0 || hi - lo < (int64_t)k) return set_error(SGC_ERR_INVALID_ARG, "no shifted window fits the read");
  *span_start = (uint32_t)(is_reverse ? read_len - hi : lo);
  *span_len = (uint32_t)(hi - lo);
  *span_offset = (uint32_t)(o - lo);
  return SGC_OK;
}

int sgc_counter_create(const sgc_library* lib, int is_reverse, uint32_t offset, int position_recursion, int rc_mode,
                       void* stream, uint64_t* d_state, sgc_counter** out) {
  if (!lib || !out) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  if (rc_mode != SGC_RC_BITTRICK && rc_mode != SGC_RC_KEEP_N) return set_error(SGC_ERR_INVALID_ARG, "bad rc_mode");
  if (offset > 0x3FFFFFFFu) return set_error(SGC_ERR_INVALID_ARG, "offset too large");
  DeviceGuard guard(lib->device);
  if (!guard.ok()) return set_error(SGC_ERR_CUDA, "cudaSetDevice failed");
  sgc_counter* c = new sgc_counter();
  c->lib = lib;
  c->device = lib->device;
  c->is_reverse = is_reverse != 0;
  c->offset = offset;
  c->recursion = position_recursion != 0;
  c->rc_mode = rc_mode;
  for (int j = 0; j < kHotGuides; ++j) c->hot[j] = -2;
  struct Cleanup {
    sgc_counter* c;
    ~Cleanup() {
      if (c) sgc_counter_destroy(c);
    }
  } cleanup{c};
  if (stream) {
    c->stream = (cudaStream_t)stream;
  } else {
    // The counter's own stream: counters of concurrent samples on one device neither serialise
    // their kernels nor wait for each other in sgc_counter_sync.  A BLOCKING stream, so that work
    // the caller queued on the legacy default stream before a submit (a memcpy, a generator
    // kernel) is still ordered before the counter's kernels, as it was with stream = NULL.
    SGC_CUDA_TRY(cudaStreamCreate(&c->stream));
    c->own_stream = true;
  }
  const size_t words = (size_t)lib->n + 2;
  if (d_state) {
    c->d_state = reinterpret_cast<unsigned long long*>(d_state);
  } else {
    SGC_CUDA_TRY(cudaMalloc(&c->d_state, words * sizeof(uint64_t)));
    c->own_state = true;
  }
  SGC_CUDA_TRY(cudaMemsetAsync(c->d_state, 0, words * sizeof(uint64_t), c->stream));
  const int want_rep = env_int("SGC_REPLICAS", 0);  // tuning build: override of sgc_counter_set_replicas
  if (want_rep > 0) {
    int rc = sgc_counter_set_replicas(c, (uint32_t)want_rep);
    if (rc) return rc;
  }
  cleanup.c = nullptr;
  *out = c;
  return SGC_OK;
}

void sgc_counter_destroy(sgc_counter* c) {
  if (!c) return;
  DeviceGuard guard(c->device);  // (not c->lib: a garbage collector may have destroyed the library first)
  cudaStreamSynchronize(c->stream);
  for (sgc_fastq_stream* s : std::vector<sgc_fastq_stream*>(c->fastq_streams)) fastq_stream_release(s);
  if (c->copy_stream) {
    cudaStreamSynchronize(c->copy_stream);
    cudaStreamDestroy(c->copy_stream);
  }
  for (int i = 0; i < 2; ++i) {
    cudaFree(c->d_stage[i]);
    cudaFree(c->d_stage_off[i]);
    if (c->copy_done[i]) cudaEventDestroy(c->copy_done[i]);
    if (c->kernel_done[i]) cudaEventDestroy(c->kernel_done[i]);
  }
  for (cudaEvent_t e : c->copy_tickets) cudaEventDestroy(e);
  for (cudaEvent_t e : c->free_tickets) cudaEventDestroy(e);
  cudaFree(c->d_rep);
  cudaFree(c->d_top);
  cudaFree(c->d_um_table);
  cudaFree(c->d_um_assign);
  cudaFree(c->d_um_tally);
  if (c->own_state) cudaFree(c->d_state);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
}

int sgc_counter_submit_device(sgc_counter* c, const uint8_t* d_lines, uint64_t n_bytes, const uint32_t* d_line_off,
                              uint32_t stride, uint32_t read_len, uint64_t n_reads, int32_t* d_assign_out) {
  int rc = check_batch(c, d_lines, n_bytes, d_line_off, stride, read_len, n_reads);
  if (rc) return rc;
  DeviceGuard guard(c->lib->device);
  return count_batch(c, d_lines, n_bytes, d_line_off, 0, stride, read_len, n_reads, d_assign_out, c->stream);
}

int sgc_counter_submit(sgc_counter* c, const uint8_t* lines, uint64_t n_bytes, const uint32_t* line_off,
                       uint32_t stride, uint32_t read_len, uint64_t n_reads) {
  int rc = check_batch(c, lines, n_bytes, line_off, stride, read_len, n_reads);
  if (rc) return rc;
  if (n_reads == 0) return SGC_OK;
  if (line_off && line_off[n_reads] > n_bytes) return set_error(SGC_ERR_INVALID_ARG, "line offsets exceed n_bytes");
  DeviceGuard guard(c->lib->device);
  if ((rc = ensure_staging(c))) return rc;
  uint64_t r0 = 0;
  while (r0 < n_reads) {
    const uint64_t r1 = host_chunk_end(line_off, stride, r0, n_reads);
    HostChunk ch;
    if ((rc = stage_host_chunk(c, c->stream, lines, n_bytes, line_off, stride, r0, r1, &ch))) return rc;
    // the chunk's offsets stay what they were in the batch: the kernel subtracts the chunk's base
    rc = count_batch(c, ch.d_lines, ch.bytes, ch.d_off, ch.off_base, stride, read_len, r1 - r0, nullptr, c->stream);
    if (rc) return rc;
    if ((rc = end_host_chunk(c, c->stream, ch))) return rc;
    r0 = r1;
  }
  return push_copy_ticket(c);
}

int sgc_counter_set_replicas(sgc_counter* c, uint32_t replicas) {
  if (!c) return set_error(SGC_ERR_INVALID_ARG, "counter is NULL");
  DeviceGuard guard(c->lib->device);
  if (replicas == 0) {  // back to the automatic plan, made again on the next large batch
    c->auto_skew = true;
    c->skew_planned = false;
    for (int j = 0; j < kHotGuides; ++j) c->hot[j] = -2;
    return alloc_replicas(c, 1, c->stream);
  }
  c->auto_skew = false;
  for (int j = 0; j < kHotGuides; ++j) c->hot[j] = -2;
  return alloc_replicas(c, replicas, c->stream);
}

int sgc_counter_set_max_shift(sgc_counter* c, uint32_t max_shift) {
  if (!c) return set_error(SGC_ERR_INVALID_ARG, "counter is NULL");
  if (max_shift < 1 || max_shift > (uint32_t)kMaxShift) return set_error(SGC_ERR_INVALID_ARG, "max_shift must be 1..16");
  if (c->submitted) return set_error(SGC_ERR_INVALID_ARG, "max_shift must be set before the counter's first submit");
  if (max_shift >= 2 && !c->recursion)
    return set_error(SGC_ERR_INVALID_ARG, "max_shift >= 2 needs position recursion");
  if (max_shift >= 2 && c->lib->opaque)
    return set_error(SGC_ERR_INVALID_ARG, "max_shift >= 2 needs a library of guides of at most 30 bases over A,C,G,T");
  c->max_shift = max_shift;
  return SGC_OK;
}

int sgc_counter_sync(sgc_counter* c) {
  if (!c) return set_error(SGC_ERR_INVALID_ARG, "counter is NULL");
  DeviceGuard guard(c->lib->device);
  SGC_CUDA_TRY(cudaStreamSynchronize(c->stream));
  return SGC_OK;
}

int sgc_counter_wait_copies(sgc_counter* c, uint32_t keep_in_flight) {
  if (!c) return set_error(SGC_ERR_INVALID_ARG, "counter is NULL");
  DeviceGuard guard(c->lib->device);
  while (c->copy_tickets.size() > keep_in_flight) {
    cudaEvent_t ticket = c->copy_tickets.front();
    SGC_CUDA_TRY(cudaEventSynchronize(ticket));
    c->copy_tickets.pop_front();
    c->free_tickets.push_back(ticket);
  }
  return SGC_OK;
}

int sgc_counter_reset(sgc_counter* c) {
  if (!c) return set_error(SGC_ERR_INVALID_ARG, "counter is NULL");
  DeviceGuard guard(c->lib->device);
  SGC_CUDA_TRY(cudaMemsetAsync(c->d_state, 0, ((size_t)c->lib->n + 2) * sizeof(uint64_t), c->stream));
  return c->um_capacity ? clear_unmatched(c) : SGC_OK;
}

int sgc_unmatched_report_bytes(uint64_t capacity, uint64_t* bytes) {
  if (!bytes) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  if (capacity == 0 || capacity > kUnmatchedMaxCapacity)
    return set_error(SGC_ERR_INVALID_ARG, "the unmatched report's capacity must be 1..2^26 windows");
  *bytes = capacity * sizeof(ulonglong2) + kUnmatchedLaunchReads * sizeof(int32_t) + kTallyWords * sizeof(uint64_t);
  return SGC_OK;
}

int sgc_counter_set_unmatched_report(sgc_counter* c, uint64_t capacity) {
  if (!c) return set_error(SGC_ERR_INVALID_ARG, "counter is NULL");
  uint64_t bytes = 0;
  if (int rc = sgc_unmatched_report_bytes(capacity, &bytes)) return rc;
  if (c->submitted) return set_error(SGC_ERR_INVALID_ARG, "the unmatched report must be set before the counter's first submit");
  if (c->lib->opaque)
    return set_error(SGC_ERR_INVALID_ARG,
                     "the unmatched report needs a library of guides of at most 30 bases over A,C,G,T");
  DeviceGuard guard(c->lib->device);
  if (capacity != c->um_capacity) {
    SGC_CUDA_TRY(cudaStreamSynchronize(c->stream));
    cudaFree(c->d_um_table);
    c->d_um_table = nullptr;
    c->um_capacity = 0;
    SGC_CUDA_TRY(cudaMalloc(&c->d_um_table, capacity * sizeof(ulonglong2)));
    c->um_capacity = capacity;
  }
  if (!c->d_um_assign) SGC_CUDA_TRY(cudaMalloc(&c->d_um_assign, kUnmatchedLaunchReads * sizeof(int32_t)));
  if (!c->d_um_tally) SGC_CUDA_TRY(cudaMalloc(&c->d_um_tally, kTallyWords * sizeof(uint64_t)));
  return clear_unmatched(c);
}

int sgc_counter_unmatched(sgc_counter* c, uint64_t max_windows, uint8_t* windows, uint64_t* counts, uint64_t* n_windows,
                          sgc_unmatched_info* info) {
  if (!c) return set_error(SGC_ERR_INVALID_ARG, "counter is NULL");
  if (!c->um_capacity) return set_error(SGC_ERR_INVALID_ARG, "the counter has no unmatched report");
  if (max_windows && (!windows || !counts)) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  DeviceGuard guard(c->lib->device);
  // the compaction goes through the assignment scratch, one piece of the table at a time
  constexpr uint64_t kPiece = kUnmatchedLaunchReads * sizeof(int32_t) / sizeof(ulonglong2);
  ulonglong2* buf = reinterpret_cast<ulonglong2*>(c->d_um_assign);
  std::vector<ulonglong2> held;
  unsigned long long tally[kTallyWords];
  uint64_t distinct = 0;
  for (uint64_t a = 0; a < c->um_capacity; a += kPiece) {
    const uint64_t n = std::min(kPiece, c->um_capacity - a);
    SGC_CUDA_TRY(cudaMemsetAsync(c->d_um_tally + kTallyCompacted, 0, sizeof(uint64_t), c->stream));
    const uint64_t blocks = std::min<uint64_t>((n + 255) / 256, (uint64_t)c->lib->sm_count * 8);
    unmatched_compact_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(static_cast<const ulonglong2*>(c->d_um_table) + a, n,
                                                                       buf, c->d_um_tally);
    SGC_CUDA_TRY(cudaGetLastError());
    SGC_CUDA_TRY(cudaMemcpyAsync(tally, c->d_um_tally, sizeof tally, cudaMemcpyDeviceToHost, c->stream));
    SGC_CUDA_TRY(cudaStreamSynchronize(c->stream));
    distinct += tally[kTallyCompacted];
    if (!max_windows) continue;  // the tallies alone
    const size_t at = held.size();
    held.resize(at + tally[kTallyCompacted]);
    SGC_CUDA_TRY(cudaMemcpyAsync(held.data() + at, buf, tally[kTallyCompacted] * sizeof(ulonglong2), cudaMemcpyDeviceToHost,
                                 c->stream));
  }
  SGC_CUDA_TRY(cudaStreamSynchronize(c->stream));
  // report order: count descending, then window ascending (the key order of one k)
  const uint64_t n_out = std::min<uint64_t>(max_windows, held.size());
  auto before = [](const ulonglong2& a, const ulonglong2& b) { return a.y != b.y ? a.y > b.y : a.x < b.x; };
  std::nth_element(held.begin(), held.begin() + n_out, held.end(), before);
  std::sort(held.begin(), held.begin() + n_out, before);
  const uint32_t k = c->lib->k;
  for (uint64_t i = 0; i < n_out; ++i) {
    for (uint32_t j = 0; j < k; ++j) windows[i * k + j] = "ACGT"[(held[i].x >> (2 * (k - 1 - j))) & 3];
    counts[i] = held[i].y;
  }
  if (n_windows) *n_windows = n_out;
  if (info) {
    info->unmatched = tally[kTallyUnmatched];
    info->short_reads = tally[kTallyShort];
    info->non_acgt = tally[kTallyNonAcgt];
    info->overflow = tally[kTallyOverflow];
    info->distinct = distinct;
  }
  return SGC_OK;
}

int sgc_counter_finish(sgc_counter* c, uint64_t* counts, uint64_t* total, uint64_t* matched) {
  if (!c) return set_error(SGC_ERR_INVALID_ARG, "counter is NULL");
  DeviceGuard guard(c->lib->device);
  const size_t n = c->lib->n;
  std::vector<uint64_t> host(n + 2);
  SGC_CUDA_TRY(cudaMemcpyAsync(host.data(), c->d_state, (n + 2) * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
  SGC_CUDA_TRY(cudaStreamSynchronize(c->stream));
  if (counts) std::copy(host.begin(), host.begin() + n, counts);
  if (total) *total = host[n];
  if (matched) *matched = host[n + 1];
  return SGC_OK;
}

int sgc_counter_state(sgc_counter* c, uint64_t** d_state, uint64_t* n_words) {
  if (!c || !d_state || !n_words) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  *d_state = reinterpret_cast<uint64_t*>(c->d_state);
  *n_words = (uint64_t)c->lib->n + 2;
  return SGC_OK;
}

int sgc_counter_launch_info(const sgc_counter* c, sgc_launch_info* out) {
  if (!c || !out) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  *out = c->last;
  return SGC_OK;
}

}  // extern "C"
