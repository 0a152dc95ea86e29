// pair.cu — dual-guide constructs from paired reads (sgc_pair_counter, include/sgcount_cuda.h).
//
// Each mate goes through its own counter's ordinary count path (count.cu count_into_scratch: line,
// shift or byte-keyed kernel, the skew plan's replicas and hot guides kept) in chunks of at most 2^24
// pairs, which writes the chunk's per-read assignments into one int32 scratch per mate.  Then
//   pair_count_kernel     one warp per 32 pairs: reads both assignment vectors coalesced, classifies
//                         every pair, looks the both-matched ones up in the construct table, counts
//                         constructs (and recombinants into the report) once per distinct key of the
//                         warp (__match_any_sync: a construct that holds most pairs costs one atomic
//                         per warp), and adds the five class tallies once per warp.
//   pair_table_build_kernel  the construct table: open addressing, {key = a1 << 32 | a2, construct},
//                         at least 2 x n_pairs slots, filled with atomicCAS; a key met twice is a
//                         duplicate entry of the list.
#include <algorithm>
#include <string>
#include <vector>

#include "internal.h"

namespace sgc {
namespace {

constexpr unsigned long long kEmpty = ~0ull;  // no key: guide indices stay below 2^22
constexpr uint64_t kMaxPairs = 1ull << 26;
constexpr uint64_t kMaxRecombinants = 1ull << 26;
constexpr int kReportProbes = 128;  // linear probes before a recombinant pair is refused
constexpr int kPairWarps = 8;
enum { kListed, kRecombined, kFirstOnly, kSecondOnly, kNeither, kOverflow, kDistinct, kDuplicate, kPairTallyWords };

__device__ __forceinline__ uint64_t home_slot(unsigned long long key, uint64_t n_slots) {
  return __umul64hi(key * 0x9E3779B97F4A7C15ull, n_slots);
}

// n_slots: a power of two >= 2 n_pairs; keys all kEmpty before the launch, tally[kDuplicate] kEmpty
__global__ void pair_table_build_kernel(const uint32_t* __restrict__ first, const uint32_t* __restrict__ second,
                                        uint64_t n_pairs, unsigned long long* __restrict__ keys,
                                        uint32_t* __restrict__ construct, uint64_t n_slots,
                                        unsigned long long* __restrict__ tally) {
  for (uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; j < n_pairs; j += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long key = ((unsigned long long)first[j] << 32) | second[j];
    for (uint64_t s = home_slot(key, n_slots);; s = (s + 1) & (n_slots - 1)) {
      const unsigned long long cur = atomicCAS(&keys[s], kEmpty, key);
      if (cur == kEmpty) {
        construct[s] = (uint32_t)j;
        break;
      }
      if (cur == key) {
        atomicMin(tally + kDuplicate, key);
        break;
      }
    }
  }
}

struct PairView {
  const int32_t* a1;
  const int32_t* a2;
  uint64_t n;
  const unsigned long long* keys;
  const uint32_t* construct;
  uint64_t n_slots;
  unsigned long long* counts;     // n_pairs construct counts
  unsigned long long* rc_keys;    // report: capacity keys (kEmpty = free) ...
  unsigned long long* rc_counts;  // ... and their counts
  uint64_t capacity;              // 0 = no report
  unsigned long long* tally;
};

__global__ void __launch_bounds__(kPairWarps * 32) pair_count_kernel(PairView p) {
  const int lane = threadIdx.x & 31;
  const uint32_t gwarp = blockIdx.x * kPairWarps + (threadIdx.x >> 5), gwarps = gridDim.x * kPairWarps;
  const int probes = p.capacity < (uint64_t)kReportProbes ? (int)p.capacity : kReportProbes;
  uint32_t t[kNeither + 1] = {0, 0, 0, 0, 0};
  uint32_t n_over = 0, n_new = 0;
  const uint64_t n_tiles = (p.n + 31) / 32;
  for (uint64_t tile = gwarp; tile < n_tiles; tile += gwarps) {
    const uint64_t i = tile * 32 + lane;
    const int32_t x = i < p.n ? __ldcs(p.a1 + i) : -1, y = i < p.n ? __ldcs(p.a2 + i) : -1;
    uint32_t hit = ~0u;  // the construct of a listed pair
    bool recombined = false;
    unsigned long long key = kEmpty;
    if (i < p.n) {
      if (x >= 0 && y >= 0) {
        key = ((unsigned long long)(uint32_t)x << 32) | (uint32_t)y;
        for (uint64_t s = home_slot(key, p.n_slots);; s = (s + 1) & (p.n_slots - 1)) {
          const unsigned long long cur = __ldg(p.keys + s);
          if (cur == key) {
            hit = __ldg(p.construct + s);
            break;
          }
          if (cur == kEmpty) break;
        }
        recombined = hit == ~0u;
        ++t[recombined ? kRecombined : kListed];
      } else {
        ++t[x >= 0 ? kFirstOnly : (y >= 0 ? kSecondOnly : kNeither)];
      }
    }
    // one count update per distinct construct of the warp
    const uint32_t listed = __ballot_sync(0xffffffffu, hit != ~0u);
    if (listed) {
      const uint32_t group = __match_any_sync(0xffffffffu, hit);
      if (hit != ~0u && lane == __ffs((int)group) - 1) atomicAdd(p.counts + hit, (unsigned long long)__popc(group));
    }
    if (p.capacity == 0) continue;
    // and one report update per distinct recombinant pair
    const uint32_t want = __ballot_sync(0xffffffffu, recombined);
    const uint32_t group = recombined ? __match_any_sync(want, key) : 0u;
    if (recombined && lane == __ffs((int)group) - 1) {
      const unsigned long long cnt = (unsigned long long)__popc(group);
      uint64_t s = home_slot(key, p.capacity);
      bool done = false;
      for (int q = 0; q < probes && !done; ++q) {
        unsigned long long cur = __ldcg(p.rc_keys + s);
        if (cur == kEmpty) {
          cur = atomicCAS(p.rc_keys + s, kEmpty, key);
          n_new += cur == kEmpty;
        }
        if (cur == kEmpty || cur == key) {
          atomicAdd(p.rc_counts + s, cnt);
          done = true;
        }
        s = s + 1 == p.capacity ? 0 : s + 1;
      }
      if (!done) n_over += (uint32_t)cnt;
    }
  }
#pragma unroll
  for (int c = 0; c <= kNeither; ++c) {
    const uint32_t v = __reduce_add_sync(0xffffffffu, t[c]);
    if (lane == 0 && v) atomicAdd(p.tally + c, (unsigned long long)v);
  }
  n_over = __reduce_add_sync(0xffffffffu, n_over);
  n_new = __reduce_add_sync(0xffffffffu, n_new);
  if (lane == 0 && n_over) atomicAdd(p.tally + kOverflow, (unsigned long long)n_over);
  if (lane == 0 && n_new) atomicAdd(p.tally + kDistinct, (unsigned long long)n_new);
}

uint64_t table_slots(uint64_t n_pairs) {
  uint64_t n = 1;
  while (n < 2 * n_pairs) n *= 2;
  return n;
}

}  // namespace
}  // namespace sgc

using namespace sgc;

struct sgc_pair_counter {
  sgc_counter* mate[2] = {nullptr, nullptr};
  int device = 0;
  int sm_count = 0;
  uint64_t n_pairs = 0, n_slots = 0, capacity = 0;
  unsigned long long* d_keys = nullptr;
  uint32_t* d_construct = nullptr;
  unsigned long long* d_counts = nullptr;
  unsigned long long* d_rc_keys = nullptr;
  unsigned long long* d_rc_counts = nullptr;
  unsigned long long* d_tally = nullptr;
  int32_t* d_assign[2] = {nullptr, nullptr};
  // the end of mate 2's earlier work (begin_submit), then the end of the pair counter's last work on mate 1's
  // stream: destroy waits for it without looking at the counters, which may be gone already
  cudaEvent_t mark = nullptr;
};

namespace {

cudaStream_t work_stream(const sgc_pair_counter* pc) { return pc->mate[0]->stream; }

// empty constructs, tallies and report
int clear_pair(sgc_pair_counter* pc) {
  cudaStream_t s = work_stream(pc);
  SGC_CUDA_TRY(cudaMemsetAsync(pc->d_counts, 0, pc->n_pairs * sizeof(uint64_t), s));
  SGC_CUDA_TRY(cudaMemsetAsync(pc->d_tally, 0, kPairTallyWords * sizeof(uint64_t), s));
  if (pc->capacity) {
    SGC_CUDA_TRY(cudaMemsetAsync(pc->d_rc_keys, 0xFF, pc->capacity * sizeof(uint64_t), s));
    SGC_CUDA_TRY(cudaMemsetAsync(pc->d_rc_counts, 0, pc->capacity * sizeof(uint64_t), s));
  }
  SGC_CUDA_TRY(cudaEventRecord(pc->mark, s));
  return SGC_OK;
}

// mate 1's stream waits for mate 2's earlier work (a reset, a standalone batch)
int begin_submit(sgc_pair_counter* pc) {
  SGC_CUDA_TRY(cudaEventRecord(pc->mark, pc->mate[1]->stream));
  SGC_CUDA_TRY(cudaStreamWaitEvent(work_stream(pc), pc->mark, 0));
  return SGC_OK;
}

// mate 2's stream waits for everything the submit enqueued
int end_submit(sgc_pair_counter* pc) {
  SGC_CUDA_TRY(cudaEventRecord(pc->mark, work_stream(pc)));
  SGC_CUDA_TRY(cudaStreamWaitEvent(pc->mate[1]->stream, pc->mark, 0));
  return SGC_OK;
}

int combine(sgc_pair_counter* pc, uint64_t n) {
  PairView v{};
  v.a1 = pc->d_assign[0];
  v.a2 = pc->d_assign[1];
  v.n = n;
  v.keys = pc->d_keys;
  v.construct = pc->d_construct;
  v.n_slots = pc->n_slots;
  v.counts = pc->d_counts;
  v.rc_keys = pc->d_rc_keys;
  v.rc_counts = pc->d_rc_counts;
  v.capacity = pc->capacity;
  v.tally = pc->d_tally;
  uint64_t blocks = (n + 32 * kPairWarps - 1) / (32 * kPairWarps);
  blocks = std::min<uint64_t>(blocks, (uint64_t)pc->sm_count * 8);
  pair_count_kernel<<<(unsigned)blocks, 32 * kPairWarps, 0, work_stream(pc)>>>(v);
  SGC_CUDA_TRY(cudaGetLastError());
  return SGC_OK;
}

struct MateBatch {
  const uint8_t* lines;
  uint64_t n_bytes;
  const uint32_t* line_off;
  uint32_t stride, read_len;
};

int check_pair_batches(const sgc_pair_counter* pc, const MateBatch* m, uint64_t n_pairs, bool host) {
  if (!pc) return set_error(SGC_ERR_INVALID_ARG, "pair counter is NULL");
  for (int i = 0; i < 2; ++i) {
    if (int rc = check_batch(pc->mate[i], m[i].lines, m[i].n_bytes, m[i].line_off, m[i].stride, m[i].read_len, n_pairs))
      return rc;
    if (host && n_pairs && m[i].line_off && m[i].line_off[n_pairs] > m[i].n_bytes)
      return set_error(SGC_ERR_INVALID_ARG, "line offsets exceed n_bytes");
  }
  return SGC_OK;
}

}  // namespace

extern "C" {

int sgc_pair_counter_bytes(uint64_t n_pairs, uint64_t recombinant_capacity, uint64_t* bytes) {
  if (!bytes) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  if (n_pairs == 0 || n_pairs > kMaxPairs) return set_error(SGC_ERR_INVALID_ARG, "a pair list must hold 1..2^26 constructs");
  if (recombinant_capacity > kMaxRecombinants)
    return set_error(SGC_ERR_INVALID_ARG, "the recombinant report's capacity must be at most 2^26 pairs");
  *bytes = table_slots(n_pairs) * (sizeof(uint64_t) + sizeof(uint32_t)) + n_pairs * sizeof(uint64_t) +
           2 * kAssignScratchReads * sizeof(int32_t) + recombinant_capacity * 2 * sizeof(uint64_t) +
           kPairTallyWords * sizeof(uint64_t);
  return SGC_OK;
}

int sgc_pair_counter_create(sgc_counter* first, sgc_counter* second, const uint32_t* pair_first,
                            const uint32_t* pair_second, uint64_t n_pairs, uint64_t recombinant_capacity,
                            sgc_pair_counter** out) {
  if (!first || !second || !pair_first || !pair_second || !out) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  uint64_t bytes = 0;
  if (int rc = sgc_pair_counter_bytes(n_pairs, recombinant_capacity, &bytes)) return rc;
  if (first == second) return set_error(SGC_ERR_INVALID_ARG, "the two mates need two counters");
  if (first->device != second->device) return set_error(SGC_ERR_INVALID_ARG, "the two counters are on different devices");
  for (const sgc_counter* c : {first, second}) {
    if (c->submitted) return set_error(SGC_ERR_INVALID_ARG, "a mate's counter has already counted");
    if (c->um_capacity) return set_error(SGC_ERR_INVALID_ARG, "a mate's counter has an unmatched report");
  }
  for (uint64_t j = 0; j < n_pairs; ++j)
    if (pair_first[j] >= first->lib->n || pair_second[j] >= second->lib->n)
      return set_error(SGC_ERR_INVALID_ARG, "pair " + std::to_string(j) + " names a guide outside its library");
  DeviceGuard guard(first->device);
  if (!guard.ok()) return set_error(SGC_ERR_CUDA, "cudaSetDevice failed");
  sgc_pair_counter* pc = new sgc_pair_counter();
  struct Cleanup {
    sgc_pair_counter* pc;
    ~Cleanup() {
      if (pc) sgc_pair_counter_destroy(pc);
    }
  } cleanup{pc};
  pc->mate[0] = first;
  pc->mate[1] = second;
  pc->device = first->device;
  pc->sm_count = first->lib->sm_count;
  pc->n_pairs = n_pairs;
  pc->n_slots = table_slots(n_pairs);
  pc->capacity = recombinant_capacity;
  cudaStream_t s = work_stream(pc);
  SGC_CUDA_TRY(cudaEventCreateWithFlags(&pc->mark, cudaEventDisableTiming));
  SGC_CUDA_TRY(cudaMalloc(&pc->d_keys, pc->n_slots * sizeof(uint64_t)));
  SGC_CUDA_TRY(cudaMalloc(&pc->d_construct, pc->n_slots * sizeof(uint32_t)));
  SGC_CUDA_TRY(cudaMalloc(&pc->d_counts, n_pairs * sizeof(uint64_t)));
  SGC_CUDA_TRY(cudaMalloc(&pc->d_tally, kPairTallyWords * sizeof(uint64_t)));
  for (int i = 0; i < 2; ++i) SGC_CUDA_TRY(cudaMalloc(&pc->d_assign[i], kAssignScratchReads * sizeof(int32_t)));
  if (pc->capacity) {
    SGC_CUDA_TRY(cudaMalloc(&pc->d_rc_keys, pc->capacity * sizeof(uint64_t)));
    SGC_CUDA_TRY(cudaMalloc(&pc->d_rc_counts, pc->capacity * sizeof(uint64_t)));
  }
  // the list is on the device only while the table is built
  uint32_t* d_list = nullptr;
  SGC_CUDA_TRY(cudaMalloc(&d_list, 2 * n_pairs * sizeof(uint32_t)));
  struct FreeList {
    uint32_t* p;
    ~FreeList() { cudaFree(p); }
  } free_list{d_list};
  SGC_CUDA_TRY(cudaMemcpyAsync(d_list, pair_first, n_pairs * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
  SGC_CUDA_TRY(cudaMemcpyAsync(d_list + n_pairs, pair_second, n_pairs * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
  SGC_CUDA_TRY(cudaMemsetAsync(pc->d_keys, 0xFF, pc->n_slots * sizeof(uint64_t), s));
  SGC_CUDA_TRY(cudaMemsetAsync(pc->d_tally + kDuplicate, 0xFF, sizeof(uint64_t), s));
  const uint64_t blocks = std::min<uint64_t>((n_pairs + 255) / 256, (uint64_t)pc->sm_count * 8);
  pair_table_build_kernel<<<(unsigned)blocks, 256, 0, s>>>(d_list, d_list + n_pairs, n_pairs, pc->d_keys, pc->d_construct,
                                                           pc->n_slots, pc->d_tally);
  SGC_CUDA_TRY(cudaGetLastError());
  unsigned long long dup = 0;
  SGC_CUDA_TRY(cudaMemcpyAsync(&dup, pc->d_tally + kDuplicate, sizeof dup, cudaMemcpyDeviceToHost, s));
  SGC_CUDA_TRY(cudaStreamSynchronize(s));
  if (dup != kEmpty) {
    const uint32_t a = (uint32_t)(dup >> 32), b = (uint32_t)dup;
    std::vector<uint64_t> at;
    for (uint64_t j = 0; j < n_pairs && at.size() < 2; ++j)
      if (pair_first[j] == a && pair_second[j] == b) at.push_back(j);
    return set_error(SGC_ERR_DUPLICATE_SEQUENCE, "pairs " + std::to_string(at[0]) + " and " + std::to_string(at[1]) +
                                                     " are both (" + std::to_string(a) + ", " + std::to_string(b) + ")");
  }
  if (int rc = clear_pair(pc)) return rc;
  cleanup.pc = nullptr;
  *out = pc;
  return SGC_OK;
}

void sgc_pair_counter_destroy(sgc_pair_counter* pc) {
  if (!pc) return;
  DeviceGuard guard(pc->device);
  if (pc->mark) cudaEventSynchronize(pc->mark);
  cudaFree(pc->d_keys);
  cudaFree(pc->d_construct);
  cudaFree(pc->d_counts);
  cudaFree(pc->d_rc_keys);
  cudaFree(pc->d_rc_counts);
  cudaFree(pc->d_tally);
  for (int i = 0; i < 2; ++i) cudaFree(pc->d_assign[i]);
  if (pc->mark) cudaEventDestroy(pc->mark);
  delete pc;
}

int sgc_pair_counter_submit(sgc_pair_counter* pc, const uint8_t* lines1, uint64_t n_bytes1, const uint32_t* line_off1,
                            uint32_t stride1, uint32_t read_len1, const uint8_t* lines2, uint64_t n_bytes2,
                            const uint32_t* line_off2, uint32_t stride2, uint32_t read_len2, uint64_t n_pairs) {
  const MateBatch m[2] = {{lines1, n_bytes1, line_off1, stride1, read_len1}, {lines2, n_bytes2, line_off2, stride2, read_len2}};
  int rc = check_pair_batches(pc, m, n_pairs, true);
  if (rc || n_pairs == 0) return rc;
  DeviceGuard guard(pc->device);
  cudaStream_t s = work_stream(pc);
  for (int i = 0; i < 2; ++i)
    if ((rc = ensure_staging(pc->mate[i]))) return rc;
  if ((rc = begin_submit(pc))) return rc;
  rc = [&]() -> int {
    int rc = SGC_OK;
    for (uint64_t r0 = 0; r0 < n_pairs;) {
      // a chunk: both mates' copies fit their staging buffers and the pairs fit the assignment scratch
      const uint64_t r1 = std::min({host_chunk_end(line_off1, stride1, r0, n_pairs), host_chunk_end(line_off2, stride2, r0, n_pairs),
                                    r0 + assign_scratch_reads()});
      HostChunk ch[2];
      for (int i = 0; i < 2; ++i)
        if ((rc = stage_host_chunk(pc->mate[i], s, m[i].lines, m[i].n_bytes, m[i].line_off, m[i].stride, r0, r1, &ch[i])))
          return rc;
      for (int i = 0; i < 2; ++i)
        if ((rc = count_into_scratch(pc->mate[i], ch[i].d_lines, ch[i].bytes, ch[i].d_off, ch[i].off_base, m[i].stride,
                                     m[i].read_len, r1 - r0, pc->d_assign[i], s)))
          return rc;
      if ((rc = combine(pc, r1 - r0))) return rc;
      for (int i = 0; i < 2; ++i)
        if ((rc = end_host_chunk(pc->mate[i], s, ch[i]))) return rc;
      r0 = r1;
    }
    for (int i = 0; i < 2; ++i)
      if ((rc = push_copy_ticket(pc->mate[i]))) return rc;
    return rc;
  }();
  // also after a failure part-way, so that destroy waits for what was enqueued
  const int rc_end = end_submit(pc);
  return rc ? rc : rc_end;
}

int sgc_pair_counter_submit_device(sgc_pair_counter* pc, const uint8_t* d_lines1, uint64_t n_bytes1,
                                   const uint32_t* d_line_off1, uint32_t stride1, uint32_t read_len1,
                                   const uint8_t* d_lines2, uint64_t n_bytes2, const uint32_t* d_line_off2,
                                   uint32_t stride2, uint32_t read_len2, uint64_t n_pairs) {
  const MateBatch m[2] = {{d_lines1, n_bytes1, d_line_off1, stride1, read_len1},
                          {d_lines2, n_bytes2, d_line_off2, stride2, read_len2}};
  int rc = check_pair_batches(pc, m, n_pairs, false);
  if (rc || n_pairs == 0) return rc;
  DeviceGuard guard(pc->device);
  if ((rc = begin_submit(pc))) return rc;
  rc = [&]() -> int {
    int rc = SGC_OK;
    for (uint64_t r0 = 0; r0 < n_pairs;) {
      const uint64_t r1 = std::min(n_pairs, r0 + assign_scratch_reads());
      for (int i = 0; i < 2; ++i) {
        // the chunk as a batch of its own: offsets keep their values, fixed-stride lines move to the chunk
        const uint8_t* lines = m[i].line_off ? m[i].lines : m[i].lines + r0 * m[i].stride;
        const uint64_t bytes = m[i].line_off ? m[i].n_bytes : m[i].n_bytes - r0 * m[i].stride;
        const uint32_t* off = m[i].line_off ? m[i].line_off + r0 : nullptr;
        if ((rc = count_into_scratch(pc->mate[i], lines, bytes, off, 0, m[i].stride, m[i].read_len, r1 - r0, pc->d_assign[i],
                                     work_stream(pc))))
          return rc;
      }
      if ((rc = combine(pc, r1 - r0))) return rc;
      r0 = r1;
    }
    return rc;
  }();
  const int rc_end = end_submit(pc);
  return rc ? rc : rc_end;
}

int sgc_pair_counter_wait_copies(sgc_pair_counter* pc, uint32_t keep_in_flight) {
  if (!pc) return set_error(SGC_ERR_INVALID_ARG, "pair counter is NULL");
  for (sgc_counter* c : pc->mate)
    if (int rc = sgc_counter_wait_copies(c, keep_in_flight)) return rc;
  return SGC_OK;
}

int sgc_pair_counter_finish(sgc_pair_counter* pc, uint64_t* construct_counts, sgc_pair_info* info) {
  if (!pc) return set_error(SGC_ERR_INVALID_ARG, "pair counter is NULL");
  DeviceGuard guard(pc->device);
  cudaStream_t s = work_stream(pc);
  unsigned long long tally[kPairTallyWords];
  if (construct_counts)
    SGC_CUDA_TRY(cudaMemcpyAsync(construct_counts, pc->d_counts, pc->n_pairs * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
  SGC_CUDA_TRY(cudaMemcpyAsync(tally, pc->d_tally, sizeof tally, cudaMemcpyDeviceToHost, s));
  SGC_CUDA_TRY(cudaStreamSynchronize(s));
  if (info) {
    info->listed = tally[kListed];
    info->recombined = tally[kRecombined];
    info->first_only = tally[kFirstOnly];
    info->second_only = tally[kSecondOnly];
    info->neither = tally[kNeither];
    info->total = info->listed + info->recombined + info->first_only + info->second_only + info->neither;
    info->overflow = tally[kOverflow];
    info->distinct = tally[kDistinct];
  }
  return SGC_OK;
}

int sgc_pair_counter_recombinants(sgc_pair_counter* pc, uint64_t max_pairs, uint32_t* first, uint32_t* second,
                                  uint64_t* counts, uint64_t* n_out) {
  if (!pc) return set_error(SGC_ERR_INVALID_ARG, "pair counter is NULL");
  if (!pc->capacity) return set_error(SGC_ERR_INVALID_ARG, "the pair counter has no recombinant report");
  if (max_pairs && (!first || !second || !counts)) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  DeviceGuard guard(pc->device);
  cudaStream_t s = work_stream(pc);
  std::vector<unsigned long long> keys(pc->capacity), cnt(pc->capacity);
  SGC_CUDA_TRY(cudaMemcpyAsync(keys.data(), pc->d_rc_keys, pc->capacity * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
  SGC_CUDA_TRY(cudaMemcpyAsync(cnt.data(), pc->d_rc_counts, pc->capacity * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
  SGC_CUDA_TRY(cudaStreamSynchronize(s));
  std::vector<std::pair<unsigned long long, unsigned long long>> held;  // (count, key)
  for (uint64_t i = 0; i < pc->capacity; ++i)
    if (keys[i] != kEmpty) held.emplace_back(cnt[i], keys[i]);
  // report order: count descending, then (first, second) ascending, which is key order
  const uint64_t n = std::min<uint64_t>(max_pairs, held.size());
  auto before = [](const auto& a, const auto& b) { return a.first != b.first ? a.first > b.first : a.second < b.second; };
  std::partial_sort(held.begin(), held.begin() + n, held.end(), before);
  for (uint64_t i = 0; i < n; ++i) {
    first[i] = (uint32_t)(held[i].second >> 32);
    second[i] = (uint32_t)held[i].second;
    counts[i] = held[i].first;
  }
  if (n_out) *n_out = n;
  return SGC_OK;
}

int sgc_pair_counter_reset(sgc_pair_counter* pc) {
  if (!pc) return set_error(SGC_ERR_INVALID_ARG, "pair counter is NULL");
  DeviceGuard guard(pc->device);
  for (sgc_counter* c : pc->mate)
    if (int rc = sgc_counter_reset(c)) return rc;
  return clear_pair(pc);
}

}  // extern "C"
