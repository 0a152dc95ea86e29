// internal.h — host-side objects behind the opaque handles of include/sgcount_cuda.h.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <deque>
#include <string>
#include <vector>

#include "../../include/sgcount_cuda.h"
#include "common.cuh"

namespace sgc {

int set_error(int code, const std::string& msg);
int cuda_error(cudaError_t e, const char* what, const char* file, int line);

#define SGC_CUDA_TRY(expr)                                                   \
  do {                                                                       \
    cudaError_t _e = (expr);                                                 \
    if (_e != cudaSuccess) return ::sgc::cuda_error(_e, #expr, __FILE__, __LINE__); \
  } while (0)

// Selects a device for the lifetime of the guard and restores the caller's device.
class DeviceGuard {
  int prev_ = -1;
  bool ok_ = false;

 public:
  explicit DeviceGuard(int device) {
    if (cudaGetDevice(&prev_) != cudaSuccess) prev_ = -1;
    ok_ = cudaSetDevice(device) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (prev_ >= 0) cudaSetDevice(prev_);
  }
  bool ok() const { return ok_; }
};

// position histogram of a batch of reads (offsetter.rs:55-79), defined in offset.cu
int position_counts_device(const uint8_t* d_lines, const uint32_t* d_line_off, uint32_t stride,
                           uint32_t read_len, uint64_t n_reads, uint32_t size, uint32_t* d_hist /* size*4, zeroed */,
                           cudaStream_t stream);

// exclusive prefix sum of cnt[0..n) into start[0..n) (library.cu);
// tile_sums: scratch of (n + 2047) / 2048 + 1 words
int exclusive_scan_u32(const uint32_t* d_cnt, uint32_t n, uint32_t* d_start, uint32_t* d_tile_sums,
                       cudaStream_t stream = nullptr);

}  // namespace sgc

struct sgc_library;
struct sgc_counter;

namespace sgc {
// opaque.cu: libraries with a byte outside A,C,G,T or guides longer than kMaxK, kept as bytes
constexpr uint32_t kMaxKOpaque = 1024;
int opaque_build(sgc_library* lib, const uint8_t* d_seqs, uint64_t* n_variants, uint64_t* n_ambiguous, uint32_t* dup_guide);
void opaque_destroy(sgc_library* lib);
int opaque_lookup_tokens(const sgc_library* lib, const uint8_t* d_tokens, uint64_t n_tokens, int32_t* d_idx, uint8_t* d_kind);
int opaque_count(const sgc_counter* c, const uint8_t* d_lines, const uint32_t* d_off, uint32_t off_base, uint32_t stride,
                 uint32_t read_len, uint64_t first, uint64_t n_reads, int32_t* d_assign, cudaStream_t stream,
                 uint32_t* grid_out);
}  // namespace sgc

struct sgc_counter {
  const sgc_library* lib = nullptr;
  int device = 0;  // lib->device, kept so that destroying the counter never looks at the library
  int is_reverse = 0;
  uint32_t offset = 0;
  int recursion = 1;
  int rc_mode = SGC_RC_BITTRICK;
  uint32_t max_shift = 1;  // sgc_counter_set_max_shift: >= 2 takes the shift kernel
  bool submitted = false;  // a batch has been submitted (max_shift is fixed from then on)
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  unsigned long long* d_state = nullptr;
  bool own_state = false;
  // skew plan (count.cu plan_skew): replicas of the count vector and guides counted in registers
  unsigned long long* d_rep = nullptr;  // n_rep x n_guides words, zero between launches
  uint32_t n_rep = 1;
  int32_t hot[4] = {-2, -2, -2, -2};
  bool auto_skew = true, skew_planned = false;
  void* d_top = nullptr;  // the plan's read-back buffer
  const uint32_t* gather_end = nullptr;  // count_gathered_lines: per-read end offsets (transient)
  // host-batch staging (sgc_counter_submit)
  cudaStream_t copy_stream = nullptr;
  uint8_t* d_stage[2] = {nullptr, nullptr};
  uint32_t* d_stage_off[2] = {nullptr, nullptr};
  size_t stage_cap = 0, stage_off_cap = 0;
  cudaEvent_t copy_done[2] = {nullptr, nullptr}, kernel_done[2] = {nullptr, nullptr};
  uint64_t chunks_submitted = 0;
  std::deque<cudaEvent_t> copy_tickets;   // one per sgc_counter_submit call whose copies may still run
  std::vector<cudaEvent_t> free_tickets;
  sgc_launch_info last{};
  // unmatched report (sgc_counter_set_unmatched_report; count.cu unmatched_collect_kernel): capacity
  // {key, count} slots, the per-read assignments of one launch (also the compaction buffer), tallies
  uint64_t um_capacity = 0;  // 0 = off
  void* d_um_table = nullptr;
  int32_t* d_um_assign = nullptr;
  unsigned long long* d_um_tally = nullptr;
  // device-ingest streams that count into this counter (gzip.cu); released with it if still open
  std::vector<struct sgc_fastq_stream*> fastq_streams;
  // pair.cu: set only while a pair counter counts one chunk of a mate (count_into_scratch): the line
  // (shift, byte-keyed) kernel writes read r's assignment to pair_assign[r]; NULL for every other caller
  int32_t* pair_assign = nullptr;
};

namespace sgc {
// count.cu: reads scattered in a device-resident text, read r = d_text[d_start[r] .. d_end[r])
int count_gathered_lines(sgc_counter* c, const uint8_t* d_text, uint64_t n_bytes, const uint32_t* d_start,
                         const uint32_t* d_end, uint64_t n_reads);
// gzip.cu: frees the device side of a stream whose counter is going away (the handle stays valid
// for sgc_fastq_stream_destroy)
void fastq_stream_release(struct sgc_fastq_stream* s);
int check_batch(const sgc_counter* c, const uint8_t* lines, uint64_t n_bytes, const uint32_t* line_off, uint32_t stride,
                uint32_t read_len, uint64_t n_reads);
// entries of a fixed per-read assignment scratch (the unmatched report's, each mate's of a pair counter)
constexpr uint64_t kAssignScratchReads = 1ull << 24;
// count.cu: reads per launch of a counter whose assignments go to such a scratch: kAssignScratchReads, fewer
// under SGC_MAX_LAUNCH_TILES (read from the environment at every call)
uint64_t assign_scratch_reads();
// count.cu: counts a device-resident batch of at most kAssignScratchReads reads on `stream` through the
// line, shift or byte-keyed kernel (the skew plan included) and writes read r's assignment to d_assign[r]
int count_into_scratch(sgc_counter* c, const uint8_t* d_lines, uint64_t n_bytes, const uint32_t* d_off, uint32_t off_base,
                       uint32_t stride, uint32_t read_len, uint64_t n_reads, int32_t* d_assign, cudaStream_t stream);
// count.cu: a host batch copied chunk by chunk into a counter's two staging buffers on its copy stream
// (sgc_counter_submit); `stream` is the stream whose kernels read the chunk
struct HostChunk {
  const uint8_t* d_lines;
  const uint32_t* d_off;
  uint64_t bytes;
  uint32_t off_base;
  int buf;
};
int ensure_staging(sgc_counter* c);
uint64_t host_chunk_end(const uint32_t* line_off, uint32_t stride, uint64_t r0, uint64_t n_reads);
int stage_host_chunk(sgc_counter* c, cudaStream_t stream, const uint8_t* lines, uint64_t n_bytes, const uint32_t* line_off,
                     uint32_t stride, uint64_t r0, uint64_t r1, HostChunk* out);
int end_host_chunk(sgc_counter* c, cudaStream_t stream, const HostChunk& ch);  // after the chunk's kernels
int push_copy_ticket(sgc_counter* c);  // at the end of a submit call
}

struct sgc_library {
  int device = 0;
  uint32_t n = 0, k = 0;
  bool with_perm = false;
  bool wide = false;
  // seed index + front table per read orientation (common.cuh): [0] forward, [1] reverse
  struct Index {
    uint64_t* d_keys = nullptr;  // n interleaved keys (hi << 32 | lo), library order
    uint64_t* d_dir64[sgc::kSeeds] = {};      // narrow keys
    ulonglong2* d_dir128[sgc::kSeeds] = {};   // wide keys
    uint64_t* d_post = nullptr;  // kSeeds lists of n postings
    uint64_t* d_front = nullptr;
  } ix[2];
  uint32_t dir_shift = 0, front_shift = 0;
  sgc::SeedParts parts{};
  size_t front_bytes = 0;
  // opaque libraries (opaque.cu): the members' bytes and the two half indexes
  bool opaque = false;
  uint8_t* d_oseqs = nullptr;
  uint32_t* d_ostart[2] = {nullptr, nullptr};
  uint32_t* d_opost[2] = {nullptr, nullptr};
  uint32_t oshift = 0;
  uint32_t* d_lib_hist = nullptr;  // k*4 positional counts over guides 1..n-1 (offsetter.rs:190-191)
  int sm_count = 0;
  sgc_library_info info{};

  sgc::LibView view() const {
    sgc::LibView v{};
    v.k = k;
    v.n = n;
    v.wide = wide ? 1u : 0u;
    v.dir_shift = dir_shift;
    v.front_shift = front_shift;
    v.parts = parts;
    sgc::IndexView* views[2] = {&v.fwd, &v.rev};
    for (int o = 0; o < 2; ++o) {
      for (int i = 0; i < sgc::kSeeds; ++i) {
        views[o]->dir64[i] = ix[o].d_dir64[i];
        views[o]->dir128[i] = ix[o].d_dir128[i];
      }
      views[o]->post = ix[o].d_post;
      views[o]->front = ix[o].d_front;
    }
    return v;
  }
};
