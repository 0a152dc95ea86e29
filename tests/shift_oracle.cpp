// shift_oracle.cpp — the staggered-read rule (max_shift S >= 2), written literally over the CPU
// oracle's own lookups (oracle/oracle.h).  TEST INFRASTRUCTURE: built and loaded by
// tests/shift_oracle.py, never by the product.
//
// The rule is this project's own, not the reference's (the reference has S = 1 only): the
// windows at offset + d for d = 0, +1, -1, ..., +S, -S, in the coordinates of the read the
// reference trims (the reverse complement of the whole read in Reverse, counter.rs:196-204), each
// looked up as counter.rs:111-117 does (Library::contains, then Permuter::contains); the first
// window that yields a guide wins, and a window that does not fit the read is skipped (no early
// return as at counter.rs:105-108).  One fresh token per probe, like the oracle.
#include <string>
#include <thread>
#include <vector>

#include "../oracle/oracle.h"

namespace {

int64_t assign_one(const orc_library* lib, const orc_permuter* perm, const uint8_t* read, size_t len,
                   int is_reverse, uint64_t offset, uint32_t max_shift, int rc_mode) {
  const size_t k = orc_library_size(lib);
  std::string src((const char*)read, len);
  if (is_reverse) orc_seq_rev_comp(read, len, rc_mode, (uint8_t*)&src[0]);
  for (uint32_t i = 0; i <= 2 * max_shift; ++i) {
    const long long d = i == 0 ? 0 : ((i & 1) ? (long long)(i + 1) / 2 : -(long long)(i / 2));
    const long long lo = (long long)offset + d;
    if (lo < 0 || (size_t)lo + k > src.size()) continue;  // skipped, not a return
    const std::string token = src.substr((size_t)lo, k);
    int64_t idx = orc_library_contains(lib, (const uint8_t*)token.data(), k);
    if (idx < 0 && perm) idx = orc_permuter_contains(perm, (const uint8_t*)token.data(), k);
    if (idx >= 0) return idx;
  }
  return -1;
}

}  // namespace

extern "C" {

int64_t shift_assign(const orc_library* lib, const orc_permuter* perm, const uint8_t* read, size_t len, int is_reverse,
                     uint64_t offset, uint32_t max_shift, int rc_mode) {
  return assign_one(lib, perm, read, len, is_reverse, offset, max_shift, rc_mode);
}

// out[i] = library index of record i, or -1; records split over n_threads threads
void shift_assign_records(const orc_records* recs, const orc_library* lib, const orc_permuter* perm, int is_reverse,
                          uint64_t offset, uint32_t max_shift, int rc_mode, int n_threads, int32_t* out) {
  const uint64_t n = orc_records_len(recs);
  if (n_threads < 1) n_threads = 1;
  auto run = [&](uint64_t a, uint64_t b) {
    for (uint64_t i = a; i < b; ++i) {
      uint64_t len = 0;
      const uint8_t* seq = orc_records_seq(recs, i, &len);
      out[i] = (int32_t)assign_one(lib, perm, seq, len, is_reverse, offset, max_shift, rc_mode);
    }
  };
  std::vector<std::thread> pool;
  for (int t = 1; t < n_threads; ++t) pool.emplace_back(run, n * t / n_threads, n * (t + 1) / n_threads);
  run(0, n / n_threads);
  for (auto& th : pool) th.join();
}

}  // extern "C"
