// library.cu — Library::from_reader + Permuter::new as device table build (kernels K2a/K2b),
// and the composed token lookup.
//
// Replaces /root/reference/src/library.rs:17-99 and permutes.rs:47-158.  The reference's
// stateful insert algorithm is order independent in its observable effect (SURVEY.md A.2):
// a token that is not a library member resolves iff exactly ONE library sequence lies at
// Hamming distance 1.  Nothing but the n members is stored (common.cuh): the build packs every
// guide 2-bit in both orientations (pack_library), sorts the members into the three seed lists
// of each orientation (seed_count / scan / seed_fill / seed_dir), fills the front tables
// (front_insert), and then asks the finished index for duplicates (duplicate_check) and for the
// Permuter's map / null sizes (variant_stats).  Variants — with or without an 'N' — are never
// materialised: a window is resolved against the members at lookup time (lookup_token).
#include <algorithm>
#include <cstdio>
#include <string>
#include <vector>

#include "internal.h"

namespace sgc {

thread_local std::string g_last_error;

int set_error(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
int cuda_error(cudaError_t e, const char* what, const char* file, int line) {
  char buf[512];
  snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d in %s", (int)e, cudaGetErrorString(e), file, line, what);
  cudaGetLastError();  // clear the sticky flag of non-fatal errors
  return set_error(SGC_ERR_CUDA, buf);
}

namespace {

struct BuildStatus {
  unsigned int bad_guide;   // smallest guide index holding a non-ACGT byte, or 0xFFFFFFFF
  unsigned int dup_guide;   // smallest guide index that duplicates an earlier sequence
  unsigned long long n_variants, n_ambiguous;
  unsigned int front_left_out;  // members that did not fit their front-table bucket
};

// K2a: one thread per guide: the interleaved key of the guide as written and of its reverse
// complement (hi << 32 | lo each).
__global__ void pack_library_kernel(const uint8_t* __restrict__ seqs, uint32_t n, uint32_t k, bool wide,
                                    uint64_t* __restrict__ keys_fwd, uint64_t* __restrict__ keys_rev, BuildStatus* st) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint8_t* s = seqs + (size_t)i * k;
  Key f{0, 0}, r{0, 0};
  bool bad = false;
  for (uint32_t j = 0; j < k; ++j) {
    const uint8_t c = s[j];
    bad |= !is_acgt(c);
    key_set_base(f, j, wide, code_of(c));
    key_set_base(r, k - 1 - j, wide, code_of(c) ^ 2u);
  }
  keys_fwd[i] = ((uint64_t)f.hi << 32) | f.lo;
  keys_rev[i] = ((uint64_t)r.hi << 32) | r.lo;
  if (bad) atomicMin(&st->bad_guide, i);
}
__device__ __forceinline__ Key as_key(uint64_t w) { return Key{(uint32_t)w, (uint32_t)(w >> 32)}; }

// ---- seed index ---------------------------------------------------------------------------
struct SeedArrays {
  uint32_t* a[kSeeds];
};

// pass 1: members per bucket
__global__ void seed_count_kernel(const uint64_t* __restrict__ keys, uint32_t n, uint32_t dir_shift, SeedParts parts,
                                  SeedArrays cnt) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Key key = as_key(keys[i]);
#pragma unroll
  for (int s = 0; s < kSeeds; ++s) atomicAdd(cnt.a[s] + (seed_hash(seed_of(parts, key, s)) >> dir_shift), 1u);
}

// pass 2: exclusive prefix sum of the counts (three small kernels: tile sums, scan of the
// tile sums by one block, tile scan + carry-in)
constexpr int kScanThreads = 256;
constexpr int kScanPerThread = 8;
constexpr int kScanTile = kScanThreads * kScanPerThread;

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total) {
  __shared__ uint32_t warp_sums[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += t;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = lane < (int)(blockDim.x >> 5) ? warp_sums[lane] : 0;
    uint32_t winc = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, winc, d);
      if (lane >= d) winc += t;
    }
    warp_sums[lane] = winc - w;  // exclusive
    if (lane == 31 && total) *total = winc;
  }
  __syncthreads();
  const uint32_t r = warp_sums[warp] + inc - v;
  __syncthreads();
  return r;
}

__global__ void __launch_bounds__(kScanThreads) scan_tile_sums_kernel(const uint32_t* __restrict__ cnt, uint32_t n,
                                                                      uint32_t* __restrict__ tile_sums) {
  const uint32_t base = blockIdx.x * kScanTile + threadIdx.x * kScanPerThread;
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < kScanPerThread; ++j)
    if (base + j < n) s += cnt[base + j];
  __shared__ uint32_t total;
  block_exclusive_scan(s, &total);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

// one block: exclusive scan of the tile sums, in place
__global__ void __launch_bounds__(kScanThreads) scan_sums_kernel(uint32_t* sums, uint32_t n_tiles) {
  __shared__ uint32_t carry, total;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (uint32_t base = 0; base < n_tiles; base += kScanThreads) {
    const uint32_t i = base + threadIdx.x;
    const uint32_t v = i < n_tiles ? sums[i] : 0;
    const uint32_t ex = block_exclusive_scan(v, &total);
    if (i < n_tiles) sums[i] = carry + ex;
    __syncthreads();
    if (threadIdx.x == 0) carry += total;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kScanThreads) scan_tiles_kernel(const uint32_t* __restrict__ cnt, uint32_t n,
                                                                  const uint32_t* __restrict__ tile_sums,
                                                                  uint32_t* __restrict__ start) {
  const uint32_t base = blockIdx.x * kScanTile + threadIdx.x * kScanPerThread;
  uint32_t v[kScanPerThread], s = 0;
#pragma unroll
  for (int j = 0; j < kScanPerThread; ++j) {
    v[j] = base + j < n ? cnt[base + j] : 0;
    s += v[j];
  }
  uint32_t run = tile_sums[blockIdx.x] + block_exclusive_scan(s, nullptr);
#pragma unroll
  for (int j = 0; j < kScanPerThread; ++j) {
    if (base + j < n) start[base + j] = run;
    run += v[j];
  }
}

// pass 3: postings.  `cursor` starts as a copy of `start`; the order inside one bucket is
// whatever the atomics give, which no lookup depends on.
template <bool WIDE>
__global__ void seed_fill_kernel(const uint64_t* __restrict__ keys, uint32_t n, uint32_t dir_shift, SeedParts parts,
                                 SeedArrays cursor, uint64_t* __restrict__ post) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t w = keys[i];
  const Key key = as_key(w);
#pragma unroll
  for (int s = 0; s < kSeeds; ++s) {
    const size_t a = (size_t)s * n + atomicAdd(cursor.a[s] + (seed_hash(seed_of(parts, key, s)) >> dir_shift), 1u);
    if (WIDE) {
      post[2 * a] = w;
      post[2 * a + 1] = i;
    } else {
      post[a] = w | ((uint64_t)i << kPostIdxShift);  // hi has 8 bits
    }
  }
}

// pass 4: directory entries; a bucket with one posting carries the posting itself.
// wide keys: two words per entry
__global__ void seed_dir128_kernel(const uint32_t* __restrict__ start, const uint32_t* __restrict__ cnt,
                                   const uint64_t* __restrict__ post, ulonglong2* __restrict__ dir, uint32_t n_entries) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_entries) return;
  const uint32_t c = cnt[i];
  ulonglong2 e{0ull, 0ull};
  if (c == 1) {
    e.x = kDirKindInline | (post[2 * (size_t)start[i]] & (kDirKindInline - 1));
    e.y = post[2 * (size_t)start[i] + 1];
  } else if (c >= 2) {
    e.x = kDirKindRun;
    e.y = start[i] | ((uint64_t)c << 22);
  }
  dir[i] = e;
}

// narrow keys: one word per entry
__global__ void seed_dir64_kernel(const uint32_t* __restrict__ start, const uint32_t* __restrict__ cnt,
                                  const uint64_t* __restrict__ post, uint64_t* __restrict__ dir, uint32_t n_entries) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_entries) return;
  const uint32_t c = cnt[i];
  uint64_t e = 0;
  if (c == 1)
    e = kDirKindInline | (post[start[i]] & (kDirKindInline - 1));
  else if (c >= 2)
    e = kDirKindRun | start[i] | ((uint64_t)c << 22);
  dir[i] = e;
}

// ---- checks and statistics through the finished (forward) index -----------------------------
// duplicate sequences (library.rs:91-95): the later of two equal records reports itself
template <bool WIDE>
__global__ void duplicate_check_kernel(LibView v, const uint64_t* __restrict__ keys, BuildStatus* st) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= v.n) return;
  const Key key = as_key(keys[i]);
  const uint64_t pol = l2_evict_last_policy();
  bool dup = false;
  for_each_posting<WIDE>(v, v.fwd, 0, key, pol, [&](Key mk, uint32_t idx) {
    if (mk.lo == key.lo && mk.hi == key.hi && idx < i) dup = true;
    return dup;
  });
  if (dup) atomicMin(&st->dup_guide, i);
}

// Permuter statistics: one thread per (guide, position) enumerates the three ACGT
// substitutions (permutes.rs:78-107 without the N column, which needs no storage) and asks
// the index who their parents are.  A variant that is itself a member is unreachable in the
// reference (SURVEY.md A.2); one parent = map entry; two or more = null set, counted once by
// its smallest parent.
template <bool WIDE>
__global__ void variant_stats_kernel(LibView v, const uint64_t* __restrict__ keys, BuildStatus* st) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned var = 0, amb = 0;
  const uint64_t pol = l2_evict_last_policy();
  if (t < (uint64_t)v.n * v.k) {
    const uint32_t i = (uint32_t)(t / v.k), pos = (uint32_t)(t % v.k);
    const Key key = as_key(keys[i]);
    const uint32_t own = key_get_base(key, pos, WIDE);
    for (uint32_t d = 1; d < 4; ++d) {
      Key q = key;
      key_set_base(q, pos, WIDE, own ^ d);
      bool member = false;
      uint32_t parents = 0, smallest = 0xFFFFFFFFu;
      for (int s = 0; s < kSeeds && !member; ++s) {
        const Key qs = seed_of(v.parts, q, s);
        for_each_posting<WIDE>(v, v.fwd, s, q, pol, [&](Key mk, uint32_t idx) {
          const Key ms = seed_of(v.parts, mk, s);
          if (ms.lo != qs.lo || ms.hi != qs.hi) return false;  // another seed in this bucket
          const Key x{mk.lo ^ q.lo, mk.hi ^ q.hi};
          if ((x.lo | x.hi) == 0) member = true;
          if (bases_differing(x) == 1) {
            ++parents;
            smallest = min(smallest, idx);
          }
          return member;
        });
      }
      if (member) continue;
      if (parents == 1) ++var;
      if (parents > 1 && smallest == i) ++amb;
    }
  }
  var = __reduce_add_sync(0xffffffffu, var);
  amb = __reduce_add_sync(0xffffffffu, amb);
  if ((threadIdx.x & 31) == 0) {
    if (var) atomicAdd(&st->n_variants, (unsigned long long)var);
    if (amb) atomicAdd(&st->n_ambiguous, (unsigned long long)amb);
  }
}

// ---- front table ------------------------------------------------------------------------------
// One thread per guide.  A member goes into the first free slot of its home bucket; if the
// bucket is full, or already holds a member with the same `lo` word (the streaming kernel
// selects a slot by `lo` alone), it is left out and the bucket is flagged.
template <bool WIDE>
__global__ void front_insert_kernel(uint64_t* table_, uint32_t front_shift, const uint64_t* __restrict__ keys,
                                    uint32_t n, BuildStatus* st) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long* table = reinterpret_cast<unsigned long long*>(table_);
  const Key key = as_key(keys[i]);
  const uint32_t b = front_hash(key.lo, key.hi) >> front_shift;
  unsigned long long* bucket = table + (size_t)b * 4;
  const uint64_t meta = kFrontOccupied | ((uint64_t)i << kFrontIdxShift);
  bool placed = false;
  if (!WIDE) {
    const uint64_t val = meta | ((uint64_t)key.hi << 32) | key.lo;
    for (int s = 0; s < 4 && !placed; ++s) {
      unsigned long long cur = atomicCAS(bucket + s, 0ull, (unsigned long long)val);
      if (cur == 0) {
        placed = true;
      } else if ((uint32_t)cur == key.lo) {
        break;  // same lo word as an earlier member: leave this one out
      }
    }
  } else {
    const uint64_t w0 = ((uint64_t)key.hi << 32) | key.lo;
    for (int s = 0; s < 2 && !placed; ++s) {
      // the meta word claims the slot; the key word is written by the claimer and read by
      // nobody until the build has finished
      unsigned long long cur = atomicCAS(bucket + 2 * s + 1, 0ull, (unsigned long long)meta);
      if (cur == 0) {
        bucket[2 * s] = w0;
        placed = true;
      }
    }
  }
  if (!placed) {
    atomicOr(bucket + (WIDE ? 1 : 0), (unsigned long long)kFrontFlag);
    atomicAdd(&st->front_left_out, 1u);
  }
}

// composed lookup of raw k-byte tokens (sgc_library_lookup)
__global__ void lookup_tokens_kernel(LibView v, bool with_perm, const uint8_t* __restrict__ tokens,
                                     uint64_t n_tokens, int32_t* __restrict__ idx_out, uint8_t* __restrict__ kind_out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_tokens) return;
  const uint8_t* s = tokens + i * v.k;
  Key key{0, 0};
  int nbad = 0;
  uint32_t bad_pos = 0;
  bool wild = false;
  for (uint32_t j = 0; j < v.k; ++j) {
    uint8_t c = s[j];
    key_set_base(key, j, v.wide, code_of(c));
    if (!is_acgt(c)) {
      ++nbad;
      bad_pos = j;
      wild = (c == 'N');
    }
  }
  int kind = 0;
  const uint64_t pol = l2_evict_last_policy();
  int32_t hit = v.wide ? window_lookup_t<true>(v, v.fwd, with_perm, key, nbad, bad_pos, wild, &kind, pol)
                       : window_lookup_t<false>(v, v.fwd, with_perm, key, nbad, bad_pos, wild, &kind, pol);
  idx_out[i] = hit;
  if (kind_out) kind_out[i] = hit == kMiss ? 0 : (uint8_t)kind;
}

template <typename T>
struct DeviceBuffer {
  T* p = nullptr;
  ~DeviceBuffer() {
    if (p) cudaFree(p);
  }
  cudaError_t alloc(size_t n) { return cudaMalloc(&p, n * sizeof(T)); }
};

inline unsigned blocks_for(uint64_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

}  // namespace
}  // namespace sgc

using namespace sgc;

extern "C" {

const char* sgc_last_error(void) { return g_last_error.c_str(); }
int sgc_abi_version(void) { return SGC_ABI_VERSION; }

int sgc_device_count(int* n) {
  if (!n) return set_error(SGC_ERR_INVALID_ARG, "n is NULL");
  SGC_CUDA_TRY(cudaGetDeviceCount(n));
  return SGC_OK;
}

int sgc_device_memory(int device, uint64_t* free_bytes, uint64_t* total_bytes) {
  if (!free_bytes || !total_bytes) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  DeviceGuard guard(device);
  if (!guard.ok()) return set_error(SGC_ERR_CUDA, "no such device");
  size_t f = 0, t = 0;
  SGC_CUDA_TRY(cudaMemGetInfo(&f, &t));
  *free_bytes = f;
  *total_bytes = t;
  return SGC_OK;
}

int sgc_host_alloc(void** ptr, size_t bytes) {
  if (!ptr) return set_error(SGC_ERR_INVALID_ARG, "ptr is NULL");
  SGC_CUDA_TRY(cudaHostAlloc(ptr, bytes, cudaHostAllocPortable));
  return SGC_OK;
}
int sgc_host_free(void* ptr) {
  SGC_CUDA_TRY(cudaFreeHost(ptr));
  return SGC_OK;
}

void sgc_library_destroy(sgc_library* lib) {
  if (!lib) return;
  DeviceGuard g(lib->device);
  for (int o = 0; o < 2; ++o) {
    for (int i = 0; i < kSeeds; ++i) {
      cudaFree(lib->ix[o].d_dir64[i]);
      cudaFree(lib->ix[o].d_dir128[i]);
    }
    cudaFree(lib->ix[o].d_post);
    cudaFree(lib->ix[o].d_front);
    cudaFree(lib->ix[o].d_keys);
  }
  opaque_destroy(lib);
  cudaFree(lib->d_lib_hist);
  delete lib;
}

}  // extern "C"

namespace sgc {
int exclusive_scan_u32(const uint32_t* d_cnt, uint32_t n, uint32_t* d_start, uint32_t* d_tile_sums, cudaStream_t stream) {
  const uint32_t tiles = (n + kScanTile - 1) / kScanTile;
  scan_tile_sums_kernel<<<tiles, kScanThreads, 0, stream>>>(d_cnt, n, d_tile_sums);
  scan_sums_kernel<<<1, kScanThreads, 0, stream>>>(d_tile_sums, tiles);
  scan_tiles_kernel<<<tiles, kScanThreads, 0, stream>>>(d_cnt, n, d_tile_sums, d_start);
  SGC_CUDA_TRY(cudaGetLastError());
  return SGC_OK;
}
}  // namespace sgc

namespace {

// temporaries of one build, allocated before the timed region
struct BuildScratch {
  DeviceBuffer<uint32_t> start[kSeeds], cur[kSeeds], cnt[kSeeds], sums;
  int alloc(uint32_t entries) {
    SGC_CUDA_TRY(sums.alloc((entries + kScanTile - 1) / kScanTile + 1));
    for (int i = 0; i < kSeeds; ++i) {
      SGC_CUDA_TRY(start[i].alloc(entries));
      SGC_CUDA_TRY(cur[i].alloc(entries));
      SGC_CUDA_TRY(cnt[i].alloc(entries));
    }
    return SGC_OK;
  }
};

// seed index + front table of one orientation
template <bool WIDE>
int build_index(sgc_library* lib, int o, BuildScratch& sc, BuildStatus* d_st) {
  const uint32_t n = lib->n;
  const unsigned T = 256;
  const uint32_t entries = 1u << (32 - lib->dir_shift);
  sgc_library::Index& ix = lib->ix[o];
  SeedArrays cnt, cursor;
  for (int i = 0; i < kSeeds; ++i) {
    SGC_CUDA_TRY(cudaMemsetAsync(sc.cnt[i].p, 0, (size_t)entries * 4, 0));
    cnt.a[i] = sc.cnt[i].p;
    cursor.a[i] = sc.cur[i].p;
  }
  seed_count_kernel<<<blocks_for(n, T), T>>>(ix.d_keys, n, lib->dir_shift, lib->parts, cnt);
  for (int i = 0; i < kSeeds; ++i) {
    int rc = exclusive_scan_u32(sc.cnt[i].p, entries, sc.start[i].p, sc.sums.p);
    if (rc) return rc;
    SGC_CUDA_TRY(cudaMemcpyAsync(sc.cur[i].p, sc.start[i].p, (size_t)entries * 4, cudaMemcpyDeviceToDevice, 0));
  }
  seed_fill_kernel<WIDE><<<blocks_for(n, T), T>>>(ix.d_keys, n, lib->dir_shift, lib->parts, cursor, ix.d_post);
  for (int i = 0; i < kSeeds; ++i) {
    if (WIDE)
      seed_dir128_kernel<<<blocks_for(entries, T), T>>>(sc.start[i].p, sc.cnt[i].p, ix.d_post + 2 * (size_t)i * n,
                                                        ix.d_dir128[i], entries);
    else
      seed_dir64_kernel<<<blocks_for(entries, T), T>>>(sc.start[i].p, sc.cnt[i].p, ix.d_post + (size_t)i * n,
                                                       ix.d_dir64[i], entries);
  }
  SGC_CUDA_TRY(cudaMemsetAsync(ix.d_front, 0, lib->front_bytes, 0));
  front_insert_kernel<WIDE><<<blocks_for(n, T), T>>>(ix.d_front, lib->front_shift, ix.d_keys, n, d_st);
  SGC_CUDA_TRY(cudaGetLastError());
  return SGC_OK;
}

template <bool WIDE>
int build_tables(sgc_library* lib, BuildScratch& sc, BuildStatus* d_st) {
  const unsigned T = 256;
  for (int o = 0; o < 2; ++o) {
    int rc = build_index<WIDE>(lib, o, sc, d_st);
    if (rc) return rc;
  }
  const LibView v = lib->view();
  duplicate_check_kernel<WIDE><<<blocks_for(lib->n, T), T>>>(v, lib->ix[0].d_keys, d_st);
  if (lib->with_perm)
    variant_stats_kernel<WIDE><<<blocks_for((uint64_t)lib->n * lib->k, T), T>>>(v, lib->ix[0].d_keys, d_st);
  SGC_CUDA_TRY(cudaGetLastError());
  return SGC_OK;
}

}  // namespace

extern "C" {

int sgc_library_create(int device, const uint8_t* seqs, uint32_t n, uint32_t k, int with_permutations,
                       sgc_library** out) {
  if (!seqs || !out) return set_error(SGC_ERR_INVALID_ARG, "seqs/out is NULL");
  if (n == 0) return set_error(SGC_ERR_EMPTY_READER, "empty library (library.rs:74 unwraps on an empty table)");
  if (k == 0 || k > kMaxKOpaque) return set_error(SGC_ERR_K_UNSUPPORTED, "guide length must be 1..1024");
  if (n > SGC_MAX_GUIDES) return set_error(SGC_ERR_TOO_MANY_GUIDES, "too many guides");
  int ndev = 0;
  SGC_CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return set_error(SGC_ERR_INVALID_ARG, "no such device");
  DeviceGuard guard(device);
  if (!guard.ok()) return set_error(SGC_ERR_CUDA, "cudaSetDevice failed");

  sgc_library* lib = new sgc_library();
  lib->device = device;
  lib->n = n;
  lib->k = k;
  lib->with_perm = with_permutations != 0;
  // The 2-bit tables hold A,C,G,T guides of up to 30 bases.  Anything else the reference accepts
  // (library.rs keeps opaque byte strings) goes through the byte-keyed index of opaque.cu.
  lib->opaque = k > kMaxK;
  for (size_t i = 0, total = (size_t)n * k; i < total && !lib->opaque; ++i) lib->opaque = !is_acgt(seqs[i]);
  lib->wide = k > kNarrowMaxK;
  if (!lib->opaque) lib->parts = make_seed_parts(k, lib->wide);
  struct Cleanup {
    sgc_library* l;
    ~Cleanup() {
      if (l) sgc_library_destroy(l);
    }
  } cleanup{lib};
  SGC_CUDA_TRY(cudaDeviceGetAttribute(&lib->sm_count, cudaDevAttrMultiProcessorCount, device));

  // each directory has a power of two of buckets, at least four per member (<= 2^24)
  uint32_t dir_bits = 8;
  while (((uint64_t)1 << dir_bits) < 4ull * n) ++dir_bits;
  lib->dir_shift = 32 - dir_bits;
  const size_t dir_entries = (size_t)1 << dir_bits;
  const size_t post_words = (size_t)n * (lib->wide ? 2 : 1);
  // front table: 32-byte buckets, a power of two of them, about one member per bucket
  // (narrow, 4 slots) or one per two buckets (wide, 2 slots)
  uint32_t log_buckets = 6;
  while (((uint64_t)1 << log_buckets) < (uint64_t)n * (lib->wide ? 2 : 1)) ++log_buckets;
  lib->front_shift = 32 - log_buckets;
  lib->front_bytes = ((size_t)1 << log_buckets) * 32;

  DeviceBuffer<uint8_t> d_seqs;
  DeviceBuffer<BuildStatus> d_st;
  BuildScratch scratch;
  SGC_CUDA_TRY(d_seqs.alloc((size_t)n * k));
  SGC_CUDA_TRY(d_st.alloc(1));
  int rc = lib->opaque ? SGC_OK : scratch.alloc((uint32_t)dir_entries);
  if (rc) return rc;
  for (int o = 0; o < 2 && !lib->opaque; ++o) {
    sgc_library::Index& ix = lib->ix[o];
    SGC_CUDA_TRY(cudaMalloc(&ix.d_keys, (size_t)n * sizeof(uint64_t)));
    for (int i = 0; i < kSeeds; ++i) {
      if (lib->wide)
        SGC_CUDA_TRY(cudaMalloc(&ix.d_dir128[i], dir_entries * 16));
      else
        SGC_CUDA_TRY(cudaMalloc(&ix.d_dir64[i], dir_entries * 8));
    }
    SGC_CUDA_TRY(cudaMalloc(&ix.d_post, kSeeds * post_words * 8));
    SGC_CUDA_TRY(cudaMalloc(&ix.d_front, lib->front_bytes));
  }
  SGC_CUDA_TRY(cudaMalloc(&lib->d_lib_hist, (size_t)k * 4 * sizeof(uint32_t)));
  SGC_CUDA_TRY(cudaMemcpy(d_seqs.p, seqs, (size_t)n * k, cudaMemcpyHostToDevice));
  BuildStatus st0{0xFFFFFFFFu, 0xFFFFFFFFu, 0, 0, 0};
  SGC_CUDA_TRY(cudaMemcpy(d_st.p, &st0, sizeof st0, cudaMemcpyHostToDevice));

  struct Events {
    cudaEvent_t a = nullptr, b = nullptr;
    ~Events() {
      if (a) cudaEventDestroy(a);
      if (b) cudaEventDestroy(b);
    }
  } events;
  SGC_CUDA_TRY(cudaEventCreate(&events.a));
  SGC_CUDA_TRY(cudaEventCreate(&events.b));
  const cudaEvent_t e0 = events.a, e1 = events.b;
  SGC_CUDA_TRY(cudaEventRecord(e0, 0));
  uint64_t o_variants = 0, o_ambiguous = 0;
  uint32_t o_dup = 0xFFFFFFFFu;
  if (lib->opaque) {
    rc = opaque_build(lib, d_seqs.p, &o_variants, &o_ambiguous, &o_dup);
  } else {
    pack_library_kernel<<<blocks_for(n, 256), 256>>>(d_seqs.p, n, k, lib->wide, lib->ix[0].d_keys, lib->ix[1].d_keys,
                                                     d_st.p);
    rc = lib->wide ? build_tables<true>(lib, scratch, d_st.p) : build_tables<false>(lib, scratch, d_st.p);
  }
  if (rc) return rc;
  // library positional histogram for the offset detector: records 1..n-1 (offsetter.rs:57,190-191)
  SGC_CUDA_TRY(cudaMemsetAsync(lib->d_lib_hist, 0, (size_t)k * 4 * sizeof(uint32_t), 0));
  if (n > 1) {
    rc = position_counts_device(d_seqs.p + k, nullptr, k, k, n - 1, k, lib->d_lib_hist, 0);
    if (rc) return rc;
  }
  SGC_CUDA_TRY(cudaEventRecord(e1, 0));
  SGC_CUDA_TRY(cudaGetLastError());
  SGC_CUDA_TRY(cudaEventSynchronize(e1));
  float ms = 0;
  SGC_CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));

  BuildStatus st;
  SGC_CUDA_TRY(cudaMemcpy(&st, d_st.p, sizeof st, cudaMemcpyDeviceToHost));
  if (lib->opaque) {
    st.dup_guide = o_dup;
    st.n_variants = o_variants;
    st.n_ambiguous = o_ambiguous;
  }
  if (st.bad_guide != 0xFFFFFFFFu) {
    char buf[160];
    snprintf(buf, sizeof buf, "library sequence %u holds a byte outside A,C,G,T", st.bad_guide);
    return set_error(SGC_ERR_NON_ACGT_LIBRARY, buf);
  }
  if (st.dup_guide != 0xFFFFFFFFu) {
    std::string s((const char*)seqs + (size_t)st.dup_guide * k, k);
    return set_error(SGC_ERR_DUPLICATE_SEQUENCE, "Unexpected duplicate sequence in library found: " + s);
  }
  lib->info.n_guides = n;
  lib->info.k = k;
  lib->info.with_permutations = lib->with_perm;
  lib->info.device = device;
  lib->info.n_variants = st.n_variants;
  lib->info.n_ambiguous = st.n_ambiguous;
  lib->info.opaque = lib->opaque;
  if (!lib->opaque) {
    lib->info.n_slots = ((size_t)1 << log_buckets) * (lib->wide ? 2 : 4);
    // what one counter touches: the directories, postings and front table of its orientation
    lib->info.table_bytes = kSeeds * (dir_entries * (lib->wide ? 16 : 8) + post_words * 8) + lib->front_bytes;
  }
  lib->info.build_ms = ms;
  lib->info.front_left_out = st.front_left_out;
  cleanup.l = nullptr;
  *out = lib;
  return SGC_OK;
}

int sgc_library_get_info(const sgc_library* lib, sgc_library_info* out) {
  if (!lib || !out) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  *out = lib->info;
  return SGC_OK;
}

int sgc_library_lookup(const sgc_library* lib, const uint8_t* tokens, uint64_t n_tokens, int32_t* idx_out,
                       uint8_t* kind_out) {
  if (!lib || !tokens || !idx_out) return set_error(SGC_ERR_INVALID_ARG, "NULL argument");
  if (n_tokens == 0) return SGC_OK;
  DeviceGuard guard(lib->device);
  DeviceBuffer<uint8_t> d_tok, d_kind;
  DeviceBuffer<int32_t> d_idx;
  SGC_CUDA_TRY(d_tok.alloc(n_tokens * lib->k));
  SGC_CUDA_TRY(d_idx.alloc(n_tokens));
  if (kind_out) SGC_CUDA_TRY(d_kind.alloc(n_tokens));
  SGC_CUDA_TRY(cudaMemcpy(d_tok.p, tokens, n_tokens * lib->k, cudaMemcpyHostToDevice));
  if (lib->opaque) {
    int rc = opaque_lookup_tokens(lib, d_tok.p, n_tokens, d_idx.p, d_kind.p);
    if (rc) return rc;
  } else {
    lookup_tokens_kernel<<<blocks_for(n_tokens, 256), 256>>>(lib->view(), lib->with_perm, d_tok.p, n_tokens, d_idx.p,
                                                              d_kind.p);
    SGC_CUDA_TRY(cudaGetLastError());
  }
  SGC_CUDA_TRY(cudaMemcpy(idx_out, d_idx.p, n_tokens * sizeof(int32_t), cudaMemcpyDeviceToHost));
  if (kind_out) SGC_CUDA_TRY(cudaMemcpy(kind_out, d_kind.p, n_tokens, cudaMemcpyDeviceToHost));
  return SGC_OK;
}

}  // extern "C"
