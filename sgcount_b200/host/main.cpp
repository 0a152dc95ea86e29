// sgcount (B200 host) — the reference's command line (main.rs:54-203) and run driver
// (count.rs:15-148) over libsgcount_cuda.so.  Everything that touches a read runs on the GPU
// through the C ABI of include/sgcount_cuda.h; this program parses FASTA/FASTQ(.gz), keeps the
// alias strings and writes the count table (results.rs:32-99, genemap.rs:53-86).
//
//   sgcount -l <library> -i <sample>... [-n names...] [-o out] [-g gene map] [-a N [-r]] [-p]
//           [-x] [-s N] [-t N] [-q] [-z]   [--gpus N] [--device D] [--rc-keep-n]
//
// Differences from the reference, all documented in DESIGN.md: rows are written in library-file
// order (the reference iterates a randomly seeded HashMap); `-t` sets the number of samples
// processed concurrently (one host pipeline and one CUDA stream per counter each), `--gpus` spreads the samples over devices and, when there are fewer
// samples than devices, cuts every sample into read shards over gpus / samples devices whose
// count vectors are summed with sgc_reduce_counts (NCCL).
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <fstream>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "../../include/sgcount_cuda.h"
#include "fastx.h"
#include "inflate.h"

namespace {

struct Fatal : std::runtime_error {
  using std::runtime_error::runtime_error;
};

[[noreturn]] void fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  throw Fatal(buf);
}

void check(int rc) {
  if (rc != SGC_OK) fail("%s", sgc_last_error());
}

struct Args {
  std::string library_path;
  std::vector<std::string> input_paths, sample_names;
  bool have_names = false;
  std::string output_path, genemap;
  bool have_offset = false;
  unsigned long offset = 0;
  bool no_position_recursion = false, reverse = false, exact = false, quiet = false, include_zero = false;
  unsigned long subsample = 5000;
  unsigned threads = 1;
  int gpus = 1, device = 0;
  unsigned read_shards = 0;     // counters per sample; 0 = gpus / samples (at least 1)
  unsigned ingest_threads = 0;  // inflate threads per sample; 0 = hardware threads / concurrent samples
  bool timing = false;
  bool whole_lines = false;  // never frame span records
  bool host_inflate = false; // never inflate on the device
  int rc_mode = SGC_RC_BITTRICK;
};

const char* kUsage =
    "Usage: sgcount [OPTIONS] --library-path <LIBRARY_PATH> --input-paths <INPUT_PATHS>...\n\n"
    "Options:\n"
    "  -l, --library-path <LIBRARY_PATH>      Filepath of the library\n"
    "  -i, --input-paths <INPUT_PATHS>...     Filepath(s) of fastx (fastq, fasta, *.gz) sequences to map\n"
    "  -n, --sample-names <SAMPLE_NAMES>...   Sample Names\n"
    "  -o, --output-path <OUTPUT_PATH>        Output filepath [default: stdout]\n"
    "  -g, --genemap <GENEMAP>                Gene to sgRNA mapping\n"
    "  -a, --offset <OFFSET>                  Adapter Offset\n"
    "  -p, --no-position-recursion            Remove Position Recursion (i.e. offseting sequences by +/- 1 on mismatch condition)\n"
    "  -r, --reverse                          Read Direction (reverse complement reads)\n"
    "  -x, --exact                            Disallow One Off Mismatch\n"
    "  -s, --subsample <SUBSAMPLE>            Number of Reads to Subsample in Determining Offset [default: 5000]\n"
    "  -t, --threads <THREADS>                Number of Threads to Use for Parallel Jobs [default: 1]; samples counted at once (at least one per device, and four per device when every input is inflated on the device, within each device's free memory)\n"
    "  -q, --quiet                            Does not show progress\n"
    "  -z, --include-zero                     Include zero count sgRNAs in output table\n"
    "      --gpus <N>                         Spread the samples (and, with fewer samples than devices, read shards of each sample) over N devices [default: 1]\n"
    "      --read-shards <N>                  Cut every sample into N read shards, dealt round the devices and summed with an NCCL reduce [default: gpus / samples when there are fewer samples than devices and an input of 1 GiB or more, else 1]\n"
    "      --device <D>                       First device to use [default: 0]\n"
    "      --ingest-threads <N>               Threads inflating the gzip members of one sample [default: cores / samples in flight]\n"
    "      --rc-keep-n                        Reverse complement keeps N (default: the fxread bit trick, N -> J)\n"
    "      --whole-lines                      Copy whole sequence lines to the device (default: for fixed-length reads, only the guide window and one byte either side)\n"
    "      --host-inflate                     Inflate and frame records on the host even for BGZF, single-member or multi-member gzip input (default: BGZF files of FASTQ, and gzip files of FASTQ that are one member, are inflated, framed and counted on the device; so are multi-member gzip files large enough and with too few members or ingest threads for the host to decode them faster side by side)\n"
    "      --timing                           Print a JSON line with the phase times to stderr\n"
    "  -h, --help                             Print help\n";

unsigned long parse_uint(const std::string& flag, const char* v) {
  char* end = nullptr;
  if (!v || !*v || *v == '-') fail("invalid value for '%s'", flag.c_str());
  unsigned long x = strtoul(v, &end, 10);
  if (*end) fail("invalid value '%s' for '%s'", v, flag.c_str());
  return x;
}

Args parse_args(int argc, char** argv) {
  Args a;
  auto is_flag = [](const char* s) { return s[0] == '-' && s[1] != '\0'; };
  for (int i = 1; i < argc; ++i) {
    std::string f = argv[i];
    auto value = [&]() -> const char* {
      if (i + 1 >= argc) fail("a value is required for '%s' but none was supplied", f.c_str());
      return argv[++i];
    };
    auto values = [&](std::vector<std::string>& out) {  // clap num_args = 1..
      while (i + 1 < argc && !is_flag(argv[i + 1])) out.push_back(argv[++i]);
      if (out.empty()) fail("a value is required for '%s' but none was supplied", f.c_str());
    };
    if (f == "-l" || f == "--library-path") a.library_path = value();
    else if (f == "-i" || f == "--input-paths") values(a.input_paths);
    else if (f == "-n" || f == "--sample-names") { values(a.sample_names); a.have_names = true; }
    else if (f == "-o" || f == "--output-path") a.output_path = value();
    else if (f == "-g" || f == "--genemap") a.genemap = value();
    else if (f == "-a" || f == "--offset") { a.offset = parse_uint(f, value()); a.have_offset = true; }
    else if (f == "-p" || f == "--no-position-recursion") a.no_position_recursion = true;
    else if (f == "-r" || f == "--reverse") a.reverse = true;
    else if (f == "-x" || f == "--exact") a.exact = true;
    else if (f == "-s" || f == "--subsample") a.subsample = parse_uint(f, value());
    else if (f == "-t" || f == "--threads") a.threads = (unsigned)parse_uint(f, value());
    else if (f == "-q" || f == "--quiet") a.quiet = true;
    else if (f == "-z" || f == "--include-zero") a.include_zero = true;
    else if (f == "--gpus") a.gpus = (int)parse_uint(f, value());
    else if (f == "--read-shards") a.read_shards = (unsigned)parse_uint(f, value());
    else if (f == "--device") a.device = (int)parse_uint(f, value());
    else if (f == "--ingest-threads") a.ingest_threads = (unsigned)parse_uint(f, value());
    else if (f == "--rc-keep-n") a.rc_mode = SGC_RC_KEEP_N;
    else if (f == "--timing") a.timing = true;
    else if (f == "--whole-lines") a.whole_lines = true;
    else if (f == "--host-inflate") a.host_inflate = true;
    else if (f == "-h" || f == "--help") { fputs(kUsage, stdout); exit(0); }
    else fail("unexpected argument '%s' found", f.c_str());
  }
  if (a.library_path.empty()) fail("the following required arguments were not provided:\n  --library-path <LIBRARY_PATH>");
  if (a.input_paths.empty()) fail("the following required arguments were not provided:\n  --input-paths <INPUT_PATHS>...");
  if (a.threads == 0) a.threads = 1;
  if (a.gpus < 1) a.gpus = 1;
  return a;
}

bool exists(const std::string& p) {
  FILE* f = fopen(p.c_str(), "rb");
  if (f) fclose(f);
  return f != nullptr;
}

// utils.rs:18-49
std::vector<std::string> generate_sample_names(const std::vector<std::string>& paths) {
  auto trim = [](std::string& s, const char* suffix) {
    const size_t n = strlen(suffix);
    while (s.size() >= n && s.compare(s.size() - n, n, suffix) == 0) s.erase(s.size() - n);  // trim_end_matches repeats
  };
  std::vector<std::string> base, simple;
  std::unordered_set<std::string> seen;
  for (size_t i = 0; i < paths.size(); ++i) {
    std::string b = paths[i].substr(paths[i].find_last_of('/') == std::string::npos ? 0 : paths[i].find_last_of('/') + 1);
    for (const char* suf : {".gz", ".fasta", ".fastq", ".fa", ".fq"}) trim(b, suf);
    base.push_back(b);
    seen.insert(b);
    simple.push_back("Sample." + std::to_string(i));
  }
  if (seen.size() == base.size()) return base;
  fprintf(stderr, "WARNING: Duplicate Basenames Detected, Using incrementing sample names\n");
  return simple;
}

// library.rs:17-99: sequences and aliases in file order
struct HostLibrary {
  std::vector<std::string> aliases;
  std::string seqs;  // n * k bytes
  uint32_t n = 0, k = 0;
};

HostLibrary load_library(const std::string& path) {
  HostLibrary lib;
  sgh::FastxReader reader(path);
  const char *id, *seq;
  size_t id_len, seq_len;
  bool inconsistent = false;
  while (reader.next(id, id_len, seq, seq_len)) {
    if (lib.n == 0) lib.k = (uint32_t)seq_len;
    if (seq_len != lib.k) inconsistent = true;
    lib.aliases.emplace_back(id, id_len);
    if (!inconsistent) lib.seqs.append(seq, seq_len);
    ++lib.n;
  }
  if (lib.n == 0) fail("empty library: %s", path.c_str());  // library.rs:74 unwraps
  if (inconsistent) fail("Library sequence sizes are inconsistent");  // library.rs:83
  return lib;
}

// genemap.rs:53-86
std::unordered_map<std::string, std::string> load_genemap(const std::string& path) {
  if (!exists(path)) fail("Provided gene mapping path doesn't exist: %s", path.c_str());
  std::ifstream in(path, std::ios::binary);
  std::unordered_map<std::string, std::string> map;
  std::string line;
  while (std::getline(in, line)) {
    if (!line.empty() && line.back() == '\r') line.pop_back();  // for_byte_line strips "\r\n" too (genemap.rs:55)
    const size_t tab = line.find('\t');
    if (tab == std::string::npos) fail("Missing '\\t' in gene map");
    std::string sgrna = line.substr(tab + 1);
    if (!map.emplace(sgrna, line.substr(0, tab)).second) fail("Duplicate sgRNA key found in gene map: %s", sgrna.c_str());
  }
  return map;
}

// The counting thread's copy of a member's sequence lines into pinned memory is the one serial
// stretch of the ingest; big copies are cut in four.
void copy_lines(uint8_t* dst, const char* src, size_t bytes) {
  constexpr size_t kParallelFrom = 8u << 20;
  constexpr int kParts = 4;
  if (bytes < kParallelFrom) {
    memcpy(dst, src, bytes);
    return;
  }
  const size_t part = (bytes / kParts + 4095) & ~(size_t)4095;
  std::thread helpers[kParts - 1];
  for (int i = 1; i < kParts; ++i) {
    const size_t at = std::min(bytes, part * i), n = std::min(bytes - at, part);
    helpers[i - 1] = std::thread([=] { memcpy(dst + at, src + at, n); });
  }
  memcpy(dst, src, std::min(bytes, part));
  for (auto& t : helpers) t.join();
}

// Sequence lines of a run of records, as the kernels take them (pinned host memory).
struct Batch {
  uint8_t* lines = nullptr;  // pinned
  size_t cap = 0, used = 0;
  std::vector<uint32_t> off;  // n + 1 line starts; kept only once the batch is not uniform
  bool uniform = true;        // every read as long as the first
  size_t first_len = 0;
  size_t stride = 0;          // bytes per record while uniform (first_len + 1, or the span stride)
  uint64_t n = 0;

  void reset() {
    used = 0;
    n = 0;
    uniform = true;
    off.clear();
  }
  bool fits(size_t bytes) const { return used + bytes <= cap && used + bytes < (1ull << 32); }
  bool push(const char* seq, size_t len) {
    if (!fits(len + 1)) return false;
    if (n == 0) {
      first_len = len;
      stride = len + 1;
    }
    if (uniform && len != first_len) {  // from here on the kernels need the line starts
      uniform = false;
      off.resize(n + 1);
      for (uint64_t i = 0; i <= n; ++i) off[i] = (uint32_t)(i * (first_len + 1));
    }
    memcpy(lines + used, seq, len);
    lines[used + len] = '\n';
    used += len + 1;
    if (!uniform) off.push_back((uint32_t)used);
    ++n;
    return true;
  }
  // Records [rec, blk.n) of a block, as many as fit; `byte` is where record `rec` starts in the
  // block.  Returns false when the batch is full before the block is used up.
  bool append(const sgh::SeqBlock& blk, uint64_t& rec, size_t& byte) {
    while (rec < blk.n) {
      if (uniform && blk.uniform && (n == 0 || (first_len == blk.first_len && stride == blk.stride))) {
        stride = blk.stride;
        size_t room = cap - used;
        if (used + room >= (1ull << 32)) room = (1ull << 32) - 1 - used;
        const uint64_t fit = std::min<uint64_t>(blk.n - rec, room / stride);
        if (fit == 0) return false;
        copy_lines(lines + used, blk.lines.data() + byte, fit * stride);
        first_len = blk.first_len;
        used += fit * stride;
        n += fit;
        rec += fit;
        byte += fit * stride;
      } else {
        const size_t l = blk.len[rec];
        if (!push(blk.lines.data() + byte, l)) return false;
        ++rec;
        byte += l + 1;
      }
    }
    return true;
  }
};

void submit(sgc_counter* c, const Batch& b) {
  if (b.n == 0) return;
  if (b.uniform)  // fixed stride selects the streaming kernel
    check(sgc_counter_submit(c, b.lines, b.used, nullptr, (uint32_t)b.stride, (uint32_t)b.first_len, b.n));
  else
    check(sgc_counter_submit(c, b.lines, b.used, b.off.data(), 0, 0, b.n));
}

struct OffsetValue {
  bool reverse;
  uint32_t index;
};
std::string to_string(const OffsetValue& o) {
  return std::string(o.reverse ? "Reverse(" : "Forward(") + std::to_string(o.index) + ")";
}

// The first `subsample` records of a sample, read ONCE: validate_library_size looks at the first
// (count.rs:62-71) and entropy_offset at all of them (offsetter.rs:192-200).
struct SampleHead {
  std::vector<uint8_t> lines;
  std::vector<uint32_t> off{0};
  size_t first_len = 0;
  bool any = false;      // the file holds at least one record
  bool fastq = false;    // '@' records (4 lines)
  bool uniform = true;   // every record read so far has first_len bases
  bool bgzf = false;     // the file begins with a BGZF block (a candidate for the device ingest)
};
// Does the file begin with a gzip member that carries a 'BC' extra subfield (BGZF)?
bool begins_with_bgzf_block(const std::string& path) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) return false;
  uint8_t b[12 + 256];
  const size_t got = fread(b, 1, sizeof b, f);
  fclose(f);
  if (got < 18 || b[0] != 0x1f || b[1] != 0x8b || b[2] != 8 || !(b[3] & 4)) return false;
  const size_t xlen = b[10] | ((size_t)b[11] << 8);
  for (size_t at = 12; at + 4 <= std::min(got, 12 + xlen);) {
    const size_t slen = b[at + 2] | ((size_t)b[at + 3] << 8);
    if (b[at] == 'B' && b[at + 1] == 'C' && slen == 2) return true;
    at += 4 + slen;
  }
  return false;
}
SampleHead read_head(const std::string& path, unsigned long records) {
  SampleHead h;
  h.bgzf = begins_with_bgzf_block(path);
  sgh::FastxReader reader(path);
  const char *id, *seq;
  size_t id_len, seq_len;
  for (unsigned long i = 0; i < std::max(records, 1ul) && reader.next(id, id_len, seq, seq_len); ++i) {
    if (i == 0) {
      h.first_len = seq_len;
      h.any = true;
    }
    h.uniform &= seq_len == h.first_len;
    h.fastq = reader.is_fastq();
    if (i >= records) break;
    h.lines.insert(h.lines.end(), seq, seq + seq_len);
    h.lines.push_back('\n');
    h.off.push_back((uint32_t)h.lines.size());
  }
  return h;
}

OffsetValue detect_offset(const sgc_library* lib, const SampleHead& h) {
  int rev = 0;
  uint32_t idx = 0;
  check(sgc_offset_detect(lib, h.lines.data(), h.lines.size(), h.off.data(), 0, 0, h.off.size() - 1, &rev, &idx));
  return OffsetValue{rev != 0, idx};
}

struct SampleResult {
  std::vector<uint64_t> counts;
  uint64_t total = 0, matched = 0;
  // where the counting thread spent its time (--timing): waiting for the inflate threads,
  // copying sequence lines into pinned memory, in sgc_counter_submit / sync / finish
  double wait_s = 0, copy_s = 0, submit_s = 0;
  unsigned shards = 1;  // devices the sample's reads were spread over
  uint64_t span_reads = 0, line_reads = 0;  // reads that travelled as span records / whole lines
  uint64_t members_adopted = 0, members_reframed = 0;  // gzip members framed by their inflate thread / again by the counting thread
  double dev_index_s = 0, dev_create_s = 0, dev_waves_s = 0, dev_finish_s = 0;  // phases of the device ingest
  bool device_ingest = false;               // inflate and record framing ran on the device (BGZF input)
  uint64_t device_blocks = 0;
  uint64_t member_pieces = 0, member_chain = 0, member_absorbed = 0;  // gzip members in pieces on the device
  uint64_t gzip_members = 0;                                          // how many (not BGZF), as the device confirmed them
  unsigned member_lanes = 0;                                          // streams that decoded them together
  std::string host_because;                 // why the device ingest was not used
};

// ---- device ingest: BGZF blocks inflated, framed and counted on the GPU (sgc_fastq_stream_*) ----
// A read-only mapping of a file.
struct MappedFile {
  const uint8_t* data = nullptr;
  size_t size = 0;
  int fd = -1;
  explicit MappedFile(const std::string& path) {
    fd = open(path.c_str(), O_RDONLY);
    struct stat st;
    if (fd < 0 || fstat(fd, &st) != 0) return;
    size = (size_t)st.st_size;
    if (size == 0) return;
    void* p = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
    if (p != MAP_FAILED) data = static_cast<const uint8_t*>(p);
  }
  ~MappedFile() {
    if (data) munmap(const_cast<uint8_t*>(data), size);
    if (fd >= 0) close(fd);
  }
};

using sgh::bgzf_index;  // fastx.h: every BGZF member carries its own size, so the blocks are walked without inflating

// One wave of the device ingest: blocks [first, first + n) of the file, of whose inflated text the
// first head_skip and the last tail_skip bytes belong to the neighbouring waves.
struct Wave {
  size_t first = 0, n = 0;
  uint32_t head_skip = 0, tail_skip = 0;
};

// Cuts the blocks into waves of about `blocks_per_wave` that each start and end on a record
// boundary, so that the waves do not depend on each other and can go to different devices.  A
// block's text starts anywhere inside a record; where a wave is to end, this thread inflates that
// ONE block (64 KB) and looks for the last complete record in it (fastq_last_record_end); the block
// then belongs to both waves, each skipping the other's part.  False when no boundary can be
// found near a cut (the caller then submits the blocks as one dependent sequence).
bool plan_waves(const uint8_t* file, const std::vector<uint64_t>& begin, const std::vector<uint32_t>& isize,
                size_t blocks_per_wave, uint64_t text_per_wave, std::vector<Wave>& waves) {
  const size_t n_blocks = isize.size();
  size_t a = 0;
  uint32_t head_skip = 0;
  while (a < n_blocks) {
    size_t b = a;
    uint64_t text = 0;
    while (b < n_blocks && b - a < blocks_per_wave && text + isize[b] < text_per_wave) text += isize[b++];
    if (b == a) b = a + 1;
    Wave w;
    w.first = a;
    w.head_skip = head_skip;
    if (b >= n_blocks) {  // the last wave runs to the end of the file
      w.n = n_blocks - a;
      waves.push_back(w);
      break;
    }
    // the last block of the wave that holds a recognisable record boundary
    size_t j = b - 1;
    size_t cut = SIZE_MAX;
    for (;; --j) {
      if (isize[j] >= 64) {
        sgh::Bytes text_j;
        size_t used = 0;
        if (!sgh::gunzip_member(file + begin[j], (size_t)(begin[j + 1] - begin[j]), text_j, used)) return false;
        cut = sgh::fastq_last_record_end(text_j.data(), text_j.size());
        if (cut != SIZE_MAX && !(j == a && cut <= head_skip)) break;  // (a cut inside the part we skip is no use)
        cut = SIZE_MAX;
      }
      if (j == a || b - j > 64) return false;
    }
    w.n = j + 1 - a;
    w.tail_skip = (uint32_t)(isize[j] - cut);
    waves.push_back(w);
    if (cut == isize[j]) {  // the block ends on a record boundary
      a = j + 1;
      head_skip = 0;
    } else {
      a = j;
      head_skip = (uint32_t)cut;
    }
  }
  return true;
}

// How many gzip members does the file hold, counting up to `cap`?  Every later position that looks like
// a member start (the host reader's signature scan: 1f 8b 08, reserved flags clear) is tried with zlib;
// in compressed data such a position is a coincidence (one in a few MB) that zlib rejects within a few
// bytes.  The device confirms the count: each member's trailer must be followed by the next header.
size_t gzip_members(const uint8_t* d, size_t n, size_t cap) {
  size_t members = 1;
  for (const uint8_t* p = d + 1; p + 4 <= d + n && members < cap; ++p) {
    p = static_cast<const uint8_t*>(memchr(p, 0x1f, (size_t)(d + n - p)));
    if (!p || p + 4 > d + n) break;
    if (p[1] != 0x8b || p[2] != 0x08 || (p[3] & 0xE0) != 0) continue;
    z_stream zs{};
    if (inflateInit2(&zs, 15 + 16) != Z_OK) return cap;
    uint8_t out[4096];
    zs.next_in = const_cast<uint8_t*>(p);
    zs.avail_in = (uInt)std::min<size_t>((size_t)(d + n - p), 1u << 20);
    zs.next_out = out;
    zs.avail_out = sizeof out;
    const int rc = inflate(&zs, Z_NO_FLUSH);
    const bool member = (rc == Z_OK || rc == Z_STREAM_END) && (zs.avail_out == 0 || rc == Z_STREAM_END);
    inflateEnd(&zs);
    members += member;
  }
  return members;
}

// Where a gzip file of several members (not BGZF) is counted.  The host decodes members side by side,
// one ingest thread each, at about one core's speed per member; the device decodes the whole file in
// pieces, but serially twice per piece, so it has a latency floor.  Both constants are measured with
// tools/multi_member_time.py (profiles/r4_multi_member_time.txt, one B200): below kMinDeviceGzipBytes of
// compressed input the host's cores finish first, and once min(members, ingest threads) exceeds
// kHostCoresPerDevice the host's threads side by side are as quick as the device.
constexpr size_t kMinDeviceGzipBytes = 64ull << 20;
constexpr size_t kHostCoresPerDevice = 3;

// Does a gzip file that is not BGZF, of `members` members (counted up to kHostCoresPerDevice + 1), go to the
// device?  `why_not`: the reason when it does not.
bool gzip_file_to_device(size_t members, uint64_t bytes, unsigned ingest_threads, std::string& why_not) {
  // (SGC_MULTI_MEMBER_DEVICE=1: every multi-member file to the device, for measurements of both paths)
  const char* force_env = getenv("SGC_MULTI_MEMBER_DEVICE");
  const bool force = force_env && atoi(force_env) != 0;
  if (members > 1 && !force && bytes < kMinDeviceGzipBytes) {
    why_not = "not BGZF, and several gzip members in a file under " + std::to_string(kMinDeviceGzipBytes >> 20) +
              " MB: the host's cores decode them sooner";
    return false;
  }
  if (members > 1 && !force && std::min<size_t>(members, ingest_threads) > kHostCoresPerDevice) {
    why_not = "not BGZF, and " + std::string(members > kHostCoresPerDevice ? "more than " + std::to_string(kHostCoresPerDevice)
                                                                            : std::to_string(members)) +
              " gzip members: the host decodes them side by side";
    return false;
  }
  return true;
}

// Device-memory admission of the device ingest.  Before a sample creates its streams on a device it
// reserves the library's bound of their scratch (sgc_fastq_stream_scratch_bound) from the device's
// budget, waiting while other samples hold too much of it, and gives it back once its streams are
// destroyed.  A sample whose bound exceeds the whole budget runs alone on its device.
struct DeviceBudget {
  std::mutex mu;
  std::condition_variable cv;
  uint64_t budget = 0, used = 0;
  unsigned running = 0, most = 0;  // samples holding a reservation now / at most
  void acquire(uint64_t bytes) {
    std::unique_lock<std::mutex> lk(mu);
    cv.wait(lk, [&] { return running == 0 || used + bytes <= budget; });
    used += bytes;
    most = std::max(most, ++running);
  }
  void release(uint64_t bytes) {
    {
      std::lock_guard<std::mutex> lk(mu);
      used -= bytes;
      --running;
    }
    cv.notify_all();
  }
};
// One sample's reservations, taken in device order (so that no two samples hold one device each and
// wait for the other's) and released when the guard goes.
struct Reservation {
  std::map<DeviceBudget*, uint64_t> held;  // (the budgets are one array: pointer order is device order)
  explicit Reservation(const std::map<DeviceBudget*, uint64_t>& want) {
    for (const auto& [b, bytes] : want) {
      b->acquire(bytes);
      held.emplace(b, bytes);
    }
  }
  ~Reservation() {
    for (const auto& [b, bytes] : held) b->release(bytes);
  }
};
// `lanes` streams of `bound` bytes each, stream d on the device of budgets[d % budgets.size()]
std::map<DeviceBudget*, uint64_t> lane_bytes(const std::vector<DeviceBudget*>& budgets, size_t lanes, uint64_t bound) {
  std::map<DeviceBudget*, uint64_t> want;
  for (size_t d = 0; d < lanes; ++d) want[budgets[d % budgets.size()]] += bound;
  return want;
}

// A gzip FASTQ that is not BGZF: one member through sgc_fastq_stream_submit_member, several (`several`)
// through sgc_fastq_stream_submit_gzip, on the first device; or, with lanes > 1, the file through
// sgc_fastq_stream_submit_gzip_split by `lanes` streams dealt over the sample's devices (lane d on
// libs[d % libs.size()]), their counters summed with sgc_reduce_counts.
bool count_member_on_device(const std::vector<const sgc_library*>& libs, const std::vector<DeviceBudget*>& budgets, size_t lanes,
                            uint32_t n_guides, const MappedFile& file, OffsetValue offset, uint32_t span_offset, uint32_t read_len,
                            uint32_t span_start, uint32_t span_len, bool variable, bool recursion, int rc_mode, bool several,
                            SampleResult& r, std::string& why_not) {
  uint64_t bound = 0;
  check(sgc_fastq_stream_scratch_bound(0, file.size, 0, variable ? 0 : read_len, span_len, &bound));
  Reservation reserved(lane_bytes(budgets, lanes, bound));  // (declared before the streams: released after them)
  const auto t0 = std::chrono::steady_clock::now();
  struct Guard {
    std::vector<sgc_counter*> c;
    std::vector<sgc_fastq_stream*> s;
    ~Guard() {
      for (auto* x : s) sgc_fastq_stream_destroy(x);
      for (auto* x : c) sgc_counter_destroy(x);
    }
  } g;
  g.c.assign(lanes, nullptr);
  g.s.assign(lanes, nullptr);
  for (size_t d = 0; d < lanes; ++d) {
    check(sgc_counter_create(libs[d % libs.size()], offset.reverse, span_offset, recursion, rc_mode, nullptr, nullptr, &g.c[d]));
    check(sgc_fastq_stream_create(g.c[d], variable ? 0 : read_len, span_start, span_len, &g.s[d]));
  }
  const auto t1 = std::chrono::steady_clock::now();
  uint64_t n_records = 0;
  int rc = lanes > 1 ? sgc_fastq_stream_submit_gzip_split(g.s.data(), (uint32_t)lanes, file.data, file.size)
           : several ? sgc_fastq_stream_submit_gzip(g.s[0], file.data, file.size)
                     : sgc_fastq_stream_submit_member(g.s[0], file.data, file.size);
  const auto t2 = std::chrono::steady_clock::now();
  for (size_t d = 0; d < lanes && rc == SGC_OK; ++d) {
    uint64_t records = 0;
    rc = sgc_fastq_stream_finish(g.s[d], &records);
    n_records += records;
  }
  if (rc == SGC_ERR_GZIP || rc == SGC_ERR_FASTQ_FORMAT) {
    why_not = sgc_last_error();
    return false;
  }
  if (rc != SGC_OK) fail("%s", sgc_last_error());
  check(sgc_fastq_stream_member_stats(g.s[0], &r.member_pieces, &r.member_chain, &r.member_absorbed));
  check(sgc_fastq_stream_gzip_members(g.s[0], &r.gzip_members));
  if (lanes > 1) check(sgc_reduce_counts(g.c.data(), (int)lanes, 0));
  r.counts.resize(n_guides);
  check(sgc_counter_finish(g.c[0], r.counts.data(), &r.total, &r.matched));
  const auto t3 = std::chrono::steady_clock::now();
  auto seconds = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
    return std::chrono::duration<double>(b - a).count();
  };
  r.span_reads = variable ? 0 : n_records;
  r.line_reads = variable ? n_records : 0;
  r.device_ingest = true;
  r.shards = (unsigned)std::min(lanes, libs.size());
  r.member_lanes = (unsigned)lanes;
  r.submit_s = seconds(t0, t3);
  r.dev_create_s = seconds(t0, t1);
  r.dev_waves_s = seconds(t1, t2);
  r.dev_finish_s = seconds(t2, t3);
  return true;
}

// One sample through the device ingest, on one device or — `libs.size()` > 1 — with its waves
// dealt to several, one host thread each, the devices' count vectors summed at the end
// (sgc_reduce_counts).  A gzip file that is not BGZF goes to the first device (count_member_on_device)
// when `member_ok` and it is one member, or several where the device is the quicker (kMinDeviceGzipBytes,
// kHostCoresPerDevice; `ingest_threads`: the host's threads for the sample).  Returns false when the file is neither or the device reports input it
// does not take — a read of another length (span mode), FASTA, a damaged block — so that the
// caller can try the other mode or the host path.
// `variable`: reads of any length (the sequence lines are counted where they lie in the inflated
// text); otherwise every read has read_len bytes and only its guide-window span is kept.
bool count_sample_on_device(const std::vector<const sgc_library*>& libs, const std::vector<DeviceBudget*>& budgets, uint32_t n_guides,
                            uint32_t k, const std::string& path, OffsetValue offset, uint32_t read_len, bool variable, bool recursion,
                            int rc_mode, bool member_ok, size_t members, unsigned ingest_threads, SampleResult& r, std::string& why_not) {
  uint32_t span_start = 0, span_len = 0, span_offset = offset.index;
  if (!variable && sgc_span_geometry(k, read_len, offset.reverse, offset.index, recursion, &span_start, &span_len,
                                     &span_offset) != SGC_OK) {
    why_not = "the guide window does not fit the reads";
    return false;
  }
  const auto t_start = std::chrono::steady_clock::now();
  auto seconds = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
    return std::chrono::duration<double>(b - a).count();
  };
  MappedFile file(path);
  if (!file.data) {
    why_not = "cannot map the file";
    return false;
  }
  std::vector<uint64_t> begin;
  std::vector<uint32_t> isize;
  if (!bgzf_index(file.data, file.size, begin, isize, std::min(8u, std::max(1u, std::thread::hardware_concurrency())))) {
    if (!member_ok) {
      why_not = "not BGZF, and read shards asked for";
      return false;
    }
    if (!gzip_file_to_device(members, file.size, ingest_threads, why_not)) return false;
    // SGC_MEMBER_LANES=n: n streams dealt over the sample's devices decode the file together (n on the
    // one device when the sample has one).  Without it the file goes to the first device alone.
    size_t lanes = 1;
    if (const char* e = getenv("SGC_MEMBER_LANES"); e && atoi(e) > 0) lanes = (size_t)atoi(e);
    return count_member_on_device(libs, budgets, lanes, n_guides, file, offset, span_offset, read_len, span_start, span_len, variable, recursion,
                                  rc_mode, members > 1, r, why_not);
  }
  const auto t_indexed = std::chrono::steady_clock::now();
  const size_t n_blocks = isize.size(), n_dev = libs.size();
  // Waves of blocks.  One device thread inflates each block and a wave takes about as long with
  // 60 000 blocks as with 10 000, so waves are large: up to 65 536 blocks / 4 GiB of text (variable-
  // length mode addresses the text with 32-bit offsets: 3 GiB), which also bounds the device
  // memory of a stream to ~6 GB however large the file.  The compressed bytes go to the device
  // straight from the mapping (page cache -> the driver's staging buffers).
  const uint64_t wave_text = variable ? (3ull << 30) : (4ull << 30);
  std::vector<Wave> waves;
  // lanes = streams that take waves side by side: one per device, or two on the only device when
  // the file is large (the copy of one wave's compressed bytes runs under the other's inflate,
  // and the buffers stay a quarter the size)
  const size_t lanes_wanted = n_dev > 1 ? n_dev : (n_blocks > 65536 ? 2 : 1);
  bool independent = lanes_wanted > 1;
  if (independent) {
    size_t per_wave = n_dev > 1 ? std::min<size_t>(65536, std::max<size_t>(16384, n_blocks / (2 * n_dev) + 1)) : 32768;
    if (const char* e = getenv("SGC_WAVE_BLOCKS"); e && atol(e) > 0) per_wave = (size_t)atol(e);  // tests: many small waves
    independent = plan_waves(file.data, begin, isize, per_wave, wave_text, waves);
    if (!independent) waves.clear();
  }
  if (!independent) {  // one device, one dependent sequence of waves (the stream carries partial records over)
    for (size_t a = 0; a < n_blocks;) {
      size_t b = a;
      uint64_t text = 0;
      while (b < n_blocks && b - a < 65536 && text + isize[b] < wave_text) text += isize[b++];
      if (b == a) b = a + 1;
      Wave w;
      w.first = a;
      w.n = b - a;
      waves.push_back(w);
      a = b;
    }
  }
  const size_t n_lanes = independent ? std::min(lanes_wanted, waves.size()) : 1;
  uint64_t wave_gz = 0, wave_text_most = 0, bound = 0;
  for (const Wave& w : waves) {
    uint64_t text = 0;
    for (size_t b = w.first; b < w.first + w.n; ++b) text += isize[b];
    wave_gz = std::max<uint64_t>(wave_gz, begin[w.first + w.n] - begin[w.first]);
    wave_text_most = std::max(wave_text_most, text);
  }
  check(sgc_fastq_stream_scratch_bound(1, wave_gz, wave_text_most, variable ? 0 : read_len, span_len, &bound));
  Reservation reserved(lane_bytes(budgets, n_lanes, bound));  // (declared before the streams: released after them)
  struct Lane {
    sgc_counter* c = nullptr;
    sgc_fastq_stream* stream = nullptr;
    uint64_t records = 0;
    int status = SGC_OK;
    std::string error;
  };
  struct Guard {
    std::vector<Lane> lanes;
    ~Guard() {
      for (auto& l : lanes) {
        sgc_fastq_stream_destroy(l.stream);
        sgc_counter_destroy(l.c);
      }
    }
  } g;
  g.lanes.resize(n_lanes);
  for (size_t d = 0; d < n_lanes; ++d) {
    check(sgc_counter_create(libs[d % n_dev], offset.reverse, span_offset, recursion, rc_mode, nullptr, nullptr, &g.lanes[d].c));
    check(sgc_fastq_stream_create(g.lanes[d].c, variable ? 0 : read_len, span_start, span_len, &g.lanes[d].stream));
  }
  const auto t_created = std::chrono::steady_clock::now();
  std::atomic<size_t> next_wave{0};
  std::atomic<bool> failed{false};
  auto run_lane = [&](Lane& l) {
    for (;;) {
      const size_t w = next_wave.fetch_add(1);
      if (w >= waves.size() || failed.load()) break;
      const Wave& wv = waves[w];
      l.status = sgc_fastq_stream_submit_range(l.stream, file.data, begin.data() + wv.first, isize.data() + wv.first,
                                               (uint32_t)wv.n, wv.head_skip, wv.tail_skip, independent ? 1 : 0);
      if (l.status != SGC_OK) {
        l.error = sgc_last_error();
        failed.store(true);
        break;
      }
    }
    if (l.status == SGC_OK && !failed.load()) {
      l.status = sgc_fastq_stream_finish(l.stream, &l.records);
      if (l.status != SGC_OK) {
        l.error = sgc_last_error();
        failed.store(true);
      }
    }
  };
  {
    std::vector<std::thread> pool;
    for (size_t d = 1; d < n_lanes; ++d) pool.emplace_back([&, d] { run_lane(g.lanes[d]); });
    run_lane(g.lanes[0]);
    for (auto& t : pool) t.join();
  }
  const auto t_waved = std::chrono::steady_clock::now();
  uint64_t n_records = 0;
  for (auto& l : g.lanes) {
    if (l.status == SGC_ERR_GZIP || l.status == SGC_ERR_FASTQ_FORMAT) {
      why_not = l.error;
      return false;
    }
    if (l.status != SGC_OK) fail("%s", l.error.c_str());
    n_records += l.records;
  }
  if (failed.load()) {
    why_not = "a wave failed";
    return false;
  }
  if (n_lanes > 1) {
    std::vector<sgc_counter*> shards;
    for (auto& l : g.lanes) shards.push_back(l.c);
    check(sgc_reduce_counts(shards.data(), (int)shards.size(), 0));
  }
  r.counts.resize(n_guides);
  check(sgc_counter_finish(g.lanes[0].c, r.counts.data(), &r.total, &r.matched));
  r.span_reads = variable ? 0 : n_records;
  r.line_reads = variable ? n_records : 0;
  r.device_ingest = true;
  r.device_blocks = n_blocks;
  r.shards = (unsigned)std::min(n_lanes, n_dev);
  const auto t_end = std::chrono::steady_clock::now();
  r.submit_s = seconds(t_start, t_end);
  r.dev_index_s = seconds(t_start, t_indexed);
  r.dev_create_s = seconds(t_indexed, t_created);
  r.dev_waves_s = seconds(t_created, t_waved);
  r.dev_finish_s = seconds(t_waved, t_end);
  return true;
}

// count_sample (count.rs:15-45).  The inflate threads hand over blocks of sequence lines in file
// order; this thread packs them into pinned batches and submits them.  With several devices the
// batches of the ONE sample go round the devices (read shards, each its own counter, stream and
// pair of pinned buffers) and the shard vectors are summed into the first one's at the end
// (sgc_reduce_counts: one NCCL reduce of n_guides + 2 words) — the reference never splits a
// sample; its per-sample Counters are simply collected (count.rs:136).
//
// When the sample's reads all have the length of its first record (`read_len`, known from the
// head the offset detector read), the inflate threads frame SPAN records — the guide window and
// one byte either side, all Counter::assign ever looks at — and those go to a second counter per
// device whose Offset addresses the window inside the span (sgc_span_geometry).  A member that
// holds a read of another length comes as whole lines and goes to the ordinary counter.
SampleResult count_sample(const std::vector<const sgc_library*>& libs, uint32_t n_guides, uint32_t k,
                          const std::string& path, OffsetValue offset, uint32_t read_len, bool recursion, int rc_mode,
                          unsigned ingest_threads, bool use_spans) {
  struct Channel {  // one counter and its pair of pinned buffers
    sgc_counter* c = nullptr;
    Batch b[2];
    int cur = 0;
    bool used = false;
  };
  struct Lane {
    Channel ch[2];  // [0] whole lines, [1] span records
  };
  struct Guard {
    std::vector<Lane> lanes;
    ~Guard() {
      for (auto& l : lanes)
        for (auto& ch : l.ch) {
          sgc_counter_destroy(ch.c);
          for (auto& x : ch.b)
            if (x.lines) sgc_host_free(x.lines);
        }
    }
  } g;
  g.lanes.resize(libs.size());
  sgh::SpanSpec spec;
  uint32_t span_offset = 0;
  if (use_spans && sgc_span_geometry(k, read_len, offset.reverse, offset.index, recursion, &spec.start, &spec.len,
                                     &span_offset) == SGC_OK) {
    spec.read_len = read_len;
    spec.stride = (spec.len + 7u) & ~7u;
    use_spans = spec.stride < read_len + 1;  // only if it sends fewer bytes
  } else {
    use_spans = false;
  }
  // blocks of packed sequence lines or span records, framed by the inflate threads (fastx.h);
  // they start inflating while the pinned buffers are being allocated
  sgh::SeqBlockReader reader(path, ingest_threads, use_spans ? &spec : nullptr);
  const size_t cap = 64u << 20;
  auto ready = [&](size_t d, int kind) -> Channel& {  // counter and pinned buffers on first use
    Channel& ch = g.lanes[d].ch[kind];
    if (ch.c) return ch;
    check(sgc_counter_create(libs[d], offset.reverse, kind ? span_offset : offset.index, recursion, rc_mode, nullptr,
                             nullptr, &ch.c));
    for (auto& b : ch.b) {
      void* p = nullptr;
      check(sgc_host_alloc(&p, cap));
      b.lines = static_cast<uint8_t*>(p);
      b.cap = cap;
      b.reset();
    }
    return ch;
  };
  sgh::SeqBlock blk;
  size_t d = 0;
  SampleResult r;
  using Clock = std::chrono::steady_clock;
  auto since = [](Clock::time_point t0) { return std::chrono::duration<double>(Clock::now() - t0).count(); };
  ready(0, use_spans ? 1 : 0);
  for (;;) {
    auto t0 = Clock::now();
    const bool more = reader.next(blk);
    r.wait_s += since(t0);
    if (!more) break;
    const int kind = blk.spans ? 1 : 0;
    (blk.spans ? r.span_reads : r.line_reads) += blk.n;
    uint64_t rec = 0;
    size_t byte = 0;
    for (;;) {
      Channel& ch = ready(d, kind);
      t0 = Clock::now();
      const bool done = ch.b[ch.cur].append(blk, rec, byte);
      r.copy_s += since(t0);
      if (done) break;
      if (ch.b[ch.cur].n == 0) fail("a sequence line longer than %zu bytes", cap);
      t0 = Clock::now();
      submit(ch.c, ch.b[ch.cur]);
      ch.used = true;
      ch.cur ^= 1;
      // the buffer about to be refilled was handed over one submit ago: its copy must have
      // finished, the copy just queued (and every kernel) may still be running
      check(sgc_counter_wait_copies(ch.c, 1));
      ch.b[ch.cur].reset();
      d = (d + 1) % g.lanes.size();  // the next batch goes to the next device
      r.submit_s += since(t0);
    }
  }
  r.members_adopted = reader.members_adopted();
  r.members_reframed = reader.members_reframed();
  auto t0 = Clock::now();
  std::vector<sgc_counter*> shards;
  unsigned devices_used = 0;
  for (auto& l : g.lanes) {
    bool any = false;
    for (auto& ch : l.ch) {
      if (!ch.c) continue;
      if (ch.b[ch.cur].n) {
        submit(ch.c, ch.b[ch.cur]);
        ch.used = true;
      }
      if (ch.used || shards.empty()) shards.push_back(ch.c);
      any |= ch.used;
    }
    devices_used += any;
  }
  r.shards = std::max(devices_used, 1u);
  if (shards.size() > 1) check(sgc_reduce_counts(shards.data(), (int)shards.size(), 0));
  r.counts.resize(n_guides);
  check(sgc_counter_finish(shards[0], r.counts.data(), &r.total, &r.matched));
  r.submit_s += since(t0);
  return r;
}

}  // namespace

int main(int argc, char** argv) {
  try {
    Args args = parse_args(argc, argv);
    const auto t_start = std::chrono::steady_clock::now();
    auto seconds_since_start = [&] { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count(); };
    double t_inputs = 0, t_tables = 0, t_offsets = 0;
    for (const auto& p : args.input_paths)
      if (!exists(p)) fail("Provided filepath does not exist: %s", p.c_str());  // main.rs:130-140
    std::vector<std::string> names;
    if (args.have_names) {
      if (args.sample_names.size() != args.input_paths.size())
        fail("Must provide as many sample names as there are input files");  // main.rs:156
      names = args.sample_names;
    } else {
      names = generate_sample_names(args.input_paths);
    }
    const size_t n_samples = args.input_paths.size();

    HostLibrary hlib = load_library(args.library_path);
    std::unordered_map<std::string, std::string> genemap;
    const bool have_genemap = !args.genemap.empty();
    if (have_genemap) {
      genemap = load_genemap(args.genemap);
      for (const auto& alias : hlib.aliases)  // count.rs:90-95
        if (!genemap.count(alias)) fail("Missing sgRNA aliases in gene map: \"%s\"", alias.c_str());
    }
    // validate_library_size (count.rs:62-71); the same records feed the offset detector below.  The heads
    // are read side by side, and so are the members of every gzip FASTQ the device ingest may take
    // counted (once: count_sample_on_device is given the count).
    std::vector<SampleHead> heads(n_samples);
    std::vector<size_t> members(n_samples, 0);
    auto device_candidate = [&](size_t i) {
      const std::string& p = args.input_paths[i];
      return !args.host_inflate && heads[i].fastq && p.size() > 3 && p.compare(p.size() - 3, 3, ".gz") == 0;
    };
    {
      std::vector<std::exception_ptr> errors(n_samples);
      std::atomic<size_t> next_head{0};
      auto read_heads = [&] {
        for (size_t i; (i = next_head.fetch_add(1)) < n_samples;) {
          try {
            heads[i] = read_head(args.input_paths[i], args.have_offset ? 0 : args.subsample);
            if (device_candidate(i) && args.read_shards <= 1) {  // (with read shards only BGZF goes to the device)
              MappedFile file(args.input_paths[i]);
              if (file.data) members[i] = gzip_members(file.data, file.size, kHostCoresPerDevice + 1);
            }
          } catch (...) {
            errors[i] = std::current_exception();
          }
        }
      };
      std::vector<std::thread> readers;
      const size_t n_readers = std::min<size_t>(n_samples, std::max(1u, std::thread::hardware_concurrency()));
      for (size_t t = 1; t < n_readers; ++t) readers.emplace_back(read_heads);
      read_heads();
      for (auto& t : readers) t.join();
      for (size_t i = 0; i < n_samples; ++i) {
        if (errors[i]) std::rethrow_exception(errors[i]);
        if (!heads[i].any) fail("empty reader: %s", args.input_paths[i].c_str());
        if (hlib.k > heads[i].first_len)
          fail("Sequences in reference library are larger than the sequences in input.\n\nConsider reducing the length of "
               "your reference sequences (i.e. extracting the variable region of the sgRNA or reducing the length of the "
               "adapters.)");
      }
    }

    t_inputs = seconds_since_start();
    int ndev = 0;
    check(sgc_device_count(&ndev));
    if (ndev == 0) fail("no CUDA device: this build has no CPU fallback");
    if (args.device >= ndev) fail("no such device: %d", args.device);
    const int gpus = std::min(args.gpus, ndev - args.device);
    // fewer samples than devices: every sample is cut into read shards over `per_sample` devices,
    // summed with NCCL at the end; its communicators are created on a side thread meanwhile
    // (only worth it for big inputs: the shards are summed with NCCL, whose start-up takes seconds)
    uint64_t largest_input = 0;
    for (const auto& p : args.input_paths) {
      struct stat st;
      if (stat(p.c_str(), &st) == 0) largest_input = std::max<uint64_t>(largest_input, (uint64_t)st.st_size);
    }
    const size_t per_sample = args.read_shards ? args.read_shards
                                               : (n_samples < (size_t)gpus && largest_input >= (1ull << 30) ? (size_t)gpus / n_samples : 1);
    std::thread nccl_warmup;
    struct JoinGuard {
      std::thread& t;
      ~JoinGuard() {
        if (t.joinable()) t.join();
      }
    } nccl_join{nccl_warmup};
    // (NCCL for inputs large enough to outlast its start-up; below that sgc_reduce_counts sums the
    // devices with peer copies)
    if (per_sample > 1 && gpus > 1 && largest_input >= (8ull << 30)) {
      nccl_warmup = std::thread([&] {
        for (size_t s = 0; s < n_samples; ++s) {  // one communicator set per distinct device group
          std::vector<int> devs;
          for (size_t j = 0; j < per_sample; ++j) devs.push_back(args.device + (int)((s * per_sample + j) % gpus));
          sgc_reduce_prepare(devs.data(), (int)devs.size());  // a failure is reported by sgc_reduce_counts itself
        }
      });
    }
    // one table per device; -x builds no Permuter (count.rs:103-107)
    std::vector<sgc_library*> libs(gpus, nullptr);
    struct LibGuard {
      std::vector<sgc_library*>& l;
      ~LibGuard() {
        for (auto* x : l) sgc_library_destroy(x);
      }
    } lib_guard{libs};
    {  // side by side: most of the time is the creation of each device's CUDA context
      std::vector<std::thread> builders;
      std::vector<std::string> errors(gpus);
      for (int d = 0; d < gpus; ++d)
        builders.emplace_back([&, d] {
          if (sgc_library_create(args.device + d, reinterpret_cast<const uint8_t*>(hlib.seqs.data()), hlib.n, hlib.k,
                                 args.exact ? 0 : 1, &libs[d]) != SGC_OK)
            errors[d] = sgc_last_error();
        });
      for (auto& t : builders) t.join();
      for (const auto& e : errors)
        if (!e.empty()) fail("%s", e.c_str());
    }

    // the budget of the device ingest on every device: its free memory now, less an eighth for the
    // counters' own buffers (SGC_DEVICE_BUDGET=bytes sets it, for tests of the admission)
    std::unique_ptr<DeviceBudget[]> budgets(new DeviceBudget[gpus]);
    for (int d = 0; d < gpus; ++d) {
      uint64_t free_bytes = 0, total_bytes = 0;
      check(sgc_device_memory(args.device + d, &free_bytes, &total_bytes));
      budgets[d].budget = free_bytes - free_bytes / 8;
      if (const char* e = getenv("SGC_DEVICE_BUDGET"); e && *e) budgets[d].budget = strtoull(e, nullptr, 10);
    }

    t_tables = seconds_since_start();
    std::vector<OffsetValue> offsets(n_samples);
    if (args.have_offset) {
      for (auto& o : offsets) o = OffsetValue{args.reverse, (uint32_t)args.offset};  // main.rs:163-170
    } else {
      for (size_t s = 0; s < n_samples; ++s) offsets[s] = detect_offset(libs[0], heads[s]);
      if (!args.quiet) {
        std::string msg = "Calculated Offsets: [";
        for (size_t s = 0; s < n_samples; ++s) msg += (s ? ", " : "") + to_string(offsets[s]);
        fprintf(stderr, "%s]\n", msg.c_str());  // main.rs:125
      }
    }

    t_offsets = seconds_since_start();
    // the reference's only fan-out: samples in parallel (count.rs:117-136)
    std::vector<SampleResult> results(n_samples);
    std::atomic<size_t> next{0};
    std::mutex err_mu, print_mu;
    std::string first_error;
    std::vector<char> finished(n_samples, 0);
    size_t next_to_print = 0;
    std::vector<uint32_t> first_len(n_samples);
    std::vector<char> head_uniform(n_samples, 0), head_fastq(n_samples, 0);  // 4-line FASTQ? head reads of one length?
    const bool member_ok = args.read_shards <= 1;  // (read shards asked for: gzip that is not BGZF keeps the host path)
    std::vector<char> candidate(n_samples, 0);
    std::vector<uint64_t> input_bytes(n_samples, 0);
    for (size_t i = 0; i < n_samples; ++i) {
      first_len[i] = (uint32_t)heads[i].first_len;
      head_fastq[i] = heads[i].fastq;
      head_uniform[i] = heads[i].fastq && heads[i].uniform;
      candidate[i] = device_candidate(i);
      struct stat st;
      if (stat(args.input_paths[i].c_str(), &st) == 0) input_bytes[i] = (uint64_t)st.st_size;
    }
    // Samples in flight: the reference's -t (count.rs:117-136), at least one per device — and, when
    // every sample is inflated, framed and counted on its device (BGZF, and gzip files that
    // count_sample_on_device takes), four per device whatever -t says.  A sample's host thread only
    // hands work over, and the device's inflate of one sample is bound by latency, not by throughput:
    // of its longest BGZF block, or of the serial passes over a plain gzip file's pieces, whose decodes
    // fill a fraction of the SMs (profiles/r7_member_samples_time.txt).  Samples side by side fill the
    // rest; the device budgets above keep their scratch within the devices' memory.
    // (SGC_DEVICE_SAMPLES_IN_FLIGHT=n replaces the four, for measurements)
    constexpr unsigned kDeviceSamplesInFlight = 4;
    unsigned device_in_flight = kDeviceSamplesInFlight;
    if (const char* e = getenv("SGC_DEVICE_SAMPLES_IN_FLIGHT"); e && atoi(e) > 0) device_in_flight = (unsigned)atoi(e);
    auto ingest_for = [&](unsigned workers) {
      return args.ingest_threads ? args.ingest_threads : std::max(1u, std::thread::hardware_concurrency() / workers);
    };
    const unsigned device_workers =
        (unsigned)std::min<size_t>(std::max(args.threads, (unsigned)gpus * device_in_flight), n_samples);
    bool all_for_the_device = per_sample == 1;
    for (size_t i = 0; i < n_samples && all_for_the_device; ++i) {
      std::string why_not;
      all_for_the_device = (!args.host_inflate && heads[i].fastq && heads[i].bgzf) ||
                           (candidate[i] && member_ok && gzip_file_to_device(members[i], input_bytes[i], ingest_for(device_workers), why_not));
    }
    heads.clear();
    const unsigned workers =
        all_for_the_device ? device_workers : (unsigned)std::min<size_t>(std::max(args.threads, (unsigned)gpus), n_samples);
    const unsigned ingest_threads = ingest_for(workers);
    auto work = [&]() {
      for (;;) {
        const size_t s = next.fetch_add(1);
        if (s >= n_samples) return;
        try {
          std::vector<const sgc_library*> sample_libs;
          std::vector<DeviceBudget*> sample_budgets;
          for (size_t j = 0; j < per_sample; ++j) {
            sample_libs.push_back(libs[(s * per_sample + j) % gpus]);
            sample_budgets.push_back(&budgets[(s * per_sample + j) % gpus]);
          }
          // BGZF input of fixed-length FASTQ: the whole ingest on the device (one device per sample);
          // anything else, or anything the device declines, through the host's inflate threads
          bool on_device = false;
          std::string why_not = "switched off";
          if (candidate[s]) {
            // fixed-length reads as span records; reads of several lengths (seen in the head, or
            // reported by the device deeper in the file) with their sequence lines in place
            bool variable = !head_uniform[s] || args.whole_lines;
            on_device = count_sample_on_device(sample_libs, sample_budgets, hlib.n, hlib.k, args.input_paths[s], offsets[s], first_len[s],
                                               variable, !args.no_position_recursion, args.rc_mode, member_ok, members[s], ingest_threads,
                                               results[s], why_not);
            if (!on_device && !variable && why_not.find("FASTQ") != std::string::npos) {
              results[s] = SampleResult();
              on_device = count_sample_on_device(sample_libs, sample_budgets, hlib.n, hlib.k, args.input_paths[s], offsets[s],
                                                 first_len[s], true, !args.no_position_recursion, args.rc_mode, member_ok, members[s],
                                                 ingest_threads, results[s], why_not);
            }
          } else if (!head_fastq[s]) {
            why_not = "not FASTQ";
          }
          if (!on_device) {
            results[s] = count_sample(sample_libs, hlib.n, hlib.k, args.input_paths[s], offsets[s], first_len[s],
                                      !args.no_position_recursion, args.rc_mode, ingest_threads, !args.whole_lines);
            results[s].host_because = why_not;
          }
          if (!args.quiet) {
            // count.rs:36-42.  The lines come out in sample order, as they do from the reference's
            // default single thread, however many samples are in flight here.
            std::lock_guard<std::mutex> lk(print_mu);
            finished[s] = 1;
            for (; next_to_print < n_samples && finished[next_to_print]; ++next_to_print) {
              const SampleResult& r = results[next_to_print];
              fprintf(stderr, "Finished: %s; Fraction mapped: %.3f [%llu / %llu]\n", names[next_to_print].c_str(),
                      r.total ? (double)r.matched / (double)r.total : 0.0 / 0.0, (unsigned long long)r.matched,
                      (unsigned long long)r.total);
            }
          }
        } catch (const std::exception& e) {
          std::lock_guard<std::mutex> lk(err_mu);
          if (first_error.empty()) first_error = e.what();
        }
      }
    };
    const auto t_count0 = std::chrono::steady_clock::now();
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < workers; ++t) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
    if (!first_error.empty()) fail("%s", first_error.c_str());
    if (args.timing) {
      const double count_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_count0).count();
      unsigned long long reads = 0;
      double wait_s = 0, copy_s = 0, submit_s = 0;
      unsigned max_shards = 1;
      unsigned long long span_reads = 0, device_blocks = 0, adopted = 0, reframed = 0, pieces = 0, chain = 0, absorbed = 0, gzip_member_count = 0;
      unsigned device_samples = 0, member_lanes = 0, in_flight = 0;
      for (int d = 0; d < gpus; ++d) in_flight = std::max(in_flight, budgets[d].most);
      std::string host_because;
      double dev_index_s = 0, dev_create_s = 0, dev_waves_s = 0, dev_finish_s = 0;
      for (const auto& r : results) {
        dev_index_s += r.dev_index_s, dev_create_s += r.dev_create_s, dev_waves_s += r.dev_waves_s, dev_finish_s += r.dev_finish_s;
        reads += r.total, wait_s += r.wait_s, copy_s += r.copy_s, submit_s += r.submit_s;
        span_reads += r.span_reads;
        adopted += r.members_adopted, reframed += r.members_reframed;
        device_samples += r.device_ingest;
        device_blocks += r.device_blocks;
        pieces += r.member_pieces, chain += r.member_chain, absorbed += r.member_absorbed, gzip_member_count += r.gzip_members;
        if (!r.device_ingest && host_because.empty()) host_because = r.host_because;
        max_shards = std::max(max_shards, r.shards);
        member_lanes = std::max(member_lanes, r.member_lanes);
      }
      fprintf(stderr, "{\"count_s\": %.6f, \"reads\": %llu, \"samples\": %zu, \"sample_workers\": %u, "
              "\"ingest_threads\": %u, \"gpus\": %d, \"read_shards_per_sample\": %u, \"span_reads\": %llu, \"device_ingest_samples\": %u, "
              "\"device_blocks\": %llu, \"device_phases_s\": [%.4f, %.4f, %.4f, %.4f], \"host_ingest_because\": \"%s\", \"members_adopted\": %llu, \"members_reframed\": %llu, \"wait_inflate_s\": %.6f, "
              "\"copy_to_pinned_s\": %.6f, \"submit_sync_s\": %.6f, \"read_inputs_s\": %.3f, "
              "\"device_tables_s\": %.3f, \"offsets_s\": %.3f, \"member_pieces\": %llu, \"member_chain\": %llu, \"member_absorbed\": %llu, \"gzip_members\": %llu, "
              "\"member_lanes\": %u, \"device_samples_in_flight\": %u}\n",
              count_s, reads, n_samples, workers, ingest_threads, gpus, max_shards, span_reads, device_samples, device_blocks,
              dev_index_s, dev_create_s, dev_waves_s, dev_finish_s, host_because.c_str(), adopted, reframed, wait_s, copy_s, submit_s, t_inputs,
              t_tables - t_inputs, t_offsets - t_tables, pieces, chain, absorbed, gzip_member_count, member_lanes, in_flight);
    }

    // write_results (results.rs:71-99).  Counts are keyed by alias (counter.rs:232-235):
    // sequences that share a header print the combined count on each of their rows.
    std::unordered_map<std::string, std::vector<uint32_t>> by_alias;
    for (uint32_t i = 0; i < hlib.n; ++i) by_alias[hlib.aliases[i]].push_back(i);
    FILE* out = args.output_path.empty() ? stdout : fopen(args.output_path.c_str(), "wb");
    if (!out) fail("cannot create %s", args.output_path.c_str());
    std::string text = "Guide";
    for (size_t s = 0; s < n_samples; ++s) {
      if (s == 0 && have_genemap) text += "\tGene";
      text += "\t" + names[s];
    }
    text += "\n";
    for (uint32_t i = 0; i < hlib.n; ++i) {
      const std::string& alias = hlib.aliases[i];
      std::string row = alias;
      unsigned long long row_total = 0;
      for (size_t s = 0; s < n_samples; ++s) {
        if (s == 0 && have_genemap) row += "\t" + genemap.at(alias);
        unsigned long long v = 0;
        for (uint32_t j : by_alias[alias]) v += results[s].counts[j];
        row += "\t" + std::to_string(v);
        row_total += v;
      }
      if (args.include_zero || row_total > 0) text += row + "\n";
    }
    fwrite(text.data(), 1, text.size(), out);
    if (out != stdout) fclose(out);
    return 0;
  } catch (const std::exception& e) {
    fprintf(stderr, "Error: %s\n", e.what());
    return 1;
  }
}
