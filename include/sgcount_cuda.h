/*
 * sgcount_cuda.h — C ABI of libsgcount_cuda.so, the B200 (sm_100a) implementation of
 * sgcount's read->guide matching and counting path.
 *
 * The reference (noamteyssier/sgcount v0.1.35, pure Rust) has no FFI boundary; this header
 * declares the entry points a Rust `sgcount-sys` crate would bind, one per reference call
 * site on the path (SURVEY.md §8b).  INTEGRATION.md shows the Rust side.
 *
 * Conventions
 *  - every function returns an int status (0 = SGC_OK) and never unwinds; the message for
 *    the last failure on the calling thread is sgc_last_error();
 *  - each status that stands for a reference panic / Err names the reference line;
 *  - the caller owns every host buffer; the library owns all device memory except a
 *    caller-provided count vector (sgc_counter_create: d_state);
 *  - a sgc_library is immutable after creation and may be shared by any number of
 *    sgc_counters on the same device (the reference shares &Library / &Option<Permuter>
 *    across rayon workers, count.rs:127-128);
 *  - a sgc_counter is used from one thread at a time, one per (GPU, sample or sample shard);
 *  - there is no CPU fallback: with no usable CUDA device every entry point fails with
 *    SGC_ERR_CUDA.
 */
#ifndef SGCOUNT_CUDA_H
#define SGCOUNT_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGC_ABI_VERSION 2

/* ---- status codes ------------------------------------------------------------------- */
#define SGC_OK 0
#define SGC_ERR_INVALID_ARG 1
#define SGC_ERR_CUDA 2
#define SGC_ERR_DUPLICATE_SEQUENCE 3 /* panic "Unexpected duplicate sequence in library", library.rs:92 */
#define SGC_ERR_NON_ACGT_LIBRARY 4   /* not returned since ABI 2: such libraries take the byte-keyed index (below) */
#define SGC_ERR_K_UNSUPPORTED 5      /* guide length outside 1..SGC_MAX_K */
#define SGC_ERR_READ_TOO_SHORT 6     /* Err "Sequences in reference library are larger...", offsetter.rs:154-156 */
#define SGC_ERR_NAN_ENTROPY 7        /* panic "Unexpected minmax error in entropy", offsetter.rs:123-141 */
#define SGC_ERR_EMPTY_READER 8       /* panic "empty reader", offsetter.rs:38 */
#define SGC_ERR_TOO_MANY_GUIDES 9    /* more than SGC_MAX_GUIDES library sequences */
#define SGC_ERR_BATCH_TOO_LARGE 10   /* a variable-length batch must stay below 4 GiB (u32 line offsets) */
#define SGC_ERR_GZIP 12              /* a gzip block did not inflate on the device (sgc_fastq_stream_*) */
#define SGC_ERR_FASTQ_FORMAT 13      /* not fixed-length 4-line FASTQ (sgc_fastq_stream_*): count it through the host path */
#define SGC_ERR_NCCL 11              /* libnccl.so.2 could not be loaded, or an NCCL call failed (sgc_reduce_counts) */

#define SGC_MAX_GUIDES 4194302u
#define SGC_MAX_K 1024u    /* guides of up to SGC_MAX_K_PACKED bases over A,C,G,T use the 2-bit tables */
#define SGC_MAX_K_PACKED 30u

/* how Record::seq_rev_comp (fxread, used at counter.rs:203) maps non-ACGT bytes; see DESIGN.md */
#define SGC_RC_BITTRICK 0 /* c&2 ? c^4 : c^21 — 'N' becomes 'J' and 'J' becomes 'N' (default) */
#define SGC_RC_KEEP_N 1   /* A<->T, C<->G, every other byte unchanged */

typedef struct sgc_library sgc_library;
typedef struct sgc_counter sgc_counter;

const char* sgc_last_error(void);
int sgc_abi_version(void);
int sgc_device_count(int* n);
/* Free and total memory of a device (cudaMemGetInfo), in bytes. */
int sgc_device_memory(int device, uint64_t* free_bytes, uint64_t* total_bytes);

/* Pinned host memory for the caller's read batches (the ingest ring buffers). */
int sgc_host_alloc(void** ptr, size_t bytes);
int sgc_host_free(void* ptr);

/* ---- Library + Permuter ---------------------------------------------------------------
 * Replaces Library::from_reader (library.rs:17-21,89-99) and Permuter::new
 * (permutes.rs:47-75, called at count.rs:56).
 *
 * seqs: n*k ASCII bytes, row-major, in LIBRARY-FILE ORDER.  Index i of this array is the
 * guide index used by every other call; index 0 is also the record the entropy routine
 * consumes without counting (offsetter.rs:57,190-191).
 * with_permutations: 0 = --exact (count.rs:103-107 passes None), 1 = build the
 * unambiguous one-mismatch variants.
 * The reference keeps sequences as opaque byte strings of any length (library.rs:65-99).  Guides
 * of up to 30 bases over A,C,G,T — every real sgRNA library — are packed 2-bit into the L2-resident
 * tables the fast kernels use; a library with any other byte (an N, lower case) or with longer
 * sequences is indexed by its bytes instead (sgc_library_info.opaque = 1): same results, a
 * simple one-thread-per-read kernel, none of the roofline claims.
 * Errors: SGC_ERR_DUPLICATE_SEQUENCE, SGC_ERR_K_UNSUPPORTED, SGC_ERR_TOO_MANY_GUIDES,
 * SGC_ERR_EMPTY_READER (n == 0; library.rs:74 unwraps).
 */
int sgc_library_create(int device, const uint8_t* seqs, uint32_t n, uint32_t k, int with_permutations,
                       sgc_library** out);
void sgc_library_destroy(sgc_library*);

typedef struct sgc_library_info {
  uint32_t n_guides;
  uint32_t k;
  int32_t with_permutations;
  int32_t device;
  uint64_t n_variants;   /* one-mismatch ACGT variants that map to exactly one parent   */
  uint64_t n_ambiguous;  /* ACGT variants shared by >= 2 parents (the reference's _null) */
  uint64_t n_slots;      /* slots of one front table (members only)                      */
  uint64_t table_bytes;  /* seed directories + postings + both front tables              */
  double build_ms;       /* device time of the build kernels                             */
  uint64_t front_left_out; /* members (x2 orientations) resolved through the seed index only */
  int32_t opaque;          /* 1: byte-keyed index (a byte outside A,C,G,T, or k > 30) */
} sgc_library_info;
int sgc_library_get_info(const sgc_library*, sgc_library_info* out);

/* Composed lookup of n_tokens k-byte tokens: Library::contains (library.rs:34-40), then
 * Permuter::contains -> Library::alias (counter.rs:111-117).  idx_out[i] = guide index or -1.
 * kind_out (optional): 0 no match, 1 library member, 2 one-mismatch variant. */
int sgc_library_lookup(const sgc_library*, const uint8_t* tokens, uint64_t n_tokens, int32_t* idx_out,
                       uint8_t* kind_out);

/* ---- Offsetter --------------------------------------------------------------------------
 * Sequence batches are passed as newline-terminated lines:
 *   line_off != NULL: read i is lines[line_off[i] .. line_off[i+1]-1)  (n_reads+1 entries)
 *   line_off == NULL: fixed stride — read i is lines[i*stride .. i*stride+read_len)
 */

/* position_counts (offsetter.rs:55-79): first read gives `size` and is not counted; a byte
 * outside A,C,G,T adds one to all four columns.  out: size*4 uint32 (row-major [pos][ACGT]),
 * capacity out_cap rows; *size receives the first read's length. */
int sgc_position_counts(int device, const uint8_t* lines, uint64_t n_bytes, const uint32_t* line_off,
                        uint32_t stride, uint32_t read_len, uint64_t n_reads, uint32_t* out,
                        uint32_t out_cap, uint32_t* size);

/* entropy_offset for one sample (offsetter.rs:167-210 with main.rs:117's subsample applied
 * by the caller: pass at most `subsample` reads, first record included).  The reference
 * entropy comes from the library handle.  Errors: SGC_ERR_READ_TOO_SHORT,
 * SGC_ERR_NAN_ENTROPY, SGC_ERR_EMPTY_READER. */
int sgc_offset_detect(const sgc_library*, const uint8_t* lines, uint64_t n_bytes, const uint32_t* line_off,
                      uint32_t stride, uint32_t read_len, uint64_t n_reads, int* is_reverse,
                      uint32_t* index);

/* ---- Counter ----------------------------------------------------------------------------
 * Replaces Counter::new / Counter::count (counter.rs:36-66,211-236) for one sample or one
 * read shard of a sample.
 *
 * is_reverse/offset: the Offset (offsetter.rs:10-15).  position_recursion: !-p.
 * rc_mode: SGC_RC_*.  stream: the cudaStream_t every kernel of this counter runs on; NULL = a
 * stream of its own, created (blocking: ordered after earlier work on the legacy default stream)
 * and destroyed with the counter, so that counters of concurrent samples neither serialise nor
 * wait for each other.
 * d_state: optional device buffer of (n_guides + 2) uint64 owned by the caller — counts in
 * guide-index order, then total_reads, then matched_reads — so a collective (NCCL) can sum
 * shards in place; NULL = owned by the counter.  The buffer is zeroed by create.
 */
int sgc_counter_create(const sgc_library*, int is_reverse, uint32_t offset, int position_recursion,
                       int rc_mode, void* stream, uint64_t* d_state, sgc_counter** out);
void sgc_counter_destroy(sgc_counter*);

/* Span records: all the counting ever looks at of a fixed-length read is the guide window and
 * one byte either side of it (counter.rs:164-174: offset, offset + 1, offset - 1).  A host that
 * knows the Offset before it frames the records (it does: offsetter.rs runs first) can cut that
 * span out of every read and send 24 bytes per read instead of 76.  For reads of `read_len`
 * bytes this returns where the span starts in the STORED read and how long it is, and the Offset
 * index that makes a counter treat the span records as (short) reads with exactly the same
 * outcome: same orientation, `span_offset`, same position_recursion; submit them with
 * read_len = span_len and any stride >= span_len.  Fails with SGC_ERR_INVALID_ARG when the
 * Centered window does not fit the read (offset + k > read_len: every read is unmatched anyway). */
int sgc_span_geometry(uint32_t k, uint32_t read_len, int is_reverse, uint32_t offset, int position_recursion,
                      uint32_t* span_start, uint32_t* span_len, uint32_t* span_offset);
/* The span for a counter with max_shift S (sgc_counter_set_max_shift).  S = 1 returns exactly what
 * sgc_span_geometry(..., position_recursion = 1, ...) returns.  S >= 2: the span is
 * [max(0, o - S), min(read_len, o + k + S)) in the coordinates of the trimmed read (the reverse
 * complement of the whole read when is_reverse), mirrored to stored coordinates for reverse reads,
 * and span_offset = o - max(0, o - S), so the span records hold exactly the windows the read holds.
 * Fails with SGC_ERR_INVALID_ARG only when no window offset + d, |d| <= S, fits the read, or when S
 * is outside 1..16. */
int sgc_span_geometry_shift(uint32_t k, uint32_t read_len, int is_reverse, uint32_t offset, uint32_t max_shift,
                            uint32_t* span_start, uint32_t* span_len, uint32_t* span_offset);

/* Count a batch held in HOST memory (pinned memory makes the copies asynchronous).  The
 * batch is cut into chunks that are copied and counted on alternating buffers so copy and
 * kernel overlap; returns after the last chunk has been enqueued.  The host buffers must
 * stay valid until sgc_counter_sync / sgc_counter_finish. */
int sgc_counter_submit(sgc_counter*, const uint8_t* lines, uint64_t n_bytes, const uint32_t* line_off,
                       uint32_t stride, uint32_t read_len, uint64_t n_reads);

/* Count a batch already resident in DEVICE memory (kernel only, asynchronous).
 * d_assign_out (optional, n_reads int32): guide index or -1 per read. */
int sgc_counter_submit_device(sgc_counter*, const uint8_t* d_lines, uint64_t n_bytes,
                              const uint32_t* d_line_off, uint32_t stride, uint32_t read_len,
                              uint64_t n_reads, int32_t* d_assign_out);

/* Skewed screens.  The reference's fold (counter.rs:232-235) costs the same whatever the guide
 * abundances; on the GPU a guide that carries a large share of the reads serialises its atomics
 * on one L2 address.  By DEFAULT (replicas = 0) a counter looks at the first 65 536 reads of its
 * first batch of >= 262 144 reads and, when a guide stands out, counts into 16 copies of the count
 * vector (folded into the state vector after every launch) and keeps the guides with >= 1 % of
 * the reads in registers; see count.cu count_hit / plan_skew for the measurements.  This call
 * overrides the plan: 1 = never, >1 = that many copies (rounded down to a power of two, at most
 * 64 copies / 64 MB), 0 = back to automatic.  The counts never depend on it. */
int sgc_counter_set_replicas(sgc_counter*, uint32_t replicas);

/* Staggered reads (amplicons sequenced with staggered primers move the guide by a few bases from
 * read to read).  max_shift = S, 1..16.  S = 1 (the default) is the reference's recursion: Centered,
 * then Plus, then Minus, returning when a trim fails (counter.rs:96-140).  S >= 2 tries the windows
 * at offset + d for d = 0, +1, -1, ..., +S, -S in the coordinates of the trimmed read (the reverse
 * complement of the whole read in Reverse), each looked up as counter.rs:111-117 does (member, then
 * the Permuter's unique one-mismatch parent); the first that yields a guide wins, and a window that
 * does not fit the read is skipped instead of ending the search.  total_reads and matched_reads keep
 * their meaning.  Must be called before the counter's first submit.  SGC_ERR_INVALID_ARG: S outside
 * 1..16, a counter that has counted, S >= 2 without position recursion or with a byte-keyed library
 * (sgc_library_info.opaque).  Span records for such a counter: sgc_span_geometry_shift. */
int sgc_counter_set_max_shift(sgc_counter*, uint32_t max_shift);

/* Unmatched report: the most frequent guide windows of the reads a counter leaves unmatched (counted in
 * total_reads, not in matched_reads), to tell a wrong offset or orientation, staggered primers, the wrong
 * library, adapter dimers or PhiX apart.  A read's window is trimmed[o, o + k): the read, or in Reverse its
 * reverse complement under the counter's rc_mode, at the counter's Offset index o, whatever the recursion
 * and max_shift.  Every unmatched read falls into one class: short_reads (o + k > read length: no window),
 * non_acgt (a window byte outside A, C, G, T, N included), or its window, tallied in library orientation.
 * So unmatched = short_reads + non_acgt + overflow + the sum of the window counts.
 * Bounded memory: the report holds at most `capacity` distinct windows.  A window that finds no slot
 * (the table is full around it) is added to overflow, and slots are never freed, so a window once refused
 * stays refused: every window the report holds has its exact count, and every other window's count is at
 * most overflow.  With overflow == 0 the report is exact.
 * The counter then counts through the line (or shift) kernel and, after each launch of at most 2^24 reads,
 * tallies the launch's unmatched reads on its stream.  Counts, totals and the skew plan do not change.
 * Call it before the counter's first submit.  SGC_ERR_INVALID_ARG: a byte-keyed library
 * (sgc_library_info.opaque), a counter that has counted, capacity 0 or above 2^26.  sgc_counter_reset
 * clears the report; sgc_reduce_counts does not merge reports (merge them on the host by window). */
int sgc_counter_set_unmatched_report(sgc_counter*, uint64_t capacity);
typedef struct sgc_unmatched_info {
  uint64_t unmatched;   /* reads counted and not matched                                  */
  uint64_t short_reads; /* of them, reads with no window at the offset                     */
  uint64_t non_acgt;    /* of them, windows with a byte outside A, C, G, T                 */
  uint64_t overflow;    /* of them, A/C/G/T windows refused for want of a slot             */
  uint64_t distinct;    /* windows the report holds                                        */
} sgc_unmatched_info;
/* Waits for the counter, then writes the first max_windows windows of the report in report order (count
 * descending, then window bytes ascending): windows = max_windows x k ASCII bytes, counts = max_windows
 * words (both may be NULL when max_windows == 0); *n_windows = how many were written.  info is optional. */
int sgc_counter_unmatched(sgc_counter*, uint64_t max_windows, uint8_t* windows, uint64_t* counts, uint64_t* n_windows,
                          sgc_unmatched_info* info);
/* Device memory one counter's report takes (its table and its per-launch assignment scratch of 64 MiB). */
int sgc_unmatched_report_bytes(uint64_t capacity, uint64_t* bytes);

int sgc_counter_sync(sgc_counter*);
/* Wait until all but the last `keep_in_flight` sgc_counter_submit calls have had their host
 * buffers copied to the device (those buffers may be refilled), without waiting for the kernels
 * that count them: with two buffers, refill one while the other's copy is still running. */
int sgc_counter_wait_copies(sgc_counter*, uint32_t keep_in_flight);
int sgc_counter_reset(sgc_counter*); /* zero the state vector */

/* Wait, then copy out counts[n_guides] (guide-index order), total_reads, matched_reads
 * (counter.rs:239-246).  The reference keys results by alias (counter.rs:232-235); the host
 * maps index -> alias and sums indices that share one. */
int sgc_counter_finish(sgc_counter*, uint64_t* counts, uint64_t* total, uint64_t* matched);

/* Device pointer / length (in uint64 words) of the state vector, for the caller's collective
 * (one process per GPU: torch.distributed / MPI / NCCL owned by the caller). */
int sgc_counter_state(sgc_counter*, uint64_t** d_state, uint64_t* n_words);

/* Read shards of ONE sample counted by several counters of THIS process (the reference collects
 * its per-sample Counters at count.rs:136; a sample cut into read shards needs them summed):
 * state[root] = sum over i of state[i], i.e. counts, total_reads and matched_reads of the whole
 * sample land in shards[root]; the other shards' vectors are left unspecified (reset them before
 * reuse).  Unmatched reports (sgc_counter_set_unmatched_report) are not merged: each shard keeps its own.  Shards that share a device are folded on that device first.  Across devices:
 *   - with NCCL communicators for the device set in place (sgc_reduce_prepare was called, or an
 *     earlier reduce created them): ONE ncclReduce(ncclUint64, ncclSum) of n_guides + 2 words over
 *     NVLink, each rank's call enqueued on its counter's own stream (libnccl.so.2 is loaded on first
 *     use; communicators are cached per device set);
 *   - otherwise (nobody asked for NCCL): every other device's vector is copied peer to peer into a
 *     scratch vector on the root's device and added there — loading NCCL and ncclCommInitAll take
 *     seconds, more than counting a whole sample of tens of millions of reads.
 * Asynchronous: sgc_counter_finish(shards[root]) waits for it.  Every counter must come from a
 * library of the same guides.  Errors: SGC_ERR_NCCL. */
int sgc_reduce_counts(sgc_counter* const* shards, int n_shards, int root);
/* Selects NCCL for every later sgc_reduce_counts of this process and creates the communicators for
 * counters on these devices (loading NCCL and ncclCommInitAll take seconds; the CLI does this on a
 * side thread, for inputs large enough to outlast it, while it builds its tables). */
int sgc_reduce_prepare(const int* devices, int n_devices);

/* ---- FASTQ straight from BGZF blocks -----------------------------------------------------------
 * The reference reads a sample through fxread::initialize_reader (count.rs:24): gzip inflate and
 * line splitting on the host.  For blocked gzip (BGZF: bgzip, sequencer output — independent
 * members of at most 64 KB that carry their size in a 'BC' extra field) the whole ingest runs on
 * the device instead: one thread inflates each block, the text is framed into records by a
 * newline scan, the guide-window span of every sequence line is cut out and counted, and the only
 * bytes that cross PCIe are the compressed ones.
 *
 * Two modes.  read_len > 0: every read has read_len bytes; `counter` was created with the SPAN
 * offset of sgc_span_geometry and the stream cuts the span [span_start, span_start + span_len) out
 * of every sequence line (the streaming count kernel).  read_len == 0 (span_* ignored): reads of
 * any length; `counter` is an ordinary counter (the sample's own Offset) and the sequence lines are
 * counted where they lie in the inflated text (the line kernel); a wave must then inflate to less
 * than 4 GiB.  The stream counts into `counter` (same device, same CUDA stream).  Only 4-line
 * FASTQ is framed here; anything else — and in the first mode a read of another length — fails
 * with SGC_ERR_FASTQ_FORMAT (a corrupt block or a CRC-32 mismatch: SGC_ERR_GZIP) and the caller
 * starts over with the other mode or with sgc_counter_submit.
 * submit: n_blocks consecutive blocks, in file order, continuing where the previous call stopped;
 * gz + block_begin[i] .. gz + block_begin[i + 1] is block i (host memory), block_isize[i] its
 * ISIZE field.  One call is one wave: it should carry thousands of blocks (one device thread
 * each; the decode of a block is a long serial chain, so a wave takes about as long
 * whether it holds ten thousand blocks or three hundred thousand) and must inflate to less than 64 GiB.  Blocks may end anywhere in a record.
 * finish: end of the input; *n_records = records counted.
 * Device memory: a stream's scratch (compressed bytes, text, span records) comes from one memory
 * pool per device through the stream-ordered allocator and goes back to it when the stream is
 * destroyed, without a device-wide synchronisation; the pool keeps up to 8 GiB of freed memory
 * for the next stream and hands the rest back to the driver at the next synchronisation. */
typedef struct sgc_fastq_stream sgc_fastq_stream;
int sgc_fastq_stream_create(sgc_counter* counter, uint32_t read_len, uint32_t span_start, uint32_t span_len,
                            sgc_fastq_stream** out);
void sgc_fastq_stream_destroy(sgc_fastq_stream*);
int sgc_fastq_stream_submit(sgc_fastq_stream*, const uint8_t* gz, const uint64_t* block_begin,
                            const uint32_t* block_isize, uint32_t n_blocks);
/* The same for a wave the caller has cut at record boundaries, so that waves do not depend on each
 * other and may go to different streams (devices): of the wave's inflated text the first head_skip
 * and the last tail_skip bytes belong to the neighbouring waves (a block that holds a cut is
 * submitted with both).  self_contained != 0 asserts that what is left starts and ends on a
 * record boundary (SGC_ERR_FASTQ_FORMAT otherwise). */
int sgc_fastq_stream_submit_range(sgc_fastq_stream*, const uint8_t* gz, const uint64_t* block_begin,
                                  const uint32_t* block_isize, uint32_t n_blocks, uint32_t head_skip,
                                  uint32_t tail_skip, int self_contained);
/* ONE gzip member that is not BGZF (what gzip and pigz write): as sgc_fastq_stream_submit_gzip,
 * except that no gzip header inside the file becomes a candidate, so a file of more than one member
 * fails with SGC_ERR_GZIP. */
int sgc_fastq_stream_submit_member(sgc_fastq_stream*, const uint8_t* gz, uint64_t n_bytes);
/* After sgc_fastq_stream_submit_member or sgc_fastq_stream_submit_gzip: candidate pieces, pieces on
 * the chain of true block boundaries, candidates the chain ran past, summed over the members. */
int sgc_fastq_stream_member_stats(const sgc_fastq_stream*, uint64_t* pieces, uint64_t* chain, uint64_t* absorbed);
/* ANY sequence of gzip members — one, several (`cat a.gz b.gz`, appending writers), or BGZF blocks —
 * the whole file, gz[0 .. n_bytes) in host memory, inflated, framed and counted on the device, once
 * per stream, then sgc_fastq_stream_finish.  The DEFLATE streams are decoded in parallel by
 * speculation: candidate dynamic-Huffman block starts every 32 KiB of compressed input, and behind
 * every gzip header in the file a candidate where a member begins; a decode without output from each
 * to the next that links the true block boundaries from the first member's first block on, stepping
 * from a member's last block over its trailer and the next header; then every linked piece decoded
 * into 16-bit symbols whose references to the unknown 32 KiB in front of it are resolved afterwards.
 * The compressed file stays on the device; the text goes in waves (the limits of the BGZF waves),
 * about 3 bytes of device memory per byte of text in a wave.  The members' texts are one byte
 * stream, as gzip -d writes it (a record may straddle two members); CRC-32 and ISIZE are checked
 * member by member.  Fails with SGC_ERR_GZIP when the boundaries cannot be followed to the end
 * (blocks other than dynamic Huffman codes over long stretches, damage), anything but a whole member
 * follows a trailer (zero padding included), a member's CRC-32 or ISIZE disagrees, or the file holds
 * more gzip headers than one per 256 bytes; with SGC_ERR_FASTQ_FORMAT as sgc_fastq_stream_submit
 * does; the caller then counts the file on the host. */
int sgc_fastq_stream_submit_gzip(sgc_fastq_stream*, const uint8_t* gz, uint64_t n_bytes);
/* One gzip file (one or several members, as sgc_fastq_stream_submit_gzip) inflated, framed and counted by
 * n_streams fresh streams together, on one device or several (streams may share a device).  Every
 * stream copies the file to its device; the candidate search and the boundary pass are split by input
 * range; the text goes in waves of about min(the one-stream wave, text / n_streams), wave k to stream
 * k mod n_streams, whose windows are relayed through the host so that no wave waits for another to
 * decode; records are framed wave after wave, the bytes after a wave's last complete record handed to
 * the next wave's stream.  The streams must share read_len / span_start / span_len, and their counters
 * must come from libraries of the same guides (else SGC_ERR_INVALID_ARG).  Each stream counts the records
 * of its own waves into its own counter: sum the counters with sgc_reduce_counts and call
 * sgc_fastq_stream_finish on every stream; the records they return add up to the file's.
 * sgc_fastq_stream_member_stats and sgc_fastq_stream_gzip_members report the whole file on every stream.
 * A file is declined as by sgc_fastq_stream_submit_gzip, and then every stream has failed.  One host
 * thread per stream, all joined before the call returns.  n_streams == 1 is sgc_fastq_stream_submit_gzip. */
int sgc_fastq_stream_submit_gzip_split(sgc_fastq_stream* const* streams, uint32_t n_streams, const uint8_t* gz, uint64_t n_bytes);
/* An upper bound of the device scratch ONE stream allocates (compressed bytes, 16-bit symbols, text,
 * span or line-offset buffers, piece tables), so that a caller running several samples on a device at
 * once can keep their sum within its memory.  bgzf != 0: sgc_fastq_stream_submit / _submit_range with
 * waves of at most gz_bytes compressed and text_bytes inflated bytes.  bgzf == 0: a gzip file of gz_bytes
 * through sgc_fastq_stream_submit_member, _submit_gzip or (per stream) _submit_gzip_split; text_bytes is
 * its text when known, else 0 (then every byte is taken to inflate to the most DEFLATE allows, up to the
 * wave limit).  It does not cover a single 32 KiB piece of input that inflates to more than a whole wave
 * (4 GiB), which no FASTQ does.  read_len / span_len: as sgc_fastq_stream_create.  Streams on several
 * threads: each stream is used by one thread at a time; distinct streams, on one device or several, may
 * submit at the same time. */
int sgc_fastq_stream_scratch_bound(int bgzf, uint64_t gz_bytes, uint64_t text_bytes, uint32_t read_len, uint32_t span_len,
                                   uint64_t* bytes);
/* Uncompressed FASTQ text, text[0 .. n_bytes) in host memory of any kind (a read-only file mapping,
 * mostly), framed and counted as the text of a BGZF wave, in the mode sgc_fastq_stream_create fixed.
 * self_contained == 0: the call continues where the previous one stopped and may end anywhere in a
 * record (the bytes after its last complete record are carried on).  self_contained != 0: the text
 * starts and ends on a record boundary and the stream holds no carried bytes (SGC_ERR_FASTQ_FORMAT
 * otherwise), so that the waves of one file may be dealt to several streams or devices.  Declines as
 * sgc_fastq_stream_submit does (a record that does not start with '@', a read of another length in the
 * first mode, a record over 64 KiB, a bad cut); a failed stream refuses later calls; n_bytes == 0 does
 * nothing.  The stream cuts a call into waves of a fixed size (64 MiB): the next wave's bytes go
 * through pinned staging (several host threads) and a copy stream of their own into a second device
 * text buffer while the current wave is framed and counted.  All host threads are joined, and the
 * caller's memory is no longer read, when the call returns.  Host memory: the stream pins two staging
 * buffers of one wave (128 MiB in all) at its first text call; a destroyed stream's buffers go to a list of
 * the process from which later streams take theirs, which keeps at most eight of them. */
int sgc_fastq_stream_submit_text(sgc_fastq_stream*, const uint8_t* text, uint64_t n_bytes, int self_contained);
/* An upper bound of the device scratch ONE stream allocates through sgc_fastq_stream_submit_text (both
 * text buffers, the chunk counts and scan, span records or line offsets of the fullest wave), as
 * sgc_fastq_stream_scratch_bound; it needs no device.  read_len / span_len: as sgc_fastq_stream_create. */
int sgc_fastq_stream_text_scratch_bound(uint32_t read_len, uint32_t span_len, uint64_t* bytes);
/* Members decoded by sgc_fastq_stream_submit_gzip (1 after sgc_fastq_stream_submit_member, else 0). */
int sgc_fastq_stream_gzip_members(const sgc_fastq_stream*, uint64_t* members);
int sgc_fastq_stream_finish(sgc_fastq_stream*, uint64_t* n_records);

/* ---- Dual-guide constructs from paired reads ------------------------------------------------------
 * Screens with two guides per vector read guide A in R1 and guide B in R2 and count the listed (A, B)
 * construct.  A pair counter joins two ordinary counters, one per mate, each with its own library,
 * Offset, position recursion, rc_mode and max_shift: mate m of pair i gets a_m[i], exactly what that
 * counter assigns to the read alone (guide index or -1).  Construct j is (pair_first[j], pair_second[j]),
 * guide indices of the two libraries.  Every pair falls into one class:
 *   listed       both mates matched and (a1, a2) is construct j: counted on j;
 *   recombined   both mates matched and (a1, a2) is not listed (template switching);
 *   first_only / second_only   only that mate matched;   neither   no mate matched.
 * total = listed + recombined + first_only + second_only + neither and listed = the sum of the construct
 * counts.  The mates' counters keep their usual state (marginal guide counts; total_reads = total), as if
 * each had counted its file alone.
 * Recombinant report (recombinant_capacity > 0): the recombined pairs keyed by (a1, a2), at most
 * `capacity` distinct; slots are never freed and a pair that finds no slot in 128 probes goes to
 * overflow, so every held count is exact and recombined = overflow + the held counts.
 * Each mate is counted in chunks of at most 2^24 pairs through the line (shift, byte-keyed) kernel into
 * pair-owned assignment scratch, then the chunk is combined; all of it runs on the first counter's
 * stream, and the second counter's stream waits for the end of every submit, so sgc_counter_finish on
 * either counter sees it.
 * create refuses (SGC_ERR_INVALID_ARG) counters on different devices, the same counter twice, a counter
 * that has counted or has an unmatched report, n_pairs outside 1..2^26, capacity above 2^26 and a guide
 * index outside its library; a (first, second) entry listed twice is SGC_ERR_DUPLICATE_SEQUENCE.  The
 * pair counter does not own the counters: destroy it first. */
typedef struct sgc_pair_counter sgc_pair_counter;
int sgc_pair_counter_create(sgc_counter* first, sgc_counter* second, const uint32_t* pair_first,
                            const uint32_t* pair_second, uint64_t n_pairs, uint64_t recombinant_capacity,
                            sgc_pair_counter** out);
void sgc_pair_counter_destroy(sgc_pair_counter*);
/* n_pairs pairs: read i of mate 1 and read i of mate 2, each in its own layout (as sgc_counter_submit:
 * fixed stride at any alignment, or u32 line offsets; span records of each mate's own geometry).  Host
 * memory, copied and counted chunk by chunk on double buffers; the buffers must stay valid until
 * sgc_pair_counter_wait_copies or sgc_pair_counter_finish. */
int sgc_pair_counter_submit(sgc_pair_counter*, const uint8_t* lines1, uint64_t n_bytes1, const uint32_t* line_off1,
                            uint32_t stride1, uint32_t read_len1, const uint8_t* lines2, uint64_t n_bytes2,
                            const uint32_t* line_off2, uint32_t stride2, uint32_t read_len2, uint64_t n_pairs);
/* The same for batches resident in device memory. */
int sgc_pair_counter_submit_device(sgc_pair_counter*, const uint8_t* d_lines1, uint64_t n_bytes1,
                                   const uint32_t* d_line_off1, uint32_t stride1, uint32_t read_len1,
                                   const uint8_t* d_lines2, uint64_t n_bytes2, const uint32_t* d_line_off2,
                                   uint32_t stride2, uint32_t read_len2, uint64_t n_pairs);
/* sgc_counter_wait_copies for both mates. */
int sgc_pair_counter_wait_copies(sgc_pair_counter*, uint32_t keep_in_flight);
typedef struct sgc_pair_info {
  uint64_t total, listed, recombined, first_only, second_only, neither;
  uint64_t overflow; /* recombined pairs the report refused for want of a slot */
  uint64_t distinct; /* recombinant pairs the report holds                     */
} sgc_pair_info;
/* Waits, then copies out construct_counts[n_pairs] (list order; may be NULL) and info (may be NULL). */
int sgc_pair_counter_finish(sgc_pair_counter*, uint64_t* construct_counts, sgc_pair_info* info);
/* Waits, then writes the first max_pairs recombinant pairs of the report in report order (count descending,
 * then (first, second) ascending); *n_out = how many were written.  SGC_ERR_INVALID_ARG without a report. */
int sgc_pair_counter_recombinants(sgc_pair_counter*, uint64_t max_pairs, uint32_t* first, uint32_t* second,
                                  uint64_t* counts, uint64_t* n_out);
/* Zeroes the construct counts, the tallies, the report and both mates' state vectors. */
int sgc_pair_counter_reset(sgc_pair_counter*);
/* Device memory one pair counter takes (construct table and counts, both mates' assignment scratch of
 * 64 MiB each, the report). */
int sgc_pair_counter_bytes(uint64_t n_pairs, uint64_t recombinant_capacity, uint64_t* bytes);

/* Statistics of the last sgc_counter_submit_device call, for benchmarking. */
typedef struct sgc_launch_info {
  uint32_t grid, block, smem_bytes;
  uint32_t kernel; /* 0 = streaming fixed-stride kernel, 1 = line kernel (any layout), 2 = byte-keyed (opaque library),
                      3 = shift kernel (max_shift >= 2, any layout) */
  uint64_t launches_total;
  uint32_t replicas;   /* copies of the count vector in use (1 = none) */
  uint32_t hot_guides; /* guides counted in registers */
} sgc_launch_info;
int sgc_counter_launch_info(const sgc_counter*, sgc_launch_info* out);

#ifdef __cplusplus
}
#endif
#endif
