// member_core_test <file.gz> <piece_bytes> <skew 0|1> [members 0|1 [waves]] — decodes a gzip file the way the
// device does (gzip.cu member_* kernels), serially, from the same csrc/inflate_core.h code: candidate
// block starts every piece_bytes of compressed input (with skew, every other candidate moved one bit on),
// the boundary pass, the chain (members_chain), 16-bit symbols with window markers, the chain cut into
// about <waves> waves (default 1) as sgc_fastq_stream_submit_gzip_split cuts it over that many streams,
// each wave's windows relayed through F_k and W_k (inflate_core.h "waves: the window relay"), CRC-32 in
// pieces joined and ISIZE, member by member.  With members = 1 every gzip header is a member-start
// candidate too, so the file may hold any number of members (sgc_fastq_stream_submit_gzip); without, it
// must be one (sgc_fastq_stream_submit_member).
// Prints "<bytes> <fnv1a> <pieces> <chain> <absorbed>" (with members = 1, then "<members>"; exit 0),
// "decline ..." when the chain does not reach the end (exit 3: the device would hand the file to the
// host), or the error (exit 4).  Test helper for tests/test_member_inflate_core.py and
// tests/test_multi_member_inflate_core.py; zlib is the comparison.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../csrc/inflate_core.h"

using namespace sgc::inflate;

int main(int argc, char** argv) {
  if (argc < 4) return 2;
  FILE* f = fopen(argv[1], "rb");
  if (!f) return 2;
  std::vector<unsigned char> data;
  unsigned char buf[1 << 16];
  for (size_t got; (got = fread(buf, 1, sizeof buf, f)) > 0;) data.insert(data.end(), buf, buf + got);
  fclose(f);
  const size_t n = data.size();
  const uint64_t piece = (uint64_t)atoll(argv[2]);
  const bool skew = atoi(argv[3]) != 0;
  const bool members = argc > 4 && atoi(argv[4]) != 0;
  const uint64_t waves = argc > 5 ? (uint64_t)atoll(argv[5]) : 1;
  if (piece < 16 || waves < 1) return 2;
  data.resize(n + 64);  // the reader's slack
  const uint8_t* in = data.data();
  PlainTableStorage storage;
  PlainTables t{&storage};

  // 1. candidate starts: the member's first block, then one per piece of input
  size_t pos = 0;
  if (int rc = gzip_header(in, n, &pos)) {
    printf("error: header status %d\n", rc);
    return 4;
  }
  std::vector<uint64_t> starts{(uint64_t)pos * 8};
  for (uint64_t j = 1; j * piece < n; ++j) {
    const uint64_t hi = (j + 1) * piece < n ? (j + 1) * piece : n;
    for (uint64_t bit = j * piece * 8; bit < hi * 8; ++bit)
      if (probe_block_start(in, n, bit, t, kProbeTrial)) {
        // (skew: every other candidate one bit late, so that the piece in front of it runs past it)
        const uint64_t s = bit + (skew && (starts.size() & 1) ? 1 : 0);
        if (s > starts.back()) starts.push_back(s);
        break;
      }
  }
  std::vector<uint8_t> is_member(starts.size(), 0);
  is_member[0] = 1;
  if (members) {  // and every gzip header
    std::vector<uint64_t> heads;
    for (size_t p = 0; p < n; ++p) {
      uint64_t bit = 0;
      if (member_start_at(in, n, p, &bit)) heads.push_back(bit);
    }
    std::vector<uint64_t> probe = starts;
    starts.resize(probe.size() + heads.size());
    is_member.resize(starts.size());
    starts.resize(merge_starts(probe.data(), (uint32_t)probe.size(), heads.data(), (uint32_t)heads.size(), starts.data(),
                               is_member.data()));
  }
  const uint32_t n_pieces = (uint32_t)starts.size();

  // 2. every piece to its first block end at or beyond the next candidate
  std::vector<PieceMeta> meta(n_pieces);
  for (uint32_t j = 0; j < n_pieces; ++j) {
    PieceMeta& m = meta[j];
    m.status = piece_boundary(in, n, starts.data(), n_pieces, j, kMaxAbsorb, t, &m.next, &m.end_bit, &m.out_len,
                              is_member[j] ? 0u : kWindow);
  }

  // 3. the chain from the first piece to the last trailer, which ends the file
  std::vector<uint32_t> chain(n_pieces), member_of(n_pieces);
  std::vector<MemberTrailer> trailers(n_pieces);
  uint32_t n_members = 0;
  uint64_t absorbed = 0;
  const uint32_t n_chain = members_chain(in, n, starts.data(), is_member.data(), meta.data(), n_pieces, chain.data(), member_of.data(),
                                         trailers.data(), &n_members, &absorbed);
  if (n_chain == 0) {
    printf("decline: the chain of pieces does not reach the member's end\n");
    return 3;
  }
  std::vector<uint64_t> off(n_chain + 1, 0), member_begin(n_members + 1, 0);
  for (uint32_t i = 0; i < n_chain; ++i) {
    if (i > 0 && member_of[i] != member_of[i - 1]) member_begin[member_of[i]] = off[i];
    off[i + 1] = off[i] + meta[chain[i]].out_len;
  }
  const uint64_t total = off[n_chain];
  member_begin[n_members] = total;

  // 4. symbols of every piece on the chain; a match may reach back to its member's first byte
  std::vector<uint16_t> sym(total + 1);
  for (uint32_t i = 0; i < n_chain; ++i) {
    const uint32_t j = chain[i];
    const uint64_t in_member = off[i] - member_begin[member_of[i]];
    MarkSink sink{sym.data() + off[i], 0, meta[j].out_len, in_member < kWindow ? in_member : kWindow};
    uint64_t e = 0;
    bool fin = false;
    const uint64_t want_end = meta[j].end_bit;
    const int rc = inflate_piece(in, n, starts[j], want_end, t, sink, [&](uint64_t b) { return b >= want_end; }, &e, &fin);
    if (rc != kOk || e != want_end || sink.op != meta[j].out_len) {
      printf("error: piece %u decodes differently the second time (status %d)\n", j, rc);
      return 4;
    }
  }

  // 5. waves of about total / waves bytes (at least one piece each); every wave sees only its own
  // symbols and the window composed from the waves before it
  std::vector<uint8_t> text(total + 1);
  const uint64_t cap = (total + waves - 1) / waves;
  std::vector<uint8_t> window(kWindow, 0), next(kWindow);  // W_0: zeros
  std::vector<uint16_t> front(kWindow);
  for (uint32_t a = 0; a < n_chain;) {
    uint32_t b = a;
    uint64_t len = 0;
    while (b < n_chain && (b == a || len + (off[b + 1] - off[b]) <= cap)) len += off[b + 1] - off[b], ++b;
    uint16_t* ws = sym.data() + off[a];  // the wave's symbols, addressed from its first byte
    uint8_t* wt = text.data() + off[a];
    auto region = [&](uint32_t i) { return off[i + 1] - off[i] > kWindow ? off[i + 1] - kWindow : off[i]; };
    for (uint32_t i = a; i < b; ++i)  // a. piece after piece
      for (uint64_t x = region(i); x < off[i + 1]; ++x) ws[x - off[a]] = relay_symbol(ws[x - off[a]], off[i] - off[a], ws);
    const uint64_t m = len < kWindow ? len : kWindow;  // b. F_k and W_{k+1}
    for (uint64_t j = 0; j < m; ++j) front[kWindow - m + j] = ws[len - m + j];
    wave_front(front.data(), len);
    compose_window(front.data(), window.data(), next.data());
    for (uint32_t i = a; i < b; ++i) {  // c. the relayed symbols, then the rest
      for (uint64_t x = region(i); x < off[i + 1]; ++x) wt[x - off[a]] = settle_symbol(ws[x - off[a]], window.data());
      for (uint64_t x = off[i]; x + kWindow < off[i + 1]; ++x)
        wt[x - off[a]] = settle_symbol(relay_symbol(ws[x - off[a]], off[i] - off[a], ws), window.data());
    }
    window.swap(next);
    a = b;
  }

  // 6. CRC-32 in pieces, joined per member
  uint32_t table[256];
  for (uint32_t i = 0; i < 256; ++i) table[i] = crc_table_entry(i);
  std::vector<uint32_t> crc(n_members, 0);
  for (uint32_t i = 0; i < n_chain; ++i) {
    const uint64_t len = off[i + 1] - off[i];
    crc[member_of[i]] = crc_combine(crc[member_of[i]], crc_bytes(text.data() + off[i], len, [&](uint32_t k) { return table[k]; }), len);
  }
  for (uint32_t m = 0; m < n_members; ++m) {
    if (crc[m] != trailers[m].crc) {
      printf("error: CRC-32 of the inflated bytes differs from the trailer of member %u\n", m);
      return 4;
    }
    if (trailers[m].isize != (uint32_t)(member_begin[m + 1] - member_begin[m])) {
      printf("error: ISIZE differs from the inflated length of member %u\n", m);
      return 4;
    }
  }
  unsigned long long h = 1469598103934665603ull;
  for (uint64_t i = 0; i < total; ++i) h = (h ^ text[i]) * 1099511628211ull;
  printf("%llu %llx %u %u %llu", (unsigned long long)total, h, n_pieces, n_chain, (unsigned long long)absorbed);
  if (members) printf(" %u", n_members);
  printf("\n");
  return 0;
}
