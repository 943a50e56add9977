// Test helper: are two indexdb file sets (prefix A = reference-built, prefix B = smr_build_index) the same index up to the
// arbitrary numbering of the unique L-mers?  Checks, for part 0..P-1:
//   .kmer      byte-identical
//   .bursttrie byte-identical except the id word of every bucket entry; the id pairs (a,b) met along the way must form a
//              bijection
//   .pos       same N; list of id a == list of id b (same order) under that bijection
//   .stats     identical apart from the embedded FASTA path and the 4 padding bytes of each index_parts_stats record
// Usage: index_equiv_check <prefixA> <prefixB> <lnwin>.  Prints "OK ..." and exits 0, or the first difference and exits 1.
//        index_equiv_check --canonical <prefix> <lnwin> <out>: writes a form of the index that equivalent indexes share (the
//        .stats FASTA size and body without path and padding, then per part the .kmer bytes, the .bursttrie with every id replaced by its
//        rank of first appearance, and the position lists in that order), so that a digest of it stands for the index.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <fstream>
#include <string>
#include <vector>

static std::vector<uint8_t> slurp(const std::string& p, bool& ok) {
  std::ifstream in(p, std::ios::binary | std::ios::ate);
  std::vector<uint8_t> v;
  ok = (bool)in;
  if (!ok) return v;
  v.resize((size_t)in.tellg());
  in.seekg(0);
  if (!v.empty()) in.read((char*)v.data(), (std::streamsize)v.size());
  return v;
}
static void die(const std::string& m) { printf("DIFF %s\n", m.c_str()); exit(1); }
static uint32_t u32(const std::vector<uint8_t>& v, size_t o) { uint32_t x; if (o + 4 > v.size()) die("truncated"); memcpy(&x, &v[o], 4); return x; }

struct Stats { uint64_t fsize; std::string name; std::vector<uint8_t> rest_wo_pad; uint16_t parts; };
static Stats parse_stats(const std::string& p) {
  bool ok; auto v = slurp(p, ok);
  if (!ok) die("cannot read " + p);
  Stats s; size_t o = 0;
  memcpy(&s.fsize, &v[o], 8); o += 8;
  uint32_t nl = u32(v, o); o += 4;
  s.name.assign((const char*)&v[o], nl); o += nl;
  size_t fixed = 32 + 8 + 4 + 8;            // freqs, full_len, lnwin, numseq
  s.rest_wo_pad.insert(s.rest_wo_pad.end(), v.begin() + o, v.begin() + o + fixed); o += fixed;
  memcpy(&s.parts, &v[o], 2); o += 2;
  for (uint16_t k = 0; k < s.parts; ++k) { s.rest_wo_pad.insert(s.rest_wo_pad.end(), v.begin() + o, v.begin() + o + 20); o += 24; }
  s.rest_wo_pad.insert(s.rest_wo_pad.end(), v.begin() + o, v.end());
  return s;
}

static int canonical(const std::string& A, uint32_t lnwin, const std::string& out_path) {
  const uint32_t limit = 1u << lnwin;
  const Stats sa = parse_stats(A + ".stats");
  std::vector<uint8_t> out((const uint8_t*)&sa.fsize, (const uint8_t*)&sa.fsize + 8);
  auto put = [&](const uint8_t* p, size_t n) { out.insert(out.end(), p, p + n); };
  put(sa.rest_wo_pad.data(), sa.rest_wo_pad.size());
  auto put32 = [&](uint32_t x) { put((const uint8_t*)&x, 4); };
  for (uint16_t part = 0; part < sa.parts; ++part) {
    const std::string ps = std::to_string(part);
    bool ok;
    auto ka = slurp(A + ".kmer_" + ps + ".dat", ok);
    if (!ok) die("kmer file missing");
    auto ta = slurp(A + ".bursttrie_" + ps + ".dat", ok);
    if (!ok) die("bursttrie file missing");
    auto pa = slurp(A + ".pos_" + ps + ".dat", ok);
    if (!ok) die("pos file missing");
    put(ka.data(), ka.size());
    const uint32_t N = u32(pa, 0);
    std::vector<uint32_t> rank(N, 0xFFFFFFFFu), order;
    size_t o = 0;
    for (uint32_t i = 0; i < limit; ++i) {
      const uint32_t sz[2] = {u32(ta, o), u32(ta, o + 4)};
      put(&ta[o], 8);
      o += 8;
      for (int j = 0; j < 2; ++j) {
        if (!sz[j]) continue;
        std::deque<uint8_t> fifo;
        for (int k = 0; k < 4; ++k) { fifo.push_back(ta[o]); put(&ta[o], 1); ++o; }
        while (!fifo.empty()) {
          const uint8_t f = fifo.front(); fifo.pop_front();
          if (f == 1) { for (int k = 0; k < 4; ++k) { fifo.push_back(ta[o]); put(&ta[o], 1); ++o; } }
          else if (f == 2) {
            const uint32_t bytes = u32(ta, o);
            put(&ta[o], 4);
            o += 4;
            for (uint32_t e = 0; e < bytes / 8; ++e, o += 8) {
              const uint32_t id = u32(ta, o + 4);
              if (id >= N) die("id out of range");
              if (rank[id] == 0xFFFFFFFFu) { rank[id] = (uint32_t)order.size(); order.push_back(id); }
              put(&ta[o], 4);
              put32(rank[id]);
            }
          } else if (f != 0) die("bad flag");
        }
      }
    }
    if (o != ta.size()) die("trailing bytes in bursttrie");
    if (order.size() != N) die("an id never appears in a bucket");
    std::vector<size_t> offa(N);
    size_t oa = 4;
    for (uint32_t i = 0; i < N; ++i) { offa[i] = oa; oa += 4 + (size_t)u32(pa, oa) * 8; }
    if (oa != pa.size()) die("pos file length");
    put32(N);
    for (uint32_t id : order) put(&pa[offa[id]], 4 + (size_t)u32(pa, offa[id]) * 8);
  }
  FILE* f = fopen(out_path.c_str(), "wb");
  if (!f || fwrite(out.data(), 1, out.size(), f) != out.size()) die("cannot write " + out_path);
  fclose(f);
  printf("OK parts=%u bytes=%zu\n", sa.parts, out.size());
  return 0;
}

int main(int argc, char** argv) {
  if (argc == 5 && std::string(argv[1]) == "--canonical") return canonical(argv[2], (uint32_t)atoi(argv[3]), argv[4]);
  if (argc < 4) { fprintf(stderr, "usage: %s prefixA prefixB lnwin\n", argv[0]); return 2; }
  const std::string A = argv[1], B = argv[2];
  const uint32_t lnwin = (uint32_t)atoi(argv[3]), limit = 1u << lnwin;
  const Stats sa = parse_stats(A + ".stats"), sb = parse_stats(B + ".stats");
  if (sa.fsize != sb.fsize) die("stats: file size");
  if (sa.parts != sb.parts) die("stats: number of parts");
  if (sa.rest_wo_pad != sb.rest_wo_pad) die("stats: body");
  uint64_t total_ids = 0, total_entries = 0;
  for (uint16_t part = 0; part < sa.parts; ++part) {
    const std::string ps = std::to_string(part);
    bool ok1, ok2;
    auto ka = slurp(A + ".kmer_" + ps + ".dat", ok1), kb = slurp(B + ".kmer_" + ps + ".dat", ok2);
    if (!ok1 || !ok2) die("kmer file missing");
    if (ka != kb) die("kmer counts differ in part " + ps);
    auto ta = slurp(A + ".bursttrie_" + ps + ".dat", ok1), tb = slurp(B + ".bursttrie_" + ps + ".dat", ok2);
    if (!ok1 || !ok2) die("bursttrie file missing");
    if (ta.size() != tb.size()) die("bursttrie size differs in part " + ps);
    auto pa = slurp(A + ".pos_" + ps + ".dat", ok1), pb = slurp(B + ".pos_" + ps + ".dat", ok2);
    if (!ok1 || !ok2) die("pos file missing");
    if (pa.size() != pb.size()) die("pos size differs in part " + ps);
    const uint32_t N = u32(pa, 0);
    if (N != u32(pb, 0)) die("number of unique L-mers differs");
    std::vector<uint32_t> a2b(N, 0xFFFFFFFFu), b2a(N, 0xFFFFFFFFu);
    // walk both trie streams in lock step
    size_t o = 0;
    for (uint32_t i = 0; i < limit; ++i) {
      uint32_t sz[2] = {u32(ta, o), u32(ta, o + 4)};
      if (sz[0] != u32(tb, o) || sz[1] != u32(tb, o + 4)) die("trie sizes differ at 9-mer " + std::to_string(i));
      o += 8;
      uint32_t cnt; memcpy(&cnt, &ka[(size_t)i * 4], 4);
      if (cnt == 0) { if (sz[0] || sz[1]) die("trie without count at 9-mer " + std::to_string(i)); continue; }
      for (int j = 0; j < 2; ++j) {
        if (!sz[j]) continue;
        std::deque<uint8_t> fifo;
        for (int k = 0; k < 4; ++k) { if (ta[o] != tb[o]) die("flag differs"); fifo.push_back(ta[o]); ++o; }
        while (!fifo.empty()) {
          const uint8_t f = fifo.front(); fifo.pop_front();
          if (f == 1) { for (int k = 0; k < 4; ++k) { if (ta[o] != tb[o]) die("flag differs"); fifo.push_back(ta[o]); ++o; } }
          else if (f == 2) {
            const uint32_t bytes = u32(ta, o);
            if (bytes != u32(tb, o)) die("bucket size differs at 9-mer " + std::to_string(i));
            o += 4;
            for (uint32_t e = 0; e < bytes / 8; ++e, o += 8) {
              if (u32(ta, o) != u32(tb, o)) die("bucket tail differs at 9-mer " + std::to_string(i));
              const uint32_t ia = u32(ta, o + 4), ib = u32(tb, o + 4);
              if (ia >= N || ib >= N) die("id out of range");
              if (a2b[ia] == 0xFFFFFFFFu && b2a[ib] == 0xFFFFFFFFu) { a2b[ia] = ib; b2a[ib] = ia; }
              else if (a2b[ia] != ib || b2a[ib] != ia) die("ids are not related by a bijection at 9-mer " + std::to_string(i));
              ++total_entries;
            }
          } else if (f != 0) die("bad flag");
        }
      }
    }
    if (o != ta.size()) die("trailing bytes in bursttrie");
    // positions: offsets per id, then compare lists under the bijection
    std::vector<size_t> offa(N), offb(N);
    size_t oa = 4, ob = 4;
    for (uint32_t i = 0; i < N; ++i) { offa[i] = oa; oa += 4 + (size_t)u32(pa, oa) * 8; }
    for (uint32_t i = 0; i < N; ++i) { offb[i] = ob; ob += 4 + (size_t)u32(pb, ob) * 8; }
    if (oa != pa.size() || ob != pb.size()) die("pos file length");
    for (uint32_t i = 0; i < N; ++i) {
      if (a2b[i] == 0xFFFFFFFFu) die("id " + std::to_string(i) + " of A never appears in a bucket");
      const size_t x = offa[i], y = offb[a2b[i]];
      const uint32_t sz = u32(pa, x);
      if (sz != u32(pb, y)) die("position list length differs for id " + std::to_string(i));
      if (memcmp(&pa[x + 4], &pb[y + 4], (size_t)sz * 8) != 0) die("position list differs for id " + std::to_string(i));
    }
    total_ids += N;
  }
  printf("OK parts=%u ids=%llu entries=%llu\n", sa.parts, (unsigned long long)total_ids, (unsigned long long)total_entries);
  return 0;
}
