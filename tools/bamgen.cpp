// bamgen — deterministic synthetic BAM + BAI writer for the `ngs qc` hot path.
//
// The reference ships no BAM fixture and `ngs generate` only emits FASTQ
// (reference src/generate/command.rs:72-75), so every input for parity tests
// and for bench.py is authored here.  Every record is a pure function of
// (seed, record index): blocks can therefore be produced by any number of
// threads, in any order, and always give the same bytes.
//
// Layout choices follow what htslib-written files look like (SURVEY App. A):
//   * header in its own BGZF block(s), records packed into 0xFF00-byte
//     payloads (records straddle blocks), 28-byte EOF marker;
//   * text header "@HD VN:1.6 SO:coordinate" + one @SQ per binary reference
//     (SURVEY App. D.11);
//   * BAI with bins/chunks, 16 kb linear index, pseudo-bin 37450 and n_no_coor.
//
// Shapes (BASELINE.json configs): 0 = C1 3-contig 2x150, 1 = WGS 25-contig
// 2x150 (C2/C3), 2 = long reads 10-50 kb on chr1-5 (C4), 3 = spliced 2x100
// RNA-seq (C5), 4 = references past 2^29 and 2^30 bases (a CSI's inputs:
// a 1.9 Gbp, a 0.8 Gbp and a 1 Mbp reference) with short, 10-50 kb and spliced
// reads, some of them across 2^29; no BAI can address it, so none is written.
//
// Exposed both as a C API (libngs_synth.so, used by tests/bench via ctypes)
// and as a CLI (`bamgen <shape> <n_records> <out.bam> [seed] [level] [threads]`).

#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

namespace {

constexpr uint32_t kPayload = 0xFF00;  // htslib BGZF_BLOCK_SIZE
constexpr uint32_t kChunkRecs = 1024;  // granularity of the size index

struct Contig {
  const char* name;
  uint32_t len;
};

const Contig kC1[] = {{"chr1", 20000000}, {"chr2", 10000000}, {"chrM", 16569}};
const Contig kBig[] = {{"chrA", 1900000000}, {"chrB", 800000000}, {"chrS", 1000000}};
const Contig kWGS[] = {
    {"chr1", 248956422},  {"chr2", 242193529},  {"chr3", 198295559},  {"chr4", 190214555},
    {"chr5", 181538259},  {"chr6", 170805979},  {"chr7", 159345973},  {"chr8", 145138636},
    {"chr9", 138394717},  {"chr10", 133797422}, {"chr11", 135086622}, {"chr12", 133275309},
    {"chr13", 114364328}, {"chr14", 107043718}, {"chr15", 101991189}, {"chr16", 90338345},
    {"chr17", 83257441},  {"chr18", 80373285},  {"chr19", 58617616},  {"chr20", 64444167},
    {"chr21", 46709983},  {"chr22", 50818468},  {"chrX", 156040895},  {"chrY", 57227415},
    {"chrM", 16569}};

inline uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

struct Rng {
  uint64_t s;
  explicit Rng(uint64_t seed) : s(seed) {}
  uint64_t next() {
    s += 0x9E3779B97F4A7C15ull;
    uint64_t x = s;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
  }
  uint32_t below(uint32_t n) { return (uint32_t)(((next() >> 32) * (uint64_t)n) >> 32); }
  uint32_t permille() { return below(1000); }
};

int reg2bin(int64_t beg, int64_t end) {
  --end;
  if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
  if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
  if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
  if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
  if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
  return 0;
}

struct Shape {
  int kind = 0;
  std::vector<Contig> contigs;
  uint64_t n = 0, n_unmapped_tail = 0;
  std::vector<uint64_t> cum;  // cum[c] = first record index of contig c; cum[n_ref] = first tail record
  uint64_t seed = 0;
  uint32_t read_len = 150;
  uint32_t read_groups = 1;  // @RG rg0..rg{K-1}; K = 1 writes the bytes of a generator without read groups
  uint64_t hot_lo = 0, hot_n = 0;  // hotspot in contig 0: records [hot_lo, hot_lo+hot_n) share one pos
  // subset generation (one shard of the logical file): global record-index ranges, ascending
  std::vector<std::pair<uint64_t, uint64_t>> ranges;
  std::vector<uint64_t> range_base;  // local ordinal of each range's first record
  uint64_t n_local = 0;
  uint64_t to_global(uint64_t q) const {
    size_t k = std::upper_bound(range_base.begin(), range_base.end(), q) - range_base.begin() - 1;
    return ranges[k].first + (q - range_base[k]);
  }
  void set_ranges(std::vector<std::pair<uint64_t, uint64_t>> r) {
    ranges.clear(); range_base.clear(); n_local = 0;
    for (auto& x : r) if (x.second > x.first) { ranges.push_back(x); range_base.push_back(n_local); n_local += x.second - x.first; }
    if (ranges.empty()) { ranges.push_back({0, 0}); range_base.push_back(0); }
  }
};

// Everything about a record except its sequence/quality bytes.
struct Meta {
  int32_t ref_id, pos, next_ref, next_pos, tlen;
  uint16_t flag, n_cigar, bin;
  uint8_t mapq;
  uint32_t l_seq, span;
  uint32_t cigar[8];      // short-read shapes: at most 8 ops
  uint32_t size;          // bytes incl. the 4-byte block_size prefix
  bool missing_qual;
  bool long_read;         // the CIGAR is a LongCigar (shape 2, and shape 4's long reads)
  uint64_t rng_state;     // state handed to the payload generator
};

constexpr uint32_t kNameLen = 20;  // "syn:%015llu" + NUL
constexpr uint32_t kAuxLen = 15;   // NM:C AS:C RG:Z:rg0

inline uint32_t op(uint32_t len, uint32_t code) { return (len << 4) | code; }
// op codes: M0 I1 D2 N3 S4 H5 P6 =7 X8

void locate(const Shape& sh, uint64_t i, int& c, uint64_t& j) {
  int n_ref = (int)sh.contigs.size();
  if (i >= sh.cum[n_ref]) {
    c = -1;
    j = i - sh.cum[n_ref];
    return;
  }
  int lo = 0;
  while (lo + 1 < n_ref && sh.cum[lo + 1] <= i) ++lo;
  c = lo;
  j = i - sh.cum[lo];
}

inline int32_t pos_of(const Shape& sh, int c, uint64_t j) {
  uint64_t n_c = sh.cum[c + 1] - sh.cum[c];
  uint64_t L = sh.contigs[c].len;
  uint64_t margin = sh.kind == 2 ? 5000 : 60;
  uint64_t range = L > margin ? L - margin : 1;
  if (c == 0 && sh.hot_n) {
    if (j >= sh.hot_lo && j < sh.hot_lo + sh.hot_n) j = sh.hot_lo;
  }
  if (j + 1 == n_c && L > 50) return (int32_t)(L - 50);  // last read overhangs the contig end (nonsensical positions)
  return (int32_t)((unsigned __int128)j * range / n_c);
}

// Long-read CIGAR: generated on the fly by both meta (for span/size) and payload.
struct LongCigar {
  Rng rng;
  uint32_t remaining;  // query bases still to emit
  bool first = true;
  explicit LongCigar(uint64_t st, uint32_t qlen) : rng(st), remaining(qlen) {}
  // returns 0 when done
  uint32_t next() {
    if (remaining == 0) return 0;
    uint32_t r = (uint32_t)rng.next();
    if (first) {
      first = false;
      if ((r & 3) == 0) {
        uint32_t l = 1 + (r >> 8) % 200;
        if (l >= remaining) l = remaining;
        remaining -= l;
        return op(l, 4);
      }
    }
    uint32_t l = 8 + (r >> 4) % 13;
    uint32_t k = (r >> 20) % 16;
    uint32_t code;
    if (k < 8) code = 0;        // M
    else if (k < 11) code = 7;  // =
    else if (k < 12) code = 8;  // X
    else if (k < 14) code = 1;  // I
    else code = 2;              // D
    if (code == 8) l = 1 + l % 3;
    if (code == 1 || code == 2) l = 1 + l % 6;
    if (code == 2) return op(l, 2);  // D consumes no query
    if (l > remaining) l = remaining;
    remaining -= l;
    return op(l, code);
  }
};

void make_meta(const Shape& sh, uint64_t i, Meta& m) {
  Rng rng(splitmix64(sh.seed ^ (i * 0xD1342543DE82EF95ull)));
  int c;
  uint64_t j;
  locate(sh, i, c, j);
  m.missing_qual = false;
  m.long_read = sh.kind == 2;
  m.n_cigar = 0;
  m.span = 0;
  uint32_t R = sh.read_len;
  if (sh.kind == 2) R = 10000 + rng.below(40001);
  if (sh.kind == 4 && rng.permille() < 10) { m.long_read = true; R = 10000 + rng.below(40001); }
  uint32_t pm = rng.permille();
  if (sh.kind != 2 && !m.long_read) {
    if (pm < 20) R = 30 + rng.below(R - 30);        // trimmed (<100 exercises GC too-short)
    else if (pm < 23) R = 100 + (pm & 1);           // exactly 100 / 101
  }
  bool rna = sh.kind == 3;
  uint16_t f = 0x1;
  uint32_t fl = rng.permille();
  f |= (rng.next() & 1) ? 0x40 : 0x80;
  if (rng.next() & 1) f |= 0x10;
  if (rng.next() & 1) f |= 0x20;
  if (rng.permille() < 920) f |= 0x2;
  if (rng.permille() < (rna ? 400u : 50u)) f |= 0x400;
  if (rng.permille() < (rna ? 80u : 10u)) f |= 0x100;
  if (rng.permille() < (rna ? 10u : 5u)) f |= 0x800;
  if (rng.permille() < 3) f |= 0x200;
  bool mate_unmapped = rng.permille() < 15;
  bool self_unmapped = false;
  if (fl < 5) {  // unpaired
    f &= ~(0x1 | 0x2 | 0x8 | 0x20 | 0x40 | 0x80);
    if (fl == 0) f |= 0x40;  // odd but legal: exercises the read-one CIGAR split
    mate_unmapped = false;
  }
  uint32_t mq = rng.permille();
  if (mq < 50) m.mapq = 0;
  else if (mq < 80) m.mapq = 1 + rng.below(4);
  else if (mq < 280) m.mapq = 5 + rng.below(55);
  else if (mq < 980) m.mapq = 60;
  else m.mapq = 255;

  if (c < 0) {  // unplaced unmapped tail
    f = (f & (0x1 | 0x40 | 0x80 | 0x200)) | 0x4;
    if (f & 0x1) f |= 0x8;
    m.ref_id = -1; m.pos = -1; m.next_ref = -1; m.next_pos = -1; m.tlen = 0;
    m.mapq = 0;
    m.bin = 4680;
    if (sh.kind == 2) R = 10000 + rng.below(2000);
    if (rng.permille() < 20) R = 0;  // empty SEQ
  } else {
    m.ref_id = c;
    m.pos = pos_of(sh, c, j);
    int n_ref = (int)sh.contigs.size();
    if ((f & 0x1) && rng.permille() < 10) {  // placed unmapped (mate mapped)
      self_unmapped = true;
      f |= 0x4;
      f &= ~0x2;
      mate_unmapped = false;
      m.mapq = 0;
    }
    if (mate_unmapped) { f |= 0x8; f &= ~0x2; }
    if (!(f & 0x1)) { m.next_ref = -1; m.next_pos = -1; m.tlen = 0; }
    else if (mate_unmapped) { m.next_ref = c; m.next_pos = m.pos; m.tlen = 0; }
    else {
      if (n_ref > 1 && rng.permille() < 30) {
        m.next_ref = (c + 1 + (int)rng.below(n_ref - 1)) % n_ref;
        m.next_pos = (int32_t)rng.below(sh.contigs[m.next_ref].len);
        m.tlen = 0;
      } else {
        m.next_ref = c;
        uint32_t t = rng.permille();
        int32_t tl;
        if (t < 20) tl = 0;
        else if (t < 50) tl = 1025 + (int32_t)rng.below(100000);
        else tl = 50 + (int32_t)(rng.below(200) + rng.below(200) + rng.below(200) + rng.below(200));
        if (t >= 990) tl = 1024 - (int32_t)(t - 990) / 5;  // pile a few on the last bins
        bool neg = (f & 0x10) != 0;
        m.tlen = neg ? -tl : tl;
        int64_t np = (int64_t)m.pos + (neg ? -(int64_t)tl : (int64_t)tl);
        if (np < 0) np = 0;
        if (np >= (int64_t)sh.contigs[c].len) np = sh.contigs[c].len - 1;
        m.next_pos = (int32_t)np;
      }
    }
  }
  m.flag = f;
  m.l_seq = R;
  m.rng_state = rng.next();

  // CIGAR
  bool mapped = c >= 0 && !self_unmapped;
  uint32_t cig_bytes = 0;
  if (mapped && R > 0) {
    if (m.long_read) {
      LongCigar lc(m.rng_state, R);
      uint32_t n = 0, span = 0;
      while (uint32_t o = lc.next()) {
        ++n;
        uint32_t code = o & 15, l = o >> 4;
        if (code == 0 || code == 2 || code == 3 || code == 7 || code == 8) span += l;
      }
      m.n_cigar = (uint16_t)n;
      m.span = span;
      cig_bytes = 4 * n;
    } else {
      uint32_t k = rng.permille();
      uint32_t* cg = m.cigar;
      uint32_t n = 0;
      if ((rna || sh.kind == 4) && k < (rna ? 600u : 300u) && R >= 40) {
        uint32_t a = 10 + rng.below(R - 20);
        // shape 4: introns up to 8 record spacings (at most 2^26), so that some spliced reads cross 2^29 at any record count
        const uint32_t spacing = sh.kind == 4 ? (uint32_t)(sh.contigs[c].len / (sh.cum[c + 1] - sh.cum[c])) : 0;
        uint32_t skip = 100 + rng.below(sh.kind == 4 ? std::min<uint32_t>(std::max<uint32_t>(199901, 8 * spacing), 1u << 26) : 199901);
        cg[n++] = op(a, 0); cg[n++] = op(skip, 3); cg[n++] = op(R - a, 0);
        if (k < 60 && R - a > 20) {  // second junction
          uint32_t b = 5 + rng.below(R - a - 10);
          cg[n - 1] = op(b, 0);
          cg[n++] = op(100 + rng.below(5000), 3);
          cg[n++] = op(R - a - b, 0);
        }
      } else if (k < 700 || R < 40) {
        cg[n++] = op(R, 0);
      } else if (k < 820) {
        uint32_t a = 1 + rng.below(R / 3);
        if (k & 1) { cg[n++] = op(a, 4); cg[n++] = op(R - a, 0); }
        else { cg[n++] = op(R - a, 0); cg[n++] = op(a, 4); }
      } else if (k < 880) {
        uint32_t b = 1 + rng.below(5), a = 5 + rng.below(R - b - 10);
        cg[n++] = op(a, 0); cg[n++] = op(b, 1); cg[n++] = op(R - a - b, 0);
      } else if (k < 940) {
        uint32_t b = 1 + rng.below(20), a = 5 + rng.below(R - 10);
        cg[n++] = op(a, 0); cg[n++] = op(b, 2); cg[n++] = op(R - a, 0);
      } else if (k < 970) {
        uint32_t b = 1 + rng.below(3), a = 5 + rng.below(R - b - 10);
        cg[n++] = op(a, 7); cg[n++] = op(b, 8); cg[n++] = op(R - a - b, 7);
      } else if (k < 990) {
        cg[n++] = op(1 + rng.below(80), 5); cg[n++] = op(R, 0);
        if (k & 1) cg[n++] = op(1 + rng.below(40), 5);
      } else {
        uint32_t a = 5 + rng.below(R - 10);
        cg[n++] = op(a, 0); cg[n++] = op(1 + rng.below(3), 6); cg[n++] = op(R - a, 0);
      }
      uint32_t span = 0;
      for (uint32_t q = 0; q < n; ++q) {
        uint32_t code = cg[q] & 15, l = cg[q] >> 4;
        if (code == 0 || code == 2 || code == 3 || code == 7 || code == 8) span += l;
      }
      m.n_cigar = (uint16_t)n;
      m.span = span;
      cig_bytes = 4 * n;
    }
  }
  if (c >= 0) {
    int64_t end = (int64_t)m.pos + (m.span ? m.span : 1);
    m.bin = (uint16_t)reg2bin(m.pos, end);
    if (end > (1 << 29)) m.bin = 4680;  // shape 4: past what the bin field addresses (reg2bin(-1, 0), as for no position)
  }
  if (R > 0 && rng.permille() < 2) m.missing_qual = true;
  m.size = 4 + 32 + kNameLen + cig_bytes + (R + 1) / 2 + R + kAuxLen;
}

inline void put32(uint8_t* p, uint32_t v) { memcpy(p, &v, 4); }
inline void put16(uint8_t* p, uint16_t v) { memcpy(p, &v, 2); }

// Writes the full record (m.size bytes) to out.
void make_record(const Shape& sh, uint64_t i, const Meta& m, uint8_t* out) {
  uint8_t* p = out;
  put32(p, m.size - 4); p += 4;
  put32(p, (uint32_t)m.ref_id); put32(p + 4, (uint32_t)m.pos);
  p[8] = kNameLen; p[9] = m.mapq; put16(p + 10, m.bin); put16(p + 12, m.n_cigar);
  put16(p + 14, m.flag); put32(p + 16, m.l_seq); put32(p + 20, (uint32_t)m.next_ref);
  put32(p + 24, (uint32_t)m.next_pos); put32(p + 28, (uint32_t)m.tlen);
  p += 32;
  char name[32];
  snprintf(name, sizeof name, "syn:%015llu", (unsigned long long)i);
  memcpy(p, name, kNameLen); p += kNameLen;
  if (m.long_read) {
    if (m.n_cigar) {
      LongCigar lc(m.rng_state, m.l_seq);
      while (uint32_t o = lc.next()) { put32(p, o); p += 4; }
    }
  } else {
    for (uint32_t q = 0; q < m.n_cigar; ++q) { put32(p, m.cigar[q]); p += 4; }
  }
  Rng rng(splitmix64(m.rng_state ^ 0xA5A5A5A5ull));
  uint32_t R = m.l_seq;
  // sequence: per-record GC fraction in [0.20, 0.70]
  uint32_t gc_thr = 13107 + rng.below(32768);  // of 65536
  uint32_t nb = (R + 1) / 2;
  uint64_t bits = 0; int have = 0;
  for (uint32_t b = 0; b < nb; ++b) {
    uint8_t byte = 0;
    for (int h = 0; h < 2; ++h) {
      if (!have) { bits = rng.next(); have = 4; }
      uint32_t r16 = bits & 0xFFFF; bits >>= 16; --have;
      uint8_t code;
      if ((r16 & 0x1FF) == 0x1FF) code = 15;             // ~0.2 % N
      else if ((r16 & 0xFFF) == 0xABC) code = 3 + (r16 >> 12) % 4 * 3;  // rare ambiguity codes
      else if (((r16 * 40503u) & 0xFFFF) < gc_thr) code = (r16 & 0x8000) ? 2 : 4;
      else code = (r16 & 0x8000) ? 1 : 8;
      if (2 * b + h >= R) code = 0;
      byte = (uint8_t)((byte << 4) | code);
    }
    *p++ = byte;
  }
  // qualities: 7-point skewed Phred table, tail degrades with position
  static const uint8_t qtab[8] = {37, 37, 37, 40, 40, 25, 11, 2};
  if (m.missing_qual) {
    memset(p, 0xFF, R);
  } else {
    for (uint32_t q = 0; q < R; q += 8) {
      uint64_t r = rng.next();
      for (uint32_t k = 0; k < 8 && q + k < R; ++k) {
        uint32_t v = (r >> (8 * k)) & 0xFF;
        uint32_t posn = q + k;
        uint32_t decay = sh.kind == 2 ? 96 : 32 + (posn * 160) / (sh.read_len ? sh.read_len : 150);
        uint32_t idx = v < decay ? 5 + (v % 3) : (v & 3) + (v >> 7);
        p[q + k] = qtab[idx & 7];
      }
    }
  }
  p += R;
  uint64_t r = rng.next();
  p[0] = 'N'; p[1] = 'M'; p[2] = 'C'; p[3] = (uint8_t)(r % 6);
  p[4] = 'A'; p[5] = 'S'; p[6] = 'C'; p[7] = (uint8_t)(100 + (r >> 8) % 51);
  memcpy(p + 8, "RGZrg0", 7);  // includes NUL
  if (sh.read_groups > 1) p[13] = (uint8_t)('0' + (r >> 32) % sh.read_groups);  // the high half of the NM / AS draw
}

struct Built {
  std::vector<uint8_t> bam, bai;
  uint64_t n_records = 0, inflated = 0, header_inflated = 0;
  uint32_t n_blocks = 0;
};

size_t bgzf_block(const uint8_t* src, uint32_t n, int level, uint8_t* dst, size_t cap) {
  z_stream zs;
  memset(&zs, 0, sizeof zs);
  if (deflateInit2(&zs, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) abort();
  zs.next_in = const_cast<uint8_t*>(src);
  zs.avail_in = n;
  zs.next_out = dst + 18;
  zs.avail_out = (uInt)(cap - 18 - 8);
  if (deflate(&zs, Z_FINISH) != Z_STREAM_END) abort();
  size_t clen = zs.total_out;
  deflateEnd(&zs);
  size_t total = 18 + clen + 8;
  if (total > 65536) abort();
  static const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
  memcpy(dst, hdr, 16);
  put16(dst + 16, (uint16_t)(total - 1));
  put32(dst + 18 + clen, (uint32_t)crc32(crc32(0, nullptr, 0), src, n));
  put32(dst + 18 + clen + 4, n);
  return total;
}

void setup_shape(Shape& sh, int kind, uint64_t n, uint64_t seed) {
  sh.kind = kind;
  sh.n = n;
  sh.seed = seed;
  sh.read_len = kind == 3 ? 100 : 150;
  if (kind == 0) sh.contigs.assign(kC1, kC1 + 3);
  else if (kind == 2) sh.contigs.assign(kWGS, kWGS + 5);
  else if (kind == 4) sh.contigs.assign(kBig, kBig + 3);
  else sh.contigs.assign(kWGS, kWGS + 25);
  size_t n_ref = sh.contigs.size();
  sh.n_unmapped_tail = n / 100;
  uint64_t nm = n - sh.n_unmapped_tail;
  long double tot = 0;
  std::vector<long double> w(n_ref);
  for (size_t c = 0; c < n_ref; ++c) {
    w[c] = sh.contigs[c].len;
    if (sh.contigs[c].len < 100000) w[c] = sh.contigs[c].len * 20.0L;  // chrM is deep in real data
    tot += w[c];
  }
  sh.cum.assign(n_ref + 1, 0);
  uint64_t used = 0;
  std::vector<uint64_t> cnt(n_ref);
  for (size_t c = 0; c < n_ref; ++c) { cnt[c] = (uint64_t)(nm * (w[c] / tot)); used += cnt[c]; }
  cnt[0] += nm - used;
  for (size_t c = 0; c < n_ref; ++c) sh.cum[c + 1] = sh.cum[c] + cnt[c];
  if (cnt[0] >= 20000 && kind != 2) { sh.hot_lo = cnt[0] / 3; sh.hot_n = 2600; }
  else if (cnt[0] >= 400) { sh.hot_lo = cnt[0] / 3; sh.hot_n = cnt[0] / 50; }
  sh.set_ranges({{0, n}});
}

std::vector<uint8_t> make_header(const Shape& sh) {
  std::string text = "@HD\tVN:1.6\tSO:coordinate\n";
  for (auto& c : sh.contigs) text += std::string("@SQ\tSN:") + c.name + "\tLN:" + std::to_string(c.len) + "\n";
  for (uint32_t k = 0; k < sh.read_groups; ++k) text += "@RG\tID:rg" + std::to_string(k) + "\tSM:synthetic\n";
  text += "@PG\tID:bamgen\tPN:bamgen\n";
  std::vector<uint8_t> h;
  auto p32 = [&](uint32_t v) { uint8_t b[4]; put32(b, v); h.insert(h.end(), b, b + 4); };
  h.insert(h.end(), {'B', 'A', 'M', 1});
  p32((uint32_t)text.size());
  h.insert(h.end(), text.begin(), text.end());
  p32((uint32_t)sh.contigs.size());
  for (auto& c : sh.contigs) {
    uint32_t l = (uint32_t)strlen(c.name) + 1;
    p32(l);
    h.insert(h.end(), c.name, c.name + l);
    p32(c.len);
  }
  return h;
}

template <class F>
void parallel_for(uint64_t n, int threads, F f) {
  std::atomic<uint64_t> next{0};
  std::vector<std::thread> ts;
  for (int t = 0; t < threads; ++t)
    ts.emplace_back([&, t] {
      for (;;) {
        uint64_t i = next.fetch_add(1);
        if (i >= n) break;
        f(i, t);
      }
    });
  for (auto& t : ts) t.join();
}

struct BaiRef {
  std::vector<std::pair<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>>> bins;  // sorted by first use
  std::vector<uint64_t> lin;
  uint64_t beg = 0, end = 0, n_mapped = 0, n_unmapped = 0;
  bool any = false;
};

void build(const Shape& sh, int level, int threads, Built& out) {
  const uint64_t N = sh.n_local;
  // pass 1: per-chunk byte totals (chunks of local ordinals)
  uint64_t n_chunks = (N + kChunkRecs - 1) / kChunkRecs;
  std::vector<uint64_t> chunk_off(n_chunks + 1, 0);
  parallel_for(n_chunks, threads, [&](uint64_t ch, int) {
    uint64_t lo = ch * kChunkRecs, hi = std::min(N, lo + kChunkRecs), s = 0;
    Meta m;
    for (uint64_t i = lo; i < hi; ++i) { make_meta(sh, sh.to_global(i), m); s += m.size; }
    chunk_off[ch + 1] = s;
  });
  for (uint64_t ch = 0; ch < n_chunks; ++ch) chunk_off[ch + 1] += chunk_off[ch];
  const uint64_t total = chunk_off[n_chunks];
  const uint64_t n_rec_blocks = (total + kPayload - 1) / kPayload;

  // header blocks
  std::vector<uint8_t> hdr = make_header(sh);
  std::vector<uint8_t> hdr_comp;
  uint32_t n_hdr_blocks = 0;
  for (size_t o = 0; o < hdr.size(); o += kPayload) {
    uint32_t n = (uint32_t)std::min<size_t>(kPayload, hdr.size() - o);
    uint8_t tmp[65536 + 64];
    size_t c = bgzf_block(hdr.data() + o, n, level, tmp, sizeof tmp);
    hdr_comp.insert(hdr_comp.end(), tmp, tmp + c);
    ++n_hdr_blocks;
  }

  // pass 2: blocks in groups, each group compressed into its own buffer
  const uint64_t kGroup = 64;
  uint64_t n_groups = (n_rec_blocks + kGroup - 1) / kGroup;
  std::vector<std::vector<uint8_t>> gbuf(n_groups);
  std::vector<uint32_t> csize(n_rec_blocks);
  parallel_for(n_groups, threads, [&](uint64_t g, int) {
    uint64_t b0 = g * kGroup, b1 = std::min(n_rec_blocks, b0 + kGroup);
    uint64_t byte0 = b0 * kPayload, byte1 = std::min(total, b1 * kPayload);
    std::vector<uint8_t> raw(byte1 - byte0 + 0);
    // find the first record overlapping byte0
    uint64_t ch = std::upper_bound(chunk_off.begin(), chunk_off.end(), byte0) - chunk_off.begin() - 1;
    if (ch >= n_chunks) ch = n_chunks - 1;
    uint64_t i = ch * kChunkRecs, off = chunk_off[ch];
    Meta m;
    std::vector<uint8_t> rec;
    while (off < byte1 && i < N) {
      const uint64_t gi = sh.to_global(i);
      make_meta(sh, gi, m);
      if (off + m.size > byte0) {
        rec.resize(m.size);
        make_record(sh, gi, m, rec.data());
        uint64_t lo = std::max(off, byte0), hi = std::min(off + m.size, byte1);
        memcpy(raw.data() + (lo - byte0), rec.data() + (lo - off), hi - lo);
      }
      off += m.size;
      ++i;
    }
    std::vector<uint8_t>& ob = gbuf[g];
    ob.resize((b1 - b0) * 65536);
    size_t w = 0;
    for (uint64_t b = b0; b < b1; ++b) {
      uint64_t lo = b * kPayload, hi = std::min(total, lo + kPayload);
      size_t c = bgzf_block(raw.data() + (lo - byte0), (uint32_t)(hi - lo), level, ob.data() + w, ob.size() - w);
      csize[b] = (uint32_t)c;
      w += c;
    }
    ob.resize(w);
    ob.shrink_to_fit();
  });
  // assemble
  std::vector<uint64_t> coff(n_rec_blocks + 1);
  coff[0] = hdr_comp.size();
  for (uint64_t b = 0; b < n_rec_blocks; ++b) coff[b + 1] = coff[b] + csize[b];
  static const uint8_t eof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  out.bam.resize(coff[n_rec_blocks] + 28);
  memcpy(out.bam.data(), hdr_comp.data(), hdr_comp.size());
  parallel_for(n_groups, threads, [&](uint64_t g, int) {
    memcpy(out.bam.data() + coff[g * kGroup], gbuf[g].data(), gbuf[g].size());
    std::vector<uint8_t>().swap(gbuf[g]);
  });
  memcpy(out.bam.data() + coff[n_rec_blocks], eof, 28);
  out.n_records = N;
  out.inflated = hdr.size() + total;
  out.header_inflated = hdr.size();
  out.n_blocks = (uint32_t)(n_hdr_blocks + n_rec_blocks + 1);

  // pass 3: BAI, one task per contig (none for shape 4: a BAI cannot address its references)
  if (sh.kind == 4) return;
  size_t n_ref = sh.contigs.size();
  std::vector<BaiRef> refs(n_ref);
  auto voff_of = [&](uint64_t stream_byte) -> uint64_t {
    uint64_t b = stream_byte / kPayload;
    if (b >= n_rec_blocks) return coff[n_rec_blocks] << 16;  // EOF block
    return (coff[b] << 16) | (stream_byte % kPayload);
  };
  parallel_for(n_ref, threads, [&](uint64_t c, int) {
    BaiRef& R = refs[c];
    uint64_t glo = sh.cum[c], ghi = sh.cum[c + 1];
    if (glo == ghi) return;
    // local ordinals of this contig (contigs are included whole or not at all)
    size_t rk = 0;
    bool present = false;
    for (; rk < sh.ranges.size(); ++rk) if (sh.ranges[rk].first <= glo && ghi <= sh.ranges[rk].second) { present = true; break; }
    if (!present) return;
    uint64_t lo = sh.range_base[rk] + (glo - sh.ranges[rk].first), hi = lo + (ghi - glo);
    uint64_t ch = lo / kChunkRecs;
    uint64_t i = ch * kChunkRecs, off = chunk_off[ch];
    Meta m;
    for (; i < lo; ++i) { make_meta(sh, sh.to_global(i), m); off += m.size; }
    R.any = true;
    R.beg = voff_of(off);
    R.lin.assign(((uint64_t)sh.contigs[c].len >> 14) + 1, 0);
    std::vector<int> bin_slot(37450, -1);
    uint32_t last_bin = 0xFFFFFFFFu;
    uint64_t save_off = R.beg;
    auto flush = [&](uint64_t end_off) {
      if (last_bin == 0xFFFFFFFFu) return;
      int& s = bin_slot[last_bin];
      if (s < 0) { s = (int)R.bins.size(); R.bins.push_back({last_bin, {}}); }
      R.bins[s].second.push_back({save_off, end_off});
    };
    for (; i < hi; ++i) {
      make_meta(sh, sh.to_global(i), m);
      uint64_t v = voff_of(off);
      if (m.bin != last_bin) { flush(v); last_bin = m.bin; save_off = v; }
      int64_t beg = m.pos, end = (int64_t)m.pos + (m.span ? m.span : 1);
      if (m.flag & 0x4) ++R.n_unmapped; else ++R.n_mapped;
      uint64_t w0 = (uint64_t)beg >> 14, w1 = (uint64_t)(end - 1) >> 14;
      if (w1 >= R.lin.size()) w1 = R.lin.size() - 1;
      for (uint64_t w = w0; w <= w1 && w < R.lin.size(); ++w)
        if (R.lin[w] == 0) R.lin[w] = v;
      off += m.size;
    }
    R.end = voff_of(off);
    flush(R.end);
    // htslib fills empty linear-index slots with the following value's predecessor; keep
    // the common "carry previous forward" convention.
    uint64_t last = 0;
    size_t used = 0;
    for (size_t w = 0; w < R.lin.size(); ++w) {
      if (R.lin[w] == 0) R.lin[w] = last; else { last = R.lin[w]; used = w + 1; }
    }
    R.lin.resize(used);
  });
  std::vector<uint8_t>& bi = out.bai;
  auto p32 = [&](uint32_t v) { uint8_t b[4]; put32(b, v); bi.insert(bi.end(), b, b + 4); };
  auto p64 = [&](uint64_t v) { uint8_t b[8]; memcpy(b, &v, 8); bi.insert(bi.end(), b, b + 8); };
  bi.insert(bi.end(), {'B', 'A', 'I', 1});
  p32((uint32_t)n_ref);
  for (size_t c = 0; c < n_ref; ++c) {
    BaiRef& R = refs[c];
    if (!R.any) { p32(0); p32(0); continue; }
    p32((uint32_t)R.bins.size() + 1);
    for (auto& b : R.bins) {
      p32(b.first);
      p32((uint32_t)b.second.size());
      for (auto& ck : b.second) { p64(ck.first); p64(ck.second); }
    }
    p32(37450); p32(2); p64(R.beg); p64(R.end); p64(R.n_mapped); p64(R.n_unmapped);
    p32((uint32_t)R.lin.size());
    for (uint64_t v : R.lin) p64(v);
  }
  p64(sh.ranges.back().second == sh.n && sh.n_local ? sh.n_unmapped_tail : 0);
}

}  // namespace

extern "C" {

struct synth_info {
  uint64_t n_records, inflated_bytes, header_bytes, bam_bytes, bai_bytes;
  uint32_t n_blocks, n_ref;
};

// Generates a BAM+BAI pair in memory. Buffers are malloc'd; release with synth_free.
int synth_bam(int shape, uint64_t n_records, uint64_t seed, int level, int threads, uint8_t** bam,
              uint8_t** bai, synth_info* info) {
  if (shape < 0 || shape > 4 || !bam || !bai) return -1;
  if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
  if (threads <= 0) threads = 1;
  Shape sh;
  setup_shape(sh, shape, n_records, seed);
  Built b;
  build(sh, level, threads, b);
  *bam = (uint8_t*)malloc(b.bam.size() ? b.bam.size() : 1);
  *bai = (uint8_t*)malloc(b.bai.size() ? b.bai.size() : 1);
  if (!*bam || !*bai) return -2;
  memcpy(*bam, b.bam.data(), b.bam.size());
  memcpy(*bai, b.bai.data(), b.bai.size());
  if (info) {
    info->n_records = b.n_records;
    info->inflated_bytes = b.inflated;
    info->header_bytes = b.header_inflated;
    info->bam_bytes = b.bam.size();
    info->bai_bytes = b.bai.size();
    info->n_blocks = b.n_blocks;
    info->n_ref = (uint32_t)sh.contigs.size();
  }
  return 0;
}

// One shard of the logical file: only the contigs whose bit is set in contig_mask (whole contigs),
// plus the unplaced-unmapped tail when with_tail != 0.  Record contents are identical to the
// corresponding records of the full file (records are pure functions of their global index).
int synth_bam_subset(int shape, uint64_t n_records, uint64_t seed, int level, int threads, uint64_t contig_mask,
                     int with_tail, uint8_t** bam, uint8_t** bai, synth_info* info) {
  if (shape < 0 || shape > 4 || !bam || !bai) return -1;
  if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
  if (threads <= 0) threads = 1;
  Shape sh;
  setup_shape(sh, shape, n_records, seed);
  std::vector<std::pair<uint64_t, uint64_t>> r;
  size_t n_ref = sh.contigs.size();
  for (size_t c = 0; c < n_ref; ++c)
    if ((contig_mask >> c) & 1) {
      if (!r.empty() && r.back().second == sh.cum[c]) r.back().second = sh.cum[c + 1];
      else r.push_back({sh.cum[c], sh.cum[c + 1]});
    }
  if (with_tail) {
    if (!r.empty() && r.back().second == sh.cum[n_ref]) r.back().second = sh.n;
    else r.push_back({sh.cum[n_ref], sh.n});
  }
  sh.set_ranges(r);
  Built b;
  build(sh, level, threads, b);
  *bam = (uint8_t*)malloc(b.bam.size() ? b.bam.size() : 1);
  *bai = (uint8_t*)malloc(b.bai.size() ? b.bai.size() : 1);
  if (!*bam || !*bai) return -2;
  memcpy(*bam, b.bam.data(), b.bam.size());
  memcpy(*bai, b.bai.data(), b.bai.size());
  if (info) {
    info->n_records = b.n_records;
    info->inflated_bytes = b.inflated;
    info->header_bytes = b.header_inflated;
    info->bam_bytes = b.bam.size();
    info->bai_bytes = b.bai.size();
    info->n_blocks = b.n_blocks;
    info->n_ref = (uint32_t)n_ref;
  }
  return 0;
}

// synth_bam with K read groups (1..10): the header declares rg0..rg{K-1} and each record's RG:Z takes its group from bits of
// the random draw its NM and AS values come from, so records keep their length; K = 1 is synth_bam.
int synth_bam_rg(int shape, uint64_t n_records, uint64_t seed, int level, int threads, uint32_t read_groups, uint8_t** bam,
                 uint8_t** bai, synth_info* info) {
  if (shape < 0 || shape > 4 || !bam || !bai || read_groups < 1 || read_groups > 10) return -1;
  if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
  if (threads <= 0) threads = 1;
  Shape sh;
  setup_shape(sh, shape, n_records, seed);
  sh.read_groups = read_groups;
  Built b;
  build(sh, level, threads, b);
  *bam = (uint8_t*)malloc(b.bam.size() ? b.bam.size() : 1);
  *bai = (uint8_t*)malloc(b.bai.size() ? b.bai.size() : 1);
  if (!*bam || !*bai) return -2;
  memcpy(*bam, b.bam.data(), b.bam.size());
  memcpy(*bai, b.bai.data(), b.bai.size());
  if (info) {
    info->n_records = b.n_records;
    info->inflated_bytes = b.inflated;
    info->header_bytes = b.header_inflated;
    info->bam_bytes = b.bam.size();
    info->bai_bytes = b.bai.size();
    info->n_blocks = b.n_blocks;
    info->n_ref = (uint32_t)sh.contigs.size();
  }
  return 0;
}

// Record counts per contig (and the tail) of the logical file: lets a planner balance shards.
int synth_layout(int shape, uint64_t n_records, uint64_t* per_contig, uint32_t cap, uint32_t* n_ref, uint64_t* tail) {
  Shape sh;
  setup_shape(sh, shape, n_records, 0);
  uint32_t n = (uint32_t)sh.contigs.size();
  if (n_ref) *n_ref = n;
  for (uint32_t c = 0; c < n && c < cap; ++c) per_contig[c] = sh.cum[c + 1] - sh.cum[c];
  if (tail) *tail = sh.n_unmapped_tail;
  return 0;
}

void synth_free(void* p) { free(p); }

}  // extern "C"

#ifdef BAMGEN_MAIN
int main(int argc, char** argv) {
  if (argc < 4) {
    fprintf(stderr, "usage: bamgen <shape 0..4> <n_records> <out.bam> [seed] [zlib level] [threads]\n");
    return 2;
  }
  int shape = atoi(argv[1]);
  uint64_t n = strtoull(argv[2], nullptr, 10);
  uint64_t seed = argc > 4 ? strtoull(argv[4], nullptr, 0) : 0x5EED0001ull + shape;
  int level = argc > 5 ? atoi(argv[5]) : 6;
  int threads = argc > 6 ? atoi(argv[6]) : 0;
  uint8_t *bam, *bai;
  synth_info info;
  if (synth_bam(shape, n, seed, level, threads, &bam, &bai, &info)) return 1;
  std::string path = argv[3];
  FILE* f = fopen(path.c_str(), "wb");
  if (!f || fwrite(bam, 1, info.bam_bytes, f) != info.bam_bytes) return 1;
  fclose(f);
  f = fopen((path + ".bai").c_str(), "wb");
  if (!f || fwrite(bai, 1, info.bai_bytes, f) != info.bai_bytes) return 1;
  fclose(f);
  fprintf(stderr, "records=%llu inflated=%llu bam=%llu bai=%llu blocks=%u\n", (unsigned long long)info.n_records,
          (unsigned long long)info.inflated_bytes, (unsigned long long)info.bam_bytes,
          (unsigned long long)info.bai_bytes, info.n_blocks);
  return 0;
}
#endif
