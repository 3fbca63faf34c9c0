// Host-side BAM/BAI handling for the CUDA qc path (reference: src/utils/formats/bam.rs:77-123,
// src/utils/pathbuf.rs:59-75).  BGZF framing (K1) and header parsing stay on the host as in the
// reference; the header blocks themselves are inflated on the GPU (ngsq_inflate_to_host), so no
// CPU inflate exists anywhere on this path.
#pragma once
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <fstream>
#include <functional>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/ngs_cuda.h"
#include "facets.hpp"

namespace ngs {

class MappedFile {
 public:
  explicit MappedFile(const std::string& path) {
    fd_ = open(path.c_str(), O_RDONLY);
    if (fd_ < 0) throw std::runtime_error("cannot open " + path);
    struct stat st;
    if (fstat(fd_, &st)) throw std::runtime_error("cannot stat " + path);
    size_ = (size_t)st.st_size;
    if (size_) {
      data_ = (const uint8_t*)mmap(nullptr, size_, PROT_READ, MAP_PRIVATE, fd_, 0);
      if (data_ == MAP_FAILED) throw std::runtime_error("cannot mmap " + path);
      madvise((void*)data_, size_, MADV_SEQUENTIAL);
    }
  }
  ~MappedFile() { if (data_ && size_) munmap((void*)data_, size_); if (fd_ >= 0) close(fd_); }
  const uint8_t* data() const { return data_; }
  size_t size() const { return size_; }

 private:
  int fd_ = -1;
  const uint8_t* data_ = nullptr;
  size_t size_ = 0;
};

struct BamHeader {
  std::string text;
  std::vector<ReferenceSequence> reference_sequences;  // binary reference list (bam.rs:109-111)
  uint64_t first_record_voffset = 0;
};

inline BamHeader read_bam_header(ngsq_engine* e, const uint8_t* bam, size_t size) {
  size_t take = 1 << 16;
  for (;;) {
    size_t n = std::min(take, size);
    uint32_t nb = 0;
    size_t used = 0;
    if (ngsq_bgzf_walk(bam, n, 0, nullptr, 0, &nb, &used)) throw std::runtime_error("malformed BGZF framing at the start of the file");
    std::vector<ngsq_block> blk(nb ? nb : 1);
    ngsq_bgzf_walk(bam, n, 0, blk.data(), nb, &nb, &used);
    std::vector<uint8_t> buf((size_t)nb * 65536 + 16);
    size_t got = 0;
    if (used) check(e, ngsq_inflate_to_host(e, bam, used, buf.data(), buf.size(), &got));
    auto need_more = [&]() {
      if (n == size) throw std::runtime_error("truncated BAM header");
      take *= 4;
    };
    auto u32 = [&](size_t o) { uint32_t v; memcpy(&v, &buf[o], 4); return v; };
    if (got < 12) { need_more(); continue; }
    if (memcmp(buf.data(), "BAM\1", 4)) throw std::runtime_error("not a BAM file (bad magic)");
    size_t o = 8 + (size_t)u32(4);
    if (got < o + 4) { need_more(); continue; }
    BamHeader h;
    h.text.assign((const char*)&buf[8], o - 8);
    uint32_t n_ref = u32(o);
    o += 4;
    bool short_read = false;
    for (uint32_t i = 0; i < n_ref; ++i) {
      if (got < o + 4) { short_read = true; break; }
      uint32_t l_name = u32(o);
      o += 4;
      if (got < o + l_name + 4) { short_read = true; break; }
      ReferenceSequence rs;
      rs.name.assign((const char*)&buf[o], l_name ? l_name - 1 : 0);
      o += l_name;
      rs.length = u32(o);
      o += 4;
      h.reference_sequences.push_back(rs);
    }
    if (short_read) { need_more(); continue; }
    uint64_t acc = 0;
    bool found = false;
    for (uint32_t i = 0; i < nb; ++i) {
      if (o < acc + blk[i].isize) { h.first_record_voffset = (blk[i].coffset << 16) | (o - acc); found = true; break; }
      acc += blk[i].isize;
    }
    if (!found) h.first_record_voffset = (uint64_t)used << 16;
    return h;
  }
}

// BAI (SAM spec 5.2): only what sharding needs — per-reference file extents from pseudo-bin 37450 and the linear index
// (ioffset of every 16 kb window: the first record overlapping it, a record start the shard planner may cut at).
struct BaiReference {
  bool has_extent = false;
  uint64_t ref_beg = 0, ref_end = 0, n_mapped = 0, n_unmapped = 0;
  uint32_t n_bins = 0, n_intv = 0;
  std::vector<uint64_t> ioffset;
};
struct BaiIndex { std::vector<BaiReference> refs; bool has_n_no_coor = false; uint64_t n_no_coor = 0; };

// IndexCheck::Full (utils/formats/bam.rs:86-96): the index must exist next to the BAM and parse.
inline BaiIndex read_bai(const std::string& path) {
  std::ifstream f(path, std::ios::binary);
  if (!f) throw std::runtime_error("Could not find BAM index at " + path + ". Please index the BAM first (`ngs index`).");
  std::vector<uint8_t> b((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  size_t o = 0;
  auto need = [&](size_t k) { if (o + k > b.size()) throw std::runtime_error("reading BAM index: truncated"); };
  need(8);
  if (memcmp(b.data(), "BAI\1", 4)) throw std::runtime_error("reading BAM index: bad magic");
  uint32_t n_ref;
  memcpy(&n_ref, &b[4], 4);
  o = 8;
  BaiIndex idx;
  for (uint32_t r = 0; r < n_ref; ++r) {
    BaiReference R;
    need(4);
    memcpy(&R.n_bins, &b[o], 4);
    o += 4;
    for (uint32_t k = 0; k < R.n_bins; ++k) {
      need(8);
      uint32_t bin, n_chunk;
      memcpy(&bin, &b[o], 4);
      memcpy(&n_chunk, &b[o + 4], 4);
      o += 8;
      need(16ull * n_chunk);
      if (bin == 37450 && n_chunk == 2) {
        memcpy(&R.ref_beg, &b[o], 8); memcpy(&R.ref_end, &b[o + 8], 8);
        memcpy(&R.n_mapped, &b[o + 16], 8); memcpy(&R.n_unmapped, &b[o + 24], 8);
        R.has_extent = R.ref_end > R.ref_beg;
      }
      o += 16ull * n_chunk;
    }
    need(4);
    memcpy(&R.n_intv, &b[o], 4);
    o += 4;
    need(8ull * R.n_intv);
    R.ioffset.resize(R.n_intv);
    if (R.n_intv) memcpy(R.ioffset.data(), &b[o], 8ull * R.n_intv);
    o += 8ull * R.n_intv;
    idx.refs.push_back(R);
  }
  if (o + 8 <= b.size()) { idx.has_n_no_coor = true; memcpy(&idx.n_no_coor, &b[o], 8); }
  return idx;
}

// CSIv1 (the CSI spec; `samtools index -c`, `ngs-cuda-qc index --csi`), UNCOMPRESSED, read into the planner's input: each
// reference's extent and counts from its pseudo-bin ((1 << 3(depth + 1)) - 1) / 7 + 1 (BAI bin 37450's fields), and as its
// ioffset the loffsets of its other bins, sorted.  A bin's loffset is the virtual offset of the first record overlapping its first
// window (htslib forward-fills empty windows, may store 0 or all ones, and folds small bins into a parent holding the minimum):
// a record start or a value bai_anchors drops.  The aux bytes (tabix meta) are skipped.  `path` names the file in errors.
inline BaiIndex parse_csi(const uint8_t* p, size_t n, const std::string& path, size_t n_ref_header) {
  size_t o = 0;
  auto fail = [&](const std::string& what) { throw std::runtime_error("reading CSI index " + path + ": " + what); };
  auto need = [&](uint64_t k, const char* field) { if (k > n - o) fail(std::string("truncated in ") + field); };
  auto i32 = [&](size_t at) { int32_t v; memcpy(&v, p + at, 4); return v; };
  need(16, "the header");
  if (memcmp(p, "CSI\1", 4)) fail("bad magic");
  const int32_t min_shift = i32(4), depth = i32(8), l_aux = i32(12);
  // bins are u32: the pseudo-bin's 1 << 3(depth + 1) fits 32 bits up to depth 9; coordinates are 64-bit
  if (depth < 0 || depth > 9 || min_shift < 0 || (int64_t)min_shift + 3 * depth > 63)
    fail("min_shift " + std::to_string(min_shift) + " with depth " + std::to_string(depth) + " overflows the bin arithmetic");
  if (l_aux < 0) fail("negative l_aux");
  o = 16;
  if ((uint64_t)l_aux > n - o) fail("l_aux " + std::to_string(l_aux) + " runs past the end");
  o += (size_t)l_aux;
  need(4, "n_ref");
  const int32_t n_ref = i32(o);
  o += 4;
  if (n_ref < 0 || (size_t)n_ref != n_ref_header)
    fail(std::to_string(n_ref) + " references, the BAM header has " + std::to_string(n_ref_header));
  const uint32_t meta = ((1u << (3 * (depth + 1))) - 1) / 7 + 1;
  BaiIndex idx;
  for (int32_t r = 0; r < n_ref; ++r) {
    BaiReference R;
    need(4, "n_bin");
    const int32_t n_bin = i32(o);
    o += 4;
    if (n_bin < 0) fail("negative n_bin");
    R.n_bins = (uint32_t)n_bin;
    for (int32_t k = 0; k < n_bin; ++k) {
      need(16, "a bin");
      uint32_t bin;
      uint64_t loffset;
      memcpy(&bin, p + o, 4);
      memcpy(&loffset, p + o + 4, 8);
      const int32_t n_chunk = i32(o + 12);
      o += 16;
      if (n_chunk < 0 || 16ull * (uint32_t)n_chunk > n - o) fail("n_chunk " + std::to_string(n_chunk) + " runs past the end");
      if (bin == meta && n_chunk == 2) {
        memcpy(&R.ref_beg, p + o, 8); memcpy(&R.ref_end, p + o + 8, 8);
        memcpy(&R.n_mapped, p + o + 16, 8); memcpy(&R.n_unmapped, p + o + 24, 8);
        R.has_extent = R.ref_end > R.ref_beg;
      } else {
        R.ioffset.push_back(loffset);
      }
      o += 16ull * (uint32_t)n_chunk;
    }
    std::sort(R.ioffset.begin(), R.ioffset.end());
    R.n_intv = (uint32_t)R.ioffset.size();
    idx.refs.push_back(std::move(R));
  }
  if (o + 8 <= n) { idx.has_n_no_coor = true; memcpy(&idx.n_no_coor, p + o, 8); }
  return idx;
}

// <BAM>.csi: BGZF framed on the host and inflated on the GPU (ngsq_inflate_to_host), like the BAM header, then parse_csi.
inline BaiIndex read_csi(ngsq_engine* e, const std::string& path, size_t n_ref_header) {
  MappedFile f(path);
  uint32_t nb = 0;
  size_t used = 0;
  if (f.size() && (ngsq_bgzf_walk(f.data(), f.size(), 0, nullptr, 0, &nb, &used) || used != f.size()))
    throw std::runtime_error("reading CSI index " + path + ": malformed BGZF framing");
  std::vector<uint8_t> payload((size_t)nb * 65536 + 16);
  size_t got = 0;
  if (used) check(e, ngsq_inflate_to_host(e, f.data(), used, payload.data(), payload.size(), &got));
  return parse_csi(payload.data(), got, path, n_ref_header);
}

// One contiguous range of the file owned by a shard.
struct Shard {
  uint64_t first_voffset = 0, end_voffset = 0;  // end 0 = to EOF
  std::vector<uint32_t> contigs;                // references whose coverage this shard owns
  bool empty = false;
};

// Contig-aligned cuts (SURVEY 8(e)): contiguous runs of contigs balanced by compressed bytes, so
// each coverage position has exactly one owner and the only exchange is the final sum-reduce.
inline std::vector<Shard> plan_shards(const BamHeader& h, const BaiIndex& bai, uint32_t n_shards, uint64_t file_size) {
  struct Span { uint32_t ref; uint64_t beg, end; };
  std::vector<Span> spans;
  for (uint32_t c = 0; c < bai.refs.size(); ++c)
    if (bai.refs[c].has_extent) spans.push_back({c, bai.refs[c].ref_beg, bai.refs[c].ref_end});
  std::sort(spans.begin(), spans.end(), [](const Span& a, const Span& b) { return a.beg < b.beg; });
  std::vector<Shard> out;
  auto all_refs = [&]() { std::vector<uint32_t> v; for (uint32_t c = 0; c < h.reference_sequences.size(); ++c) v.push_back(c); return v; };
  if (n_shards <= 1 || spans.size() < 2) {
    Shard s;
    s.first_voffset = h.first_record_voffset;
    s.contigs = all_refs();
    out.push_back(s);
  } else {
    const uint64_t base = h.first_record_voffset >> 16;
    const double total = (double)(file_size - base);
    Shard cur;
    cur.first_voffset = h.first_record_voffset;
    for (size_t i = 0; i < spans.size(); ++i) {
      cur.contigs.push_back(spans[i].ref);
      size_t contigs_left = spans.size() - i - 1;
      size_t shards_left = n_shards - out.size() - 1;
      double done = (double)((spans[i].end >> 16) - base);
      double target = total * (double)(out.size() + 1) / (double)n_shards;
      if (shards_left > 0 && contigs_left > 0 && (done >= target || contigs_left <= shards_left)) {
        cur.end_voffset = spans[i + 1].beg;
        out.push_back(cur);
        cur = Shard();
        cur.first_voffset = spans[i + 1].beg;
      }
    }
    out.push_back(cur);  // last shard runs to EOF: covers the unplaced-unmapped tail
    // references without records: coverage never touches them; give them to shard 0 for completeness
  }
  while (out.size() < n_shards) { Shard s; s.empty = true; out.push_back(s); }
  return out;
}

// Cuts inside contigs (SURVEY 8(e), DESIGN 5): shards balanced by compressed bytes, cut at record starts the BAI names.
// The anchors are every contig's first record (pseudo-bin 37450) and its linear-index ioffsets; the linear index is
// non-decreasing in file order, so each anchor is the start of a record.  A contig with records on both sides of a cut is
// a split reference: every engine must declare it (ngsq_split_reference) and the merge resolves it once, on the root.
struct ShardPlan {
  std::vector<Shard> shards;
  std::vector<uint32_t> split;  // split references, ascending
  bool split_plan = false;      // plan_shards_split's plan (choose_shards), or plan_shards_unindexed's
  uint32_t dropped = 0;         // plan_shards_unindexed: cuts left out (no record found, or an anchor repeated)
};

// Record starts the planner may cut at, ascending and distinct: zeros, entries below their contig's first record and
// repeats (long reads make consecutive windows share an offset) are dropped.
inline std::vector<uint64_t> bai_anchors(const BaiIndex& bai) {
  std::vector<uint64_t> a;
  for (const BaiReference& r : bai.refs) {
    if (!r.has_extent) continue;
    a.push_back(r.ref_beg);
    for (uint64_t v : r.ioffset)
      if (v && v >= r.ref_beg && v < r.ref_end) a.push_back(v);
  }
  std::sort(a.begin(), a.end());
  a.erase(std::unique(a.begin(), a.end()), a.end());
  return a;
}

inline ShardPlan plan_shards_split(const BamHeader& h, const BaiIndex& bai, uint32_t n_shards, uint64_t file_size) {
  ShardPlan plan;
  const uint64_t first = h.first_record_voffset;
  std::vector<uint64_t> cand;  // possible cuts: anchors after the first record
  for (uint64_t v : bai_anchors(bai)) if (v > first) cand.push_back(v);
  const uint64_t base = first >> 16;
  const double total = (double)(file_size > base ? file_size - base : 0);
  std::vector<uint64_t> cuts;
  const size_t m = cand.size();
  const size_t n_cuts = std::min<size_t>(n_shards ? n_shards - 1 : 0, m);
  size_t lo = 0;  // first candidate the next cut may take
  for (size_t k = 1; k <= n_cuts; ++k) {
    const double target = total * (double)k / (double)n_shards;
    const size_t hi = m - (n_cuts - k);  // leave one candidate for every later cut
    // the candidate nearest the target (ties: the earlier one) within [lo, hi)
    size_t j = (size_t)(std::lower_bound(cand.begin() + lo, cand.begin() + hi, target,
                                         [&](uint64_t v, double t) { return (double)((v >> 16) - base) < t; }) - cand.begin());
    if (j == hi || (j > lo && target - (double)((cand[j - 1] >> 16) - base) <= (double)((cand[j] >> 16) - base) - target)) --j;
    cuts.push_back(cand[j]);
    lo = j + 1;
  }
  std::vector<uint64_t> bounds{first};
  bounds.insert(bounds.end(), cuts.begin(), cuts.end());
  for (size_t i = 0; i < bounds.size(); ++i) {
    Shard s;
    s.first_voffset = bounds[i];
    s.end_voffset = i + 1 < bounds.size() ? bounds[i + 1] : 0;  // the last shard runs to EOF: the unplaced tail
    for (uint32_t c = 0; c < bai.refs.size(); ++c) {
      const BaiReference& r = bai.refs[c];
      if (r.has_extent && r.ref_end > s.first_voffset && (s.end_voffset == 0 || r.ref_beg < s.end_voffset)) s.contigs.push_back(c);
    }
    plan.shards.push_back(s);
  }
  for (uint32_t c = 0; c < bai.refs.size(); ++c) {
    const BaiReference& r = bai.refs[c];
    for (uint64_t v : cuts)
      if (r.has_extent && r.ref_beg < v && v < r.ref_end) { plan.split.push_back(c); break; }
  }
  while (plan.shards.size() < n_shards) { Shard s; s.empty = true; plan.shards.push_back(s); }
  plan.split_plan = true;
  return plan;
}

// Compressed bytes a shard covers, for balancing: from its first record's block to the block of its end (or EOF).
inline uint64_t shard_compressed_bytes(const Shard& s, uint64_t file_size) {
  if (s.empty) return 0;
  const uint64_t lo = s.first_voffset >> 16, hi = s.end_voffset ? s.end_voffset >> 16 : file_size;
  return hi > lo ? hi - lo : 0;
}

// Bytes the merge moves per rank for a split plan: every split contig's int32 difference array (L + 2) and tile sums, and
// its touched word (Edits adds two u32 counters per position; not counted).
inline uint64_t split_reduce_bytes(const BamHeader& h, const std::vector<uint32_t>& split) {
  uint64_t b = 0;
  for (uint32_t c : split) {
    const uint64_t L = c < h.reference_sequences.size() ? h.reference_sequences[c].length : 0;
    b += (L + 2) * 4 + (L + 4096) / 4096 * 4 + 8;
  }
  return b;
}

// The plan `ngs qc` runs.  The split plan is taken when the contig-aligned one leaves a device without a shard.  When every
// device has one, it is taken for balance only if the largest contig-aligned shard holds more than 25 % above the mean
// compressed bytes AND the split plan's merge moves at most twice a balanced shard's compressed bytes per rank
// (split_reduce_bytes).  Measured on one B200 with every shard run alone (DESIGN 6, profiles/split_bench_1gpu.json): where
// the second condition fails, on the 25-contig WGS shape at 8 shards (26 % imbalance, 7 split contigs, 4.2 GB of difference
// arrays per rank), the split plan saves 0.5 ms of the slowest shard's 27 ms including the root's 2.5 ms resolve, before the
// reduce itself; where it holds (shape 2 at 2 and 4 shards, shape 0 at 2) the split plan is 18-36 % faster.  The ncclReduce
// of the split arrays has not been timed on several GPUs.
constexpr double kSplitImbalance = 1.25;
constexpr double kSplitReduceShards = 2.0;
inline ShardPlan choose_shards(const BamHeader& h, const BaiIndex& bai, uint32_t n_shards, uint64_t file_size) {
  ShardPlan plan;
  plan.shards = plan_shards(h, bai, n_shards, file_size);
  if (n_shards <= 1) return plan;
  uint64_t total = 0, most = 0;
  bool all_live = true;
  for (const Shard& s : plan.shards) {
    const uint64_t b = shard_compressed_bytes(s, file_size);
    total += b;
    most = std::max(most, b);
    all_live = all_live && !s.empty;
  }
  const double mean = (double)total / (double)n_shards;
  if (all_live && (double)most <= kSplitImbalance * mean) return plan;
  ShardPlan split = plan_shards_split(h, bai, n_shards, file_size);
  if (all_live && (double)split_reduce_bytes(h, split.split) > kSplitReduceShards * mean) return plan;
  return split;
}

// ---- cuts without an index (DESIGN 5): a freshly sorted BAM has no .bai, so the anchors come from the records themselves
// BGZF header of a block that carries only the BC subfield: magic, CM = 8, FLG = FEXTRA, XLEN = 6, 'B' 'C', SLEN = 2
inline bool bgzf_signature(const uint8_t* p) {
  return p[0] == 0x1f && p[1] == 0x8b && p[2] == 8 && p[3] == 4 && p[10] == 6 && p[11] == 0 && p[12] == 'B' && p[13] == 'C' && p[14] == 2 && p[15] == 0;
}

// The first block start at or after `from`: a signature confirmed by a chain of whole blocks behind it (at least three, or
// exactly to the end of the file), so that a signature inside a block's payload is skipped.  file_size when there is none.
constexpr uint32_t kChainConfirm = 3;
inline uint64_t next_block_start(const uint8_t* bam, uint64_t file_size, uint64_t from) {
  for (uint64_t q = from; q + 18 <= file_size; ++q) {
    if (!bgzf_signature(bam + q)) continue;
    const uint64_t len = std::min<uint64_t>(file_size - q, (uint64_t)(kChainConfirm + 1) << 16);
    uint32_t n = 0;
    size_t used = 0;
    if (ngsq_bgzf_walk(bam + q, len, q, nullptr, 0, &n, &used)) continue;
    if (n >= kChainConfirm || q + used == file_size) return q;
  }
  return file_size;
}

// The record anchor finder (ngsq_find_record on an engine; a fake in the CPU tests): whole BGZF blocks `bgzf` at file
// offset `file_off` -> the first record start in them as a virtual offset and its reference id, 0 when there is none.
using FindRecord = std::function<void(const uint8_t* bgzf, size_t nbytes, uint64_t file_off, uint64_t* voffset, int32_t* ref_id)>;
constexpr uint32_t kFindBlocks = 4;        // first window of the finder, in blocks
constexpr uint32_t kFindBlocksMax = 4096;  // its largest window (256 MiB inflated): a read longer than that leaves the cut out

// Cuts at targets first_record_coffset + (file_size - that) * k / n, each snapped to the next block start and moved to the
// first record the finder sees from there (its window doubles until it sees one).  A cut is dropped when no record is found
// or when its anchor does not lie strictly behind the previous one; its device gets an empty shard.  The anchors are
// speculative until the range in front of each closes on it (run_parts in the driver).  Only the reference of the first
// record behind a cut can have records on both sides of it (sorted input), so those references are the split set; the
// driver declares them whether or not Coverage processes them, because Edits keeps per-position counters of every contig.
inline ShardPlan plan_shards_unindexed(const BamHeader& h, const uint8_t* bam, uint64_t file_size, uint32_t n_shards, const FindRecord& find) {
  ShardPlan plan;
  plan.split_plan = true;
  const uint64_t first = h.first_record_voffset, base = std::min<uint64_t>(first >> 16, file_size);
  std::vector<uint64_t> bounds{first};
  std::vector<uint32_t> split;
  std::vector<ngsq_block> tmp(kFindBlocksMax);
  for (uint32_t k = 1; k < n_shards; ++k) {
    const uint64_t target = base + (uint64_t)((unsigned __int128)(file_size - base) * k / n_shards);
    const uint64_t p = next_block_start(bam, file_size, target);
    uint64_t anchor = 0;
    int32_t ref = -1;
    for (uint32_t nb = kFindBlocks; p < file_size && nb <= kFindBlocksMax; nb *= 2) {
      uint32_t n = 0;
      size_t used = 0;
      const uint64_t len = std::min<uint64_t>(file_size - p, (uint64_t)nb << 16);
      if (ngsq_bgzf_walk(bam + p, len, p, tmp.data(), nb, &n, &used) || !used) break;
      find(bam + p, used, p, &anchor, &ref);
      if (anchor || p + used == file_size) break;
    }
    if (!anchor || anchor <= bounds.back()) { ++plan.dropped; continue; }
    bounds.push_back(anchor);
    if (ref >= 0) split.push_back((uint32_t)ref);
  }
  for (size_t i = 0; i < bounds.size(); ++i) {
    Shard s;
    s.first_voffset = bounds[i];
    s.end_voffset = i + 1 < bounds.size() ? bounds[i + 1] : 0;
    plan.shards.push_back(s);
  }
  std::sort(split.begin(), split.end());
  split.erase(std::unique(split.begin(), split.end()), split.end());
  plan.split = split;
  while (plan.shards.size() < n_shards) { Shard s; s.empty = true; plan.shards.push_back(s); }
  return plan;
}

// Compressed byte range [lo, hi) a shard submits: through the block that holds end_voffset.
inline void shard_bytes(const Shard& s, const uint8_t* bam, uint64_t file_size, uint64_t* lo, uint64_t* hi) {
  *lo = s.first_voffset >> 16;
  if (s.end_voffset == 0) { *hi = file_size; return; }
  uint64_t co = s.end_voffset >> 16, uo = s.end_voffset & 0xFFFF;
  if (uo == 0) { *hi = co; return; }
  ngsq_block b;
  uint32_t n = 0;
  size_t used = 0;
  if (ngsq_bgzf_walk(bam + co, std::min<uint64_t>(file_size - co, 1 << 17), co, &b, 1, &n, &used) || n == 0)
    throw std::runtime_error("shard end does not address a BGZF block");
  *hi = co + b.csize;
}

}  // namespace ngs
