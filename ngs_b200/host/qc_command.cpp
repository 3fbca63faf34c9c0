// ngs-cuda-qc — host driver of the CUDA `ngs qc` path.  Mirrors the reference's subcommand
// (src/qc/command.rs): QcArgs (36-102), qc() (109-218), app() (226-421).  Same positional
// arguments and flags, same checks in the same order, same output file; the two hot loops of
// app() (305-316 and 350-397) are replaced by one pass of the CUDA engine per GPU.  `index` builds the
// BAI that `qc` needs (src/index/bam.rs:39-109) in one pass of the engine on one GPU.
//
// A BAM without an index is cut between GPUs at record anchors the engine finds (ngsq_find_record), each GPU indexes its part
// (NGSQ_F_INDEX_PART) and the host joins the parts (ngsq_join_bai): `index --cuda-devices`, and `qc --cuda-build-index`,
// which writes the missing index (.bai, or .csi with --cuda-csi) in the same pass as the results.  `qc` plans its shards from
// <BAM>.bai, or from <BAM>.csi when there is no .bai (the reference needs the .bai).
//
//   ngs-cuda-qc qc <BAM> <REFERENCE_GENOME> [-n N] [-o DIR] [-p PREFIX] [--only FACET]
//               [--cuda-devices 0,1,..] [--cuda-build-index [--cuda-csi [--cuda-min-shift N]]] [--cuda-gc-seed S]
//               [--cuda-no-crc] [--cuda-chunk-mb M] [--cuda-buffered-io] [--cuda-perf]
//   ngs-cuda-qc index <BAM> [--csi [-m|--min-shift N]] [--cuda-device N | --cuda-devices 0,1,..] [--cuda-no-crc] [--cuda-chunk-mb M]
//                     [--cuda-buffered-io]
#include <cerrno>
#include <cstdio>
#include <cstdlib>
#include <filesystem>
#include <iostream>
#include <optional>
#include <sstream>
#include <chrono>
#include <thread>

#include <fcntl.h>
#include <unistd.h>

#include "bam.hpp"
#include "facets.hpp"

using namespace ngs;

namespace {

// command.rs:36-102
struct QcArgs {
  std::string src;
  std::string reference_genome;
  std::optional<std::string> features_gff, reference_fasta, output_prefix, output_directory, only_facet, vaf_file_path;
  std::optional<uint64_t> num_records;
  FeatureNames feature_names;  // command.rs:78-101
  // engine-only knobs (not part of the reference CLI)
  std::vector<int> devices{0};
  uint64_t gc_seed = 0;
  bool verify_crc = true;
  size_t chunk_mb = 64;
  bool direct_io = true;
  bool perf = false;
  bool build_index = false;  // a missing index is built in the same pass and written next to the BAM
  bool csi = false;          // --cuda-csi: that index is <BAM>.csi instead of <BAM>.bai
  uint32_t min_shift = 14;   // --cuda-min-shift (CSI); the depth follows samtools' rule
};

void info(const std::string& s) { std::cerr << "INFO " << s << "\n"; }

// "  [*] Processed 1,000,000 records." (display.rs:43-52: RecordCounter::inc logs every millionth record; Locale::en)
std::string with_commas(uint64_t v) {
  std::string d = std::to_string(v), out;
  for (size_t i = 0; i < d.size(); ++i) {
    out += d[i];
    const size_t left = d.size() - 1 - i;
    if (left && left % 3 == 0) out += ',';
  }
  return out;
}

struct Progress {
  uint64_t logged = 0;  // millions already reported
  void report(ngsq_engine* e) {
    uint64_t n = 0;
    if (ngsq_progress(e, &n)) return;
    for (; (logged + 1) * 1000000ull <= n; ++logged) info("  [*] Processed " + with_commas((logged + 1) * 1000000ull) + " records.");
  }
};

// The shard's bytes, read with O_DIRECT into a ring of page-locked buffers and handed to the engine chunk by chunk:
// the file read of chunk k+2, the PCIe copy of chunk k+1 and the kernels of chunk k overlap, and the page cache is
// left alone (the reference reads through a BufReader, bam.rs:41-44).  A chunk ends on a BGZF block boundary; the
// partial block behind it moves in front of the next read.
class ChunkReader {
 public:
  static constexpr size_t kLead = 1 << 17;  // room in front of every buffer for the previous chunk's partial block
  ChunkReader(const std::string& path, size_t chunk_bytes, bool direct) : chunk_((chunk_bytes + 4095) & ~size_t(4095)) {
    fd_ = -1;
#ifdef O_DIRECT
    if (direct) fd_ = open(path.c_str(), O_RDONLY | O_DIRECT);
    direct_ = fd_ >= 0;
#endif
    if (fd_ < 0) fd_ = open(path.c_str(), O_RDONLY);
    if (fd_ < 0) throw std::runtime_error("cannot open " + path);
    for (auto& b : buf_) {
      b = (uint8_t*)ngsq_host_alloc(kLead + chunk_ + 4096);
      if (!b) throw std::runtime_error("cannot allocate pinned staging buffers");
    }
  }
  ~ChunkReader() {
    for (auto& b : buf_) if (b) ngsq_host_free(b);
    if (fd_ >= 0) close(fd_);
  }
  bool direct() const { return direct_; }

  // streams file bytes [lo, hi) (lo on a block boundary) into e
  void run(ngsq_engine* e, uint64_t lo, uint64_t hi, Progress* progress) {
    uint64_t pos = lo & ~uint64_t(4095);  // aligned file position of the next read
    size_t skip = (size_t)(lo - pos);     // bytes of the first read that precede the shard
    size_t carry = 0;                     // bytes of a partial block kept from the previous chunk
    const uint8_t* carry_src = nullptr;
    uint32_t submits = 0;
    int32_t used_by[kBufs];
    for (auto& u : used_by) u = -1;
    uint64_t file_off = lo;               // file offset of the next byte to submit
    for (uint32_t k = 0; pos < hi; ++k) {
      const uint32_t bi = k % kBufs;
      if (used_by[bi] >= 0) check(e, ngsq_wait_copied(e, (uint32_t)used_by[bi]));  // its last copy must have left the buffer
      uint8_t* base = buf_[bi] + kLead;
      size_t want = (size_t)std::min<uint64_t>(chunk_, ((hi + 4095) & ~uint64_t(4095)) - pos);
      size_t got = 0;
      while (got < want) {
        ssize_t r = pread(fd_, base + got, want - got, (off_t)(pos + got));
        if (r < 0) {
          if (direct_ && got == 0) {  // a file system that refuses O_DIRECT reads: fall back to buffered reads once
            int fd2 = open_again_buffered();
            if (fd2 >= 0) { close(fd_); fd_ = fd2; direct_ = false; continue; }
          }
          throw std::runtime_error("read error on the BAM file");
        }
        if (r == 0) break;
        got += (size_t)r;
      }
      uint8_t* begin = base + skip;
      size_t n = got > skip ? got - skip : 0;
      if (pos + got > hi) n -= (size_t)std::min<uint64_t>(n, pos + got - hi);
      if (carry) {
        begin -= carry;
        memcpy(begin, carry_src, carry);
        n += carry;
      }
      pos += got;
      skip = 0;
      const bool last = pos >= hi || got < want;
      uint32_t nb = 0;
      size_t used = 0;
      if (ngsq_bgzf_walk(begin, n, file_off, nullptr, 0, &nb, &used)) throw std::runtime_error("malformed BGZF framing");
      if (last && used != n) throw std::runtime_error("truncated BGZF block at end of file");
      if (used) {
        check(e, ngsq_submit(e, begin, used, file_off));
        used_by[bi] = (int32_t)submits++;
        file_off += used;
      }
      carry = n - used;
      carry_src = begin + used;
      if (carry > kLead) throw std::runtime_error("BGZF block larger than 128 KiB");
      if (progress) progress->report(e);
      if (got < want) break;
    }
  }

 private:
  int open_again_buffered() {
    char link[64], path[4096];
    snprintf(link, sizeof link, "/proc/self/fd/%d", fd_);
    ssize_t n = readlink(link, path, sizeof path - 1);
    if (n <= 0) return -1;
    path[n] = 0;
    return open(path, O_RDONLY);
  }
  static constexpr int kBufs = 3;
  int fd_ = -1;
  bool direct_ = false;
  size_t chunk_;
  uint8_t* buf_[kBufs] = {nullptr, nullptr, nullptr};
};

void run_shard(ngsq_engine* e, const std::string& path, const MappedFile& file, const Shard& shard, size_t chunk_bytes, bool direct, bool log_progress,
               std::string* err, int* code) {
  try {
    if (shard.empty) { check(e, ngsq_set_range(e, 0, 0)); check(e, ngsq_finish(e)); return; }
    uint64_t lo, hi;
    shard_bytes(shard, file.data(), file.size(), &lo, &hi);
    ChunkReader reader(path, chunk_bytes, direct);
    for (int attempt = 0;; ++attempt) {
      check(e, ngsq_set_range(e, shard.first_voffset, shard.end_voffset));
      Progress progress;
      reader.run(e, lo, hi, log_progress ? &progress : nullptr);
      const int rc = ngsq_finish(e);
      if (rc == NGSQ_E_QUAL_CAP && attempt == 0) {
        // a read longer than the quality-by-position table (131072 positions by default): size the table for the
        // longest read the scan met and stream the shard again — the engine keeps nothing of a file it has streamed
        ngsq_stats st;
        check(e, ngsq_get_stats(e, &st));
        info("  [*] Reads of up to " + std::to_string(st.max_read_len) + " bases: enlarging the quality table and reading the file again.");
        check(e, ngsq_reset(e));
        check(e, ngsq_set_quality_positions(e, (uint32_t)st.max_read_len + 1));
        continue;
      }
      if (code) *code = rc;
      check(e, rc);
      if (log_progress) progress.report(e);
      break;
    }
  } catch (const std::exception& ex) {
    *err = ex.what();
  }
}

// The parts of a file cut without an index (plan_shards_unindexed), one thread per engine.  An anchor is proven when the
// range in front of it closes on it; the first record after the header is proven, so the cuts are proven in file order: a
// part whose start is proven and that fails with NGSQ_E_CHAIN or NGSQ_E_TRUNCATED, with a next part behind it, ends on a
// false anchor.  That cut is dropped: the part is run again over both ranges, the next engine over an empty one.  Any other
// failure is the file's and is reported.  On return every engine has finished; shards holds the ranges that ran.
void run_parts(const std::vector<ngsq_engine*>& engines, std::vector<Shard>& shards, const std::string& path, const MappedFile& file,
               size_t chunk_bytes, bool direct) {
  const size_t n = engines.size();
  std::vector<std::string> errs(n);
  std::vector<int> codes(n, 0);
  {
    std::vector<std::thread> ts;
    for (size_t i = 0; i < n; ++i)
      ts.emplace_back(run_shard, engines[i], std::cref(path), std::cref(file), std::cref(shards[i]), chunk_bytes, direct, i == 0, &errs[i], &codes[i]);
    for (auto& t : ts) t.join();
  }
  for (size_t k = 0; k < n; ++k) {
    while (!errs[k].empty()) {
      size_t j = k + 1;  // the next live part: its start is the cut in question
      while (j < n && shards[j].empty) ++j;
      if (j == n || (codes[k] != NGSQ_E_CHAIN && codes[k] != NGSQ_E_TRUNCATED)) throw std::runtime_error(errs[k]);
      info("  [*] The record anchor at virtual offset " + std::to_string(shards[j].first_voffset) +
           " is not a record start: dropping that cut and reading the range again.");
      shards[k].end_voffset = shards[j].end_voffset;
      shards[j] = Shard();
      shards[j].empty = true;
      for (size_t i : {k, j}) {
        check(engines[i], ngsq_reset(engines[i]));
        errs[i].clear();
        codes[i] = 0;
      }
      run_shard(engines[j], path, file, shards[j], chunk_bytes, direct, false, &errs[j], &codes[j]);
      if (!errs[j].empty()) throw std::runtime_error(errs[j]);
      run_shard(engines[k], path, file, shards[k], chunk_bytes, direct, false, &errs[k], &codes[k]);
    }
  }
}

// The record anchor finder of plan_shards_unindexed on engine e (after ngsq_set_references)
FindRecord engine_finder(ngsq_engine* e) {
  return [e](const uint8_t* p, size_t n, uint64_t off, uint64_t* voff, int32_t* ref) { check(e, ngsq_find_record(e, p, n, off, voff, ref)); };
}

// The parts' .bai (or uncompressed .csi), in file order (engines with an empty range hold no part)
std::vector<uint8_t> join_parts(const std::vector<ngsq_engine*>& engines, const std::vector<Shard>& shards, bool csi = false) {
  std::vector<ngsq_engine*> parts;
  for (size_t i = 0; i < engines.size(); ++i)
    if (!shards[i].empty) parts.push_back(engines[i]);
  auto join = csi ? ngsq_join_csi : ngsq_join_bai;
  size_t n = 0;
  check(parts[0], join(parts.data(), (uint32_t)parts.size(), nullptr, 0, &n));
  std::vector<uint8_t> bai(n);
  check(parts[0], join(parts.data(), (uint32_t)parts.size(), bai.data(), bai.size(), &n));
  return bai;
}

// A .csi file is BGZF: the payload in blocks of at most 0xFF00 bytes, each deflated at level 6 (as htslib writes them), then
// the 28-byte EOF block.
std::vector<uint8_t> bgzf_compress(const std::vector<uint8_t>& data) {
  static const uint8_t kEof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  std::vector<uint8_t> out;
  uint8_t blk[65536];
  for (size_t o = 0; o < data.size(); o += 0xFF00) {
    const uInt n = (uInt)std::min<size_t>(0xFF00, data.size() - o);
    z_stream zs{};
    if (deflateInit2(&zs, 6, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) throw std::runtime_error("deflateInit2 failed");
    zs.next_in = const_cast<uint8_t*>(data.data() + o);
    zs.avail_in = n;
    zs.next_out = blk + 18;
    zs.avail_out = sizeof blk - 26;
    const int rc = deflate(&zs, Z_FINISH);
    const size_t clen = zs.total_out;
    deflateEnd(&zs);
    if (rc != Z_STREAM_END || 26 + clen > sizeof blk) throw std::runtime_error("BGZF block does not fit in 64 KiB");
    static const uint8_t kHdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
    memcpy(blk, kHdr, 16);
    const uint16_t bsize = (uint16_t)(26 + clen - 1);
    const uint32_t crc = (uint32_t)crc32(crc32(0, nullptr, 0), data.data() + o, n), isize = n;
    memcpy(blk + 16, &bsize, 2);
    memcpy(blk + 18 + clen, &crc, 4);
    memcpy(blk + 22 + clen, &isize, 4);
    out.insert(out.end(), blk, blk + 26 + clen);
  }
  out.insert(out.end(), kEof, kEof + 28);
  return out;
}

// The .bai next to the BAM.  O_EXCL: an index that appeared while the file was read is not replaced either.
void write_index(const std::string& dst, const std::vector<uint8_t>& bai) {
  info("Writing index to " + dst + ".");
  const int fd = open(dst.c_str(), O_WRONLY | O_CREAT | O_EXCL, 0644);
  if (fd < 0) throw std::runtime_error("cannot create " + dst + (errno == EEXIST ? ": index file already exists" : ""));
  size_t done = 0;
  while (done < bai.size()) {
    const ssize_t w = write(fd, bai.data() + done, bai.size() - done);
    if (w <= 0) { close(fd); std::filesystem::remove(dst); throw std::runtime_error("write error on " + dst); }
    done += (size_t)w;
  }
  if (close(fd)) { std::filesystem::remove(dst); throw std::runtime_error("write error on " + dst); }
}

void log_dropped_cuts(const ShardPlan& plan) {
  if (plan.dropped) info("  [*] " + std::to_string(plan.dropped) + " cut(s) left out: no record start found behind the target, or the anchor repeats.");
}

// command.rs:226-421
int app(const QcArgs& args, const ReferenceGenome& genome, const std::string& output_prefix, const std::string& output_directory) {
  // open_and_parse(src, IndexCheck::Full): bam.rs:77-123
  if (args.src.size() < 4 || args.src.substr(args.src.size() - 4) != ".bam")
    throw std::runtime_error("could not open " + args.src + ": expected a .bam file");
  MappedFile file(args.src);
  const std::string bai_path = args.src + ".bai";  // pathbuf.rs:59-75: x.bam -> x.bam.bai
  const std::string csi_path = args.src + ".csi";  // x.bam -> x.bam.csi: planned from when there is no .bai
  const bool have_bai = std::filesystem::exists(bai_path), have_csi = !have_bai && std::filesystem::exists(csi_path);
  // --cuda-build-index: an existing index (.bai, else .csi) is used as it is; a missing one is built by this pass
  const bool build_index = args.build_index && !have_bai && !have_csi;
  const bool build_csi = build_index && args.csi;
  // the .csi is BGZF: it is read once an engine can inflate it (below); without any index read_bai reports the missing .bai
  BaiIndex bai = build_index || have_csi ? BaiIndex{} : read_bai(bai_path);
  const uint32_t n_dev = (uint32_t)args.devices.size();

  // facets first (cheap) so `--only` errors surface before any device work.  The two optional facets read their
  // inputs here, like GenomicFeaturesFacet::try_from / EditsFacet::try_from do inside get_qc_facets (qc.rs:68-94).
  std::unique_ptr<GenomicFeaturesFacet> features_facet;
  std::unique_ptr<EditsFacet> edits_facet;
  if (args.features_gff) features_facet = std::make_unique<GenomicFeaturesFacet>(GenomicFeaturesFacet::try_from(*args.features_gff, args.feature_names, genome));
  if (args.reference_fasta) edits_facet = std::make_unique<EditsFacet>(EditsFacet::try_from(*args.reference_fasta, args.vaf_file_path));
  FacetSet facets = get_qc_facets(genome, args.only_facet, std::move(features_facet), std::move(edits_facet));
  GenomicFeaturesFacet* features = nullptr;
  EditsFacet* edits = nullptr;
  bool coverage = false, record_defaults = false;
  for (auto& f : facets.record_based) { if (auto* g = dynamic_cast<GenomicFeaturesFacet*>(f.get())) features = g; else record_defaults = true; }
  for (auto& f : facets.sequence_based) { if (auto* g = dynamic_cast<EditsFacet*>(f.get())) edits = g; else coverage = true; }
  uint32_t flags = 0;
  if (record_defaults) flags |= NGSQ_F_RECORD_FACETS;
  if (coverage) flags |= NGSQ_F_COVERAGE;
  if (features) flags |= NGSQ_F_FEATURES;
  if (edits) flags |= NGSQ_F_EDITS;
  if (args.verify_crc) flags |= NGSQ_F_VERIFY_CRC;
  if (build_index) flags |= (n_dev > 1 ? NGSQ_F_INDEX_PART : NGSQ_F_INDEX) | (build_csi ? NGSQ_F_INDEX_CSI : 0u);
  if (args.num_records && n_dev > 1) throw std::runtime_error("-n needs a single device (records are counted in file order)");

  std::vector<ngsq_engine*> engines(n_dev, nullptr);
  struct Cleanup { std::vector<ngsq_engine*>& v; ~Cleanup() { for (auto* e : v) if (e) ngsq_destroy(e); } } cleanup{engines};
  for (uint32_t i = 0; i < n_dev; ++i) {
    ngsq_config cfg{};
    cfg.struct_size = sizeof cfg;
    cfg.flags = flags;
    cfg.gc_seed = args.gc_seed;
    cfg.max_records = args.num_records.value_or(0);
    if (ngsq_create(args.devices[i], &cfg, &engines[i])) throw std::runtime_error(std::string("CUDA engine: ") + ngsq_last_error(nullptr));
    if (build_csi) check(engines[i], ngsq_set_index_binning(engines[i], args.min_shift, 0));  // before any ngsq_set_references
  }
  BamHeader header = read_bam_header(engines[0], file.data(), file.size());
  if (have_csi) bai = read_csi(engines[0], csi_path, header.reference_sequences.size());

  if (!std::filesystem::exists(output_directory)) std::filesystem::create_directories(output_directory);

  // reference sequence concordance check: command.rs:258-272
  std::vector<Sequence> supported = get_all_sequences(genome);
  for (auto& rs : header.reference_sequences) {
    bool ok = false;
    for (auto& s : supported) if (s.name == rs.name) { ok = true; break; }
    if (!ok) throw std::runtime_error("Sequence \"" + rs.name + "\" not found in specified reference genome. Did you set the correct reference genome?");
  }

  for (auto& f : facets.record_based) info(std::string("  [*] ") + f->name() + ", " + to_string(f->computational_load()));
  for (auto& f : facets.sequence_based) info(std::string("  [*] ") + f->name() + ", " + to_string(f->computational_load()));

  // shards: contig-aligned file ranges from the index (BAI or CSI), or ranges cut inside contigs when those leave a device idle or
  // unbalanced (choose_shards); a contig cut between shards is declared on every engine and merged by ngsq_reduce
  std::vector<uint32_t> ref_len;
  for (auto& rs : header.reference_sequences) ref_len.push_back(rs.length);
  ShardPlan plan;
  if (build_index && n_dev > 1) {
    // no index to cut at: anchors from the records (the finder needs the references; every engine sets them again below)
    check(engines[0], ngsq_set_references(engines[0], (uint32_t)ref_len.size(), ref_len.data(), std::vector<uint8_t>(ref_len.size(), 0).data()));
    plan = plan_shards_unindexed(header, file.data(), file.size(), n_dev, engine_finder(engines[0]));
    log_dropped_cuts(plan);
  } else {
    plan = choose_shards(header, bai, n_dev, file.size());
  }
  std::vector<Shard> shards = plan.shards;
  if (plan.split_plan) {
    std::string names;
    for (uint32_t c : plan.split) names += (names.empty() ? "" : ", ") + header.reference_sequences[c].name;
    info("  [*] Sharding inside contigs: " + std::to_string(n_dev) + " shards" + (names.empty() ? std::string() : ", split: " + names) + ".");
  }
  for (uint32_t i = 0; i < n_dev; ++i) {
    // the same mask on every engine: the packed result buffer (the NCCL payload) is laid out from it, and a
    // contig outside an engine's shard simply stays untouched there (ngsq_reduce rejects differing layouts)
    std::vector<uint8_t> enabled(ref_len.size(), 0);
    for (auto& f : facets.sequence_based)
      for (uint32_t c = 0; c < ref_len.size(); ++c)
        if (f.get() != edits && f->supports_sequence_name(header.reference_sequences[c].name)) enabled[c] = 1;  // the Coverage mask
    check(engines[i], ngsq_set_references(engines[i], (uint32_t)ref_len.size(), ref_len.data(), enabled.data()));
    if (features) features->upload(engines[i], header.reference_sequences);
    if (edits) edits->upload(engines[i], header.reference_sequences);
    for (uint32_t c : plan.split) check(engines[i], ngsq_split_reference(engines[i], c));
  }
  if (n_dev > 1) {
    char id[128];
    if (ngsq_nccl_unique_id(id)) throw std::runtime_error(std::string("NCCL: ") + ngsq_last_error(nullptr));
    std::vector<std::thread> ts;
    std::vector<std::string> errs(n_dev);
    for (uint32_t i = 0; i < n_dev; ++i)
      ts.emplace_back([&, i] { if (ngsq_comm_init(engines[i], (int)n_dev, (int)i, id)) errs[i] = ngsq_last_error(engines[i]); });
    for (auto& t : ts) t.join();
    for (auto& s : errs) if (!s.empty()) throw std::runtime_error("NCCL: " + s);
  }

  // the hot path: one thread per GPU
  info("Starting CUDA pass for QC stats.");
  const auto t_hot = std::chrono::steady_clock::now();
  if (build_index && n_dev > 1) {
    run_parts(engines, shards, args.src, file, args.chunk_mb << 20, args.direct_io);
  } else {
    std::vector<std::thread> ts;
    std::vector<std::string> errs(n_dev);
    for (uint32_t i = 0; i < n_dev; ++i)
      ts.emplace_back(run_shard, engines[i], std::cref(args.src), std::cref(file), std::cref(shards[i]), args.chunk_mb << 20, args.direct_io, i == 0, &errs[i], nullptr);
    for (auto& t : ts) t.join();
    for (auto& s : errs) if (!s.empty()) throw std::runtime_error(s);
  }
  if (n_dev > 1) {
    std::vector<std::thread> ts;
    std::vector<std::string> errs(n_dev);
    for (uint32_t i = 0; i < n_dev; ++i) ts.emplace_back([&, i] { if (ngsq_reduce(engines[i], 0)) errs[i] = ngsq_last_error(engines[i]); });
    for (auto& t : ts) t.join();
    for (auto& s : errs) if (!s.empty()) throw std::runtime_error("NCCL: " + s);
  }
  // the index of this pass: joined (and its order checked) before any output is written
  std::vector<uint8_t> new_index;
  if (build_index && n_dev > 1) new_index = join_parts(engines, shards, build_csi);
  else if (build_index) {
    auto get = build_csi ? ngsq_get_csi : ngsq_get_bai;
    size_t n = 0;
    check(engines[0], get(engines[0], nullptr, 0, &n));
    new_index.resize(n);
    check(engines[0], get(engines[0], new_index.data(), new_index.size(), &n));
  }
  const double hot_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_hot).count();
  ngsq_engine* root = engines[0];
  uint64_t n_records = 0;
  for (auto* e : engines) { ngsq_stats st; ngsq_get_stats(e, &st); n_records += st.records; }
  {
    std::ostringstream os;
    os << "Processed " << n_records << " records.";
    info(os.str());
  }

  // first pass: summarize (command.rs:328-330)
  for (auto& f : facets.record_based) { f->ingest(root); f->summarize(); }
  // second pass: per sequence in header order setup -> (process on the device) -> teardown (command.rs:356-396)
  if (edits) edits->set_engines(engines);  // the VAF file reads every engine's per-position counters
  for (auto& f : facets.sequence_based) f->ingest_global(root);
  for (uint32_t c = 0; c < header.reference_sequences.size(); ++c) {
    const ReferenceSequence& seq = header.reference_sequences[c];
    for (auto& f : facets.sequence_based) {
      if (!f->supports_sequence_name(seq.name)) continue;
      f->setup(seq);
      f->ingest(root, c, seq);
      f->teardown(seq);
    }
  }
  // finalize: command.rs:406-418
  info("Aggregating results.");
  Results results;
  for (auto& f : facets.record_based) f->aggregate(results);
  for (auto& f : facets.sequence_based) f->aggregate(results);
  info("Writing output.");
  results.write(output_prefix, output_directory);
  if (build_index) write_index(build_csi ? csi_path : bai_path, build_csi ? bgzf_compress(new_index) : new_index);

  if (args.perf) {
    std::ofstream pf(output_directory + "/" + output_prefix + ".perf.json");
    pf << "[";
    for (uint32_t i = 0; i < n_dev; ++i) {
      ngsq_stats st;
      ngsq_get_stats(engines[i], &st);
      pf << (i ? "," : "") << "{\"device\":" << args.devices[i] << ",\"records\":" << st.records << ",\"blocks\":" << st.blocks
         << ",\"compressed_bytes\":" << st.compressed_bytes << ",\"inflated_bytes\":" << st.inflated_bytes << ",\"ms_inflate\":" << st.ms_inflate
         << ",\"ms_crc\":" << st.ms_crc << ",\"ms_scan\":" << st.ms_scan << ",\"ms_facets\":" << st.ms_facets << ",\"ms_coverage\":" << st.ms_coverage
         << ",\"ms_total\":" << st.ms_total << ",\"ms_tail\":" << st.ms_tail << ",\"waves\":" << st.waves << ",\"wall_ms_file_to_results\":" << hot_ms << "}";
    }
    pf << "]\n";
  }
  return 0;
}

// command.rs:109-218
int qc(const QcArgs& args) {
  info("Starting qc command...");
  auto genome = get_reference_genome(args.reference_genome);
  if (!genome)
    throw std::runtime_error("reference genome is not supported: " + args.reference_genome +
                             ". Did you set the correct reference genome?. Use the `list genomes` subcommand to see supported reference genomes.");
  std::string prefix = args.output_prefix.value_or(std::filesystem::path(args.src).filename().string());
  std::string outdir = args.output_directory.value_or(std::filesystem::current_path().string());
  return app(args, *genome, prefix, outdir);
}

// `ngs index` for a BAM (src/index/bam.rs:39-109): the header, then every record through the engine's NGSQ_F_INDEX pass, and
// the .bai next to the file (utils/pathbuf.rs:59-75: x.bam -> x.bam.bai).  Like the reference (bam.rs:52-58) it never
// overwrites an existing index.
struct IndexArgs {
  std::string src;
  bool csi = false;          // --csi: <BAM>.csi (BGZF) instead of <BAM>.bai
  uint32_t min_shift = 14;   // -m / --min-shift (CSI); the depth follows samtools' rule
  int device = 0;
  std::vector<int> devices;  // --cuda-devices: several engines, one part of the file each
  bool verify_crc = true;
  size_t chunk_mb = 64;
  bool direct_io = true;
};

// the index file of the engine(s): the .bai as it is, the .csi payload BGZF-compressed
void write_index_file(const IndexArgs& a, const std::string& dst, const std::vector<uint8_t>& payload) {
  write_index(dst, a.csi ? bgzf_compress(payload) : payload);
}

int index_bam(const IndexArgs& a) {
  info("Starting index command...");
  const std::string dst = a.src + (a.csi ? ".csi" : ".bai");
  if (std::filesystem::exists(dst)) throw std::runtime_error("index file already exists: " + dst);
  MappedFile file(a.src);
  ngsq_config cfg{};
  cfg.struct_size = sizeof cfg;
  cfg.flags = NGSQ_F_INDEX | (a.verify_crc ? NGSQ_F_VERIFY_CRC : 0u) | (a.csi ? NGSQ_F_INDEX_CSI : 0u);
  ngsq_engine* e = nullptr;
  if (ngsq_create(a.device, &cfg, &e)) throw std::runtime_error(std::string("CUDA engine: ") + ngsq_last_error(nullptr));
  struct Cleanup { ngsq_engine* e; ~Cleanup() { ngsq_destroy(e); } } cleanup{e};
  BamHeader header = read_bam_header(e, file.data(), file.size());
  std::vector<uint32_t> ref_len;
  for (auto& rs : header.reference_sequences) ref_len.push_back(rs.length);
  std::vector<uint8_t> no_coverage(ref_len.size(), 0);
  if (a.csi) check(e, ngsq_set_index_binning(e, a.min_shift, 0));
  check(e, ngsq_set_references(e, (uint32_t)ref_len.size(), ref_len.data(), no_coverage.data()));
  check(e, ngsq_set_range(e, header.first_record_voffset, 0));
  info("Indexing BAM file.");
  {
    ChunkReader reader(a.src, a.chunk_mb << 20, a.direct_io);
    Progress progress;
    reader.run(e, std::min<uint64_t>(header.first_record_voffset >> 16, file.size()), file.size(), &progress);
    check(e, ngsq_finish(e));
    progress.report(e);
  }
  ngsq_stats st;
  check(e, ngsq_get_stats(e, &st));
  info("Processed " + std::to_string(st.records) + " records.");
  auto get = a.csi ? ngsq_get_csi : ngsq_get_bai;
  size_t n = 0;
  check(e, get(e, nullptr, 0, &n));
  std::vector<uint8_t> bai(n);
  check(e, get(e, bai.data(), bai.size(), &n));
  write_index_file(a, dst, bai);
  return 0;
}

// `index` on several devices: the file cut at record anchors, one NGSQ_F_INDEX_PART engine and one thread per part, the parts
// joined on the host.  No collective is involved, so a device may repeat.
int index_bam_parts(const IndexArgs& a) {
  info("Starting index command...");
  const std::string dst = a.src + (a.csi ? ".csi" : ".bai");
  if (std::filesystem::exists(dst)) throw std::runtime_error("index file already exists: " + dst);
  MappedFile file(a.src);
  const size_t n_dev = a.devices.size();
  std::vector<ngsq_engine*> engines(n_dev, nullptr);
  struct Cleanup { std::vector<ngsq_engine*>& v; ~Cleanup() { for (auto* e : v) if (e) ngsq_destroy(e); } } cleanup{engines};
  for (size_t i = 0; i < n_dev; ++i) {
    ngsq_config cfg{};
    cfg.struct_size = sizeof cfg;
    cfg.flags = NGSQ_F_INDEX_PART | (a.verify_crc ? NGSQ_F_VERIFY_CRC : 0u) | (a.csi ? NGSQ_F_INDEX_CSI : 0u);
    if (ngsq_create(a.devices[i], &cfg, &engines[i])) throw std::runtime_error(std::string("CUDA engine: ") + ngsq_last_error(nullptr));
  }
  BamHeader header = read_bam_header(engines[0], file.data(), file.size());
  std::vector<uint32_t> ref_len;
  for (auto& rs : header.reference_sequences) ref_len.push_back(rs.length);
  std::vector<uint8_t> no_coverage(ref_len.size(), 0);
  for (auto* e : engines) {
    if (a.csi) check(e, ngsq_set_index_binning(e, a.min_shift, 0));
    check(e, ngsq_set_references(e, (uint32_t)ref_len.size(), ref_len.data(), no_coverage.data()));
  }
  ShardPlan plan = plan_shards_unindexed(header, file.data(), file.size(), (uint32_t)n_dev, engine_finder(engines[0]));
  log_dropped_cuts(plan);
  info("Indexing BAM file in " + std::to_string(n_dev - plan.dropped) + " parts.");
  run_parts(engines, plan.shards, a.src, file, a.chunk_mb << 20, a.direct_io);
  uint64_t records = 0;
  for (auto* e : engines) { ngsq_stats st; check(e, ngsq_get_stats(e, &st)); records += st.records; }
  info("Processed " + std::to_string(records) + " records.");
  write_index_file(a, dst, join_parts(engines, plan.shards, a.csi));
  return 0;
}

int index_main(int argc, char** argv, int i) {
  IndexArgs a;
  bool min_shift_set = false;
  std::vector<std::string> pos;
  for (; i < argc; ++i) {
    std::string s = argv[i];
    auto val = [&]() -> std::string { if (i + 1 >= argc) throw std::runtime_error("missing value for " + s); return argv[++i]; };
    if (s == "--cuda-device") a.device = std::stoi(val());
    else if (s == "--cuda-devices") { a.devices.clear(); std::stringstream ss(val()); std::string t; while (std::getline(ss, t, ',')) a.devices.push_back(std::stoi(t)); }
    else if (s == "--cuda-no-crc") a.verify_crc = false;
    else if (s == "--cuda-chunk-mb") a.chunk_mb = std::stoull(val());
    else if (s == "--cuda-buffered-io") a.direct_io = false;
    else if (s == "--csi") a.csi = true;
    else if (s == "-m" || s == "--min-shift") { a.min_shift = (uint32_t)std::stoul(val()); min_shift_set = true; }
    else if (!s.empty() && s[0] == '-' && s != "-") throw std::runtime_error("unknown flag " + s);
    else pos.push_back(s);
  }
  if (min_shift_set && !a.csi) throw std::runtime_error("--min-shift sets the binning of a CSI: use it with --csi");
  if (pos.size() != 1 || !a.chunk_mb) return -1;
  a.src = pos[0];
  if (a.devices.size() > 1) return index_bam_parts(a);
  if (a.devices.size() == 1) a.device = a.devices[0];
  return index_bam(a);
}

void usage() {
  std::cerr << "usage: ngs-cuda-qc qc <BAM> <REFERENCE_GENOME> [-n N] [-o DIR] [-p PREFIX] [--only FACET]\n"
               "                  [--cuda-devices 0,1,..] [--cuda-build-index [--cuda-csi [--cuda-min-shift N]]] [--cuda-gc-seed S]\n"
               "                  [--cuda-no-crc] [--cuda-chunk-mb M] [--cuda-buffered-io] [--cuda-perf]\n"
               "                  (the index is <BAM>.bai, or <BAM>.csi when there is no .bai; --cuda-build-index: without either,\n"
               "                  build <BAM>.bai, or with --cuda-csi <BAM>.csi (min_shift N, default 14), in the same pass and write it\n"
               "                  once the run succeeded)\n"
               "       ngs-cuda-qc index <BAM> [--csi [-m|--min-shift N]] [--cuda-device N | --cuda-devices 0,1,..] [--cuda-no-crc] [--cuda-chunk-mb M]\n"
               "                  [--cuda-buffered-io]\n"
               "                  (writes <BAM>.bai, or with --csi <BAM>.csi (min_shift N, default 14); an existing index is never overwritten;\n"
               "                  several devices index one part of the file each)\n";
}

}  // namespace

extern "C" int ngs_cuda_qc_main(int argc, char** argv) {
  try {
    QcArgs a;
    bool min_shift_set = false;
    std::vector<std::string> pos;
    int i = 1;
    if (i < argc && std::string(argv[i]) == "index") {
      const int rc = index_main(argc, argv, i + 1);
      if (rc < 0) { usage(); return 2; }
      return rc;
    }
    if (i < argc && std::string(argv[i]) == "qc") ++i;
    for (; i < argc; ++i) {
      std::string s = argv[i];
      auto val = [&]() -> std::string { if (i + 1 >= argc) throw std::runtime_error("missing value for " + s); return argv[++i]; };
      if (s == "-n" || s == "--num-records") a.num_records = std::stoull(val());
      else if (s == "-o" || s == "--output-directory") a.output_directory = val();
      else if (s == "-p" || s == "--output-prefix") a.output_prefix = val();
      else if (s == "-f" || s == "--features-gff") a.features_gff = val();
      else if (s == "-r" || s == "--reference-fasta") a.reference_fasta = val();
      else if (s == "--only") a.only_facet = val();
      else if (s == "--vaf-file" || s == "--vaf-file-path") a.vaf_file_path = val();
      else if (s == "--five-prime-utr-feature-name") a.feature_names.slot[0] = val();
      else if (s == "--three-prime-utr-feature-name") a.feature_names.slot[1] = val();
      else if (s == "--coding-sequence-feature-name") a.feature_names.slot[2] = val();
      else if (s == "--exon-feature-name") a.feature_names.slot[3] = val();
      else if (s == "--gene-feature-name") a.feature_names.slot[4] = val();
      else if (s == "--cuda-devices") { a.devices.clear(); std::stringstream ss(val()); std::string t; while (std::getline(ss, t, ',')) a.devices.push_back(std::stoi(t)); }
      else if (s == "--cuda-gc-seed") a.gc_seed = std::stoull(val(), nullptr, 0);
      else if (s == "--cuda-no-crc") a.verify_crc = false;
      else if (s == "--cuda-chunk-mb") a.chunk_mb = std::stoull(val());
      else if (s == "--cuda-perf") a.perf = true;
      else if (s == "--cuda-build-index") a.build_index = true;
      else if (s == "--cuda-csi") a.csi = true;
      else if (s == "--cuda-min-shift") { a.min_shift = (uint32_t)std::stoul(val()); min_shift_set = true; }
      else if (s == "--cuda-buffered-io") a.direct_io = false;
      else if (s == "-h" || s == "--help") { usage(); return 0; }
      else if (!s.empty() && s[0] == '-' && s != "-") throw std::runtime_error("unknown flag " + s);
      else pos.push_back(s);
    }
    if (pos.size() != 2 || a.devices.empty()) { usage(); return 2; }
    if (a.build_index && a.num_records) throw std::runtime_error("--cuda-build-index cannot be combined with -n: an index covers every record of the file");
    if (a.csi && !a.build_index) throw std::runtime_error("--cuda-csi sets the format of the index --cuda-build-index writes: use it with --cuda-build-index");
    if (min_shift_set && !a.csi) throw std::runtime_error("--cuda-min-shift sets the binning of a CSI: use it with --cuda-csi");
    a.src = pos[0];
    a.reference_genome = pos[1];
    return qc(a);
  } catch (const std::exception& ex) {
    std::cerr << "Error: " << ex.what() << "\n";
    return 1;
  }
}

#ifndef NGS_CUDA_QC_NO_MAIN
int main(int argc, char** argv) { return ngs_cuda_qc_main(argc, argv); }
#endif
